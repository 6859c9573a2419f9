// Stage 3 of the AVDN hot path: the warp-level kernels of the episodic
// cross-modal transformer ("ET", src/models/ET_haa.py, enc_vl.py, encodings.py,
// model_util.py) around the tensor-core GEMMs:
//
//   frame_attn   SoftDotAttention(49) over the 512 channels of every frame + fc2
//                (ET_haa.py:54-74,138-144), forward and backward
//   embed        positional encoding + [lang ; frames ; directions] concat +
//                direction embedding (encodings.py:22-49, enc_vl.py:71-83, ET_haa.py:147)
//   layernorm    (residual add +) LayerNorm(768), forward/backward
//   softmax      masked softmax of the attention scores; the block-causal mask
//                (model_util.py:213-241) and the key-padding mask (enc_vl.py:44-55)
//                are evaluated as a predicate from (L, T, len_b) -- never materialised
//   build_masks  materialises both masks for the bit-exact parity tests
//   heads        row gather + waypoint MLP + saliency FC (ET_haa.py:157-167)
//   colsum       bias gradients
//
// d_model is 768 (asserted by the host: the reference hard-codes it).
#include "common.cuh"

namespace {

constexpr int E = 768;
constexpr int EPL = E / 32;      // 24 elements per lane
constexpr int NCH = 512;         // trunk channels
constexpr int NSP = 49;          // 7x7 positions

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ------------------------------------------------------------- frame attention
// One CTA (256 threads = 8 warps) per (b,t).  ctx = frames[b,t] is [512][49] fp32.
//   target = W_in h ; logit_c = ctx_c . target ; attn = softmax_c ; wc = sum_c attn_c ctx_c
//   e49 = tanh(W_out [wc ; h]) ; out768 = fc2_w e49 + fc2_b
__global__ void __launch_bounds__(256) frame_attn_fwd_kernel(
    const float* __restrict__ frames, const float* __restrict__ lang_cls, const float* __restrict__ w_in,
    const float* __restrict__ w_out, const float* __restrict__ fc2_w, const float* __restrict__ fc2_b, int T,
    float* __restrict__ attn_out, float* __restrict__ wc_out, float* __restrict__ e49_out,
    float* __restrict__ emb_out) {
  __shared__ float s_h[NSP], s_t[NSP], s_logit[NCH], s_wc[NSP], s_e[NSP], s_red[8][NSP + 1];
  __shared__ float s_max, s_sum;
  const int bt = blockIdx.x, b = bt / T;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const float* ctx = frames + (size_t)bt * NCH * NSP;
  if (tid < NSP) s_h[tid] = lang_cls[b * NSP + tid];
  __syncthreads();
  if (tid < NSP) {
    float a = 0.f;
    for (int j = 0; j < NSP; ++j) a = fmaf(w_in[tid * NSP + j], s_h[j], a);
    s_t[tid] = a;
  }
  __syncthreads();
  for (int c = warp; c < NCH; c += 8) {
    float a = 0.f;
    for (int j = lane; j < NSP; j += 32) a = fmaf(ctx[c * NSP + j], s_t[j], a);
    a = warp_sum(a);
    if (lane == 0) s_logit[c] = a;
  }
  __syncthreads();
  if (warp == 0) {
    float m = -INFINITY;
    for (int c = lane; c < NCH; c += 32) m = fmaxf(m, s_logit[c]);
    m = warp_max(m);
    float s = 0.f;
    for (int c = lane; c < NCH; c += 32) s += __expf(s_logit[c] - m);
    s = warp_sum(s);
    if (lane == 0) { s_max = m; s_sum = s; }
  }
  __syncthreads();
  for (int c = tid; c < NCH; c += 256) {
    const float a = __expf(s_logit[c] - s_max) / s_sum;
    s_logit[c] = a;
    attn_out[(size_t)bt * NCH + c] = a;
  }
  __syncthreads();
  // wc[j] = sum_c attn[c] * ctx[c][j] : warp w takes channels w, w+8, ...; lanes over j
  {
    float a0 = 0.f, a1 = 0.f;
    for (int c = warp; c < NCH; c += 8) {
      const float a = s_logit[c];
      a0 = fmaf(a, ctx[c * NSP + lane], a0);
      if (lane + 32 < NSP) a1 = fmaf(a, ctx[c * NSP + lane + 32], a1);
    }
    s_red[warp][lane] = a0;
    if (lane + 32 < NSP) s_red[warp][lane + 32] = a1;
  }
  __syncthreads();
  if (tid < NSP) {
    float a = 0.f;
    for (int w = 0; w < 8; ++w) a += s_red[w][tid];
    s_wc[tid] = a;
    wc_out[(size_t)bt * NSP + tid] = a;
  }
  __syncthreads();
  if (tid < NSP) {
    float a = 0.f;
    for (int j = 0; j < NSP; ++j) a = fmaf(w_out[tid * 2 * NSP + j], s_wc[j], a);
    for (int j = 0; j < NSP; ++j) a = fmaf(w_out[tid * 2 * NSP + NSP + j], s_h[j], a);
    a = tanhf(a);
    s_e[tid] = a;
    e49_out[(size_t)bt * NSP + tid] = a;
  }
  __syncthreads();
  if (fc2_w == nullptr) return;          // SoftDotAttention only (ViT_LSTM)
  for (int o = tid; o < E; o += 256) {
    float a = fc2_b[o];
    for (int j = 0; j < NSP; ++j) a = fmaf(fc2_w[o * NSP + j], s_e[j], a);
    emb_out[(size_t)bt * E + o] = a;
  }
}

__global__ void __launch_bounds__(256) frame_attn_bwd_kernel(
    const float* __restrict__ frames, const float* __restrict__ lang_cls, const float* __restrict__ w_in,
    const float* __restrict__ w_out, const float* __restrict__ fc2_w, int T, const float* __restrict__ attn,
    const float* __restrict__ wc, const float* __restrict__ e49, const float* __restrict__ d_emb,
    float* __restrict__ d_frames, float* __restrict__ d_w_in, float* __restrict__ d_w_out,
    float* __restrict__ d_fc2_w, float* __restrict__ d_fc2_b, float* __restrict__ d_lang_cls) {
  __shared__ float s_h[NSP], s_t[NSP], s_wc[NSP], s_e[NSP], s_de[NSP], s_dpre[NSP], s_dwc[NSP], s_dt[NSP];
  __shared__ float s_demb[E], s_attn[NCH], s_dattn[NCH], s_red[8][NSP + 1];
  __shared__ float s_dot;
  const int bt = blockIdx.x, b = bt / T;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const float* ctx = frames + (size_t)bt * NCH * NSP;
  float* dctx = d_frames + (size_t)bt * NCH * NSP;
  if (tid < NSP) {
    s_h[tid] = lang_cls[b * NSP + tid];
    s_wc[tid] = wc[(size_t)bt * NSP + tid];
    s_e[tid] = e49[(size_t)bt * NSP + tid];
  }
  if (fc2_w) {
    for (int o = tid; o < E; o += 256) s_demb[o] = d_emb[(size_t)bt * E + o];
  }
  for (int c = tid; c < NCH; c += 256) s_attn[c] = attn[(size_t)bt * NCH + c];
  __syncthreads();
  if (tid < NSP) {
    float a = 0.f;
    for (int j = 0; j < NSP; ++j) a = fmaf(w_in[tid * NSP + j], s_h[j], a);
    s_t[tid] = a;
  }
  if (fc2_w) {
    // fc2: d_e[j] = sum_o fc2_w[o][j] d_emb[o]   (d_fc2_w / d_fc2_b: frame_attn_fc2_grad_kernel)
    float a0 = 0.f, a1 = 0.f;       // warp w: rows o = w, w+8, ... ; lanes over j
    for (int o = warp; o < E; o += 8) {
      const float g = s_demb[o];
      a0 = fmaf(g, fc2_w[o * NSP + lane], a0);
      if (lane + 32 < NSP) a1 = fmaf(g, fc2_w[o * NSP + lane + 32], a1);
    }
    s_red[warp][lane] = a0;
    if (lane + 32 < NSP) s_red[warp][lane + 32] = a1;
  }
  __syncthreads();
  if (tid < NSP) {
    float a = 0.f;
    if (fc2_w) {
      for (int w = 0; w < 8; ++w) a += s_red[w][tid];
    } else {
      a = d_emb[(size_t)bt * NSP + tid];                   // no fc2 (ViT_LSTM): d_emb is d_e49 [B*T,49]
    }
    s_de[tid] = a;
    s_dpre[tid] = a * (1.f - s_e[tid] * s_e[tid]);       // tanh'
  }
  __syncthreads();
  // linear_out: d_w_out[i][j] += dpre[i] * [wc;h][j] ; d_wc[j] = sum_i w_out[i][j] dpre[i]
  for (int idx = tid; idx < NSP * 2 * NSP; idx += 256) {
    const int i = idx / (2 * NSP), j = idx % (2 * NSP);
    const float in = j < NSP ? s_wc[j] : s_h[j - NSP];
    atomicAdd(&d_w_out[idx], s_dpre[i] * in);
  }
  if (tid < NSP) {
    float a = 0.f;
    for (int i = 0; i < NSP; ++i) a = fmaf(w_out[i * 2 * NSP + tid], s_dpre[i], a);
    s_dwc[tid] = a;
  }
  __syncthreads();
  // d_attn[c] = ctx_c . d_wc
  for (int c = warp; c < NCH; c += 8) {
    float a = 0.f;
    for (int j = lane; j < NSP; j += 32) a = fmaf(ctx[c * NSP + j], s_dwc[j], a);
    a = warp_sum(a);
    if (lane == 0) s_dattn[c] = a;
  }
  __syncthreads();
  if (warp == 0) {
    float a = 0.f;
    for (int c = lane; c < NCH; c += 32) a = fmaf(s_attn[c], s_dattn[c], a);
    a = warp_sum(a);
    if (lane == 0) s_dot = a;
  }
  __syncthreads();
  for (int c = tid; c < NCH; c += 256) s_dattn[c] = s_attn[c] * (s_dattn[c] - s_dot);     // d_logit
  __syncthreads();
  // d_ctx[c][j] = attn[c]*d_wc[j] + d_logit[c]*target[j] ; d_target[j] = sum_c d_logit[c] ctx[c][j]
  {
    float a0 = 0.f, a1 = 0.f;
    for (int c = warp; c < NCH; c += 8) {
      const float at = s_attn[c], dl = s_dattn[c];
      const float x0 = ctx[c * NSP + lane];
      dctx[c * NSP + lane] = fmaf(at, s_dwc[lane], dl * s_t[lane]);
      a0 = fmaf(dl, x0, a0);
      if (lane + 32 < NSP) {
        const float x1 = ctx[c * NSP + lane + 32];
        dctx[c * NSP + lane + 32] = fmaf(at, s_dwc[lane + 32], dl * s_t[lane + 32]);
        a1 = fmaf(dl, x1, a1);
      }
    }
    s_red[warp][lane] = a0;
    if (lane + 32 < NSP) s_red[warp][lane + 32] = a1;
  }
  __syncthreads();
  if (tid < NSP) {
    float a = 0.f;
    for (int w = 0; w < 8; ++w) a += s_red[w][tid];
    s_dt[tid] = a;
  }
  __syncthreads();
  for (int idx = tid; idx < NSP * NSP; idx += 256) atomicAdd(&d_w_in[idx], s_dt[idx / NSP] * s_h[idx % NSP]);
  // gradient of the query h = lang_cls (it feeds linear_in and the second half of linear_out's input);
  // accumulated over the T frames of the sample
  if (d_lang_cls != nullptr && tid < NSP) {
    float a = 0.f;
    for (int i = 0; i < NSP; ++i) a = fmaf(w_in[i * NSP + tid], s_dt[i], fmaf(w_out[i * 2 * NSP + NSP + tid], s_dpre[i], a));
    atomicAdd(&d_lang_cls[b * NSP + tid], a);
  }
}

// d_fc2_w[o][j] += sum_bt d_emb[bt][o] * e49[bt][j] ; d_fc2_b[o] += sum_bt d_emb[bt][o].  A block owns 16 output rows
// and a slice of the frames; one thread per (o, j), column 49 = the bias.  (Summed by every (b,t) CTA of
// frame_attn_bwd_kernel with global atomics this was 24 M atomic adds per step at B = 64.)
constexpr int FC2_ROWS = 16, FC2_SLICES = 4;
__global__ void __launch_bounds__(FC2_ROWS * (NSP + 1)) frame_attn_fc2_grad_kernel(const float* __restrict__ d_emb,
                                                                                  const float* __restrict__ e49, int BT,
                                                                                  float* __restrict__ d_fc2_w,
                                                                                  float* __restrict__ d_fc2_b) {
  const int o = blockIdx.x * FC2_ROWS + threadIdx.x / (NSP + 1), j = threadIdx.x % (NSP + 1);
  const int per = (BT + FC2_SLICES - 1) / FC2_SLICES;
  const int lo = blockIdx.y * per, hi = min(BT, lo + per);
  float a0 = 0.f, a1 = 0.f;
  int bt = lo;
  for (; bt + 1 < hi; bt += 2) {
    a0 = fmaf(d_emb[(size_t)bt * E + o], j < NSP ? e49[(size_t)bt * NSP + j] : 1.f, a0);
    a1 = fmaf(d_emb[(size_t)(bt + 1) * E + o], j < NSP ? e49[(size_t)(bt + 1) * NSP + j] : 1.f, a1);
  }
  if (bt < hi) a0 = fmaf(d_emb[(size_t)bt * E + o], j < NSP ? e49[(size_t)bt * NSP + j] : 1.f, a0);
  if (j < NSP) atomicAdd(&d_fc2_w[o * NSP + j], a0 + a1);
  else atomicAdd(&d_fc2_b[o], a0 + a1);
}

// ------------------------------------------------------------------ embedding
// v[b,s,:] = row + pe[pos]/sqrt(768): lang rows (s<L, pos=s), frame rows (pos=L+t),
// direction rows (pos=L+t, row = W_d dir + b_d).  One warp per row.
__global__ void __launch_bounds__(256) embed_fwd_kernel(const float* __restrict__ lang,
                                                        const float* __restrict__ emb_frames,
                                                        const float* __restrict__ dirs, const float* __restrict__ wd,
                                                        const float* __restrict__ bd, const float* __restrict__ pe,
                                                        int B, int L, int T, float* __restrict__ v) {
  const int S = L + 2 * T;
  const long long row = blockIdx.x * 8LL + (threadIdx.x >> 5);
  if (row >= (long long)B * S) return;
  const int lane = threadIdx.x & 31;
  const int b = (int)(row / S), s = (int)(row % S);
  const float inv = 0.03608439182435161f;        // 1/sqrt(768)
  float* o = v + row * E;
  if (s < L) {
    const float* src = lang + ((size_t)b * L + s) * E;
    for (int j = lane; j < E; j += 32) o[j] = src[j] + pe[(size_t)s * E + j] * inv;
  } else if (s < L + T) {
    const int t = s - L;
    const float* src = emb_frames + ((size_t)b * T + t) * E;
    for (int j = lane; j < E; j += 32) o[j] = src[j] + pe[(size_t)(L + t) * E + j] * inv;
  } else {
    const int t = s - L - T;
    if (wd == nullptr) {          // dirs already embedded: [B,T,768] (EncoderVL.forward's emb_directions)
      const float* src = dirs + ((size_t)b * T + t) * E;
      for (int j = lane; j < E; j += 32) o[j] = src[j] + pe[(size_t)(L + t) * E + j] * inv;
    } else {
      const float d0 = dirs[((size_t)b * T + t) * 2], d1 = dirs[((size_t)b * T + t) * 2 + 1];
      for (int j = lane; j < E; j += 32)
        o[j] = fmaf(wd[j * 2], d0, fmaf(wd[j * 2 + 1], d1, bd[j])) + pe[(size_t)(L + t) * E + j] * inv;
    }
  }
}

// backward of the direction embedding: d_wd[j][k] += sum dv[b,L+T+t,j]*dir[b,t,k]; d_bd[j] += sum dv
__global__ void __launch_bounds__(256) embed_dir_bwd_kernel(const float* __restrict__ dv,
                                                            const float* __restrict__ dirs, int B, int L, int T,
                                                            float* __restrict__ d_wd, float* __restrict__ d_bd) {
  const int S = L + 2 * T;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= E) return;
  float a0 = 0.f, a1 = 0.f, ab = 0.f;
  for (int b = 0; b < B; ++b)
    for (int t = 0; t < T; ++t) {
      const float g = dv[((size_t)b * S + L + T + t) * E + j];
      a0 = fmaf(g, dirs[((size_t)b * T + t) * 2], a0);
      a1 = fmaf(g, dirs[((size_t)b * T + t) * 2 + 1], a1);
      ab += g;
    }
  d_wd[j * 2] += a0;
  d_wd[j * 2 + 1] += a1;
  d_bd[j] += ab;
}

// ------------------------------------------------------------------ LayerNorm
// v = a (+ b) ; y = LN(v)*gamma + beta ; writes v (if b), y (f32), y16 (bf16), mean, rstd
__global__ void __launch_bounds__(256) ln_fwd_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                     const float* __restrict__ gamma, const float* __restrict__ beta,
                                                     long long M, float eps, float* __restrict__ v_out,
                                                     float* __restrict__ y, __nv_bfloat16* __restrict__ y16,
                                                     float* __restrict__ mean, float* __restrict__ rstd,
                                                     unsigned int dthr, float dscale, unsigned long long seed,
                                                     unsigned int site) {
  const long long row = blockIdx.x * 8LL + (threadIdx.x >> 5);
  if (row >= M) return;
  const int lane = threadIdx.x & 31;
  float x[EPL];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < EPL; ++i) {
    const int j = lane + 32 * i;
    float t = a[row * E + j];
    if (b) {
      float bv = b[row * E + j];
      if (dthr) bv = avdn_drop_keep(seed, site, (unsigned long long)(row * E + j), dthr) ? bv * dscale : 0.f;
      t += bv;
    }
    x[i] = t;
    s += t;
  }
  const float mu = warp_sum(s) * (1.f / E);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < EPL; ++i) { const float d = x[i] - mu; q = fmaf(d, d, q); }
  const float rs = rsqrtf(warp_sum(q) * (1.f / E) + eps);
#pragma unroll
  for (int i = 0; i < EPL; ++i) {
    const int j = lane + 32 * i;
    const float o = (x[i] - mu) * rs * gamma[j] + beta[j];
    if (v_out) v_out[row * E + j] = x[i];
    if (y) y[row * E + j] = o;
    if (y16) y16[row * E + j] = __float2bfloat16_rn(o);
  }
  if (lane == 0) { mean[row] = mu; rstd[row] = rs; }
}

// dv = rstd * (g - mean(g) - xhat*mean(g*xhat)), g = dy*gamma ; dgamma += dy*xhat ; dbeta += dy
// dy = dy1 (+ dy2).  Persistent over rows so that the parameter gradients leave as one
// atomic per (warp, column).
__global__ void __launch_bounds__(256) ln_bwd_kernel(const float* __restrict__ dy1, const float* __restrict__ dy2,
                                                     const float* __restrict__ v, const float* __restrict__ mean,
                                                     const float* __restrict__ rstd, const float* __restrict__ gamma,
                                                     long long M, float* __restrict__ dv,
                                                     __nv_bfloat16* __restrict__ dv16, float* __restrict__ dgamma,
                                                     float* __restrict__ dbeta, unsigned int dthr, float dscale,
                                                     unsigned long long seed, unsigned int site) {
  const int lane = threadIdx.x & 31;
  const long long w0 = blockIdx.x * 8LL + (threadIdx.x >> 5), nw = gridDim.x * 8LL;
  float dg[EPL], db[EPL], gm[EPL];
#pragma unroll
  for (int i = 0; i < EPL; ++i) { dg[i] = 0.f; db[i] = 0.f; gm[i] = gamma[lane + 32 * i]; }
  for (long long row = w0; row < M; row += nw) {
    const float mu = mean[row], rs = rstd[row];
    float xh[EPL], g[EPL];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < EPL; ++i) {
      const int j = lane + 32 * i;
      float d = dy1[row * E + j];
      if (dy2) d += dy2[row * E + j];
      xh[i] = (v[row * E + j] - mu) * rs;
      dg[i] = fmaf(d, xh[i], dg[i]);
      db[i] += d;
      g[i] = d * gm[i];
      s1 += g[i];
      s2 = fmaf(g[i], xh[i], s2);
    }
    s1 = warp_sum(s1) * (1.f / E);
    s2 = warp_sum(s2) * (1.f / E);
#pragma unroll
    for (int i = 0; i < EPL; ++i) {
      const int j = lane + 32 * i;
      const float o = rs * (g[i] - s1 - xh[i] * s2);
      if (dv) dv[row * E + j] = o;
      if (dv16) {
        // gradient of the dropped branch b of v = a + dropout(b)
        float ob = o;
        if (dthr) ob = avdn_drop_keep(seed, site, (unsigned long long)(row * E + j), dthr) ? o * dscale : 0.f;
        dv16[row * E + j] = __float2bfloat16_rn(ob);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < EPL; ++i) {
    atomicAdd(&dgamma[lane + 32 * i], dg[i]);
    atomicAdd(&dbeta[lane + 32 * i], db[i]);
  }
}

// ------------------------------------------------------------ masked softmax
// may query row q attend key k in sample with `len` valid steps?  (model_util.py:213-241
// + enc_vl.py:48-55; L language tokens, T = max length)
__device__ __forceinline__ bool may_attend(int q, int k, int L, int T, int len) {
  if (T == 0) return k < len;        // key-padding mask only (BERT: len = number of real tokens of the sample)
  if (k < L) return true;            // everyone sees language
  if (q < L) return false;           // language sees only language
  const int tk = (k - L) % T, tq = (q - L) % T;
  return tk <= tq && tk < len;       // causal over steps, padded steps masked
}

// scores [B,H,S,Sp] fp32 -> P [B,H,S,Sp] bf16 (0 where masked / padded).  One warp per row.
__global__ void __launch_bounds__(256) softmax_fwd_kernel(const float* __restrict__ scores,
                                                          const int* __restrict__ lens, int B, int H, int L, int T,
                                                          int Sp, __nv_bfloat16* __restrict__ P,
                                                          __nv_bfloat16* __restrict__ P_full, unsigned int dthr,
                                                          float dscale, unsigned long long seed, unsigned int site) {
  const int S = L + 2 * T;
  const long long row = blockIdx.x * 8LL + (threadIdx.x >> 5);
  if (row >= (long long)B * H * S) return;
  const int lane = threadIdx.x & 31;
  const int q = (int)(row % S), b = (int)(row / ((long long)S * H));
  const int len = lens[b];
  const float* sr = scores + row * Sp;
  __nv_bfloat16* pr = P + row * Sp;
  float m = -INFINITY;
  for (int k = lane; k < S; k += 32)
    if (may_attend(q, k, L, T, len)) m = fmaxf(m, sr[k]);
  m = warp_max(m);
  float s = 0.f;
  for (int k = lane; k < S; k += 32)
    if (may_attend(q, k, L, T, len)) s += __expf(sr[k] - m);
  s = 1.f / warp_sum(s);
  for (int k = lane; k < Sp; k += 32) {
    float p = 0.f;
    if (k < S && may_attend(q, k, L, T, len)) p = __expf(sr[k] - m) * s;
    if (dthr) {
      // attention dropout (nn.MultiheadAttention(dropout=p)): the PV GEMM consumes the dropped
      // probabilities, the softmax backward needs the full ones
      P_full[row * Sp + k] = __float2bfloat16_rn(p);
      p = avdn_drop_keep(seed, site, (unsigned long long)(row * Sp + k), dthr) ? p * dscale : 0.f;
    }
    pr[k] = __float2bfloat16_rn(p);
  }
}

// The same, one pass: a lane keeps its NP column pairs (k = 2*lane + 64*i) in registers, so a row is read once
// (float2) and written once (bf16x2); the mask of a column costs a compare, not a modulo.  Sp <= 64 * NP, Sp even.
template <int NP>
__global__ void __launch_bounds__(256) softmax_fwd_regs_kernel(const float* __restrict__ scores,
                                                               const int* __restrict__ lens, int B, int H, int L, int T,
                                                               int Sp, __nv_bfloat16* __restrict__ P,
                                                               __nv_bfloat16* __restrict__ P_full, unsigned int dthr,
                                                               float dscale, unsigned long long seed, unsigned int site) {
  const int S = L + 2 * T;
  const long long row = blockIdx.x * 8LL + (threadIdx.x >> 5);
  if (row >= (long long)B * H * S) return;
  const int lane = threadIdx.x & 31;
  const int q = (int)(row % S), b = (int)(row / ((long long)S * H));
  const int len = lens[b];
  // columns a query may attend: [0, k_all) all of them, then k in [L, S) with step(k) <= tq and step(k) < len
  int k_all, tq = -1;
  if (T == 0) k_all = len;                               // key-padding mask only
  else {
    k_all = L;
    if (q >= L) tq = (q - L) >= T ? q - L - T : q - L;
  }
  const int tmax = tq < len - 1 ? tq : len - 1;          // largest step that may be attended (-1: none)
  auto allowed = [&](int k) -> bool {
    if (k < k_all) return true;
    if (T == 0 || k >= S) return false;
    const int d = k - L, tk = d >= T ? d - T : d;
    return tk <= tmax;
  };
  const float2* sr = reinterpret_cast<const float2*>(scores + row * Sp);
  float2 v[NP];
  unsigned int ok = 0u;
  float m = -INFINITY;
#pragma unroll
  for (int i = 0; i < NP; ++i) {
    const int k = 2 * lane + 64 * i;
    v[i] = make_float2(0.f, 0.f);
    if (k < Sp) {
      v[i] = sr[lane + 32 * i];
      if (allowed(k)) { ok |= 1u << (2 * i); m = fmaxf(m, v[i].x); }
      if (allowed(k + 1)) { ok |= 2u << (2 * i); m = fmaxf(m, v[i].y); }
    }
  }
  m = warp_max(m);
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < NP; ++i) {
    v[i].x = (ok >> (2 * i)) & 1u ? __expf(v[i].x - m) : 0.f;
    v[i].y = (ok >> (2 * i)) & 2u ? __expf(v[i].y - m) : 0.f;
    sum += v[i].x + v[i].y;
  }
  sum = 1.f / warp_sum(sum);
  __nv_bfloat162* pr = reinterpret_cast<__nv_bfloat162*>(P + row * Sp);
  __nv_bfloat162* pf = reinterpret_cast<__nv_bfloat162*>(P_full + row * Sp);
#pragma unroll
  for (int i = 0; i < NP; ++i) {
    const int k = 2 * lane + 64 * i;
    if (k < Sp) {
      const float p0f = (ok >> (2 * i)) & 1u ? v[i].x * sum : 0.f, p1f = (ok >> (2 * i)) & 2u ? v[i].y * sum : 0.f;
      float p0 = p0f, p1 = p1f;
      if (dthr) {
        pf[lane + 32 * i] = __floats2bfloat162_rn(p0, p1);
        const unsigned long long idx = (unsigned long long)(row * Sp + k);
        p0 = avdn_drop_keep(seed, site, idx, dthr) ? p0 * dscale : 0.f;
        p1 = avdn_drop_keep(seed, site, idx + 1, dthr) ? p1 * dscale : 0.f;
      }
      pr[lane + 32 * i] = __floats2bfloat162_rn(p0, p1);
    }
  }
}

// dS = alpha * P * (dP - sum_k P*dP)  (bf16 out, 0 in the padding)
__global__ void __launch_bounds__(256) softmax_bwd_kernel(const __nv_bfloat16* __restrict__ P,
                                                          const float* __restrict__ dP, long long rows, int S, int Sp,
                                                          float alpha, __nv_bfloat16* __restrict__ dS,
                                                          unsigned int dthr, float dscale, unsigned long long seed,
                                                          unsigned int site) {
  const long long row = blockIdx.x * 8LL + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const __nv_bfloat16* pr = P + row * Sp;
  const float* dr = dP + row * Sp;
  // with attention dropout, dP arrives w.r.t. the dropped probabilities: d(full) = keep ? d * scale : 0
  auto dp_at = [&](int k) {
    float d = dr[k];
    if (dthr) d = avdn_drop_keep(seed, site, (unsigned long long)(row * Sp + k), dthr) ? d * dscale : 0.f;
    return d;
  };
  float dot = 0.f;
  for (int k = lane; k < S; k += 32) dot = fmaf(__bfloat162float(pr[k]), dp_at(k), dot);
  dot = warp_sum(dot);
  for (int k = lane; k < Sp; k += 32) {
    float o = 0.f;
    if (k < S) o = alpha * __bfloat162float(pr[k]) * (dp_at(k) - dot);
    dS[row * Sp + k] = __float2bfloat16_rn(o);
  }
}

template <int NP>
__global__ void __launch_bounds__(256) softmax_bwd_regs_kernel(const __nv_bfloat16* __restrict__ P,
                                                               const float* __restrict__ dP, long long rows, int S, int Sp,
                                                               float alpha, __nv_bfloat16* __restrict__ dS,
                                                               unsigned int dthr, float dscale, unsigned long long seed,
                                                               unsigned int site) {
  const long long row = blockIdx.x * 8LL + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const __nv_bfloat162* pr = reinterpret_cast<const __nv_bfloat162*>(P + row * Sp);
  const float2* dr = reinterpret_cast<const float2*>(dP + row * Sp);
  float2 p[NP], d[NP];
  float dot = 0.f;
#pragma unroll
  for (int i = 0; i < NP; ++i) {
    const int k = 2 * lane + 64 * i;
    p[i] = make_float2(0.f, 0.f);
    d[i] = make_float2(0.f, 0.f);
    if (k < Sp) {
      p[i] = __bfloat1622float2(pr[lane + 32 * i]);
      d[i] = dr[lane + 32 * i];
      if (dthr) {
        const unsigned long long idx = (unsigned long long)(row * Sp + k);
        d[i].x = avdn_drop_keep(seed, site, idx, dthr) ? d[i].x * dscale : 0.f;
        d[i].y = avdn_drop_keep(seed, site, idx + 1, dthr) ? d[i].y * dscale : 0.f;
      }
      if (k >= S) p[i].x = d[i].x = 0.f;          // the padding columns of dP hold whatever the GEMM left there
      if (k + 1 >= S) p[i].y = d[i].y = 0.f;
      dot = fmaf(p[i].x, d[i].x, dot);
      dot = fmaf(p[i].y, d[i].y, dot);
    }
  }
  dot = warp_sum(dot);
  __nv_bfloat162* o = reinterpret_cast<__nv_bfloat162*>(dS + row * Sp);
#pragma unroll
  for (int i = 0; i < NP; ++i) {
    const int k = 2 * lane + 64 * i;
    if (k < Sp) o[lane + 32 * i] = __floats2bfloat162_rn(alpha * p[i].x * (d[i].x - dot), alpha * p[i].y * (d[i].y - dot));
  }
}


// Incremental ("decode") attention of the ET inference path.  Rows of earlier steps never change (the mask is
// causal over steps and LayerNorm / FFN are row-wise), so a rollout step only computes its R = 2 new rows per
// sample (frame t, direction t); they attend to the first n rows of the layer's K|V cache (language rows, then
// frame/direction rows of steps 0..t interleaved).  One warp per (sample, head, new row); fp32 online softmax.
//   qkv_new [B*R, 2304] bf16 (q | k | v of the new rows; q is read), cache [B, Lc, 1536] bf16 (k | v),
//   ctx [B*R, 768] bf16.
__global__ void __launch_bounds__(256) attn_decode_kernel(const __nv_bfloat16* __restrict__ qkv_new,
                                                          const __nv_bfloat16* __restrict__ cache, int B, int R, int H,
                                                          int Lc, int n, float scale, __nv_bfloat16* __restrict__ ctx) {
  const long long w = blockIdx.x * 8LL + (threadIdx.x >> 5);
  if (w >= (long long)B * H * R) return;
  const int lane = threadIdx.x & 31;
  const int r = (int)(w % R), h = (int)((w / R) % H), b = (int)(w / ((long long)R * H));
  const __nv_bfloat162 q2 = *reinterpret_cast<const __nv_bfloat162*>(qkv_new + ((size_t)b * R + r) * (3 * E) + h * 64 + 2 * lane);
  const float q0 = __low2float(q2) * scale, q1 = __high2float(q2) * scale;
  const __nv_bfloat16* kv = cache + (size_t)b * Lc * (2 * E) + h * 64 + 2 * lane;
  float m = -INFINITY, l = 0.f, a0 = 0.f, a1 = 0.f;
  for (int j = 0; j < n; ++j) {
    const __nv_bfloat162 k2 = *reinterpret_cast<const __nv_bfloat162*>(kv + (size_t)j * (2 * E));
    const __nv_bfloat162 v2 = *reinterpret_cast<const __nv_bfloat162*>(kv + (size_t)j * (2 * E) + E);
    const float sc = warp_sum(fmaf(q0, __low2float(k2), q1 * __high2float(k2)));
    const float mn = fmaxf(m, sc);
    const float corr = __expf(m - mn), pj = __expf(sc - mn);
    l = fmaf(l, corr, pj);
    a0 = fmaf(a0, corr, pj * __low2float(v2));
    a1 = fmaf(a1, corr, pj * __high2float(v2));
    m = mn;
  }
  const float inv = 1.f / l;
  *reinterpret_cast<__nv_bfloat162*>(ctx + ((size_t)b * R + r) * E + h * 64 + 2 * lane) =
      __floats2bfloat162_rn(a0 * inv, a1 * inv);
}

// materialised masks for the bit-exact parity tests (E3 / E5)
__global__ void build_masks_kernel(const int* __restrict__ lens, int B, int L, int T, uint8_t* __restrict__ mask_pad,
                                   float* __restrict__ mask_attn) {
  const int S = L + 2 * T;
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < (long long)B * S) {
    const int b = (int)(i / S), k = (int)(i % S);
    mask_pad[i] = (k >= L && ((k - L) % T) >= lens[b]) ? 1 : 0;
  }
  if (i < (long long)S * S) {
    const int q = (int)(i / S), k = (int)(i % S);
    mask_attn[i] = may_attend(q, k, L, T, T) ? 0.f : -INFINITY;
  }
}

// ----------------------------------------------------------------- col sums
// out[n] += sum_m in[m][n]  (bias gradients).  in is bf16 or f32 with row pitch ld.
template <typename TIn>
__global__ void __launch_bounds__(256) colsum_kernel(const TIn* __restrict__ in, long long M, int N, long long ld,
                                                     float* __restrict__ out, int rows_per_block) {
  const int n = blockIdx.x * 32 + (threadIdx.x & 31);
  const int ry = threadIdx.x >> 5;
  const long long r0 = (long long)blockIdx.y * rows_per_block;
  const long long r1 = min(M, r0 + rows_per_block);
  float a = 0.f;
  if (n < N)
    for (long long r = r0 + ry; r < r1; r += 8) a += (float)in[r * ld + n];
  __shared__ float sm[8][33];
  sm[ry][threadIdx.x & 31] = a;
  __syncthreads();
  if (ry == 0 && n < N) {
    float t = 0.f;
    for (int y = 0; y < 8; ++y) t += sm[y][threadIdx.x & 31];
    atomicAdd(&out[n], t);
  }
}

// -------------------------------------------------------------------- heads
// One CTA per sample.  dir row -> 768->256 relu ->32 relu ->4 ; vis row -> 768->64 relu.
__global__ void __launch_bounds__(256) heads_fwd_kernel(const float* __restrict__ x, int S, int row_vis, int row_dir,
                                                        const float* __restrict__ w0, const float* __restrict__ b0,
                                                        const float* __restrict__ w1, const float* __restrict__ b1,
                                                        const float* __restrict__ w2, const float* __restrict__ b2,
                                                        const float* __restrict__ wf, const float* __restrict__ bf,
                                                        float* __restrict__ h0_out, float* __restrict__ h1_out,
                                                        float* __restrict__ output, float* __restrict__ h_sali,
                                                        unsigned int dthr, float dscale, unsigned long long seed,
                                                        unsigned int site) {
  // train mode: Dropout(0.2) after both hidden ReLUs of decoder_2_action_full (sites site, site+1) and
  // between fc's Linear and ReLU (site+2) -- ET_haa.py:98-119.  relu(dropout(z)) == dropout(relu(z)).
  __shared__ float s_dir[E], s_vis[E], s_h0[256], s_h1[32];
  const int b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int j = tid; j < E; j += 256) {
    s_dir[j] = x[((size_t)b * S + row_dir) * E + j];
    s_vis[j] = x[((size_t)b * S + row_vis) * E + j];
  }
  __syncthreads();
  for (int o = warp; o < 256; o += 8) {
    float a = 0.f;
    for (int j = lane; j < E; j += 32) a = fmaf(w0[(size_t)o * E + j], s_dir[j], a);
    a = warp_sum(a);
    if (lane == 0) {
      a = fmaxf(a + b0[o], 0.f);
      if (dthr) a = avdn_drop_keep(seed, site, (unsigned long long)(b * 256 + o), dthr) ? a * dscale : 0.f;
      s_h0[o] = a; h0_out[b * 256 + o] = a;
    }
  }
  for (int o = warp; o < 64; o += 8) {
    float a = 0.f;
    for (int j = lane; j < E; j += 32) a = fmaf(wf[(size_t)o * E + j], s_vis[j], a);
    a = warp_sum(a);
    if (lane == 0) {
      a = fmaxf(a + bf[o], 0.f);
      if (dthr) a = avdn_drop_keep(seed, site + 2, (unsigned long long)(b * 64 + o), dthr) ? a * dscale : 0.f;
      h_sali[b * 64 + o] = a;
    }
  }
  __syncthreads();
  for (int o = warp; o < 32; o += 8) {
    float a = 0.f;
    for (int j = lane; j < 256; j += 32) a = fmaf(w1[o * 256 + j], s_h0[j], a);
    a = warp_sum(a);
    if (lane == 0) {
      a = fmaxf(a + b1[o], 0.f);
      if (dthr) a = avdn_drop_keep(seed, site + 1, (unsigned long long)(b * 32 + o), dthr) ? a * dscale : 0.f;
      s_h1[o] = a; h1_out[b * 32 + o] = a;
    }
  }
  __syncthreads();
  if (warp < 4) {
    float a = w2[warp * 32 + lane] * s_h1[lane];
    a = warp_sum(a);
    if (lane == 0) output[b * 4 + warp] = a + b2[warp];
  }
}

// backward: d_output [B,4], d_h_sali [B,64] -> dx rows (zero elsewhere: caller zero-fills dx) + param grads
__global__ void __launch_bounds__(256) heads_bwd_kernel(
    const float* __restrict__ x, int S, int row_vis, int row_dir, const float* __restrict__ w0,
    const float* __restrict__ w1, const float* __restrict__ w2, const float* __restrict__ wf,
    const float* __restrict__ h0, const float* __restrict__ h1, const float* __restrict__ h_sali,
    const float* __restrict__ d_output, const float* __restrict__ d_h_sali, float* __restrict__ dx,
    float* __restrict__ dw0, float* __restrict__ db0, float* __restrict__ dw1, float* __restrict__ db1,
    float* __restrict__ dw2, float* __restrict__ db2, float* __restrict__ dwf, float* __restrict__ dbf,
    float dscale) {
  // dscale = 1/(1-p) of the heads' dropout (1 in eval mode): a dropped activation was stored as 0, so the
  // ReLU mask already removes it; kept ones carry the factor.
  __shared__ float s_dir[E], s_vis[E], s_h0[256], s_h1[32], s_d2[4], s_d1[32], s_d0[256], s_ds[64];
  const int b = blockIdx.x, tid = threadIdx.x;
  for (int j = tid; j < E; j += 256) {
    s_dir[j] = x[((size_t)b * S + row_dir) * E + j];
    s_vis[j] = x[((size_t)b * S + row_vis) * E + j];
  }
  s_h0[tid] = h0[b * 256 + tid];
  if (tid < 32) s_h1[tid] = h1[b * 32 + tid];
  if (tid < 4) s_d2[tid] = d_output[b * 4 + tid];
  if (tid < 64) s_ds[tid] = h_sali[b * 64 + tid] > 0.f ? d_h_sali[b * 64 + tid] * dscale : 0.f;
  __syncthreads();
  if (tid < 4) atomicAdd(&db2[tid], s_d2[tid]);
  if (tid < 128) atomicAdd(&dw2[tid], s_d2[tid >> 5] * s_h1[tid & 31]);
  if (tid < 32) {
    float a = 0.f;
    for (int o = 0; o < 4; ++o) a = fmaf(w2[o * 32 + tid], s_d2[o], a);
    a = s_h1[tid] > 0.f ? a * dscale : 0.f;
    s_d1[tid] = a;
    atomicAdd(&db1[tid], a);
  }
  if (tid < 64) atomicAdd(&dbf[tid], s_ds[tid]);
  __syncthreads();
  for (int idx = tid; idx < 32 * 256; idx += 256) atomicAdd(&dw1[idx], s_d1[idx >> 8] * s_h0[idx & 255]);
  {
    float a = 0.f;
    for (int o = 0; o < 32; ++o) a = fmaf(w1[o * 256 + tid], s_d1[o], a);
    a = s_h0[tid] > 0.f ? a * dscale : 0.f;
    s_d0[tid] = a;
    atomicAdd(&db0[tid], a);
  }
  __syncthreads();
  // dw0[o][j] += d0[o]*dir[j] ; d_dir[j] = sum_o w0[o][j] d0[o]
  for (int j = tid; j < E; j += 256) {
    float a = 0.f;
    for (int o = 0; o < 256; ++o) {
      const float g = s_d0[o];
      a = fmaf(w0[(size_t)o * E + j], g, a);
      if (g != 0.f) atomicAdd(&dw0[(size_t)o * E + j], g * s_dir[j]);
    }
    dx[((size_t)b * S + row_dir) * E + j] = a;
    float v = 0.f;
    for (int o = 0; o < 64; ++o) {
      const float g = s_ds[o];
      v = fmaf(wf[(size_t)o * E + j], g, v);
      if (g != 0.f) atomicAdd(&dwf[(size_t)o * E + j], g * s_vis[j]);
    }
    dx[((size_t)b * S + row_vis) * E + j] = v;
  }
}

// in-place dropout of a bf16 tensor (the FFN hidden activation after ReLU)
__global__ void __launch_bounds__(256) dropout_bf16_kernel(__nv_bfloat16* __restrict__ x, long long n, unsigned int dthr,
                                                           float dscale, unsigned long long seed, unsigned int site) {
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const float v = __bfloat162float(x[i]);
    x[i] = __float2bfloat16_rn(avdn_drop_keep(seed, site, (unsigned long long)i, dthr) ? v * dscale : 0.f);
  }
}

// in-place dropout of an fp32 tensor, optionally refreshing its bf16 shadow (embedding dropout, head dropout)
__global__ void __launch_bounds__(256) dropout_f32_kernel(float* __restrict__ x, __nv_bfloat16* __restrict__ x16,
                                                          long long n, unsigned int dthr, float dscale,
                                                          unsigned long long seed, unsigned int site) {
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const float v = avdn_drop_keep(seed, site, (unsigned long long)i, dthr) ? x[i] * dscale : 0.f;
    x[i] = v;
    if (x16) x16[i] = __float2bfloat16_rn(v);
  }
}

// out = dropout'(a + b): the gradient entering a dropout site whose output fed two consumers.  Element i draws the
// mask of element idx0 + i of its site, so a slice of a larger tensor gets that tensor's mask.
__global__ void __launch_bounds__(256) add_dropout_f32_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                              float* __restrict__ out, long long n, unsigned long long idx0,
                                                              unsigned int dthr, float dscale, unsigned long long seed,
                                                              unsigned int site) {
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    const float v = a[i] + (b ? b[i] : 0.f);
    out[i] = (!dthr || avdn_drop_keep(seed, site, idx0 + (unsigned long long)i, dthr)) ? v * dscale : 0.f;
  }
}

// the keep-scale factor (0 or 1/(1-p)) of every element of a site, for tests and debugging
__global__ void __launch_bounds__(256) dropout_keep_scale_kernel(float* __restrict__ out, long long n, unsigned int dthr,
                                                                 float dscale, unsigned long long seed,
                                                                 unsigned int site) {
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += (long long)gridDim.x * 256)
    out[i] = avdn_drop_keep(seed, site, (unsigned long long)i, dthr) ? dscale : 0.f;
}

inline int rows_grid(long long rows) { return (int)((rows + 7) / 8); }
inline bool drop_ok(float p) { return p >= 0.f && p < 1.f; }
inline float drop_scale(float p) { return 1.0f / (1.0f - p); }

}  // namespace

// ===================================================================== C ABI
extern "C" int avdn_frame_attn_fwd(const float* frames, const float* lang_cls, const float* w_in,
                                   const float* w_out, const float* fc2_w, const float* fc2_b, int B, int T,
                                   float* attn, float* wc, float* e49, float* emb, avdn_stream_t stream) {
  AVDN_REQUIRE(frames && lang_cls && w_in && w_out && attn && wc && e49, "avdn_frame_attn_fwd: null pointer");
  AVDN_REQUIRE(!fc2_w || (fc2_b && emb), "avdn_frame_attn_fwd: fc2 needs its bias and the emb output");
  if (B * T == 0) return AVDN_OK;
  frame_attn_fwd_kernel<<<B * T, 256, 0, avdn::to_cuda(stream)>>>(frames, lang_cls, w_in, w_out, fc2_w, fc2_b, T,
                                                                attn, wc, e49, emb);
  return avdn::check_launch("avdn_frame_attn_fwd");
}

extern "C" int avdn_frame_attn_bwd(const float* frames, const float* lang_cls, const float* w_in,
                                   const float* w_out, const float* fc2_w, int B, int T, const float* attn,
                                   const float* wc, const float* e49, const float* d_emb, float* d_frames,
                                   float* d_w_in, float* d_w_out, float* d_fc2_w, float* d_fc2_b,
                                   avdn_stream_t stream) {
  return avdn_frame_attn_bwd_cls(frames, lang_cls, w_in, w_out, fc2_w, B, T, attn, wc, e49, d_emb, d_frames, d_w_in,
                                 d_w_out, d_fc2_w, d_fc2_b, nullptr, stream);
}

extern "C" int avdn_frame_attn_bwd_cls(const float* frames, const float* lang_cls, const float* w_in,
                                       const float* w_out, const float* fc2_w, int B, int T, const float* attn,
                                       const float* wc, const float* e49, const float* d_emb, float* d_frames,
                                       float* d_w_in, float* d_w_out, float* d_fc2_w, float* d_fc2_b,
                                       float* d_lang_cls, avdn_stream_t stream) {
  AVDN_REQUIRE(frames && lang_cls && w_in && w_out && attn && wc && e49 && d_emb && d_frames && d_w_in && d_w_out &&
                   (!fc2_w || (d_fc2_w && d_fc2_b)),
               "avdn_frame_attn_bwd: null pointer");
  if (B * T == 0) return AVDN_OK;
  static_assert(E % FC2_ROWS == 0, "fc2 gradient blocks tile the 768 rows");
  if (fc2_w)
    frame_attn_fc2_grad_kernel<<<dim3(E / FC2_ROWS, FC2_SLICES), FC2_ROWS * (NSP + 1), 0, avdn::to_cuda(stream)>>>(
        d_emb, e49, B * T, d_fc2_w, d_fc2_b);
  frame_attn_bwd_kernel<<<B * T, 256, 0, avdn::to_cuda(stream)>>>(frames, lang_cls, w_in, w_out, fc2_w, T, attn, wc,
                                                                e49, d_emb, d_frames, d_w_in, d_w_out, d_fc2_w,
                                                                d_fc2_b, d_lang_cls);
  return avdn::check_launch("avdn_frame_attn_bwd");
}

extern "C" int avdn_embed_fwd(const float* lang, const float* emb_frames, const float* dirs, const float* wd,
                              const float* bd, const float* pe, int B, int L, int T, float* v,
                              avdn_stream_t stream) {
  AVDN_REQUIRE((lang || L == 0) && emb_frames && dirs && pe && v && (wd == nullptr || bd != nullptr),
               "avdn_embed_fwd: null pointer");
  AVDN_REQUIRE(B > 0 && L >= 0 && T >= 1, "avdn_embed_fwd: bad shape");
  embed_fwd_kernel<<<rows_grid((long long)B * (L + 2 * T)), 256, 0, avdn::to_cuda(stream)>>>(
      lang, emb_frames, dirs, wd, bd, pe, B, L, T, v);
  return avdn::check_launch("avdn_embed_fwd");
}

extern "C" int avdn_embed_dir_bwd(const float* dv, const float* dirs, int B, int L, int T, float* d_wd, float* d_bd,
                                  avdn_stream_t stream) {
  AVDN_REQUIRE(dv && dirs && d_wd && d_bd, "avdn_embed_dir_bwd: null pointer");
  embed_dir_bwd_kernel<<<(E + 127) / 128, 128, 0, avdn::to_cuda(stream)>>>(dv, dirs, B, L, T, d_wd, d_bd);
  return avdn::check_launch("avdn_embed_dir_bwd");
}

extern "C" int avdn_ln_fwd_drop(const float* a, const float* b, const float* gamma, const float* beta, long long M,
                                int D, float eps, float* v_out, float* y, void* y16, float* mean, float* rstd,
                                float p, unsigned long long seed, unsigned int site, avdn_stream_t stream) {
  AVDN_REQUIRE(D == E, "avdn_ln_fwd: d_model must be 768 (got %d)", D);
  AVDN_REQUIRE(a && gamma && beta && mean && rstd && M > 0, "avdn_ln_fwd: bad argument");
  AVDN_REQUIRE(drop_ok(p) && (p == 0.f || b), "avdn_ln_fwd: dropout p in [0,1) and needs the branch operand b");
  ln_fwd_kernel<<<rows_grid(M), 256, 0, avdn::to_cuda(stream)>>>(a, b, gamma, beta, M, eps, v_out, y,
                                                               reinterpret_cast<__nv_bfloat16*>(y16), mean, rstd,
                                                               avdn_drop_thresh(p), drop_scale(p), seed, site);
  return avdn::check_launch("avdn_ln_fwd");
}

extern "C" int avdn_ln_fwd(const float* a, const float* b, const float* gamma, const float* beta, long long M, int D,
                           float eps, float* v_out, float* y, void* y16, float* mean, float* rstd,
                           avdn_stream_t stream) {
  return avdn_ln_fwd_drop(a, b, gamma, beta, M, D, eps, v_out, y, y16, mean, rstd, 0.f, 0ull, 0u, stream);
}

extern "C" int avdn_ln_bwd(const float* dy1, const float* dy2, const float* v, const float* mean, const float* rstd,
                           const float* gamma, long long M, int D, float* dv, void* dv16, float* dgamma, float* dbeta,
                           avdn_stream_t stream) {
  return avdn_ln_bwd_drop(dy1, dy2, v, mean, rstd, gamma, M, D, dv, dv16, dgamma, dbeta, 0.f, 0ull, 0u, stream);
}

extern "C" int avdn_ln_bwd_drop(const float* dy1, const float* dy2, const float* v, const float* mean,
                                const float* rstd, const float* gamma, long long M, int D, float* dv, void* dv16,
                                float* dgamma, float* dbeta, float p, unsigned long long seed, unsigned int site,
                                avdn_stream_t stream) {
  AVDN_REQUIRE(drop_ok(p), "avdn_ln_bwd: dropout p must be in [0,1)");
  AVDN_REQUIRE(D == E, "avdn_ln_bwd: d_model must be 768 (got %d)", D);
  AVDN_REQUIRE(dy1 && v && mean && rstd && gamma && dgamma && dbeta && M > 0, "avdn_ln_bwd: bad argument");
  long long blocks = rows_grid(M);
  const long long cap = (long long)avdn::sm_count() * 4;
  if (blocks > cap) blocks = cap;
  ln_bwd_kernel<<<(unsigned)blocks, 256, 0, avdn::to_cuda(stream)>>>(dy1, dy2, v, mean, rstd, gamma, M, dv,
                                                                   reinterpret_cast<__nv_bfloat16*>(dv16), dgamma,
                                                                   dbeta, avdn_drop_thresh(p), drop_scale(p), seed,
                                                                   site);
  return avdn::check_launch("avdn_ln_bwd");
}

extern "C" int avdn_softmax_fwd_drop(const float* scores, const int* lens, int B, int H, int L, int T, int Sp, void* P,
                                     void* P_full, float p, unsigned long long seed, unsigned int site,
                                     avdn_stream_t stream) {
  AVDN_REQUIRE(scores && lens && P && T >= 0 && Sp >= L + 2 * T, "avdn_softmax_fwd: bad argument");
  AVDN_REQUIRE(drop_ok(p) && (p == 0.f || P_full), "avdn_softmax_fwd: dropout p in [0,1) and needs P_full");
  const unsigned grid = rows_grid((long long)B * H * (L + 2 * T));
  cudaStream_t s = avdn::to_cuda(stream);
  __nv_bfloat16 *Pb = reinterpret_cast<__nv_bfloat16*>(P), *Pf = reinterpret_cast<__nv_bfloat16*>(P_full);
  const unsigned int dthr = avdn_drop_thresh(p);
  const float dsc = drop_scale(p);
  const bool vec = Sp % 2 == 0 && (reinterpret_cast<uintptr_t>(scores) % 8 == 0) && (reinterpret_cast<uintptr_t>(P) % 4 == 0) &&
                   (reinterpret_cast<uintptr_t>(P_full) % 4 == 0);
  if (vec && Sp <= 128) softmax_fwd_regs_kernel<2><<<grid, 256, 0, s>>>(scores, lens, B, H, L, T, Sp, Pb, Pf, dthr, dsc, seed, site);
  else if (vec && Sp <= 320) softmax_fwd_regs_kernel<5><<<grid, 256, 0, s>>>(scores, lens, B, H, L, T, Sp, Pb, Pf, dthr, dsc, seed, site);
  else if (vec && Sp <= 512) softmax_fwd_regs_kernel<8><<<grid, 256, 0, s>>>(scores, lens, B, H, L, T, Sp, Pb, Pf, dthr, dsc, seed, site);
  else softmax_fwd_kernel<<<grid, 256, 0, s>>>(scores, lens, B, H, L, T, Sp, Pb, Pf, dthr, dsc, seed, site);
  return avdn::check_launch("avdn_softmax_fwd");
}

extern "C" int avdn_softmax_fwd(const float* scores, const int* lens, int B, int H, int L, int T, int Sp, void* P,
                                avdn_stream_t stream) {
  return avdn_softmax_fwd_drop(scores, lens, B, H, L, T, Sp, P, nullptr, 0.f, 0ull, 0u, stream);
}

extern "C" int avdn_softmax_bwd_drop(const void* P, const float* dP, long long rows, int S, int Sp, float alpha,
                                     void* dS, float p, unsigned long long seed, unsigned int site,
                                     avdn_stream_t stream) {
  AVDN_REQUIRE(P && dP && dS && rows > 0, "avdn_softmax_bwd: bad argument");
  AVDN_REQUIRE(drop_ok(p), "avdn_softmax_bwd: dropout p must be in [0,1)");
  const unsigned grid = rows_grid(rows);
  cudaStream_t s = avdn::to_cuda(stream);
  const __nv_bfloat16* Pb = reinterpret_cast<const __nv_bfloat16*>(P);
  __nv_bfloat16* dSb = reinterpret_cast<__nv_bfloat16*>(dS);
  const unsigned int dthr = avdn_drop_thresh(p);
  const float dsc = drop_scale(p);
  const bool vec = Sp % 2 == 0 && (reinterpret_cast<uintptr_t>(dP) % 8 == 0) && (reinterpret_cast<uintptr_t>(P) % 4 == 0) &&
                   (reinterpret_cast<uintptr_t>(dS) % 4 == 0);
  if (vec && Sp <= 128) softmax_bwd_regs_kernel<2><<<grid, 256, 0, s>>>(Pb, dP, rows, S, Sp, alpha, dSb, dthr, dsc, seed, site);
  else if (vec && Sp <= 320) softmax_bwd_regs_kernel<5><<<grid, 256, 0, s>>>(Pb, dP, rows, S, Sp, alpha, dSb, dthr, dsc, seed, site);
  else if (vec && Sp <= 512) softmax_bwd_regs_kernel<8><<<grid, 256, 0, s>>>(Pb, dP, rows, S, Sp, alpha, dSb, dthr, dsc, seed, site);
  else softmax_bwd_kernel<<<grid, 256, 0, s>>>(Pb, dP, rows, S, Sp, alpha, dSb, dthr, dsc, seed, site);
  return avdn::check_launch("avdn_softmax_bwd");
}

extern "C" int avdn_softmax_bwd(const void* P, const float* dP, long long rows, int S, int Sp, float alpha, void* dS,
                                avdn_stream_t stream) {
  return avdn_softmax_bwd_drop(P, dP, rows, S, Sp, alpha, dS, 0.f, 0ull, 0u, stream);
}

extern "C" int avdn_dropout_bf16(void* x, long long n, float p, unsigned long long seed, unsigned int site,
                                 avdn_stream_t stream) {
  AVDN_REQUIRE(x && n >= 0 && drop_ok(p), "avdn_dropout_bf16: bad argument");
  if (n == 0 || p == 0.f) return AVDN_OK;
  long long blocks = (n + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  dropout_bf16_kernel<<<(unsigned)blocks, 256, 0, avdn::to_cuda(stream)>>>(reinterpret_cast<__nv_bfloat16*>(x), n,
                                                                         avdn_drop_thresh(p), drop_scale(p), seed, site);
  return avdn::check_launch("avdn_dropout_bf16");
}

extern "C" int avdn_dropout_f32(float* x, void* x16, long long n, float p, unsigned long long seed, unsigned int site,
                                avdn_stream_t stream) {
  AVDN_REQUIRE(x && n >= 0 && drop_ok(p), "avdn_dropout_f32: bad argument");
  if (n == 0 || p == 0.f) return AVDN_OK;
  long long blocks = (n + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  dropout_f32_kernel<<<(unsigned)blocks, 256, 0, avdn::to_cuda(stream)>>>(x, reinterpret_cast<__nv_bfloat16*>(x16), n,
                                                                        avdn_drop_thresh(p), drop_scale(p), seed, site);
  return avdn::check_launch("avdn_dropout_f32");
}

static void add_dropout_f32_launch(const float* a, const float* b, float* out, long long n, long long idx0, float p,
                                   unsigned long long seed, unsigned int site, avdn_stream_t stream) {
  long long blocks = (n + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  add_dropout_f32_kernel<<<(unsigned)blocks, 256, 0, avdn::to_cuda(stream)>>>(
      a, b, out, n, (unsigned long long)idx0, avdn_drop_thresh(p), p == 0.f ? 1.f : drop_scale(p), seed, site);
}

extern "C" int avdn_add_dropout_f32(const float* a, const float* b, float* out, long long n, float p,
                                    unsigned long long seed, unsigned int site, avdn_stream_t stream) {
  AVDN_REQUIRE(a && out && n >= 0 && drop_ok(p), "avdn_add_dropout_f32: bad argument");
  if (n == 0) return AVDN_OK;
  add_dropout_f32_launch(a, b, out, n, 0, p, seed, site, stream);
  return avdn::check_launch("avdn_add_dropout_f32");
}

extern "C" int avdn_add_dropout_f32_at(const float* a, const float* b, float* out, long long n, long long idx0,
                                       float p, unsigned long long seed, unsigned int site, avdn_stream_t stream) {
  AVDN_REQUIRE(a && out, "avdn_add_dropout_f32_at: null pointer");
  AVDN_REQUIRE(n >= 0 && idx0 >= 0 && drop_ok(p), "avdn_add_dropout_f32_at: bad argument");
  if (n == 0) return AVDN_OK;
  add_dropout_f32_launch(a, b, out, n, idx0, p, seed, site, stream);
  return avdn::check_launch("avdn_add_dropout_f32_at");
}

extern "C" int avdn_dropout_keep_scale(float* out, long long n, float p, unsigned long long seed, unsigned int site,
                                       avdn_stream_t stream) {
  AVDN_REQUIRE(out && n >= 0 && drop_ok(p), "avdn_dropout_keep_scale: bad argument");
  if (n == 0) return AVDN_OK;
  long long blocks = (n + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  dropout_keep_scale_kernel<<<(unsigned)blocks, 256, 0, avdn::to_cuda(stream)>>>(out, n, avdn_drop_thresh(p),
                                                                               drop_scale(p), seed, site);
  return avdn::check_launch("avdn_dropout_keep_scale");
}

extern "C" int avdn_attn_decode(const void* qkv_new, const void* cache, int B, int R, int H, int Lc, int n, float scale,
                                void* ctx, avdn_stream_t stream) {
  AVDN_REQUIRE(qkv_new && cache && ctx && B > 0 && R > 0 && H * 64 == E && n >= 1 && n <= Lc,
               "avdn_attn_decode: bad argument (d_model 768 = H x 64, 1 <= n <= Lc)");
  attn_decode_kernel<<<rows_grid((long long)B * H * R), 256, 0, avdn::to_cuda(stream)>>>(
      reinterpret_cast<const __nv_bfloat16*>(qkv_new), reinterpret_cast<const __nv_bfloat16*>(cache), B, R, H, Lc, n,
      scale, reinterpret_cast<__nv_bfloat16*>(ctx));
  return avdn::check_launch("avdn_attn_decode");
}

extern "C" int avdn_build_masks(const int* lens, int B, int L, int T, uint8_t* mask_pad, float* mask_attn,
                                avdn_stream_t stream) {
  AVDN_REQUIRE(lens && mask_pad && mask_attn && T >= 1, "avdn_build_masks: bad argument");
  const long long S = L + 2 * T;
  const long long n = (B * S > S * S) ? B * S : S * S;
  build_masks_kernel<<<(unsigned)((n + 255) / 256), 256, 0, avdn::to_cuda(stream)>>>(lens, B, L, T, mask_pad,
                                                                                    mask_attn);
  return avdn::check_launch("avdn_build_masks");
}

extern "C" int avdn_colsum(const void* in, int in_dtype, long long M, int N, long long ld, float* out,
                           avdn_stream_t stream) {
  AVDN_REQUIRE(in && out && M > 0 && N > 0, "avdn_colsum: bad argument");
  long long yb = (M + 255) / 256;
  if (yb > 4 * avdn::sm_count()) yb = 4 * avdn::sm_count();
  const int rpb = (int)((M + yb - 1) / yb);
  dim3 grid((N + 31) / 32, (unsigned)yb);
  if (in_dtype == AVDN_DT_BF16)
    colsum_kernel<__nv_bfloat16><<<grid, 256, 0, avdn::to_cuda(stream)>>>(
        reinterpret_cast<const __nv_bfloat16*>(in), M, N, ld, out, rpb);
  else
    colsum_kernel<float><<<grid, 256, 0, avdn::to_cuda(stream)>>>(reinterpret_cast<const float*>(in), M, N, ld, out,
                                                                   rpb);
  return avdn::check_launch("avdn_colsum");
}

extern "C" int avdn_heads_fwd(const float* x, int B, int S, int row_vis, int row_dir, const float* w0,
                              const float* b0, const float* w1, const float* b1, const float* w2, const float* b2,
                              const float* wf, const float* bf, float* h0, float* h1, float* output, float* h_sali,
                              avdn_stream_t stream) {
  return avdn_heads_fwd_drop(x, B, S, row_vis, row_dir, w0, b0, w1, b1, w2, b2, wf, bf, h0, h1, output, h_sali, 0.f,
                             0ull, 0u, stream);
}

extern "C" int avdn_heads_fwd_drop(const float* x, int B, int S, int row_vis, int row_dir, const float* w0,
                                   const float* b0, const float* w1, const float* b1, const float* w2,
                                   const float* b2, const float* wf, const float* bf, float* h0, float* h1,
                                   float* output, float* h_sali, float p, unsigned long long seed,
                                   unsigned int site, avdn_stream_t stream) {
  AVDN_REQUIRE(drop_ok(p), "avdn_heads_fwd: dropout p must be in [0,1)");
  AVDN_REQUIRE(x && w0 && b0 && w1 && b1 && w2 && b2 && wf && bf && h0 && h1 && output && h_sali,
               "avdn_heads_fwd: null pointer");
  AVDN_REQUIRE(row_vis >= 0 && row_vis < S && row_dir >= 0 && row_dir < S, "avdn_heads_fwd: row out of range");
  if (B == 0) return AVDN_OK;
  heads_fwd_kernel<<<B, 256, 0, avdn::to_cuda(stream)>>>(x, S, row_vis, row_dir, w0, b0, w1, b1, w2, b2, wf, bf, h0,
                                                       h1, output, h_sali, avdn_drop_thresh(p), drop_scale(p), seed,
                                                       site);
  return avdn::check_launch("avdn_heads_fwd");
}

extern "C" int avdn_heads_bwd(const float* x, int B, int S, int row_vis, int row_dir, const float* w0,
                              const float* w1, const float* w2, const float* wf, const float* h0, const float* h1,
                              const float* h_sali, const float* d_output, const float* d_h_sali, float* dx,
                              float* dw0, float* db0, float* dw1, float* db1, float* dw2, float* db2, float* dwf,
                              float* dbf, avdn_stream_t stream) {
  return avdn_heads_bwd_drop(x, B, S, row_vis, row_dir, w0, w1, w2, wf, h0, h1, h_sali, d_output, d_h_sali, dx, dw0,
                             db0, dw1, db1, dw2, db2, dwf, dbf, 0.f, stream);
}

extern "C" int avdn_heads_bwd_drop(const float* x, int B, int S, int row_vis, int row_dir, const float* w0,
                                   const float* w1, const float* w2, const float* wf, const float* h0,
                                   const float* h1, const float* h_sali, const float* d_output,
                                   const float* d_h_sali, float* dx, float* dw0, float* db0, float* dw1, float* db1,
                                   float* dw2, float* db2, float* dwf, float* dbf, float p, avdn_stream_t stream) {
  AVDN_REQUIRE(drop_ok(p), "avdn_heads_bwd: dropout p must be in [0,1)");
  AVDN_REQUIRE(x && w0 && w1 && w2 && wf && h0 && h1 && h_sali && d_output && d_h_sali && dx && dw0 && db0 && dw1 &&
                   db1 && dw2 && db2 && dwf && dbf,
               "avdn_heads_bwd: null pointer");
  if (B == 0) return AVDN_OK;
  heads_bwd_kernel<<<B, 256, 0, avdn::to_cuda(stream)>>>(x, S, row_vis, row_dir, w0, w1, w2, wf, h0, h1, h_sali,
                                                       d_output, d_h_sali, dx, dw0, db0, dw1, db1, dw2, db2, dwf,
                                                       dbf, drop_scale(p));
  return avdn::check_launch("avdn_heads_bwd");
}
