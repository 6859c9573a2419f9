// Config 5 of the AVDN hot path: the recurrent "ViT_LSTM" policy step
// (src/models/vln_model.py:163-250) and the simulator update of the greedy rollout
// (src/xview_lstm/agent.py:592-602,700-730; move_view_corners src/xview_et/agent.py:285-384).
//
// Per rollout step and sample the policy is ~3 MFLOP (two LSTM cells, two soft-dot attentions, two
// small MLPs) next to 15.3 GFLOP of trunk: these kernels only have to be exact and launch-cheap.
// They are plain fp32 CUDA-core kernels (the reference runs this part in fp32 too):
//
//   linear_f32     y (+)= act(x W^T + b)              smem-tiled SGEMM, 64x64x16 tiles
//   lstm_cell      nn.LSTMCell pointwise part (gate order i,f,g,o)
//   lang_attn      SoftDotAttention(768) over the dialog tokens: scores, softmax over L, weighted sum
//   waypoint_step  agent.py:637-653,700-730 + move_view_corners, one thread per sample, float64
// and the backward of the training rollout (ViT_LSTM.train_engine): lstm_cell_bwd, lang_attn_bwd and
// direction_embed_bwd.  The weight gradients of the linear layers go through avdn_linear_f32_bwd (bert.cu).
#include "common.cuh"

namespace {

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

// ---------------------------------------------------------------- linear_f32
// y[m][n] (+)= act( sum_k x[m][k] * w[n][k] + b[n] ).  64x64 output tile per CTA, 256 threads,
// 4x4 micro-tile per thread, k-steps of 16 staged through shared memory.
constexpr int LT = 64, LK = 16;

__global__ void __launch_bounds__(256) linear_f32_kernel(const float* __restrict__ x, long long ldx,
                                                         const float* __restrict__ w, long long ldw,
                                                         const float* __restrict__ b, float* __restrict__ y,
                                                         long long ldy, int M, int N, int K, int act, int accumulate) {
  __shared__ float sx[LK][LT + 1], sw[LK][LT + 1];
  const int m0 = blockIdx.y * LT, n0 = blockIdx.x * LT;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;      // 16 x 16 threads
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int k0 = 0; k0 < K; k0 += LK) {
    for (int i = threadIdx.x; i < LT * LK; i += 256) {
      const int r = i / LK, kk = i % LK;
      const int m = m0 + r, n = n0 + r, k = k0 + kk;
      sx[kk][r] = (m < M && k < K) ? x[(long long)m * ldx + k] : 0.f;
      sw[kk][r] = (n < N && k < K) ? w[(long long)n * ldw + k] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < LK; ++kk) {
      float a[4], c[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = sx[kk][ty * 4 + i]; c[i] = sw[kk][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], c[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int m = m0 + ty * 4 + i, n = n0 + tx * 4 + j;
      if (m < M && n < N) {
        float v = acc[i][j] + (b ? b[n] : 0.f);
        if (accumulate) v += y[(long long)m * ldy + n];
        if (act == 1) v = fmaxf(v, 0.f);
        else if (act == 2) v = tanhf(v);
        y[(long long)m * ldy + n] = v;
      }
    }
}

// Second version for the rollout's shapes (M = 256 episodes, N = 4..2304, K = 32..1536, everything K-contiguous and
// 16-byte aligned): 32 x 64 output tile per 128-thread CTA (2-3x the CTAs of the 64 x 64 tiling on these skinny
// problems), k-steps of 32, operands fetched as float4 along k into REGISTERS one k-step ahead of the FMAs (the first
// version waited for every k-step's loads between two barriers: ~1 us per 16 k), shared-memory reads as float4.
// Every output is the same chain of fmaf over ascending k as in linear_f32_kernel, so the two agree bit for bit.
constexpr int L2_BM = 32, L2_BN = 64, L2_BK = 32, L2_THREADS = 128;

__global__ void __launch_bounds__(L2_THREADS) linear_f32_v2_kernel(const float* __restrict__ x, long long ldx,
                                                                   const float* __restrict__ w, long long ldw,
                                                                   const float* __restrict__ b, float* __restrict__ y,
                                                                   long long ldy, int M, int N, int K, int act,
                                                                   int accumulate) {
  __shared__ __align__(16) float sx[L2_BK][L2_BM + 4];
  __shared__ __align__(16) float sw[L2_BK][L2_BN + 4];
  const int m0 = blockIdx.y * L2_BM, n0 = blockIdx.x * L2_BN;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;      // 16 x 8 threads, 4 x 4 outputs each
  // global -> register mapping: float4 number idx of a tile = (row idx >> 3, k-chunk idx & 7): eight consecutive
  // lanes read 128 contiguous bytes of one row
  float4 rx[2], rw[4];
  const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
  auto fetch = [&](int k0) {
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int idx = tid + j * L2_THREADS, r = idx >> 3, k = k0 + (idx & 7) * 4, m = m0 + r;
      rx[j] = (m < M && k < K) ? __ldg(reinterpret_cast<const float4*>(x + (long long)m * ldx + k)) : zero4;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int idx = tid + j * L2_THREADS, r = idx >> 3, k = k0 + (idx & 7) * 4, n = n0 + r;
      rw[j] = (n < N && k < K) ? __ldg(reinterpret_cast<const float4*>(w + (long long)n * ldw + k)) : zero4;
    }
  };
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  fetch(0);
  for (int k0 = 0; k0 < K; k0 += L2_BK) {
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int idx = tid + j * L2_THREADS, r = idx >> 3, kk = (idx & 7) * 4;
      sx[kk][r] = rx[j].x; sx[kk + 1][r] = rx[j].y; sx[kk + 2][r] = rx[j].z; sx[kk + 3][r] = rx[j].w;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int idx = tid + j * L2_THREADS, r = idx >> 3, kk = (idx & 7) * 4;
      sw[kk][r] = rw[j].x; sw[kk + 1][r] = rw[j].y; sw[kk + 2][r] = rw[j].z; sw[kk + 3][r] = rw[j].w;
    }
    __syncthreads();
    if (k0 + L2_BK < K) fetch(k0 + L2_BK);         // in flight under the FMAs below
#pragma unroll
    for (int kk = 0; kk < L2_BK; ++kk) {
      const float4 a4 = *reinterpret_cast<const float4*>(&sx[kk][ty * 4]);
      const float4 c4 = *reinterpret_cast<const float4*>(&sw[kk][tx * 4]);
      const float a[4] = {a4.x, a4.y, a4.z, a4.w}, c[4] = {c4.x, c4.y, c4.z, c4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], c[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int m = m0 + ty * 4 + i, n = n0 + tx * 4 + j;
      if (m < M && n < N) {
        float v = acc[i][j] + (b ? b[n] : 0.f);
        if (accumulate) v += y[(long long)m * ldy + n];
        if (act == 1) v = fmaxf(v, 0.f);
        else if (act == 2) v = tanhf(v);
        y[(long long)m * ldy + n] = v;
      }
    }
}

// ------------------------------------------------------------------ lstm_cell
// gates [B,4H] = W_ih x + b_ih + W_hh h + b_hh (order i,f,g,o); c_prev may be NULL (zero state).
__global__ void lstm_cell_kernel(const float* __restrict__ gates, const float* __restrict__ c_prev,
                                 float* __restrict__ h_out, long long ldh, float* __restrict__ c_out, int B, int H) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * H) return;
  const int b = i / H, j = i - b * H;
  const float* g = gates + (size_t)b * 4 * H;
  const float ig = 1.f / (1.f + expf(-g[j]));
  const float fg = 1.f / (1.f + expf(-g[H + j]));
  const float gg = tanhf(g[2 * H + j]);
  const float og = 1.f / (1.f + expf(-g[3 * H + j]));
  const float c = fg * (c_prev ? c_prev[i] : 0.f) + ig * gg;
  c_out[i] = c;
  h_out[(size_t)b * ldh + j] = og * tanhf(c);
}

// Backward of lstm_cell_kernel from the saved pre-activations and cell state (autograd of nn.LSTMCell's pointwise
// part): dc = dh * o * (1 - tanh(c)^2) + dc_next; dgates = (dc g i(1-i), dc c_prev f(1-f), dc i (1-g^2),
// dh tanh(c) o(1-o)); dc_prev = dc f.  The gate activations are recomputed exactly as the forward computes them.
// dc_next and dc_prev are not __restrict__: a caller may pass one buffer for both (same element read, then written).
__global__ void lstm_cell_bwd_kernel(const float* __restrict__ gates, const float* __restrict__ c_prev,
                                     const float* __restrict__ c, const float* __restrict__ dh, long long lddh,
                                     const float* dc_next, float* __restrict__ dgates, float* dc_prev, int B, int H) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * H) return;
  const int b = i / H, j = i - b * H;
  const float* g = gates + (size_t)b * 4 * H;
  const float ig = 1.f / (1.f + expf(-g[j]));
  const float fg = 1.f / (1.f + expf(-g[H + j]));
  const float gg = tanhf(g[2 * H + j]);
  const float og = 1.f / (1.f + expf(-g[3 * H + j]));
  const float tc = tanhf(c[i]);
  const float cp = c_prev ? c_prev[i] : 0.f;
  const float d_h = dh[(size_t)b * lddh + j];
  const float dc = d_h * og * (1.f - tc * tc) + (dc_next ? dc_next[i] : 0.f);
  float* dg = dgates + (size_t)b * 4 * H;
  dg[j] = dc * gg * ig * (1.f - ig);
  dg[H + j] = dc * cp * fg * (1.f - fg);
  dg[2 * H + j] = dc * ig * (1.f - gg * gg);
  dg[3 * H + j] = d_h * tc * og * (1.f - og);
  if (c_prev) dc_prev[i] = dc * fg;
}

// direction_embedding([sin, cos](d / 180 * 3.14159)) (vln_model.py:228-229), float32 as torch evaluates it
__device__ __forceinline__ float direction_angle(float deg) { return __fmul_rn(__fdiv_rn(deg, 180.f), 3.14159f); }

__global__ void direction_embed_kernel(const float* __restrict__ deg, const float* __restrict__ w,
                                       const float* __restrict__ b, float* __restrict__ out, int B, int N) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * N) return;
  const int s = i / N, n = i - s * N;
  const float a = direction_angle(deg[s]);
  out[i] = __fadd_rn(__fadd_rn(__fmul_rn(w[n * 2], sinf(a)), __fmul_rn(w[n * 2 + 1], cosf(a))), b[n]);
}

// Its parameter gradient: one thread per (n, k), k = 0 (weight of sin), 1 (weight of cos), 2 (bias), summing over the
// B rows.  The sin / cos are the forward's (same expression, same translation unit, same flags), so the gradient
// sees exactly the inputs the forward used.
__global__ void direction_embed_bwd_kernel(const float* __restrict__ deg, const float* __restrict__ d_out, int B, int N,
                                           float* __restrict__ d_w, float* __restrict__ d_b) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 3 * N) return;
  const int n = i / 3, k = i - n * 3;
  float acc = 0.f;
  for (int s = 0; s < B; ++s) {
    const float a = direction_angle(deg[s]);
    const float v = k == 0 ? sinf(a) : (k == 1 ? cosf(a) : 1.f);
    acc = fmaf(d_out[(size_t)s * N + n], v, acc);
  }
  if (k < 2) d_w[n * 2 + k] += acc;
  else d_b[n] += acc;
}

// ------------------------------------------------------------------ lang_attn
// SoftDotAttention (vln_model.py:26-46) without the two Linear layers: one CTA per sample.
//   scores_l = ctx[b,l,:] . target[b,:] ; attn = softmax_l ; weighted = sum_l attn_l ctx[b,l,:]
__global__ void __launch_bounds__(256) lang_attn_kernel(const float* __restrict__ ctx, const float* __restrict__ target,
                                                        int L, int D, float* __restrict__ attn_out,
                                                        float* __restrict__ weighted, long long ldw) {
  extern __shared__ float sm[];            // [D] target, [L] scores
  float* s_t = sm;
  float* s_s = sm + D;
  __shared__ float s_max, s_sum;
  const int b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const float* c = ctx + (size_t)b * L * D;
  for (int d = tid; d < D; d += 256) s_t[d] = target[(size_t)b * D + d];
  __syncthreads();
  for (int l = warp; l < L; l += 8) {
    float a = 0.f;
    for (int d = lane; d < D; d += 32) a = fmaf(c[(size_t)l * D + d], s_t[d], a);
    a = warp_sum(a);
    if (lane == 0) s_s[l] = a;
  }
  __syncthreads();
  if (warp == 0) {
    float m = -INFINITY;
    for (int l = lane; l < L; l += 32) m = fmaxf(m, s_s[l]);
    m = warp_max(m);
    float s = 0.f;
    for (int l = lane; l < L; l += 32) s += expf(s_s[l] - m);
    s = warp_sum(s);
    if (lane == 0) { s_max = m; s_sum = s; }
  }
  __syncthreads();
  for (int l = tid; l < L; l += 256) {
    const float a = expf(s_s[l] - s_max) / s_sum;
    s_s[l] = a;
    if (attn_out) attn_out[(size_t)b * L + l] = a;
  }
  __syncthreads();
  for (int d = tid; d < D; d += 256) {
    float a = 0.f;
    for (int l = 0; l < L; ++l) a = fmaf(s_s[l], c[(size_t)l * D + d], a);
    weighted[(size_t)b * ldw + d] = a;
  }
}

// Second version, for D % 4 == 0 and D <= 1024 (the rollout's D = 768): the first version kept one 4-byte load per
// lane in flight (8 warps x 128 B per CTA) while streaming 768 KB of context per sample twice.  Here every load is a
// float4 and the loads of TWO rows x NQ float4 columns (scores) or EIGHT rows (weighted sum) are issued before they
// are used: 48 KB / 24 KB in flight per CTA.  A lane now sums the columns 4q..4q+3 of q = lane, lane + 32, ... (not
// d = lane, lane + 32, ...), so the results agree with the first version to fp32 summation order, not bit for bit.
template <int NQ>      // NQ = ceil(D / 4 / 32) <= 8 float4 columns per lane
__global__ void __launch_bounds__(256) lang_attn_v2_kernel(const float* __restrict__ ctx, const float* __restrict__ target,
                                                           int L, int D, float* __restrict__ attn_out,
                                                           float* __restrict__ weighted, long long ldw) {
  extern __shared__ float4 sm4[];          // [D] target, [L] scores
  float* s_t = reinterpret_cast<float*>(sm4);
  float* s_s = s_t + D;
  __shared__ float s_max, s_sum;
  const int b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int D4 = D >> 2;
  const float4* c4 = reinterpret_cast<const float4*>(ctx + (size_t)b * L * D);
  const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int d = tid; d < D; d += 256) s_t[d] = target[(size_t)b * D + d];
  __syncthreads();
  float4 t4[NQ];
#pragma unroll
  for (int i = 0; i < NQ; ++i) {
    const int q = lane + 32 * i;
    t4[i] = q < D4 ? *reinterpret_cast<const float4*>(&s_t[4 * q]) : zero4;
  }
  for (int l0 = warp; l0 < L; l0 += 16) {          // rows l0 and l0 + 8 of this warp at once
    float4 v[2][NQ];
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
      for (int i = 0; i < NQ; ++i) {
        const int q = lane + 32 * i, l = l0 + 8 * r;
        v[r][i] = (q < D4 && l < L) ? __ldg(c4 + (size_t)l * D4 + q) : zero4;
      }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      float a = 0.f;
#pragma unroll
      for (int i = 0; i < NQ; ++i) {
        a = fmaf(v[r][i].x, t4[i].x, a);
        a = fmaf(v[r][i].y, t4[i].y, a);
        a = fmaf(v[r][i].z, t4[i].z, a);
        a = fmaf(v[r][i].w, t4[i].w, a);
      }
      a = warp_sum(a);
      if (lane == 0 && l0 + 8 * r < L) s_s[l0 + 8 * r] = a;
    }
  }
  __syncthreads();
  if (warp == 0) {
    float m = -INFINITY;
    for (int l = lane; l < L; l += 32) m = fmaxf(m, s_s[l]);
    m = warp_max(m);
    float s = 0.f;
    for (int l = lane; l < L; l += 32) s += expf(s_s[l] - m);
    s = warp_sum(s);
    if (lane == 0) { s_max = m; s_sum = s; }
  }
  __syncthreads();
  for (int l = tid; l < L; l += 256) {
    const float a = expf(s_s[l] - s_max) / s_sum;
    s_s[l] = a;
    if (attn_out) attn_out[(size_t)b * L + l] = a;
  }
  __syncthreads();
  if (tid < D4) {                                   // one float4 column per thread (D <= 1024)
    float4 acc = zero4;
    int l = 0;
    for (; l + 8 <= L; l += 8) {
      float4 u[8];
#pragma unroll
      for (int r = 0; r < 8; ++r) u[r] = __ldg(c4 + (size_t)(l + r) * D4 + tid);
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const float p = s_s[l + r];
        acc.x = fmaf(p, u[r].x, acc.x); acc.y = fmaf(p, u[r].y, acc.y);
        acc.z = fmaf(p, u[r].z, acc.z); acc.w = fmaf(p, u[r].w, acc.w);
      }
    }
    for (; l < L; ++l) {
      const float p = s_s[l];
      const float4 u = __ldg(c4 + (size_t)l * D4 + tid);
      acc.x = fmaf(p, u.x, acc.x); acc.y = fmaf(p, u.y, acc.y);
      acc.z = fmaf(p, u.z, acc.z); acc.w = fmaf(p, u.w, acc.w);
    }
    float* o = weighted + (size_t)b * ldw + 4 * tid;      // ldw need not be a multiple of 4: scalar stores
    o[0] = acc.x; o[1] = acc.y; o[2] = acc.z; o[3] = acc.w;
  }
}

// Backward of lang_attn (autograd of vln_model.py:33-42 between the two Linear layers), one CTA per sample:
//   d_attn_l = ctx_l . d_weighted ; d_score_l = attn_l (d_attn_l - sum_l' attn_l' d_attn_l')
//   d_target = sum_l d_score_l ctx_l ; d_ctx_l += attn_l d_weighted + d_score_l target
// Two passes over the sample's context: the row dots (a warp per row), then one thread per column walks the rows
// for d_target and the d_ctx update together.
__global__ void __launch_bounds__(256) lang_attn_bwd_kernel(const float* __restrict__ ctx,
                                                            const float* __restrict__ target,
                                                            const float* __restrict__ attn,
                                                            const float* __restrict__ d_weighted, long long lddw,
                                                            int L, int D, float* __restrict__ d_target,
                                                            float* __restrict__ d_ctx) {
  extern __shared__ float sm[];            // [D] d_weighted, [D] target, [L] attn, [L] d_attn -> d_score
  float* s_dw = sm;
  float* s_t = sm + D;
  float* s_a = s_t + D;
  float* s_ds = s_a + L;
  __shared__ float s_dot;
  const int b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const float* c = ctx + (size_t)b * L * D;
  for (int d = tid; d < D; d += 256) {
    s_dw[d] = d_weighted[(size_t)b * lddw + d];
    s_t[d] = target[(size_t)b * D + d];
  }
  for (int l = tid; l < L; l += 256) s_a[l] = attn[(size_t)b * L + l];
  __syncthreads();
  for (int l = warp; l < L; l += 8) {
    float a = 0.f;
    for (int d = lane; d < D; d += 32) a = fmaf(c[(size_t)l * D + d], s_dw[d], a);
    a = warp_sum(a);
    if (lane == 0) s_ds[l] = a;
  }
  __syncthreads();
  if (warp == 0) {
    float a = 0.f;
    for (int l = lane; l < L; l += 32) a = fmaf(s_a[l], s_ds[l], a);
    a = warp_sum(a);
    if (lane == 0) s_dot = a;
  }
  __syncthreads();
  for (int l = tid; l < L; l += 256) s_ds[l] = s_a[l] * (s_ds[l] - s_dot);
  __syncthreads();
  float* dc = d_ctx ? d_ctx + (size_t)b * L * D : nullptr;
  for (int d = tid; d < D; d += 256) {
    const float wd = s_dw[d], td = s_t[d];
    float acc = 0.f;
    for (int l = 0; l < L; ++l) {
      const float ds = s_ds[l];
      acc = fmaf(ds, c[(size_t)l * D + d], acc);
      if (dc) dc[(size_t)l * D + d] += fmaf(s_a[l], wd, ds * td);
    }
    d_target[(size_t)b * D + d] = acc;
  }
}

// -------------------------------------------------------------- waypoint_step
struct P2 { double x, y; };
__device__ __forceinline__ P2 sub(P2 a, P2 b) { return {__dsub_rn(a.x, b.x), __dsub_rn(a.y, b.y)}; }
__device__ __forceinline__ double nrm(P2 a) { return sqrt(__dadd_rn(__dmul_rn(a.x, a.x), __dmul_rn(a.y, a.y))); }
// p + d / n * change   (numpy evaluates (d / n) * change element-wise, then adds)
__device__ __forceinline__ P2 push(P2 p, P2 d, double n, double change) {
  return {__dadd_rn(p.x, __dmul_rn(__ddiv_rn(d.x, n), change)), __dadd_rn(p.y, __dmul_rn(__ddiv_rn(d.y, n), change))};
}
__device__ __forceinline__ bool inside(P2 p, const double* bd) {
  return p.x > bd[0] && p.x < bd[2] && p.y > bd[1] && p.y < bd[3];
}
// src/xview_et/agent.py:83-101
__device__ double get_direction(P2 start, P2 end) {
  const double v0 = __dsub_rn(end.x, start.x), v1 = __dsub_rn(end.y, start.y);
  double ang;
  if (v1 > 0) ang = atan(v0 / v1) / 1.57 * 90;
  else if (v1 < 0) ang = atan(v0 / v1) / 1.57 * 90 + 180;
  else ang = (v0 > 0) ? 90.0 : 270.0;
  return fmod(360 - ang + 90, 360.0);      // operands are >= 0 here: fmod == python %
}
__device__ __forceinline__ double pymod360(double a) {
  double r = fmod(a, 360.0);
  if (r < 0) r += 360.0;
  return r;
}

// One thread per sample: post-process the 4 predicted scalars (agent.py:637-653,745-752), decide whether
// the sample stops (xview_lstm/agent.py:700-709), otherwise zoom / rotate / move the view corners
// (move_view_corners).  `ended` is sticky; a sample that stopped earlier but predicts progress below the
// threshold again IS moved, exactly as the reference loop does (it only skips on the current step's test).
__global__ void waypoint_step_kernel(const float* __restrict__ output, double* __restrict__ corners,
                                     const double* __restrict__ bounds, double* __restrict__ cur_dir,
                                     uint8_t* __restrict__ ended, int B, float stop_threshold, int last_step,
                                     int* __restrict__ angle_deg, double* __restrict__ dist_out,
                                     int* __restrict__ altitude_m) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  float x = output[i * 4], y = output[i * 4 + 1];
  const float m = fmaxf(fmaxf(fabsf(x), fabsf(y)), 1.f);
  x = __fdiv_rn(x, m);
  y = __fdiv_rn(y, m);
  const float a = fminf(1.f, fmaxf(0.f, output[i * 4 + 2]));
  const float p = fminf(1.f, fmaxf(0.f, output[i * 4 + 3]));
  // math.atan2 on float32 elements promoted to python floats (float64)
  double a_dir = (atan2((double)x, (double)y) / 3.14159 + 2.0) / 2.0;
  a_dir = a_dir - floor(a_dir);
  int angle = __double2int_rn(a_dir * 360.0);
  const int altitude = __double2int_rn((double)a * 360.0) + 40;
  P2 c[4];
  double* cp = corners + (size_t)i * 8;
#pragma unroll
  for (int k = 0; k < 4; ++k) c[k] = {cp[2 * k], cp[2 * k + 1]};
  const float nrm_xy = sqrtf(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)));     // np.linalg.norm of a float32 pair
  const double distance = (double)nrm_xy * (nrm(sub(c[0], c[1])) / 2.0);
  if (angle_deg) angle_deg[i] = angle;
  if (dist_out) dist_out[i] = distance;
  if (altitude_m) altitude_m[i] = altitude;
  if (p > stop_threshold || last_step) { ended[i] = 1; return; }

  const double* bd = bounds + (size_t)i * 4;          // gps_botm_left (2), gps_top_right (2)
  const P2 mean0 = {(c[0].x + c[1].x + c[2].x + c[3].x) / 4.0, (c[0].y + c[1].y + c[2].y + c[3].y) / 4.0};
  const P2 front = {(c[0].x + c[1].x) / 2.0, (c[0].y + c[1].y) / 2.0};
  const double cur = pymod360((double)__double2int_rn(get_direction(mean0, front)));
  double ang = (double)angle;
  const double in_dir = cur_dir[i];
  if (fabs(in_dir - cur) > 2) ang += in_dir;
  // ---- zoom ----
  const double edge = nrm(sub(c[1], c[0])) * 11.13 * 1e4;
  const double ch = 0.5 * ((double)altitude - edge) / 11.13 / 1e4;
  P2 z[4];
  const double n01 = nrm(sub(c[1], c[0])), n03 = nrm(sub(c[3], c[0])), n12 = nrm(sub(c[2], c[1])), n23 = nrm(sub(c[2], c[3]));
  z[0] = push(push(c[0], sub(c[0], c[1]), n01, ch), sub(c[0], c[3]), n03, ch);
  z[1] = push(push(c[1], sub(c[1], c[0]), n01, ch), sub(c[1], c[2]), n12, ch);
  z[2] = push(push(c[2], sub(c[2], c[3]), n23, ch), sub(c[2], c[1]), n12, ch);
  z[3] = push(push(c[3], sub(c[3], c[2]), n23, ch), sub(c[3], c[0]), n03, ch);
  if (!(inside(z[0], bd) && inside(z[1], bd) && inside(z[2], bd) && inside(z[3], bd))) { cur_dir[i] = cur; return; }
  // ---- rotate by -ang about the centre (pi = 3.14159) ----
  const P2 ctr = {(z[0].x + z[1].x + z[2].x + z[3].x) / 4.0, (z[0].y + z[1].y + z[2].y + z[3].y) / 4.0};
  const double th = -ang / 180 * 3.14159, cs = cos(th), sn = sin(th);
  P2 r[4];
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const P2 d = sub(z[k], ctr);
    r[k] = {__dadd_rn(ctr.x, __dadd_rn(__dmul_rn(cs, d.x), __dmul_rn(sn, d.y))),
            __dadd_rn(ctr.y, __dadd_rn(__dmul_rn(-sn, d.x), __dmul_rn(cs, d.y)))};
    ok = ok && inside(r[k], bd);
  }
  if (!ok) {
#pragma unroll
    for (int k = 0; k < 4; ++k) { cp[2 * k] = z[k].x; cp[2 * k + 1] = z[k].y; }
    cur_dir[i] = cur;
    return;
  }
  // ---- move forward ----
  const double m03 = nrm(sub(r[3], r[0])), m12 = nrm(sub(r[2], r[1]));
  P2 f[4];
  f[0] = push(r[0], sub(r[0], r[3]), m03, distance);
  f[1] = push(r[1], sub(r[1], r[2]), m12, distance);
  f[2] = push(r[2], sub(r[1], r[2]), m12, distance);
  f[3] = push(r[3], sub(r[0], r[3]), m03, distance);
  const bool ok2 = inside(f[0], bd) && inside(f[1], bd) && inside(f[2], bd) && inside(f[3], bd);
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    cp[2 * k] = ok2 ? f[k].x : r[k].x;
    cp[2 * k + 1] = ok2 ? f[k].y : r[k].y;
  }
  cur_dir[i] = pymod360(cur + ang);
}

}  // namespace

// ===================================================================== C ABI
// Which kernels serve avdn_linear_f32 / avdn_lang_attn_fwd: 2 = the register-prefetching / float4 versions (default),
// 1 = the first versions (kept: unaligned or K % 4 != 0 / D % 4 != 0 shapes always use them, and the tests compare).
// AVDN_LSTM_KERNELS in the environment sets the initial value; the argument 0 only queries.
static int& lstm_kernels_version() {
  static int v = [] {
    const char* e = getenv("AVDN_LSTM_KERNELS");
    return (e && e[0] == '1') ? 1 : 2;
  }();
  return v;
}
extern "C" int avdn_lstm_set_kernels(int version) {
  int& v = lstm_kernels_version();
  const int old = v;
  if (version == 1 || version == 2) v = version;
  return old;
}

extern "C" int avdn_linear_f32(const float* x, long long ldx, const float* w, long long ldw, const float* b, float* y,
                               long long ldy, int M, int N, int K, int act, int accumulate, avdn_stream_t stream) {
  AVDN_REQUIRE(x && w && y && M > 0 && N > 0 && K > 0, "avdn_linear_f32: bad argument");
  AVDN_REQUIRE(act >= 0 && act <= 2, "avdn_linear_f32: act must be 0 (none), 1 (relu) or 2 (tanh)");
  const bool vec = (K % 4 == 0) && (ldx % 4 == 0) && (ldw % 4 == 0) &&
                   (reinterpret_cast<uintptr_t>(x) % 16 == 0) && (reinterpret_cast<uintptr_t>(w) % 16 == 0);
  if (lstm_kernels_version() >= 2 && vec) {
    dim3 grid((N + L2_BN - 1) / L2_BN, (M + L2_BM - 1) / L2_BM);
    linear_f32_v2_kernel<<<grid, L2_THREADS, 0, avdn::to_cuda(stream)>>>(x, ldx, w, ldw, b, y, ldy, M, N, K, act,
                                                                        accumulate);
    return avdn::check_launch("avdn_linear_f32 (v2)");
  }
  dim3 grid((N + LT - 1) / LT, (M + LT - 1) / LT);
  linear_f32_kernel<<<grid, 256, 0, avdn::to_cuda(stream)>>>(x, ldx, w, ldw, b, y, ldy, M, N, K, act, accumulate);
  return avdn::check_launch("avdn_linear_f32");
}

extern "C" int avdn_lstm_cell(const float* gates, const float* c_prev, float* h_out, long long ldh, float* c_out,
                              int B, int H, avdn_stream_t stream) {
  AVDN_REQUIRE(gates && h_out && c_out && B > 0 && H > 0 && ldh >= H, "avdn_lstm_cell: bad argument");
  lstm_cell_kernel<<<(B * H + 255) / 256, 256, 0, avdn::to_cuda(stream)>>>(gates, c_prev, h_out, ldh, c_out, B, H);
  return avdn::check_launch("avdn_lstm_cell");
}

extern "C" int avdn_direction_embed(const float* deg, const float* w, const float* b, float* out, int B, int N,
                                    avdn_stream_t stream) {
  AVDN_REQUIRE(deg && w && b && out && B > 0 && N > 0, "avdn_direction_embed: bad argument");
  direction_embed_kernel<<<(B * N + 127) / 128, 128, 0, avdn::to_cuda(stream)>>>(deg, w, b, out, B, N);
  return avdn::check_launch("avdn_direction_embed");
}

extern "C" int avdn_lang_attn_fwd(const float* ctx, const float* target, int B, int L, int D, float* attn,
                                  float* weighted, long long ldw, avdn_stream_t stream) {
  AVDN_REQUIRE(ctx && target && weighted && B > 0 && L > 0 && D > 0 && ldw >= D, "avdn_lang_attn_fwd: bad argument");
  const size_t smem = (size_t)(D + L) * sizeof(float);
  AVDN_REQUIRE(smem <= 48 * 1024, "avdn_lang_attn_fwd: D + L = %d too large", D + L);
  cudaStream_t s = avdn::to_cuda(stream);
  const int nq = (D / 4 + 31) / 32;
  if (lstm_kernels_version() >= 2 && D % 4 == 0 && nq <= 8 && reinterpret_cast<uintptr_t>(ctx) % 16 == 0) {
#define AVDN_LANG_ATTN_CASE(NQ) \
  case NQ: lang_attn_v2_kernel<NQ><<<B, 256, smem, s>>>(ctx, target, L, D, attn, weighted, ldw); break;
    switch (nq) {
      AVDN_LANG_ATTN_CASE(1) AVDN_LANG_ATTN_CASE(2) AVDN_LANG_ATTN_CASE(3) AVDN_LANG_ATTN_CASE(4)
      AVDN_LANG_ATTN_CASE(5) AVDN_LANG_ATTN_CASE(6) AVDN_LANG_ATTN_CASE(7) AVDN_LANG_ATTN_CASE(8)
    }
#undef AVDN_LANG_ATTN_CASE
    return avdn::check_launch("avdn_lang_attn_fwd (v2)");
  }
  lang_attn_kernel<<<B, 256, smem, s>>>(ctx, target, L, D, attn, weighted, ldw);
  return avdn::check_launch("avdn_lang_attn_fwd");
}

extern "C" int avdn_lstm_cell_bwd(const float* gates, const float* c_prev, const float* c, const float* dh,
                                  long long lddh, const float* dc_next, float* dgates, float* dc_prev, int B, int H,
                                  avdn_stream_t stream) {
  AVDN_REQUIRE(gates && c && dh && dgates && B > 0 && H > 0 && lddh >= H, "avdn_lstm_cell_bwd: bad argument");
  AVDN_REQUIRE(!c_prev || dc_prev, "avdn_lstm_cell_bwd: dc_prev is required when c_prev is given");
  lstm_cell_bwd_kernel<<<(B * H + 255) / 256, 256, 0, avdn::to_cuda(stream)>>>(gates, c_prev, c, dh, lddh, dc_next,
                                                                              dgates, dc_prev, B, H);
  return avdn::check_launch("avdn_lstm_cell_bwd");
}

extern "C" int avdn_direction_embed_bwd(const float* deg, const float* d_out, int B, int N, float* d_w, float* d_b,
                                        avdn_stream_t stream) {
  AVDN_REQUIRE(deg && d_out && d_w && d_b && B > 0 && N > 0, "avdn_direction_embed_bwd: bad argument");
  direction_embed_bwd_kernel<<<(3 * N + 127) / 128, 128, 0, avdn::to_cuda(stream)>>>(deg, d_out, B, N, d_w, d_b);
  return avdn::check_launch("avdn_direction_embed_bwd");
}

extern "C" int avdn_lang_attn_bwd(const float* ctx, const float* target, const float* attn, const float* d_weighted,
                                  long long lddw, int B, int L, int D, float* d_target, float* d_ctx,
                                  avdn_stream_t stream) {
  AVDN_REQUIRE(ctx && target && attn && d_weighted && d_target && B > 0 && L > 0 && D > 0 && lddw >= D,
               "avdn_lang_attn_bwd: bad argument");
  const size_t smem = (size_t)(2 * D + 2 * L) * sizeof(float);
  AVDN_REQUIRE(smem <= 48 * 1024, "avdn_lang_attn_bwd: D + L = %d too large", D + L);
  lang_attn_bwd_kernel<<<B, 256, smem, avdn::to_cuda(stream)>>>(ctx, target, attn, d_weighted, lddw, L, D, d_target,
                                                               d_ctx);
  return avdn::check_launch("avdn_lang_attn_bwd");
}

extern "C" int avdn_waypoint_step(const float* output, double* corners, const double* bounds, double* cur_dir,
                                  uint8_t* ended, int B, float stop_threshold, int last_step, int* angle_deg,
                                  double* dist, int* altitude_m, avdn_stream_t stream) {
  AVDN_REQUIRE(output && corners && bounds && cur_dir && ended && B > 0, "avdn_waypoint_step: bad argument");
  waypoint_step_kernel<<<(B + 127) / 128, 128, 0, avdn::to_cuda(stream)>>>(output, corners, bounds, cur_dir, ended, B,
                                                                          stop_threshold, last_step, angle_deg, dist,
                                                                          altitude_m);
  return avdn::check_launch("avdn_waypoint_step");
}
