// Agent slice of the AVDN hot path (src/xview_et/agent.py): the per-step loss
// (four MSE-sum terms, the angular term and the NSS human-attention loss with
// the 8x8 -> 224x224 bilinear upsample fused in, forward AND backward in one
// kernel), waypoint post-processing / discretisation, and the optimiser step
// (global-norm clip + AdamW over a flat parameter arena).
#include "common.cuh"

namespace {

constexpr int VIEW = AVDN_VIEW;
constexpr int NPX = VIEW * VIEW;
constexpr float PI_REF = 3.14159f;      // the reference's pi (agent.py:606,666,745)

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// F.interpolate(bilinear, align_corners=False) source taps of destination index d (8 -> 224)
__device__ __forceinline__ void bilin_tap(int d, int* i0, int* i1, float* l1) {
  const float scale = 8.0f / 224.0f;
  float src = scale * ((float)d + 0.5f) - 0.5f;
  if (src < 0.f) src = 0.f;
  const int a = (int)src;
  *i0 = a;
  *i1 = a + (a < 7 ? 1 : 0);
  *l1 = src - (float)a;
}

__device__ __forceinline__ float ang_ref(float v0, float v1) {
  // ((atan2(v0, v1) / 3.14159 + 2) / 2) % 1   in float32, as torch evaluates it
  const float a = (atan2f(v0, v1) / PI_REF + 2.0f) / 2.0f;
  return a - floorf(a);
}

// One CTA per sample: loss_i and its gradient w.r.t. output[i,:] and h_sali[i,:].
//   agent.py:663-669  4 x MSELoss(reduction='sum') + angular term
//   agent.py:673-681  nss_w * NSS(pred_saliency[i], gt_saliency[i]) when sum(gt) > 0
//   agent.py:883-885  loss += ml_loss * train_ml / batch_size   (== `scale`)
//
// NSS without ever forming the 224x224 prediction: the upsample is linear and separable,
//   p[y,x] = sum_ab Wy[y,a] Wx[x,b] h[a,b]        (Wy = Wx = W, the 224x8 bilinear tap matrix)
// so with c[a] = sum_y W[y,a], G[a,a'] = sum_y W[y,a] W[y,a'] (constants) and ONE pass over the
// fixation map f for F[a,b] = sum_yx W[y,a] W[x,b] f[y,x] and SF = sum f:
//   sum p   = sum_ab h[a,b] c[a] c[b]          sum p^2 = sum_ab h[a,b] (G h G^T)[a,b]
//   sum p f = sum_ab h[a,b] F[a,b]
//   dL/dh[a,b] = k1 (F[a,b] - fm c[a] c[b]) - k2 ((G h G^T)[a,b] - m c[a] c[b])
// (the adjoint of the upsample applied to the per-pixel gradient k1 (f - fm) - k2 (p - m)).
__global__ void __launch_bounds__(256) loss_kernel(const float* __restrict__ output, const float* __restrict__ h_sali,
                                                   const float* __restrict__ gt_xy, const float* __restrict__ gt_alt,
                                                   const float* __restrict__ gt_prog, const uint8_t* __restrict__ att,
                                                   const float* __restrict__ jitter, float nss_w, int nss_r,
                                                   double scale, double* __restrict__ loss_total,
                                                   double* __restrict__ loss_i, float* __restrict__ d_output,
                                                   float* __restrict__ d_h_sali) {
  __shared__ float s_h[64];
  __shared__ float s_dh[64];
  __shared__ double s_c[8], s_G[8][8], s_F[8][8], s_GhG[8][8], s_T[8][8];
  __shared__ double s_col[8][VIEW];          // per-column partial sums A[a][x] = sum_y W[y,a] f[y,x]
  __shared__ double s_red[8];
  __shared__ double s_stat[6];
  const int b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid < 64) {
    s_h[tid] = h_sali[b * 64 + tid]; s_dh[tid] = 0.f;
    (&s_G[0][0])[tid] = 0.0; (&s_F[0][0])[tid] = 0.0;
  }
  if (tid < 8) s_c[tid] = 0.0;
  __syncthreads();
  double nss_term = 0.0;
  bool use_nss = false;
  if (att != nullptr && nss_w != 0.f) {
    const uint8_t* f = att + (size_t)b * NPX;
    int t0 = 0, t1 = 0; float tl = 0.f;
    double sf = 0.0;
    if (tid < VIEW) {
      bilin_tap(tid, &t0, &t1, &tl);           // this thread's taps, as a row (for c, G) and as a column
      const double w0 = (double)(1.f - tl), w1 = (double)tl;
      atomicAdd(&s_c[t0], w0); atomicAdd(&s_c[t1], w1);
      atomicAdd(&s_G[t0][t0], w0 * w0); atomicAdd(&s_G[t0][t1], w0 * w1);
      atomicAdd(&s_G[t1][t0], w1 * w0); atomicAdd(&s_G[t1][t1], w1 * w1);
#pragma unroll
      for (int a = 0; a < 8; ++a) s_col[a][tid] = 0.0;
      // column pass: coalesced byte loads (thread = x), weights of row y into its two tap cells
      for (int y = 0; y < VIEW; ++y) {
        int y0, y1; float ly;
        bilin_tap(y, &y0, &y1, &ly);           // warp-uniform
        const double fv = (double)f[y * VIEW + tid] / 255.0;
        sf += fv;
        s_col[y0][tid] += (double)(1.f - ly) * fv;
        s_col[y1][tid] += (double)ly * fv;
      }
#pragma unroll
      for (int a = 0; a < 8; ++a) {
        const double v = s_col[a][tid];
        atomicAdd(&s_F[a][t0], v * w0);
        atomicAdd(&s_F[a][t1], v * w1);
      }
    }
    sf = warp_sum_d(sf);
    if (lane == 0) s_red[warp] = sf;
    __syncthreads();
    if (tid < 64) {                            // T = G h  (rows), then GhG = T G^T (columns)
      const int a = tid >> 3, c2 = tid & 7;
      double t = 0.0;
#pragma unroll
      for (int k = 0; k < 8; ++k) t += s_G[a][k] * (double)s_h[k * 8 + c2];
      s_T[a][c2] = t;
    }
    __syncthreads();
    if (tid < 64) {
      const int a = tid >> 3, c2 = tid & 7;
      double t = 0.0;
#pragma unroll
      for (int k = 0; k < 8; ++k) t += s_T[a][k] * s_G[c2][k];
      s_GhG[a][c2] = t;
    }
    __syncthreads();
    if (tid == 0) {
      double SF = 0.0;
      for (int w = 0; w < 8; ++w) SF += s_red[w];
      double sp = 0.0, spp = 0.0, spf = 0.0;
      for (int a = 0; a < 8; ++a)
        for (int c2 = 0; c2 < 8; ++c2) {
          const double h = (double)s_h[a * 8 + c2];
          sp += h * s_c[a] * s_c[c2];
          spp += h * s_GhG[a][c2];
          spf += h * s_F[a][c2];
        }
      const double m = sp / NPX;
      double var = (spp - NPX * m * m) / (NPX - 1);
      if (var < 0) var = 0;
      s_stat[0] = m; s_stat[1] = sqrt(var); s_stat[2] = SF; s_stat[3] = spf;
    }
    __syncthreads();
    const double m = s_stat[0], sd = s_stat[1], SF = s_stat[2], SPF = s_stat[3];
    if (SF > 0.0 && sd > 0.0) {
      use_nss = true;
      const double half = (nss_r == 0) ? 1.0 : 0.5;
      const double A = SPF - m * SF;
      const double Fe = SF + 0.001;
      double sum_nf = half * A / sd;
      if (nss_r == 1) sum_nf += SF;
      else if (nss_r == -1) sum_nf -= SF;
      nss_term = -(double)nss_w * sum_nf / Fe;
      // per pixel: d/dp = c * [ (f - SF/N)/sd - A (p - m) / ((N-1) sd^3) ]; its upsample adjoint:
      const double c = -(double)nss_w * half / Fe * scale;
      const double k1 = c / sd, k2 = c * A / ((NPX - 1.0) * sd * sd * sd), fm = SF / NPX;
      if (tid < 64) {
        const int a = tid >> 3, c2 = tid & 7;
        const double cc = s_c[a] * s_c[c2];
        s_dh[tid] = (float)(k1 * (s_F[a][c2] - fm * cc) - k2 * (s_GhG[a][c2] - m * cc));
      }
    }
  }
  __syncthreads();
  if (tid < 64) d_h_sali[b * 64 + tid] = s_dh[tid];
  if (tid == 0) {
    const float px = output[b * 4], py = output[b * 4 + 1], pa = output[b * 4 + 2], pp = output[b * 4 + 3];
    const float gx = gt_xy[b * 2], gy = gt_xy[b * 2 + 1];
    const float j = jitter ? jitter[b] : 0.f;
    const float pyj = py + j;
    const float dax = px - gx, day = py - gy, dalt = pa - gt_alt[b], dpr = pp - gt_prog[b];
    const float dang = ang_ref(px, pyj) - ang_ref(gx, gy);
    const float mse = dax * dax + day * day;
    double l = (double)mse + (double)(dang * dang) + (double)(dalt * dalt) + (double)(dpr * dpr);
    if (use_nss) l += nss_term;
    loss_i[b] = l;
    atomicAdd(loss_total, l * scale);
    const float r2 = px * px + pyj * pyj;
    const float k = r2 > 0.f ? (2.f * dang) / (2.f * PI_REF * r2) : 0.f;
    const float sc = (float)scale;
    d_output[b * 4] = sc * (2.f * dax + k * pyj);
    d_output[b * 4 + 1] = sc * (2.f * day - k * px);
    d_output[b * 4 + 2] = sc * 2.f * dalt;
    d_output[b * 4 + 3] = sc * 2.f * dpr;
  }
}

// ------------------------------------------------------- supervision geometry (N3)
// compute_iou (src/xview_et/agent.py:46-78) and teacher_action with student feedback (agent.py:386-507), which the
// reference evaluates per sample with shapely/GEOS on the host.  For the convex quadrilaterals of the simulator
// those calls reduce to: convex hulls (monotone chain), the intersection of two convex polygons
// (Sutherland-Hodgman), shoelace areas, and the point where the segment centre -> goal leaves the view quad.
// One thread per sample, float64.
struct P2 { double x, y; };
__device__ __forceinline__ double cross3(P2 o, P2 a, P2 b) { return (a.x - o.x) * (b.y - o.y) - (a.y - o.y) * (b.x - o.x); }
__device__ double poly_area(const P2* p, int n) {
  double s = 0.0;
  for (int i = 0; i < n; ++i) { const P2 a = p[i], b = p[(i + 1) % n]; s += a.x * b.y - b.x * a.y; }
  return 0.5 * s;
}
// Andrew's monotone chain, counter-clockwise output; n <= 8
__device__ int hull_ccw(const P2* in, int n, P2* out) {
  P2 pts[8];
  for (int i = 0; i < n; ++i) pts[i] = in[i];
  for (int i = 1; i < n; ++i) {                       // insertion sort, lexicographic (x, y)
    const P2 k = pts[i];
    int j = i - 1;
    while (j >= 0 && (pts[j].x > k.x || (pts[j].x == k.x && pts[j].y > k.y))) { pts[j + 1] = pts[j]; --j; }
    pts[j + 1] = k;
  }
  if (n <= 2) { for (int i = 0; i < n; ++i) out[i] = pts[i]; return n; }
  P2 h[18];
  int m = 0;
  for (int i = 0; i < n; ++i) {
    while (m >= 2 && cross3(h[m - 2], h[m - 1], pts[i]) <= 0) --m;
    h[m++] = pts[i];
  }
  const int lo = m + 1;
  for (int i = n - 2; i >= 0; --i) {
    while (m >= lo && cross3(h[m - 2], h[m - 1], pts[i]) <= 0) --m;
    h[m++] = pts[i];
  }
  --m;                                                // the last point repeats the first
  for (int i = 0; i < m; ++i) out[i] = h[i];
  return m;
}
// intersection of two CCW convex polygons (<= 8 vertices each) -> up to 16 vertices
__device__ int clip_convex(const P2* subj, int ns, const P2* clip, int nc, P2* out) {
  P2 a_[16], b_[16];
  P2* cur = a_; P2* nxt = b_;
  int n = ns;
  for (int i = 0; i < ns; ++i) cur[i] = subj[i];
  for (int e = 0; e < nc && n > 0; ++e) {
    const P2 a = clip[e], b = clip[(e + 1) % nc];
    int m = 0;
    for (int j = 0; j < n; ++j) {
      const P2 p = cur[j], q = cur[(j + 1) % n];
      const double sp = (b.x - a.x) * (p.y - a.y) - (b.y - a.y) * (p.x - a.x);
      const double sq = (b.x - a.x) * (q.y - a.y) - (b.y - a.y) * (q.x - a.x);
      if (sp >= 0) nxt[m++] = p;
      if ((sp >= 0) != (sq >= 0)) {
        const double t = sp / (sp - sq);
        nxt[m].x = p.x + t * (q.x - p.x);
        nxt[m].y = p.y + t * (q.y - p.y);
        ++m;
      }
    }
    P2* tmp = cur; cur = nxt; nxt = tmp;
    n = m;
  }
  for (int i = 0; i < n; ++i) out[i] = cur[i];
  return n;
}
__device__ double quad_iou(const P2* a, const P2* b) {
  P2 ha[8], hb[8], inter[16], all[8], hu[8];
  const int na = hull_ccw(a, 4, ha), nb = hull_ccw(b, 4, hb);
  const int ni = clip_convex(ha, na, hb, nb, inter);
  if (ni < 3) return 0.0;
  for (int i = 0; i < 4; ++i) { all[i] = a[i]; all[4 + i] = b[i]; }
  const int nu = hull_ccw(all, 8, hu);
  const double ua = fabs(poly_area(hu, nu));
  return ua == 0.0 ? 0.0 : fabs(poly_area(inter, ni)) / ua;
}

__global__ void teacher_action_kernel(const double* __restrict__ corners, const double* __restrict__ gt, int pmax,
                                      const int32_t* __restrict__ gt_len, const uint8_t* __restrict__ ended, int B,
                                      int teacher_feedback, float* __restrict__ ratio, float* __restrict__ altitude,
                                      float* __restrict__ progress) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  P2 c[4], g[4];
  for (int k = 0; k < 4; ++k) { c[k].x = corners[(i * 4 + k) * 2]; c[k].y = corners[(i * 4 + k) * 2 + 1]; }
  const int n = gt_len[i];
  if (n < 1 || n > pmax) {                       // no ground-truth path: nothing to supervise
    ratio[2 * i] = 0.f; ratio[2 * i + 1] = 0.f; altitude[i] = 0.f; progress[i] = 0.f;
    return;
  }
  const double* gl = gt + ((size_t)i * pmax + (n - 1)) * 8;
  for (int k = 0; k < 4; ++k) { g[k].x = gl[2 * k]; g[k].y = gl[2 * k + 1]; }
  P2 cur;
  cur.x = (((c[0].x + c[1].x) + c[2].x) + c[3].x) / 4.0;
  cur.y = (((c[0].y + c[1].y) + c[2].y) + c[3].y) / 4.0;
  const float prog = (float)quad_iou(c, g);                       // progress[i] = np.float32(iou)
  progress[i] = prog;
  // teacher altitude: the ground-truth step whose centre is closest to the current position (later steps win ties)
  double min_dis = 1000.0;
  int closest = 0;
  for (int j = n - 1; j >= 0; --j) {
    const double* q = gt + ((size_t)i * pmax + j) * 8;
    const double mx = (((q[0] + q[2]) + q[4]) + q[6]) / 4.0 - cur.x, my = (((q[1] + q[3]) + q[5]) + q[7]) / 4.0 - cur.y;
    const double dis = sqrt(mx * mx + my * my);
    if (dis + 0.00001 < min_dis) { min_dis = dis; closest = j; }
  }
  {
    const double* q = gt + ((size_t)i * pmax + closest) * 8;
    const double ex = q[0] - q[2], ey = q[1] - q[3];
    altitude[i] = (float)((sqrt(ex * ex + ey * ey) * 11.13 * 1e4 - 40.0) / (400.0 - 40.0));
  }
  if (ended[i] || prog > 0.5f) { ratio[2 * i] = 0.f; ratio[2 * i + 1] = 0.f; return; }
  // the part of the segment centre -> goal centre inside the view: its end point closest to the goal
  P2 goal;
  goal.x = (((g[0].x + g[1].x) + g[2].x) + g[3].x) / 4.0;
  goal.y = (((g[0].y + g[1].y) + g[2].y) + g[3].y) / 4.0;
  P2 poly[4];
  const bool ccw = poly_area(c, 4) >= 0;
  for (int k = 0; k < 4; ++k) poly[k] = ccw ? c[k] : c[3 - k];
  double xx = 0.0, xy = 0.0;
  bool found = false;
  if (teacher_feedback) {
    // the point of (ground-truth path  intersected with  view) closest to the goal (agent.py:441-466): the end
    // points of the clipped path segments (Cyrus-Beck) are the boundary crossings and the path vertices inside
    double best = 1.0;
    P2 p;
    {
      const double* q0 = gt + (size_t)i * pmax * 8;
      p.x = (((q0[0] + q0[2]) + q0[4]) + q0[6]) / 4.0; p.y = (((q0[1] + q0[3]) + q0[5]) + q0[7]) / 4.0;
    }
    for (int j = 1; j < n; ++j) {
      const double* q1 = gt + ((size_t)i * pmax + j) * 8;
      P2 q;
      q.x = (((q1[0] + q1[2]) + q1[4]) + q1[6]) / 4.0; q.y = (((q1[1] + q1[3]) + q1[5]) + q1[7]) / 4.0;
      double t0 = 0.0, t1 = 1.0;
      bool miss = false;
      const double dx = q.x - p.x, dy = q.y - p.y;
      for (int k = 0; k < 4 && !miss; ++k) {
        const P2 a = poly[k], b = poly[(k + 1) & 3];
        const double ex = b.x - a.x, ey = b.y - a.y;
        const double s0 = ex * (p.y - a.y) - ey * (p.x - a.x);
        const double ds = ex * dy - ey * dx;
        if (ds == 0.0) { if (s0 < 0) miss = true; continue; }
        const double t = -s0 / ds;
        if (ds > 0) t0 = fmax(t0, t); else t1 = fmin(t1, t);
      }
      if (!miss && t0 <= t1) {
        const double tt[2] = {t0, t1};
        for (int e = 0; e < 2; ++e) {
          const double cx = p.x + tt[e] * dx, cy = p.y + tt[e] * dy;
          const double dist = sqrt((cx - goal.x) * (cx - goal.x) + (cy - goal.y) * (cy - goal.y));
          if (dist < best) { best = dist; xx = cx; xy = cy; found = true; }
        }
      }
      p = q;
    }
  }
  if (!found) {
    double t_exit = 1.0;
    for (int k = 0; k < 4; ++k) {
      const P2 a = poly[k], b = poly[(k + 1) & 3];
      const double ex = b.x - a.x, ey = b.y - a.y;
      const double s0 = ex * (cur.y - a.y) - ey * (cur.x - a.x);
      const double s1 = ex * (goal.y - a.y) - ey * (goal.x - a.x);
      if (s1 < 0 && s0 >= 0) t_exit = fmin(t_exit, s0 / (s0 - s1));
    }
    xx = cur.x + t_exit * (goal.x - cur.x);
    xy = cur.y + t_exit * (goal.y - cur.y);
  }
  // local frame of the view (agent.py:481-487): integer-rounded half-edge vectors, 2x2 solve with partial pivoting
  const double b0 = 1e5 * (xx - cur.x), b1 = 1e5 * (xy - cur.y);
  const double ny0 = rint(1e5 * ((c[0].x + c[1].x) / 2 - cur.x)), ny1 = rint(1e5 * ((c[0].y + c[1].y) / 2 - cur.y));
  const double nx0 = rint(1e5 * ((c[1].x + c[2].x) / 2 - cur.x)), nx1 = rint(1e5 * ((c[1].y + c[2].y) / 2 - cur.y));
  double a00 = nx0, a01 = ny0, a10 = nx1, a11 = ny1, r0b = b0, r1b = b1;
  if (fabs(a10) > fabs(a00)) { double t;  t = a00; a00 = a10; a10 = t;  t = a01; a01 = a11; a11 = t;  t = r0b; r0b = r1b; r1b = t; }
  const double l = a10 / a00;
  const double u11 = a11 - l * a01;
  const double r1 = (r1b - l * r0b) / u11;
  const double r0 = (r0b - a01 * r1) / a00;
  const double m = fmax(fmax(fabs(r0), fabs(r1)), 1.0);
  ratio[2 * i] = (float)(r0 / m);
  ratio[2 * i + 1] = (float)(r1 / m);
}

// Pixel (y, x) of the 8x8 -> 224x224 bilinear upsample of h [64].  Not inlined: upsample_kernel and
// saliency_metrics_kernel run the same machine code, so their pixel values are bit-identical.
__device__ __noinline__ float upsample_px(const float* h, int y, int x) {
  int y0, y1, x0, x1; float ly, lx;
  bilin_tap(y, &y0, &y1, &ly);
  bilin_tap(x, &x0, &x1, &lx);
  return (1.f - ly) * ((1.f - lx) * h[y0 * 8 + x0] + lx * h[y0 * 8 + x1]) +
         ly * ((1.f - lx) * h[y1 * 8 + x0] + lx * h[y1 * 8 + x1]);
}

// 8x8 -> 224x224 bilinear upsample (pred_saliency of the reference API)
__global__ void upsample_kernel(const float* __restrict__ h_sali, int B, float* __restrict__ pred) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= (long long)B * NPX) return;
  const int b = (int)(i / NPX), r = (int)(i % NPX), y = r / VIEW, x = r - y * VIEW;
  pred[i] = upsample_px(h_sali + b * 64, y, x);
}

// Sum of one double over the 256 threads of a CTA in a fixed order (xor tree per warp, then the 8 warps in order);
// every thread gets the result.  `red` holds 8 doubles.
__device__ __forceinline__ double block_sum_256(double v, double* red) {
  v = warp_sum_d(v);
  __syncthreads();                               // red may still be read from the previous call
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
#pragma unroll
  for (int w = 0; w < 8; ++w) t += red[w];
  return t;
}

// Human-attention validation scores of one row per CTA (xview_et/agent.py:683-693 per sample): sal = the upsample of
// h_sali[row], gt = att[row] / 255, p = clip(sal, 0, 1).  Two passes over the 224x224 pixels in float64: sums of sal,
// gt, p, p*gt, then the centred sums of (sal - mean)^2 and (sal - mean)*gt (torch.std's unbiased variance and the
// NSS numerator without the cancellation of a one-pass formula).
__global__ void __launch_bounds__(256) saliency_metrics_kernel(const float* __restrict__ h_sali,
                                                               const uint8_t* __restrict__ att, int nss_r,
                                                               double* __restrict__ out) {
  __shared__ float s_h[64];
  __shared__ double s_red[8];
  const int row = blockIdx.x, tid = threadIdx.x;
  if (tid < 64) s_h[tid] = h_sali[(size_t)row * 64 + tid];
  __syncthreads();
  const uint8_t* f = att + (size_t)row * NPX;
  double ss = 0.0, sg = 0.0, sp = 0.0, spg = 0.0;
  for (int i = tid; i < NPX; i += 256) {
    const int y = i / VIEW, x = i - y * VIEW;
    const float s = upsample_px(s_h, y, x);
    const double g = (double)f[i] / 255.0;
    const double p = (double)fminf(fmaxf(s, 0.f), 1.f);
    ss += (double)s; sg += g; sp += p; spg += p * g;
  }
  ss = block_sum_256(ss, s_red);
  sg = block_sum_256(sg, s_red);
  sp = block_sum_256(sp, s_red);
  spg = block_sum_256(spg, s_red);
  const double m = ss / NPX;
  double dd = 0.0, dg = 0.0;
  for (int i = tid; i < NPX; i += 256) {
    const int y = i / VIEW, x = i - y * VIEW;
    const double d = (double)upsample_px(s_h, y, x) - m;
    dd += d * d; dg += d * ((double)f[i] / 255.0);
  }
  dd = block_sum_256(dd, s_red);
  dg = block_sum_256(dg, s_red);
  if (tid == 0) {
    const double sd = sqrt(dd / (NPX - 1));
    // sum_px n_sal * gt with n_sal = (sal - m) / sd, then nss_r's affine map (n/2 + 1 or n/2 - 1)
    double sns = dg / sd;
    if (nss_r == 1) sns = sns / 2 + sg;
    else if (nss_r == -1) sns = sns / 2 - sg;
    double* o = out + (size_t)row * 4;
    o[0] = sp != 0.0 ? spg / sp : 0.0;
    o[1] = sg > 0.0 ? spg / sg : 0.0;
    o[2] = -(sns / (sg + 0.001));
    o[3] = sg;
  }
}

// adjoint of the upsample: d_h_sali[b][64] = sum_pixels w * d_pred.  One CTA per sample.
__global__ void __launch_bounds__(256) upsample_bwd_kernel(const float* __restrict__ d_pred,
                                                           float* __restrict__ d_h_sali) {
  __shared__ float s_dh[64];
  const int b = blockIdx.x, tid = threadIdx.x;
  if (tid < 64) s_dh[tid] = 0.f;
  __syncthreads();
  const float* g = d_pred + (size_t)b * NPX;
  for (int i = tid; i < NPX; i += 256) {
    const int y = i / VIEW, x = i - y * VIEW;
    int y0, y1, x0, x1; float ly, lx;
    bilin_tap(y, &y0, &y1, &ly);
    bilin_tap(x, &x0, &x1, &lx);
    const float v = g[i];
    atomicAdd(&s_dh[y0 * 8 + x0], v * (1.f - ly) * (1.f - lx));
    atomicAdd(&s_dh[y0 * 8 + x1], v * (1.f - ly) * lx);
    atomicAdd(&s_dh[y1 * 8 + x0], v * ly * (1.f - lx));
    atomicAdd(&s_dh[y1 * 8 + x1], v * ly * lx);
  }
  __syncthreads();
  if (tid < 64) d_h_sali[b * 64 + tid] = s_dh[tid];
}

// agent.py:637-653,738,745-752: normalise, clamp, discretise.  Integers are bit-exact with the
// host code: float32 element arithmetic, then float64 for the literal-constant expressions.
__global__ void postprocess_kernel(const float* __restrict__ output, const double* __restrict__ edge_len, int B,
                                   float stop_threshold, int* __restrict__ angle_deg, double* __restrict__ dist,
                                   int* __restrict__ altitude_m, uint8_t* __restrict__ stop,
                                   float* __restrict__ xy_norm) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  float x = output[i * 4], y = output[i * 4 + 1];
  const float m = fmaxf(fmaxf(fabsf(x), fabsf(y)), 1.f);
  x = __fdiv_rn(x, m);
  y = __fdiv_rn(y, m);
  const float a = fminf(1.f, fmaxf(0.f, output[i * 4 + 2]));
  const float p = fminf(1.f, fmaxf(0.f, output[i * 4 + 3]));
  // np.arctan2 on float32 scalars -> float32; the python-float constants promote to float64
  const double at = (double)atan2f(x, y);
  double a_dir = (at / 3.14159 + 2.0) / 2.0;
  a_dir = a_dir - floor(a_dir);
  angle_deg[i] = __double2int_rn(a_dir * 360.0);
  // np.linalg.norm of a float32 pair -> float32
  const float nrm = sqrtf(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y)));
  dist[i] = (double)nrm * (edge_len[i] / 2.0);
  altitude_m[i] = __double2int_rn((double)a * 360.0) + 40;
  stop[i] = p > stop_threshold ? 1 : 0;
  if (xy_norm) { xy_norm[i * 2] = x; xy_norm[i * 2 + 1] = y; }
}

// ----------------------------------------------------------------- optimiser
__global__ void __launch_bounds__(256) sumsq_kernel(const float* __restrict__ g, long long n, double* __restrict__ out) {
  double a = 0.0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float v = g[i];
    a += (double)v * v;
  }
  a = warp_sum_d(a);
  __shared__ double sm[8];
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = a;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0;
    for (int w = 0; w < 8; ++w) t += sm[w];
    atomicAdd(out, t);
  }
}

// torch.optim.AdamW step over a flat arena; grads are first scaled by
// min(1, max_norm / (sqrt(*sumsq) + 1e-6)) when sumsq != NULL (clip_grad_norm_).
__global__ void __launch_bounds__(256) adamw_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                    float* __restrict__ m, float* __restrict__ v, long long n, float lr,
                                                    float beta1, float beta2, float eps, float wd, float bias1,
                                                    float bias2_sqrt, const double* __restrict__ sumsq, float max_norm,
                                                    float grad_scale) {
  float coef = grad_scale;
  if (sumsq) {
    const float nrm = (float)sqrt(*sumsq) * grad_scale;
    const float c = max_norm / (nrm + 1e-6f);
    if (c < 1.f) coef *= c;
  }
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float gi = g[i] * coef;
    float pi = p[i] * (1.f - lr * wd);
    const float mi = beta1 * m[i] + (1.f - beta1) * gi;
    const float vi = beta2 * v[i] + (1.f - beta2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bias2_sqrt + eps;
    pi -= (lr / bias1) * (mi / denom);
    p[i] = pi;
  }
}

}  // namespace

extern "C" int avdn_teacher_action(const double* corners, const double* gt_path_corners, int pmax, const int32_t* gt_len,
                                   const uint8_t* ended, int B, int teacher_feedback, float* next_pos_ratio,
                                   float* altitude, float* progress, avdn_stream_t stream) {
  AVDN_REQUIRE(corners && gt_path_corners && gt_len && ended && next_pos_ratio && altitude && progress && pmax >= 1,
               "avdn_teacher_action: bad argument");
  if (B <= 0) return AVDN_OK;
  teacher_action_kernel<<<(B + 63) / 64, 64, 0, avdn::to_cuda(stream)>>>(corners, gt_path_corners, pmax, gt_len, ended, B,
                                                                       teacher_feedback, next_pos_ratio, altitude,
                                                                       progress);
  return avdn::check_launch("avdn_teacher_action");
}

extern "C" int avdn_loss(const float* output, const float* h_sali, const float* gt_xy, const float* gt_alt,
                         const float* gt_prog, const uint8_t* att, const float* jitter, int B, float nss_w, int nss_r,
                         double scale, double* loss_total, double* loss_i, float* d_output, float* d_h_sali,
                         avdn_stream_t stream) {
  AVDN_REQUIRE(output && h_sali && gt_xy && gt_alt && gt_prog && loss_total && loss_i && d_output && d_h_sali,
               "avdn_loss: null pointer");
  AVDN_REQUIRE(nss_r >= -1 && nss_r <= 1, "avdn_loss: nss_r must be -1, 0 or 1");
  if (B == 0) return AVDN_OK;
  loss_kernel<<<B, 256, 0, avdn::to_cuda(stream)>>>(output, h_sali, gt_xy, gt_alt, gt_prog, att, jitter, nss_w, nss_r,
                                                  scale, loss_total, loss_i, d_output, d_h_sali);
  return avdn::check_launch("avdn_loss");
}

extern "C" int avdn_upsample_saliency(const float* h_sali, int B, float* pred, avdn_stream_t stream) {
  AVDN_REQUIRE(h_sali && pred, "avdn_upsample_saliency: null pointer");
  if (B == 0) return AVDN_OK;
  const long long n = (long long)B * NPX;
  upsample_kernel<<<(unsigned)((n + 255) / 256), 256, 0, avdn::to_cuda(stream)>>>(h_sali, B, pred);
  return avdn::check_launch("avdn_upsample_saliency");
}

extern "C" int avdn_saliency_metrics(const float* h_sali, const uint8_t* att, int N, int nss_r, double* out,
                                     avdn_stream_t stream) {
  AVDN_REQUIRE(h_sali && att && out, "avdn_saliency_metrics: null pointer");
  AVDN_REQUIRE(N >= 0, "avdn_saliency_metrics: N must be >= 0");
  AVDN_REQUIRE(nss_r >= -1 && nss_r <= 1, "avdn_saliency_metrics: nss_r must be -1, 0 or 1");
  if (N == 0) return AVDN_OK;
  saliency_metrics_kernel<<<N, 256, 0, avdn::to_cuda(stream)>>>(h_sali, att, nss_r, out);
  return avdn::check_launch("avdn_saliency_metrics");
}

extern "C" int avdn_upsample_saliency_bwd(const float* d_pred, int B, float* d_h_sali, avdn_stream_t stream) {
  AVDN_REQUIRE(d_pred && d_h_sali, "avdn_upsample_saliency_bwd: null pointer");
  if (B == 0) return AVDN_OK;
  upsample_bwd_kernel<<<B, 256, 0, avdn::to_cuda(stream)>>>(d_pred, d_h_sali);
  return avdn::check_launch("avdn_upsample_saliency_bwd");
}

extern "C" int avdn_postprocess_waypoints(const float* output, const double* edge_len, int B, float stop_threshold,
                                          int* angle_deg, double* dist, int* altitude_m, uint8_t* stop,
                                          float* xy_norm, avdn_stream_t stream) {
  AVDN_REQUIRE(output && edge_len && angle_deg && dist && altitude_m && stop, "avdn_postprocess_waypoints: null pointer");
  if (B == 0) return AVDN_OK;
  postprocess_kernel<<<(B + 127) / 128, 128, 0, avdn::to_cuda(stream)>>>(output, edge_len, B, stop_threshold,
                                                                        angle_deg, dist, altitude_m, stop, xy_norm);
  return avdn::check_launch("avdn_postprocess_waypoints");
}

extern "C" int avdn_sumsq(const float* g, long long n, double* out, avdn_stream_t stream) {
  AVDN_REQUIRE(g && out && n >= 0, "avdn_sumsq: bad argument");
  if (n == 0) return AVDN_OK;
  long long blocks = (n + 255) / 256;
  const long long cap = (long long)avdn::sm_count() * 8;
  if (blocks > cap) blocks = cap;
  sumsq_kernel<<<(unsigned)blocks, 256, 0, avdn::to_cuda(stream)>>>(g, n, out);
  return avdn::check_launch("avdn_sumsq");
}

extern "C" int avdn_adamw(float* p, const float* g, float* m, float* v, long long n, float lr, float beta1,
                          float beta2, float eps, float wd, int step, const double* sumsq, float max_norm,
                          float grad_scale, avdn_stream_t stream) {
  AVDN_REQUIRE(p && g && m && v && n >= 0 && step >= 1, "avdn_adamw: bad argument");
  if (n == 0) return AVDN_OK;
  const float bias1 = 1.f - powf(beta1, (float)step);
  const float bias2_sqrt = sqrtf(1.f - powf(beta2, (float)step));
  long long blocks = (n + 255) / 256;
  const long long cap = (long long)avdn::sm_count() * 8;
  if (blocks > cap) blocks = cap;
  adamw_kernel<<<(unsigned)blocks, 256, 0, avdn::to_cuda(stream)>>>(p, g, m, v, n, lr, beta1, beta2, eps, wd, bias1,
                                                                  bias2_sqrt, sumsq, max_norm, grad_scale);
  return avdn::check_launch("avdn_adamw");
}
