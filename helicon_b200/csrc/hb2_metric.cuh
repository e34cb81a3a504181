// 2-D score metrics of a grid search (hb2_batch_score_metric): SSIM, MS-SSIM and mutual information of every
// candidate's reprojection against the reference region, the restatements of imageprep.py / _metric_2d run on the device.
//
// Images are float64 [H = L2 rows][W = D2 columns]; image slot nc of every buffer is the reference region (it is the same
// for all candidates), slots 0..nc-1 the candidates' pred_2d.  All candidates are scored in one launch per stage, grid
// (tiles, images).  Per-CTA partials are combined in a fixed order, so a candidate's value does not depend on its batch.
//
// Formulas (scipy 1.x, numpy 2.x; checked against scipy by tests/test_score_metric_cpu.py):
//  * uniform_filter(size 7, mode "reflect"): only the map cropped by 3 on each side is averaged, and its 7 x 7 windows
//    never leave the image, so no boundary rule is needed.  Means = (column sum / 7), then (row sum / 7).
//  * _rescale(img, 0.5, order=1), per axis with n = input side:
//      out = round_half_even(n / 2);  z = n / out (float64);  sigma = max(0, (z - 1) / 2);  r = int(4 sigma + 0.5)
//      gaussian weights g[k] = exp(-0.5 / sigma^2 * k^2) / sum_{|k|<=r} (k = -r..r), applied along axis 0 then axis 1 as
//      correlate1d does for symmetric weights: o[i] = in[i] g[0] + sum_{k=r..1} (in[i-k] + in[i+k]) g[k], with the
//      half-sample reflection in[-1-i] = in[i], in[n+i] = in[n-1-i];
//      zoom(order 1, grid_mode): for output index o, c = ((o + 0.5) z) - 0.5, i0 = floor(c), t = c - i0,
//      w0 = 1 - t, w1 = 1 - w0; value = sum over (a, b) in C order of ((in[i0+a][j0+b] wy[a]) wx[b]).  For n >= 8,
//      z > 1 keeps 0 <= i0 and i0 + 1 <= n - 1, so no boundary rule is needed; then clip to the input's [min, max].
//  * histogramdd(bins=64) of float32 samples: edges are float32, e[i] = fl(fl(i * step) + lo), step = fl(hi - lo) / 64,
//    e[64] = hi, with (lo, hi) = (min, max), widened to (min - 0.5, max + 0.5) in float32 when min == max; a sample's
//    bin is (number of edges <= v) - 1, and v == e[64] goes to bin 63.  density=True divides every count by the float32
//    edge widths dx[i] dy[j] (and then by the total), which the entropies keep.
#pragma once

#include <cassert>

#include "hb2_kernels.cuh"

#define MET_T 16                     // SSIM output tile (MET_T x MET_T outputs per CTA)
#define MET_IN (MET_T + 6)           // input tile with the 3-pixel halo
#define MET_GMAX 4                   // largest Gaussian radius of a 0.5 rescale of a side >= 8 is 3
#define MET_HIST_PIX 4096            // pixels per CTA of the joint histogram
#define MET_MAX_SCALES 5

struct MetCand {
  int active;       // still scored at the current scale (0 after a zero data range)
  int nv;           // MS-SSIM scales reached
  double vals[MET_MAX_SCALES];
  double ssim;      // SSIM at scale 0
  double mi;
  double c1, c2;    // scale-0 constants (float32 arithmetic of the host, see hb2_batch_score_metric)
};

struct MetGauss {
  double w[MET_GMAX + 1];  // w[0] centre, w[k] = weight of offset +-k
  int r;
};

__device__ __forceinline__ double met_block_sum(double v, double* sh) {
  // fixed-order tree over HB2_BLOCK threads; result in thread 0
  sh[threadIdx.x] = v;
  __syncthreads();
  for (int s = HB2_BLOCK / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) sh[threadIdx.x] = __dadd_rn(sh[threadIdx.x], sh[threadIdx.x + s]);
    __syncthreads();
  }
  return sh[0];
}

// pred_2d of every candidate: the last writer of each pixel (or 0), clipped at 0 when clip
__global__ void __launch_bounds__(HB2_BLOCK) k_met_gather(const BD B, const int* __restrict__ rows, int HW, int clip,
                                                          double* __restrict__ img, long long stride) {
  const int c = blockIdx.y;
  const int p = blockIdx.x * HB2_BLOCK + threadIdx.x;
  if (p >= HW) return;
  const int r = rows[(size_t)c * HW + p];
  assert(r < B.cand_mdata[c]);
  float v = 0.f;
  if (r >= 0) {
    v = B.u[B.cand_uoff[c] + r];
    if (clip) v = fmaxf(v, 0.f);
  }
  img[(size_t)c * stride + p] = (double)v;
}

// reference: ref_2d[k][j] = pix[j][k] (the problem's crop, [D2][L2])
__global__ void __launch_bounds__(HB2_BLOCK) k_met_ref(const float* __restrict__ pix, int H, int W, double* __restrict__ img) {
  const int p = blockIdx.x * HB2_BLOCK + threadIdx.x;
  if (p >= H * W) return;
  const int k = p / W, j = p % W;
  img[p] = (double)pix[(size_t)j * H + k];
}

// min / max of every active image at the current scale (slot nc: the reference)
__global__ void __launch_bounds__(HB2_BLOCK) k_met_range(const double* __restrict__ img, long long stride, int HW, int nc,
                                                         const MetCand* __restrict__ st, double2* __restrict__ rng) {
  const int c = blockIdx.x;
  if (c < nc && !st[c].active) return;
  const double* a = img + (size_t)c * stride;
  double lo = a[0], hi = a[0];
  for (int p = threadIdx.x; p < HW; p += HB2_BLOCK) {
    lo = fmin(lo, a[p]);
    hi = fmax(hi, a[p]);
  }
  __shared__ double sl[HB2_BLOCK], sh[HB2_BLOCK];
  sl[threadIdx.x] = lo; sh[threadIdx.x] = hi;
  __syncthreads();
  for (int s = HB2_BLOCK / 2; s > 0; s >>= 1) {
    if (threadIdx.x < s) {
      sl[threadIdx.x] = fmin(sl[threadIdx.x], sl[threadIdx.x + s]);
      sh[threadIdx.x] = fmax(sh[threadIdx.x], sh[threadIdx.x + s]);
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) rng[c] = make_double2(sl[0], sh[0]);
}

// after a rescale: a candidate whose data range (float64, both images) is 0 stops (ms_ssim_score's break)
__global__ void k_met_check(MetCand* st, const double2* __restrict__ rng, int nc) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= nc || !st[c].active) return;
  const double R = fmax(rng[c].y - rng[c].x, rng[nc].y - rng[nc].x);
  if (R == 0.0) st[c].active = 0;
}

// SSIM map of one 16 x 16 tile of the cropped region + its partial sum; grid (tiles x, tiles y, nc)
__global__ void __launch_bounds__(HB2_BLOCK) k_met_ssim(const double* __restrict__ img, long long stride, int H, int W,
                                                        int scale, int nc, const MetCand* __restrict__ st,
                                                        const double2* __restrict__ rng, double* __restrict__ part) {
  const int c = blockIdx.z;
  if (!st[c].active) return;
  __shared__ double sa[MET_IN][MET_IN], sb[MET_IN][MET_IN];
  __shared__ double sv[5][MET_T][MET_IN];
  __shared__ double red[HB2_BLOCK];
  const double* a = img + (size_t)c * stride;
  const double* b = img + (size_t)nc * stride;
  const int y0 = blockIdx.y * MET_T, x0 = blockIdx.x * MET_T;
  for (int i = threadIdx.x; i < MET_IN * MET_IN; i += HB2_BLOCK) {
    const int ly = i / MET_IN, lx = i % MET_IN, y = y0 + ly, x = x0 + lx;
    const bool in = y < H && x < W;
    sa[ly][lx] = in ? a[(size_t)y * W + x] : 0.0;
    sb[ly][lx] = in ? b[(size_t)y * W + x] : 0.0;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < MET_T * MET_IN; i += HB2_BLOCK) {  // axis 0: means over 7 rows
    const int ly = i / MET_IN, lx = i % MET_IN;
    double mx = 0, my = 0, mxx = 0, myy = 0, mxy = 0;
#pragma unroll
    for (int k = 0; k < 7; ++k) {
      const double x = sa[ly + k][lx], y = sb[ly + k][lx];
      mx += x; my += y; mxx += x * x; myy += y * y; mxy += x * y;
    }
    sv[0][ly][lx] = mx / 7.0; sv[1][ly][lx] = my / 7.0; sv[2][ly][lx] = mxx / 7.0;
    sv[3][ly][lx] = myy / 7.0; sv[4][ly][lx] = mxy / 7.0;
  }
  __syncthreads();
  double C1, C2;
  if (scale == 0) {
    C1 = st[c].c1; C2 = st[c].c2;
  } else {
    const double R = fmax(rng[c].y - rng[c].x, rng[nc].y - rng[nc].x);
    C1 = (0.01 * R) * (0.01 * R); C2 = (0.03 * R) * (0.03 * R);
  }
  const int ly = threadIdx.x / MET_T, lx = threadIdx.x % MET_T;
  const int y = y0 + ly + 3, x = x0 + lx + 3;
  double S = 0.0;
  if (y < H - 3 && x < W - 3) {
    double m[5];
#pragma unroll
    for (int q = 0; q < 5; ++q) {
      double s = 0;
#pragma unroll
      for (int k = 0; k < 7; ++k) s += sv[q][ly][lx + k];
      m[q] = s / 7.0;
    }
    const double cov_norm = 49.0 / 48.0;
    const double ux = m[0], uy = m[1];
    const double vx = cov_norm * (m[2] - ux * ux), vy = cov_norm * (m[3] - uy * uy), vxy = cov_norm * (m[4] - ux * uy);
    S = ((2 * ux * uy + C1) * (2 * vxy + C2)) / ((ux * ux + uy * uy + C1) * (vx + vy + C2));
  }
  const double t = met_block_sum(S, red);
  if (threadIdx.x == 0) part[(size_t)c * gridDim.x * gridDim.y + blockIdx.y * gridDim.x + blockIdx.x] = t;
}

// mean of the cropped SSIM map from the partials (fixed order); scale 0 keeps it as the SSIM score, ms_take appends
// max(mean, 0) to the MS-SSIM scales
__global__ void __launch_bounds__(HB2_BLOCK) k_met_ssim_fin(const double* __restrict__ part, int ntiles, double count,
                                                            int scale, int ms_take, MetCand* st) {
  const int c = blockIdx.x;
  if (!st[c].active) return;
  __shared__ double red[HB2_BLOCK];
  double s = 0.0;
  for (int i = threadIdx.x; i < ntiles; i += HB2_BLOCK) s += part[(size_t)c * ntiles + i];
  const double t = met_block_sum(s, red);
  if (threadIdx.x == 0) {
    const double mean = t / count;
    if (scale == 0) st[c].ssim = mean;
    if (ms_take) st[c].vals[st[c].nv++] = fmax(mean, 0.0);
  }
}

// Gaussian pre-filter of the rescale along one axis (correlate1d order, reflect); grid (tiles, nc + 1)
template <int AXIS>
__global__ void __launch_bounds__(HB2_BLOCK) k_met_gauss(const double* __restrict__ in, long long in_stride,
                                                         double* __restrict__ out, long long out_stride, int H, int W,
                                                         const MetGauss g, int nc, const MetCand* __restrict__ st) {
  const int c = blockIdx.y;
  if (c < nc && !st[c].active) return;
  const int p = blockIdx.x * HB2_BLOCK + threadIdx.x;
  if (p >= H * W) return;
  const double* a = in + (size_t)c * in_stride;
  const int y = p / W, x = p % W;
  const int n = AXIS == 0 ? H : W, i = AXIS == 0 ? y : x;
  auto at = [&](int k) {
    k = k < 0 ? -k - 1 : (k >= n ? 2 * n - k - 1 : k);
    return AXIS == 0 ? a[(size_t)k * W + x] : a[(size_t)y * W + k];
  };
  double o = __dmul_rn(at(i), g.w[0]);
  for (int k = g.r; k >= 1; --k) o = __dadd_rn(o, __dmul_rn(__dadd_rn(at(i - k), at(i + k)), g.w[k]));
  out[(size_t)c * out_stride + p] = o;
}

// linear zoom (grid_mode) of the filtered image to (Ho, Wo), clipped to the unfiltered input's [min, max]
__global__ void __launch_bounds__(HB2_BLOCK) k_met_zoom(const double* __restrict__ in, long long in_stride, int H, int W,
                                                        double* __restrict__ out, long long out_stride, int Ho, int Wo,
                                                        double zy, double zx, int nc, const MetCand* __restrict__ st,
                                                        const double2* __restrict__ rng) {
  const int c = blockIdx.y;
  if (c < nc && !st[c].active) return;
  const int p = blockIdx.x * HB2_BLOCK + threadIdx.x;
  if (p >= Ho * Wo) return;
  const int oy = p / Wo, ox = p % Wo;
  const double cy = __dadd_rn(__dmul_rn(__dadd_rn((double)oy, 0.5), zy), -0.5);
  const double cx = __dadd_rn(__dmul_rn(__dadd_rn((double)ox, 0.5), zx), -0.5);
  const double fy = floor(cy), fx = floor(cx);
  const int iy = (int)fy, ix = (int)fx;
  assert(iy >= 0 && iy + 1 < H && ix >= 0 && ix + 1 < W);
  double wy[2], wx[2];
  wy[0] = 1.0 - (cy - fy); wy[1] = 1.0 - wy[0];
  wx[0] = 1.0 - (cx - fx); wx[1] = 1.0 - wx[0];
  const double* a = in + (size_t)c * in_stride;
  double t = 0.0;
#pragma unroll
  for (int q = 0; q < 2; ++q)
#pragma unroll
    for (int r = 0; r < 2; ++r) t = __dadd_rn(t, __dmul_rn(__dmul_rn(a[(size_t)(iy + q) * W + ix + r], wy[q]), wx[r]));
  t = fmin(fmax(t, rng[c].x), rng[c].y);
  out[(size_t)c * out_stride + p] = t;
}

__device__ __forceinline__ float met_edge(int i, double2 r) {
  // edge i of np.linspace(lo, hi, 65) in float32 as histogramdd computes it (see the header)
  float lo = (float)r.x, hi = (float)r.y;
  if (lo == hi) { lo = __fsub_rn(lo, 0.5f); hi = __fadd_rn(hi, 0.5f); }
  const float step = __fdiv_rn(__fsub_rn(hi, lo), 64.0f);
  return i == 64 ? hi : __fadd_rn(__fmul_rn((float)i, step), lo);
}

// edges of the candidate (ex) and of the reference (ey)
__device__ __forceinline__ void met_edges(const double2* rng, int c, int nc, float* ex, float* ey) {
  for (int i = threadIdx.x; i < 130; i += blockDim.x) {
    if (i < 65) ex[i] = met_edge(i, rng[c]);
    else ey[i - 65] = met_edge(i - 65, rng[nc]);
  }
}

__device__ __forceinline__ int met_bin(float v, const float* e) {
  if (v == e[64]) return 63;
  int lo = 0, hi = 65;  // first edge > v (searchsorted right), minus 1
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (e[mid] <= v) lo = mid + 1; else hi = mid;
  }
  return lo - 1;
}

// 64 x 64 joint histogram of (pred, ref) at scale 0: integer counts in shared memory, then into the candidate's
// global histogram (integer atomics: the counts do not depend on the order); grid (tiles, nc)
__global__ void __launch_bounds__(HB2_BLOCK) k_met_hist(const double* __restrict__ img, long long stride, int HW, int nc,
                                                        const double2* __restrict__ rng, int* __restrict__ hist) {
  const int c = blockIdx.y;
  __shared__ int h[64 * 64];
  __shared__ float ex[65], ey[65];
  for (int i = threadIdx.x; i < 64 * 64; i += HB2_BLOCK) h[i] = 0;
  met_edges(rng, c, nc, ex, ey);
  __syncthreads();
  const double* a = img + (size_t)c * stride;
  const double* b = img + (size_t)nc * stride;
  const int p0 = blockIdx.x * MET_HIST_PIX, p1 = min(HW, p0 + MET_HIST_PIX);
  for (int p = p0 + threadIdx.x; p < p1; p += HB2_BLOCK) {
    const int bx = met_bin((float)a[p], ex), by = met_bin((float)b[p], ey);
    atomicAdd(&h[bx * 64 + by], 1);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 64 * 64; i += HB2_BLOCK)
    if (h[i]) atomicAdd(&hist[(size_t)c * 4096 + i], h[i]);
}

// (H(X) + H(Y)) / H(X, Y) - 1 of the density histogram; one CTA per candidate, fixed-order sums
__global__ void __launch_bounds__(HB2_BLOCK) k_met_mi(const int* __restrict__ hist, int nc, const double2* __restrict__ rng,
                                                      MetCand* st) {
  const int c = blockIdx.x;
  __shared__ float ex[65], ey[65];
  __shared__ double hd[64 * 64];
  __shared__ double red[HB2_BLOCK];
  __shared__ double marg[2][64];
  met_edges(rng, c, nc, ex, ey);
  __syncthreads();
  double tot = 0.0;
  for (int q = threadIdx.x; q < 4096; q += HB2_BLOCK) {
    const int i = q / 64, j = q % 64;
    const double dx = (double)__fsub_rn(ex[i + 1], ex[i]), dy = (double)__fsub_rn(ey[j + 1], ey[j]);
    const double v = ((double)hist[(size_t)c * 4096 + q] / dx) / dy;
    hd[q] = v;
    tot += v;
  }
  const double T = met_block_sum(tot, red);
  __syncthreads();
  if (threadIdx.x < 128) {  // marginals: sums over the other index
    const int s = threadIdx.x / 64, k = threadIdx.x % 64;
    double m = 0.0;
    for (int l = 0; l < 64; ++l) m += s == 0 ? hd[l * 64 + k] : hd[k * 64 + l];
    marg[s][k] = m;
  }
  double hj = 0.0;
  for (int q = threadIdx.x; q < 4096; q += HB2_BLOCK) {
    const double p = hd[q] / T;
    if (p > 0) hj -= p * log(p);
  }
  __syncthreads();
  const double Hxy = met_block_sum(hj, red);
  __syncthreads();
  if (threadIdx.x == 0) {
    double hm[2];
    for (int s = 0; s < 2; ++s) {
      double ms = 0.0, e = 0.0;
      for (int k = 0; k < 64; ++k) ms += marg[s][k];
      for (int k = 0; k < 64; ++k) {
        const double p = marg[s][k] / ms;
        if (p > 0) e -= p * log(p);
      }
      hm[s] = e;
    }
    // Python raises ZeroDivisionError for H(X, Y) = 0 and the host metric returns 0.0
    st[c].mi = Hxy == 0.0 ? 0.0 : (hm[0] + hm[1]) / Hxy - 1.0;
  }
}

// the metric's value into d_score (float32, as res["score"] stores it) and, when parts, [cosine, ssim, ms_ssim, mi]
__global__ void k_met_final(const MetCand* __restrict__ st, int nc, int metric, const float* __restrict__ cos,
                            float* __restrict__ score, double* __restrict__ parts) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= nc) return;
  const MetCand& S = st[c];
  const double cosv = (double)cos[c];
  const double wall[MET_MAX_SCALES] = {0.0448, 0.2856, 0.3001, 0.2363, 0.1333};
  double ms = 0.0;
  if (S.nv > 0) {
    double wsum = 0.0;
    for (int i = 0; i < S.nv; ++i) wsum += wall[i];
    ms = 1.0;
    for (int i = 0; i < S.nv; ++i) ms *= pow(S.vals[i], wall[i] / wsum);
  }
  const double v[4] = {cosv, S.ssim, ms, S.mi};
  const double comp = (((v[0] + v[1]) + v[2]) + v[3]) / 4.0;
  if (parts)
    for (int q = 0; q < 4; ++q) parts[(size_t)c * 4 + q] = v[q];
  score[c] = (float)(metric == HB2_METRIC_SSIM ? v[1] : metric == HB2_METRIC_MS_SSIM ? v[2]
                     : metric == HB2_METRIC_MI ? v[3] : comp);
}
