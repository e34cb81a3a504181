// Bounded branch of the solve: scipy.optimize.lsq_linear(method='trf', lsq_solver='lsmr')
// as the reference calls it (SLR:246-270): reflective trust-region iterations in
// float64 (scipy/optimize/_lsq/trf_linear.py:147-249, common.py) with an inner
// float64 LSMR on [A D; diag(sqrt(diag_h))].  Batched: every kernel covers all
// candidates and consults per-candidate activity flags; data-dependent decisions
// are taken by one-thread-per-candidate scalar kernels.
#pragma once
#include "hb2_kernels.cuh"

#define TRF_NRED 8  // reduction slots per CTA
#define TRF_EPT 16  // elements per thread of the element-wise passes
#define TRF_SPAN (HB2_BLOCK * TRF_EPT)

struct Lsmr64 {  // lsmr.py:197-480, all float64
  double alpha, beta, normb;
  double zetabar, alphabar, rho, rhobar, cbar, sbar;
  double betadd, betad, rhodold, tautildeold, thetatilde, zeta, d;
  double normA2, maxrbar, minrbar, normA, normr, normar, normx, condA, rhotemp;
  double cf_hbar, cf_x, cf_h, inv_alpha, inv_beta;
  int minrbar_inf, itn, istop, active, skip_adj;
};

struct TrfState {
  double lb, ub, tol;
  double cost, g_norm, theta, lsmr_tol, p_dot_g, p_stride, r_stride_u, r_stride_l, r_stride, ag_stride;
  double cost_change;
  double coef_p, coef_r, coef_ag;  // step = D*(coef_p*PH + coef_r*RH + coef_ag*(-GH))
  double acc[TRF_NRED];            // last reduction (sums 0..5, min 6, max 7)
  double qn[5];                    // n-space dots of build_quadratic_1d / evaluate_quadratic (EW_STEP2)
  double r_value, p_value, ag_n0, ag_n1, ag_min;
  int active;      // outer loop still running
  int needed;      // bounded branch taken at all
  int status, nit, stop_next, full_step;
  Lsmr64 in;
  double ag_value;
  double trace[24][8];  // per outer iteration: cost, g_norm, inner itn, kind(0 full,1 p,2 r,3 ag), p/r/ag value, cost_change
};

struct TD {  // device buffers of the bounded branch
  TrfState* st;
  double *G, *D, *DH, *PH, *RH, *V, *H, *HBAR, *XIN, *W, *UN;  // [nc][npad]
  // sources of the select_step forwards A*(D*PH) and A*(-D*D*G).  They share storage with HBAR and H, which the
  // inner solve re-initialises at its first step and which are dead from EW_STEP1 to the next outer iteration.
  double *W2, *AG;
  // rows layout of u (u_total).  In select_step Y holds A*(D*RH), YP A*(D*PH) and YAG A*(-D*D*G); the step's A*step
  // is their combination (no forward of the step itself).
  double *R, *UM, *Y, *YP, *YAG;
  double* red;      // [nc][red_slots][TRF_NRED]
  int red_slots;
  int gn, gm;       // CTAs of an n-space / m-space pass (TRF_SPAN elements each)
  int* nactive;
  int* ninner;
};

HB2_HD void sym_ortho64_(double a, double b, double& c, double& s, double& r) {
  if (b == 0.0) { c = a > 0 ? 1.0 : (a < 0 ? -1.0 : 0.0); s = 0.0; r = fabs(a); }
  else if (a == 0.0) { c = 0.0; s = b > 0 ? 1.0 : -1.0; r = fabs(b); }
  else if (fabs(b) > fabs(a)) { double tau = a / b; s = (b > 0 ? 1.0 : -1.0) / sqrt(1 + tau * tau); c = s * tau; r = b / s; }
  else { double tau = b / a; c = (a > 0 ? 1.0 : -1.0) / sqrt(1 + tau * tau); s = c * tau; r = a / c; }
}
HB2_HD void lsmr64_init_(Lsmr64& S, double alpha, double beta) {
  S.alpha = alpha; S.beta = beta; S.normb = beta;
  S.zetabar = alpha * beta; S.alphabar = alpha; S.rho = 1; S.rhobar = 1; S.cbar = 1; S.sbar = 0;
  S.betadd = beta; S.betad = 0; S.rhodold = 1; S.tautildeold = 0; S.thetatilde = 0; S.zeta = 0; S.d = 0;
  S.normA2 = alpha * alpha; S.maxrbar = 0; S.minrbar = 0; S.minrbar_inf = 1; S.normA = sqrt(S.normA2);
  S.condA = 1; S.normx = 0; S.normr = beta; S.normar = alpha * beta; S.itn = 0; S.istop = 0; S.skip_adj = 0;
  S.cf_hbar = S.cf_x = S.cf_h = 0; S.rhotemp = 0;
  S.inv_alpha = alpha > 0 ? 1.0 / alpha : 1.0;
  S.inv_beta = beta > 0 ? 1.0 / beta : 0.0;
  S.active = (S.normar != 0.0 && beta != 0.0) ? 1 : 0;
}
HB2_HD void lsmr64_rotate_(Lsmr64& S, double alpha, double beta) {
  S.itn += 1; S.alpha = alpha; S.beta = beta;
  double chat = S.alphabar > 0 ? 1.0 : (S.alphabar < 0 ? -1.0 : 0.0), alphahat = fabs(S.alphabar);
  double rhoold = S.rho, c, s;
  sym_ortho64_(alphahat, beta, c, s, S.rho);
  double thetanew = s * alpha;
  S.alphabar = c * alpha;
  double rhobarold = S.rhobar, zetaold = S.zeta, thetabar = S.sbar * S.rho;
  S.rhotemp = S.cbar * S.rho;
  double cb, sb, rb;
  sym_ortho64_(S.cbar * S.rho, thetanew, cb, sb, rb);
  S.cbar = cb; S.sbar = sb; S.rhobar = rb;
  S.zeta = S.cbar * S.zetabar; S.zetabar = -S.sbar * S.zetabar;
  S.cf_hbar = -(thetabar * S.rho / (rhoold * rhobarold));
  S.cf_x = S.zeta / (S.rho * S.rhobar);
  S.cf_h = -(thetanew / S.rho);
  double betaacute = chat * S.betadd, betahat = c * betaacute;
  S.betadd = -s * betaacute;
  double thetatildeold = S.thetatilde, ct, st, rt;
  sym_ortho64_(S.rhodold, thetabar, ct, st, rt);
  S.thetatilde = st * S.rhobar; S.rhodold = ct * S.rhobar;
  S.betad = -st * S.betad + ct * betahat;
  S.tautildeold = (zetaold - thetatildeold * S.tautildeold) / rt;
  double taud = (S.zeta - S.thetatilde * S.tautildeold) / S.rhodold;
  S.normr = sqrt(S.d + (S.betad - taud) * (S.betad - taud) + S.betadd * S.betadd);
  S.normA2 += beta * beta; S.normA = sqrt(S.normA2); S.normA2 += alpha * alpha;
  S.maxrbar = fmax(S.maxrbar, rhobarold);
  if (S.itn > 1) { S.minrbar = S.minrbar_inf ? rhobarold : fmin(S.minrbar, rhobarold); S.minrbar_inf = 0; }
  double mn = S.minrbar_inf ? S.rhotemp : fmin(S.minrbar, S.rhotemp);
  S.condA = fmax(S.maxrbar, S.rhotemp) / mn;
  S.normar = fabs(S.zetabar);
  S.inv_alpha = alpha > 0 ? 1.0 / alpha : 1.0;
}
HB2_HD int lsmr64_test_(Lsmr64& S, double normx, double atol, double btol, double conlim, int maxiter) {
  S.normx = normx;
  double test1 = S.normr / S.normb;
  double test2 = (S.normA * S.normr) != 0 ? S.normar / (S.normA * S.normr) : INFINITY;
  double test3 = 1 / S.condA;
  double t1 = test1 / (1 + S.normA * normx / S.normb);
  double rtol = btol + atol * S.normA * normx / S.normb;
  double ctol = conlim > 0 ? 1 / conlim : 0;
  int istop = 0;
  if (S.itn >= maxiter) istop = 7;
  if (1 + test3 <= 1) istop = 6;
  if (1 + test2 <= 1) istop = 5;
  if (1 + t1 <= 1) istop = 4;
  if (test3 <= ctol) istop = 3;
  if (test2 <= atol) istop = 2;
  if (test1 <= rtol) istop = 1;
  S.istop = istop;
  return istop;
}

// gate: 0 outer-active, 1 inner-active, 2 outer-active and reflective part needed
__device__ __forceinline__ bool trf_gate(const TrfState& S, int gate) {
  if (!S.active) return false;
  if (gate == 1) return S.in.active != 0;
  if (gate == 2) return S.full_step == 0;
  return true;
}

// ---------------------------------------------------------------------------
// float64 operators (plain): rows <- A w ; w <- A^T rows.  Same maps as the
// float32 kernels; gathers in double.
// ---------------------------------------------------------------------------
template <typename IdxT>
__global__ void __launch_bounds__(HB2_BLOCK) k_fwd64_data(BD B, TD T, const double* __restrict__ src, double* __restrict__ dst,
                                                         int inner) {
  const int ntiles = (B.D2 + HB2_TILE_RAYS - 1) / HB2_TILE_RAYS;
  const int view = blockIdx.x / ntiles, tile = blockIdx.x % ntiles;
  const int c = B.view_cand[view];
  if (B.view_tie && B.view_tie[view] >= 0) return;  // tie views: k_fwd_tie<double>
  const TrfState& S = T.st[c];
  if (!trf_gate(S, inner)) return;
  __shared__ int s_colk[HB2_MAX_ZMC];
  for (int e = threadIdx.x; e < B.ZMC; e += HB2_BLOCK) s_colk[e] = B.colk[B.view_colbegin[view] + e];
  __syncthreads();
  const int a = B.view_angle[view];
  const int D2 = B.D2, L3 = B.L3, L3P = B.L3P, MC = B.MC, ZMP = B.ZMP;
  const IdxT* __restrict__ fm = (const IdxT*)B.fmap + (size_t)a * D2 * D2;
  const double* __restrict__ vsrc = src + (size_t)c * B.npad;
  double* urow = dst + B.view_uoff[view];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q = lane & 3, sg = lane >> 2;
  const uint8_t* __restrict__ pm = cand_mask(B, c);
  for (int r = warp; r < HB2_TILE_RAYS; r += HB2_BLOCK / 32) {
    const int j = tile * HB2_TILE_RAYS + r;
    if (j >= D2) break;
    if (!B.rayvalid[a * D2 + j]) continue;
    const IdxT* __restrict__ fj = fm + (size_t)j * D2;
    for (int z0 = 0; z0 < L3P; z0 += 16) {
      // lane (sg, q): the 4 consecutive slices z0 + 4q ... + 3 of every 8th sample, two 128-bit loads per sample and
      // four samples in flight (same lane layout as the float32 kernel)
      double acc[4] = {0, 0, 0, 0};
      const int zq = z0 + 4 * q;
      if (zq < L3P) {
        const double* __restrict__ vb = vsrc + zq;
        for (int i0 = sg; i0 < D2; i0 += 32) {
          IdxT ids[4];
#pragma unroll
          for (int w = 0; w < 4; ++w) ids[w] = (i0 + 8 * w < D2) ? fj[i0 + 8 * w] : Sent<IdxT>::v;
          double2 ta[4], tb[4];
#pragma unroll
          for (int w = 0; w < 4; ++w) {
            if (ids[w] != Sent<IdxT>::v) {
              const double2* vp = reinterpret_cast<const double2*>(vb + (size_t)ids[w] * L3P);
              ta[w] = __ldg(vp); tb[w] = __ldg(vp + 1);
            } else {
              ta[w] = make_double2(0.0, 0.0); tb[w] = make_double2(0.0, 0.0);
            }
          }
#pragma unroll
          for (int w = 0; w < 4; ++w)
            if (ids[w] != Sent<IdxT>::v) { acc[0] += ta[w].x; acc[1] += ta[w].y; acc[2] += tb[w].x; acc[3] += tb[w].y; }
        }
      }
#pragma unroll
      for (int o = 4; o < 32; o <<= 1)
#pragma unroll
        for (int t = 0; t < 4; ++t) acc[t] += __shfl_xor_sync(0xffffffffu, acc[t], o);
      if (sg < 4) {
        const int z = zq + sg;
        if (z < L3) {
          const double sum = sg == 0 ? acc[0] : (sg == 1 ? acc[1] : (sg == 2 ? acc[2] : acc[3]));
          for (int mc = 0; mc < MC; ++mc) {
            const int zm = z * MC + mc;
            if (s_colk[zm] >= 0 && !(pm && !pm[(size_t)s_colk[zm] * D2 + j])) urow[(size_t)j * ZMP + zm] = sum;
          }
        }
      }
    }
  }
}

__global__ void __launch_bounds__(HB2_BLOCK) k_fwd64_sym(BD B, TD T, const double* __restrict__ src, double* __restrict__ dst,
                                                        int inner) {
  const int c = blockIdx.y;
  const TrfState& S = T.st[c];
  if (!trf_gate(S, inner)) return;
  const int m = B.cand_msym[c];
  const double* __restrict__ vsrc = src + (size_t)c * B.npad;
  double* us = dst + B.cand_uoff[c] + B.cand_mdata[c];
  const int* __restrict__ sa = B.sym_a + B.cand_symoff[c];
  const int* __restrict__ sb = B.sym_b + B.cand_symoff[c];
  for (int r = blockIdx.x * HB2_BLOCK * 4 + threadIdx.x, qq = 0; qq < 4; ++qq, r += HB2_BLOCK)
    if (r < m) us[r] = __ldg(vsrc + sa[r]) - __ldg(vsrc + sb[r]);
}

// same lane layout as k_adj: one thread = (voxel p, slice quad q)
__global__ void __launch_bounds__(HB2_BLOCK) k_adj64(BD B, TD T, const double* __restrict__ rows, double* __restrict__ dst,
                                                    int inner) {
  const int c = blockIdx.y;
  const TrfState& S = T.st[c];
  if (!trf_gate(S, inner) || (inner == 1 && S.in.skip_adj)) return;
  const int L3 = B.L3, L3P = B.L3P, ZMP = B.ZMP, ndisk = B.ndisk, K = B.K, MC = B.MC;
  const int NQ = L3P >> 2;
  const int t = blockIdx.x * HB2_BLOCK + threadIdx.x;
  const int p = t / NQ, q = t - p * NQ;
  if (p >= ndisk) return;
  const int slot = B.aslot[p];
  const int z0 = 4 * q;
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  const int vb = B.cand_view_begin[c], nv = B.cand_view_count[c];
  for (int vi = 0; vi < nv; ++vi) {
    const int view = vb + vi;
    if (B.view_tie && B.view_tie[view] >= 0) continue;  // tie views: k_adj_tie<double> (BD::vtie64)
    const int a = __ldg(B.view_angle + view);
    const double* __restrict__ ub = rows + __ldg(B.view_uoff + view) + z0 * MC;
    const uint16_t* __restrict__ am = B.amap + (size_t)a * K * B.apitch + slot;
    for (int k = 0; k < K; ++k) {
      const uint16_t j = am[(size_t)k * B.apitch];
      if (j != 0xFFFFu) {
        const double* __restrict__ uj = ub + (size_t)j * ZMP;
        if (MC == 1) {
          const double2 r0 = __ldg(reinterpret_cast<const double2*>(uj));
          const double2 r1 = __ldg(reinterpret_cast<const double2*>(uj) + 1);
          acc[0] += r0.x; acc[1] += r0.y; acc[2] += r1.x; acc[3] += r1.y;
        } else {
#pragma unroll
          for (int zz = 0; zz < 4; ++zz)
            if (z0 + zz < L3)
              for (int mc = 0; mc < MC; ++mc) acc[zz] += __ldg(uj + zz * MC + mc);
        }
      }
    }
  }
  const int* __restrict__ ptr = B.csc_ptr + (size_t)c * (B.npad + 1);
  const int* __restrict__ ent = B.csc_ent + B.cand_cscoff[c];
  const double* __restrict__ us = rows + B.cand_uoff[c] + B.cand_mdata[c];
  double* vdst = dst + (size_t)c * B.npad + (size_t)p * L3P + z0;
  if (B.vtie64 && B.cand_tie_count[c] > 0) {
    const double* vt = B.vtie64 + (size_t)c * B.npad + (size_t)p * L3P + z0;
#pragma unroll
    for (int zz = 0; zz < 4; ++zz) acc[zz] += vt[zz];
  }
#pragma unroll
  for (int zz = 0; zz < 4; ++zz) {
    double a2 = acc[zz];
    if (z0 + zz < L3) {
      const int g = p * L3P + z0 + zz;
      for (int e = ptr[g]; e < ptr[g + 1]; ++e) {
        int en = ent[e];
        double val = __ldg(us + (en & 0x7fffffff));
        a2 += en < 0 ? -val : val;
      }
    }
    vdst[zz] = a2;
  }
}

// ---------------------------------------------------------------------------
// reductions: each CTA of a pass writes the partials of the slots its op uses
// (sums 0..5, min 6, max 7) to a fixed slot of the candidate; k_trf_reduce
// combines a candidate's slots in a fixed order into TrfState::acc and then takes
// the candidate's scalar decision.  No atomics, and a candidate's arithmetic does
// not depend on which other candidates share the batch.
// ---------------------------------------------------------------------------
__device__ __forceinline__ double trf_combine(int k, double a, double b) {
  return k < 6 ? a + b : (k == 6 ? fmin(a, b) : fmax(a, b));
}
__device__ __forceinline__ double trf_identity(int k) { return k < 6 ? 0.0 : (k == 6 ? INFINITY : -INFINITY); }

// block-wide combination of the slots in mask; thread 0 gets the results.  One barrier for all slots.
__device__ __forceinline__ void trf_block_reduce(double (&v)[TRF_NRED], unsigned mask, double (*shd)[HB2_BLOCK / 32]) {
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
#pragma unroll
  for (int k = 0; k < TRF_NRED; ++k) {
    if (!(mask >> k & 1u)) continue;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[k] = trf_combine(k, v[k], __shfl_xor_sync(0xffffffffu, v[k], o));
    if (l == 0) shd[k][w] = v[k];
  }
  __syncthreads();
  if (w == 0) {
#pragma unroll
    for (int k = 0; k < TRF_NRED; ++k) {
      if (!(mask >> k & 1u)) continue;
      double x = l < HB2_BLOCK / 32 ? shd[k][l] : trf_identity(k);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) x = trf_combine(k, x, __shfl_xor_sync(0xffffffffu, x, o));
      v[k] = x;
    }
  }
}

__device__ __forceinline__ double step_to_bound(double x, double s, double lb, double ub) {
  if (s == 0.0) return INFINITY;  // common.py:372-399, one component
  return fmax((lb - x) / s, (ub - x) / s);
}

// passes: n-space (unknowns of the candidate), m-space (its rows), or both in one launch (the first gn CTAs take the
// n-range, the next gm the m-range)
enum {
  EW_START = 0,   // reduction: min/max of x_lsq (in_bounds test, lsq_linear.py:328)
  EW_START_APPLY, // x <- make_strictly_feasible(reflective_transformation(x_lsq), rstep=0.1) ; W = x   (trf_linear.py:150-151)
  EW_PREP,        // Coleman-Li scaling from (x, g): D = sqrt(v), DH = g*dv ; reduction: max |g v|   (trf_linear.py:183-199)
                  // + first LSMR vector: V = D*G (D*(A^T r), u_n = 0), UN = 0 ; reduction: sum V^2
                  // + ag = -D*D*G of select_step (it depends on x and g only): its two n-space dots and min step_to_bound(x, ag)
  EW_INNER_V,     // v~ = (D*W + sqrt(DH)*u~_n)*inv_beta - beta*V ; reduction: sum v~^2
  EW_INNER_UPD,   // V = v~/alpha ; hbar, xin, h ; W = D*V ; reduction: sum xin^2
  EW_STEP1,       // PH = -XIN ; reductions: in_bounds(x + D*PH), min step_size_to_bound(x,p), p.g
  EW_STEP2,       // RH = reflected PH, PH *= p_stride ; W = D*RH, W2 = D*PH, AG = -D*D*G ; reductions: min step_size_to_bound(x+p, r),
                  // n-space dots of build_quadratic_1d / evaluate_quadratic.  Full-step candidates: W2 = D*PH only.
  EW_XUPD,        // X = make_strictly_feasible(X + step, rstep=0) ; W = X
  EW_FINAL,       // xs = float32(X)   (SLR:270)
  MW_RESID,       // R = A x - b ; u~_m = R (right-hand side of the next inner solve) ; sum R^2
  MW_DOTS,        // dots of Y = A_h r_h, YP = A_h p_h, YAG = A_h ag_h
  NM_INNER_U,     // n: u~_n = sqrt(DH)*V - alpha*(u~_n*inv_beta) ; m: u~_m = Y - alpha*(u~_m*inv_beta) ; sum of both squared
  NM_STEP         // n: step.g with step = D*(cp*PH + cr*RH - cag*D*G) ; m: |A step|^2, A step = cp*YP + cr*Y + cag*YAG
};
__host__ __device__ constexpr bool trf_has_n(int op) { return op < MW_RESID || op >= NM_INNER_U; }
__host__ __device__ constexpr bool trf_has_m(int op) { return op >= MW_RESID; }
__host__ __device__ constexpr unsigned trf_mask(int op) {  // reduction slots an op fills
  return op == EW_START ? 0xC0u : op == EW_PREP ? 0xC7u : op == EW_STEP1 ? 0xE0u : op == EW_STEP2 ? 0x9Fu
       : op == MW_DOTS ? 0x0Fu : op == NM_STEP ? 0x03u
       : (op == EW_START_APPLY || op == EW_XUPD || op == EW_FINAL) ? 0u : 0x01u;
}
__host__ __device__ constexpr unsigned trf_blocks(int op, unsigned gn, unsigned gm) {
  return (trf_has_n(op) ? gn : 0u) + (trf_has_m(op) ? gm : 0u);
}

// gate: 0 outer-active, 1 inner-active, 2 outer-active and reflective part needed
__device__ __forceinline__ bool trf_pass_active(const TrfState& S, int op) {
  switch (op) {
    case EW_START: case EW_FINAL: return S.needed != 0;
    case EW_START_APPLY: return S.active != 0;
    case EW_INNER_UPD: return S.active && (S.in.active || S.in.itn == 0);
    case NM_INNER_U: return trf_gate(S, 1);
    case EW_INNER_V: return trf_gate(S, 1) && !S.in.skip_adj;
    case MW_DOTS: return trf_gate(S, 2);
    default: return trf_gate(S, 0);
  }
}

// the step of trf_linear.py:219-225 rebuilt from PH, RH, D and G (it is never stored)
__device__ __forceinline__ double trf_step(const TrfState& S, const TD& T, size_t e) {
  const double d = T.D[e];
  return d * (S.coef_p * T.PH[e] + S.coef_r * T.RH[e] - S.coef_ag * (d * T.G[e]));
}

template <int OP>
__device__ __forceinline__ void trf_n_elem(const BD& B, const TD& T, const TrfState& S, double* X, int i, size_t e,
                                           double (&red)[TRF_NRED]) {
  const double lb = S.lb, ub = S.ub;
  if constexpr (OP == EW_START) {
    double y = X[i];
    red[6] = fmin(red[6], y); red[7] = fmax(red[7], y);
  } else if constexpr (OP == EW_START_APPLY) {
    const double y = X[i], dd = ub - lb;
    double t = fmod(y - lb, 2 * dd);
    if (t < 0) t += 2 * dd;  // np.remainder takes the sign of the divisor (common.py:535)
    double x = lb + fmin(t, 2 * dd - t);
    // make_strictly_feasible(rstep=0.1): common.py:440-464 with find_active_constraints (:401-437)
    double ld = x - lb, udist = ub - x;
    double lth = 0.1 * fmax(1.0, fabs(lb)), uth = 0.1 * fmax(1.0, fabs(ub));
    bool la = ld <= fmin(udist, lth), ua = udist <= fmin(ld, uth);
    if (la) x = lb + 0.1 * fmax(1.0, fabs(lb));
    if (ua) x = ub - 0.1 * fmax(1.0, fabs(ub));
    if (x < lb || x > ub) x = 0.5 * (lb + ub);
    X[i] = x;
    T.W[e] = x;
  } else if constexpr (OP == EW_PREP) {
    double x = X[i], g = T.G[e], v = 1.0, dv = 0.0;
    if (g < 0) { v = ub - x; dv = -1.0; }
    if (g > 0) { v = x - lb; dv = 1.0; }
    const double d = sqrt(v), dh = g * dv;
    T.D[e] = d; T.DH[e] = dh;
    red[7] = fmax(red[7], fabs(g * v));
    const double gh = d * g;  // = D*(A^T r): the inner solve's first v (before 1/beta)
    T.UN[e] = 0.0; T.V[e] = gh; red[0] += gh * gh;
    const double agh = -gh, ag = d * agh;
    red[1] += agh * dh * agh; red[2] += gh * agh;
    red[6] = fmin(red[6], step_to_bound(x, ag, lb, ub));
  } else if constexpr (OP == EW_INNER_V) {
    double vt = (T.D[e] * T.W[e] + sqrt(T.DH[e]) * T.UN[e]) * S.in.inv_beta - S.in.beta * T.V[e];
    T.V[e] = vt; red[0] += vt * vt;
  } else if constexpr (OP == EW_INNER_UPD) {
    double vn = T.V[e];
    if (S.in.itn == 0 || !S.in.skip_adj) { vn *= S.in.inv_alpha; T.V[e] = vn; }
    if (S.in.itn == 0) { T.H[e] = vn; T.HBAR[e] = 0.0; T.XIN[e] = 0.0; }
    else {
      double ho = T.H[e];
      double hb = T.HBAR[e] * S.in.cf_hbar + ho;
      T.HBAR[e] = hb;
      double xn = T.XIN[e] + S.in.cf_x * hb;
      T.XIN[e] = xn;
      T.H[e] = ho * S.in.cf_h + vn;
      red[0] += xn * xn;
    }
    T.W[e] = T.D[e] * vn;
  } else if constexpr (OP == EW_STEP1) {
    double ph = -T.XIN[e];
    T.PH[e] = ph;
    double x = X[i], p = T.D[e] * ph, xp = x + p;
    red[6] = fmin(red[6], fmin(xp - lb, ub - xp));
    red[5] += p * T.G[e];
    red[7] = fmax(red[7], -step_to_bound(x, p, lb, ub));
  } else if constexpr (OP == EW_STEP2) {
    const double ph = T.PH[e], d = T.D[e];
    if (S.full_step) { T.W2[e] = d * ph; return; }
    const double x = X[i], p = d * ph;
    const double st = step_to_bound(x, p, lb, ub);
    const double rh = (st == S.p_stride && p != 0.0) ? -ph : ph;  // hits -> reflect (trf_linear.py:97-99)
    const double phs = ph * S.p_stride;
    T.RH[e] = rh; T.PH[e] = phs;
    const double xb = x + p * S.p_stride, r = d * rh;
    red[7] = fmax(red[7], -step_to_bound(xb, r, lb, ub));
    T.W[e] = r; T.W2[e] = d * phs;
    const double dh = T.DH[e], gh = d * T.G[e];
    red[0] += rh * dh * rh; red[1] += gh * rh; red[2] += phs * dh * rh; red[3] += gh * phs; red[4] += phs * dh * phs;
    T.AG[e] = d * -gh;
  } else if constexpr (OP == EW_XUPD) {
    double x = X[i];
    if (S.cost_change >= 0) {  // else: scipy's backtracking() hands back the OLD x (trf_linear.py:69-88)
      x = x + trf_step(S, T, e);
      if (x <= lb) x = nextafter(lb, ub);
      if (x >= ub) x = nextafter(ub, lb);
      if (x < lb || x > ub) x = 0.5 * (lb + ub);
      X[i] = x;
    }
    T.W[e] = x;
  } else if constexpr (OP == EW_FINAL) {
    B.xs[e] = (float)X[i];
  } else if constexpr (OP == NM_INNER_U) {
    double un = sqrt(T.DH[e]) * T.V[e] - S.in.alpha * (T.UN[e] * S.in.inv_beta);
    T.UN[e] = un; red[0] += un * un;
  } else if constexpr (OP == NM_STEP) {
    red[1] += trf_step(S, T, e) * T.G[e];
  }
}

template <int OP>
__device__ __forceinline__ void trf_m_elem(const BD& B, const TD& T, const TrfState& S, int c, long long r, size_t e,
                                           double (&red)[TRF_NRED]) {
  if constexpr (OP == MW_RESID) {
    double bb = r < B.cand_mdata[c] ? (double)B.b[e] : 0.0;
    double res = T.Y[e] - bb;
    T.R[e] = res; T.UM[e] = res; red[0] += res * res;
  } else if constexpr (OP == NM_INNER_U) {
    double un = T.Y[e] - S.in.alpha * (T.UM[e] * S.in.inv_beta);
    T.UM[e] = un; red[0] += un * un;
  } else if constexpr (OP == MW_DOTS) {
    double v1 = T.Y[e], u1 = T.YP[e], a = T.YAG[e];
    red[0] += v1 * v1; red[1] += u1 * v1; red[2] += u1 * u1; red[3] += a * a;
  } else if constexpr (OP == NM_STEP) {  // at most two coefficients are non-zero; the others' vectors are not read
    double v = 0.0;
    if (S.coef_p != 0.0) v += S.coef_p * T.YP[e];
    if (S.coef_r != 0.0) v += S.coef_r * T.Y[e];
    if (S.coef_ag != 0.0) v += S.coef_ag * T.YAG[e];
    red[0] += v * v;
  }
}

template <int OP>
__global__ void __launch_bounds__(HB2_BLOCK) k_trf_pass(BD B, TD T) {
  const int c = blockIdx.y;
  const TrfState& S = T.st[c];
  if (!trf_pass_active(S, OP)) return;
  double red[TRF_NRED];
#pragma unroll
  for (int k = 0; k < TRF_NRED; ++k) red[k] = trf_identity(k);
  if (trf_has_n(OP) && (!trf_has_m(OP) || (int)blockIdx.x < T.gn)) {
    const size_t o = (size_t)c * B.npad;
    double* X = B.x + o;
    const int i0 = blockIdx.x * TRF_SPAN + threadIdx.x;
#pragma unroll 4
    for (int k = 0; k < TRF_EPT; ++k) {
      const int i = i0 + k * HB2_BLOCK;
      if (i >= B.npad || (i % B.L3P) >= B.L3) continue;  // padded slices are not unknowns
      trf_n_elem<OP>(B, T, S, X, i, o + i, red);
    }
  } else if (trf_has_m(OP)) {
    const long long m = (long long)B.cand_mdata[c] + B.cand_msym[c];
    const size_t o = (size_t)B.cand_uoff[c];
    const long long r0 = (long long)(blockIdx.x - (trf_has_n(OP) ? T.gn : 0)) * TRF_SPAN + threadIdx.x;
#pragma unroll 4
    for (int k = 0; k < TRF_EPT; ++k) {
      const long long r = r0 + (long long)k * HB2_BLOCK;
      if (r >= m) continue;
      trf_m_elem<OP>(B, T, S, c, r, o + r, red);
    }
  }
  constexpr unsigned mask = trf_mask(OP);
  if constexpr (mask != 0) {
    __shared__ double shd[TRF_NRED][HB2_BLOCK / 32];
    trf_block_reduce(red, mask, shd);
    if (threadIdx.x == 0) {
      double* dst = T.red + ((size_t)c * T.red_slots + blockIdx.x) * TRF_NRED;
#pragma unroll
      for (int k = 0; k < TRF_NRED; ++k)
        if (mask >> k & 1u) dst[k] = red[k];
    }
  }
}

// scalar decisions: thread 0 of k_trf_reduce, after the candidate's partials are combined into TrfState::acc ------
enum {
  SC_START = 0, SC_RESID0, SC_PREP, SC_INNER_BETA, SC_INNER_ROT, SC_INNER_TEST, SC_STEP1, SC_STEP2, SC_SELECT, SC_CC,
  SC_RESID
};
__device__ __forceinline__ bool trf_scal_active(const TrfState& S, int op) {
  if (op == SC_START) return S.needed != 0;
  if (op == SC_INNER_BETA || op == SC_INNER_ROT || op == SC_INNER_TEST) return trf_gate(S, 1);
  if (op == SC_STEP2 || op == SC_SELECT) return trf_gate(S, 2);
  return trf_gate(S, 0);
}
__device__ __forceinline__ void min_quadratic_1d(double a, double b, double lo, double hi, double c, double& t, double& y) {
  // common.py:302-322
  double tt[3] = {lo, hi, 0};
  int n = 2;
  if (a != 0) {
    double ext = -0.5 * b / a;
    if (lo < ext && ext < hi) tt[n++] = ext;
  }
  t = tt[0]; y = tt[0] * (a * tt[0] + b) + c;
  for (int k = 1; k < n; ++k) {
    double yy = tt[k] * (a * tt[k] + b) + c;
    if (yy < y) { y = yy; t = tt[k]; }  // np.argmin keeps the first minimum
  }
}
__device__ void trf_scalar(const TD& T, TrfState& S, int op, double eps, int lsmr_maxiter, int max_iter) {
  const double* r = S.acc;
  switch (op) {
    case SC_START: {
      bool inb = r[6] >= S.lb && r[7] <= S.ub;  // unconstrained solution already feasible (lsq_linear.py:328)
      S.active = inb ? 0 : 1; S.status = inb ? 3 : 0; S.nit = 0; S.stop_next = 0; S.full_step = 0;
      if (!inb) atomicAdd(T.nactive, 1);
    } break;
    case SC_RESID0: S.cost = 0.5 * r[0]; break;
    case SC_PREP: {
      S.g_norm = r[7];
      bool stop = S.stop_next != 0;
      if (S.g_norm < S.tol) { S.status = 1; stop = true; }
      if (!stop && S.nit >= max_iter) stop = true;
      if (stop) { S.active = 0; if (S.nit < max_iter) S.nit += 1; atomicSub(T.nactive, 1); break; }  // nit = iteration + 1
      S.nit += 1;
      if (S.nit <= 24) { S.trace[S.nit - 1][0] = S.cost; S.trace[S.nit - 1][1] = S.g_norm; }
      double eta = 1e-2 * fmin(0.5, S.g_norm);
      S.lsmr_tol = fmax(eps, fmin(0.1, eta * S.g_norm));
      S.theta = 1 - fmin(0.005, S.g_norm);
      S.full_step = 0;
      // inner LSMR on [A D; sqrt(diag_h)] p_h = -[r; 0]: V holds D*(A^T r) (not yet divided by beta)
      const double beta = sqrt(2 * S.cost), nv = sqrt(r[0]);
      lsmr64_init_(S.in, nv * (beta > 0 ? 1.0 / beta : 0.0), beta);
      S.in.inv_alpha = nv > 0 ? 1.0 / nv : 1.0;
      if (S.in.active) atomicAdd(T.ninner, 1);
      S.ag_n0 = r[1]; S.ag_n1 = r[2]; S.ag_min = r[6];  // ag = -D*D*G (select_step)
    } break;
    case SC_INNER_BETA: {
      S.in.beta = sqrt(r[0]);
      if (S.in.beta > 0) { S.in.inv_beta = 1.0 / S.in.beta; S.in.skip_adj = 0; } else S.in.skip_adj = 1;
    } break;
    case SC_INNER_ROT: lsmr64_rotate_(S.in, S.in.skip_adj ? S.in.alpha : sqrt(r[0]), S.in.beta); break;
    case SC_INNER_TEST: {
      int istop = lsmr64_test_(S.in, sqrt(r[0]), S.lsmr_tol, S.lsmr_tol, 1e8, lsmr_maxiter);
      if (istop > 0) { S.in.active = 0; atomicSub(T.ninner, 1); }
    } break;
    case SC_STEP1: {
      S.p_dot_g = r[5];
      if (S.p_dot_g > 0) { S.status = -1; S.stop_next = 1; }
      S.full_step = r[6] >= 0.0 ? 1 : 0;
      S.p_stride = -r[7];
      if (S.full_step) { S.coef_p = 1.0; S.coef_r = 0.0; S.coef_ag = 0.0; }
    } break;
    case SC_STEP2: {
      double rsu = -r[7];
      S.r_stride_l = (1 - S.theta) * rsu;
      S.r_stride_u = rsu * S.theta;
      for (int k = 0; k < 5; ++k) S.qn[k] = r[k];
    } break;
    case SC_SELECT: {
      // build_quadratic_1d(A_h, g_h, r_h, s0=p_h, diag=diag_h), common.py:251-299
      const double* q = S.qn;
      const double m0 = r[0], m1 = r[1], m2 = r[2];
      double a = 0.5 * (m0 + q[0]);
      double b = q[1] + m1 + q[2];
      double cc = 0.5 * m2 + q[3] + 0.5 * q[4];
      if (S.r_stride_u > 0) min_quadratic_1d(a, b, S.r_stride_l, S.r_stride_u, cc, S.r_stride, S.r_value);
      else { S.r_value = INFINITY; S.r_stride = 0; }
      double th = S.theta;  // p_h *= theta ; evaluate_quadratic(A_h, g_h, p_h, diag_h)
      S.p_value = 0.5 * (th * th * m2 + th * th * q[4]) + th * q[3];
      // anti-gradient step
      a = 0.5 * (r[3] + S.ag_n0); b = S.ag_n1;
      double ag_value;
      min_quadratic_1d(a, b, 0.0, S.ag_min * S.theta, 0.0, S.ag_stride, ag_value);
      S.ag_value = ag_value;
      if (S.p_value < S.r_value && S.p_value < ag_value) { S.coef_p = S.theta; S.coef_r = 0; S.coef_ag = 0; }
      else if (S.r_value < S.p_value && S.r_value < ag_value) { S.coef_p = 1.0; S.coef_r = S.r_stride; S.coef_ag = 0; }
      else { S.coef_p = 0; S.coef_r = 0; S.coef_ag = S.ag_stride; }
    } break;
    case SC_CC: {
      S.cost_change = -(0.5 * r[0] + r[1]);  // -evaluate_quadratic(A, g, step)
      if (S.nit <= 24) {
        double* t = S.trace[S.nit - 1];
        t[2] = S.in.itn;
        t[3] = S.full_step ? 0 : (S.coef_ag != 0 ? 3 : (S.coef_r != 0 ? 2 : 1));
        t[4] = S.p_value; t[5] = S.r_value; t[6] = S.ag_value; t[7] = S.cost_change;
      }
    } break;
    case SC_RESID: {
      if (S.cost_change < S.tol * S.cost) { S.status = 2; S.stop_next = 1; }
      S.cost = 0.5 * r[0];
    } break;
  }
}

// one CTA per candidate: combine the nslots partials of the slots in mask in a fixed order, then decide (op)
__global__ void __launch_bounds__(HB2_BLOCK) k_trf_reduce(BD B, TD T, int nslots, unsigned mask, int op, double eps,
                                                          int lsmr_maxiter, int max_iter) {
  const int c = blockIdx.x;
  __shared__ double shd[TRF_NRED][HB2_BLOCK / 32];
  TrfState& S = T.st[c];
  if (!trf_scal_active(S, op)) return;
  double v[TRF_NRED];
#pragma unroll
  for (int k = 0; k < TRF_NRED; ++k) v[k] = trf_identity(k);
  for (int s2 = threadIdx.x; s2 < nslots; s2 += HB2_BLOCK) {
    const double* p = T.red + ((size_t)c * T.red_slots + s2) * TRF_NRED;
#pragma unroll
    for (int k = 0; k < TRF_NRED; ++k)
      if (mask >> k & 1u) v[k] = trf_combine(k, v[k], p[k]);
  }
  trf_block_reduce(v, mask, shd);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int k = 0; k < TRF_NRED; ++k)
      if (mask >> k & 1u) S.acc[k] = v[k];
    trf_scalar(T, S, op, eps, lsmr_maxiter, max_iter);
  }
}
