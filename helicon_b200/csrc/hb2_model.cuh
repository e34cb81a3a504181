// ElasticNet / Lasso / Ridge (SLR:272-342) for every candidate of a batch at once: the algorithms of
// helicon_b200/regularized.py as a device state machine.  The X / X^T products are the batch's MODE_PLAIN projector
// kernels over all candidates (launch_fwd_data / launch_fwd_sym / launch_adj, only_cand = -1); the kernels here do the
// element-wise and reduction work in float64:
//   centred operator   X_c w = mask*(A w - xbar.w),   X_c^T r = A^T(mask*r) - xbar*sum(r),   xbar = A^T mask / m
//   power iteration    20 steps on the host's start vector, x1.05                      (_CenteredOperator.lipschitz)
//   FISTA + O'Donoghue-Candes restart, duality gap every 10 iterations       (_enet, _enet_gap; _ridge when positive)
//   CG on the normal equations                                                         (_ridge without the bound)
//   refit of an all-zero elastic-net / lasso solution with alpha x 0.1                        (SLR:331-335)
// Vectors: w in B.x, z (FISTA) / p (CG) in B.hbar, both [nc][npad] float64; the float32 input and output of every
// product is B.xs (n-space) and B.u (rows).  Each pass writes per-CTA partials that k_mdl_reduce combines in a fixed
// order (the pattern of k_trf_pass / k_trf_reduce), so a candidate's bits do not depend on the batch it is solved in.
#pragma once
#include "hb2_trf.cuh"

#define MDL_EPT 8
#define MDL_SPAN (HB2_BLOCK * MDL_EPT)
#define MDL_MAX_REFITS 30  // alpha x 1e-30: a right-hand side without any signal; the fit ends NOT_CONVERGED

enum { MDL_FISTA_ENET = 0, MDL_FISTA_RIDGE = 1, MDL_CG_RIDGE = 2 };

struct ModelState {
  int kind, positive, in_power, active, wait, zero_now, lip_zero, not_conv, it, refits, stop;
  double m, ybar, yy, alpha, l1_ratio, alpha_s, beta_s, lip, L, step, tol_gap;
  double t, t_new, restart;       // FISTA
  double s, sr;                   // xbar.q of the product's input, sum of its centred row vector
  double rs, rs0, a, beta;        // CG
  double gap, dw, lam;
  double acc[TRF_NRED];
};

struct MD {
  ModelState* st;
  const uint8_t* real;  // [u_total] real rows (hb2_batch_set_real_rows)
  double* xbar;         // [nc][npad]
  double* wn;           // [nc][npad] w_new (FISTA) / A p (CG) / X_c^T X_c v (power iteration)
  double* rhs;          // [nc][npad] X_c^T y_c (ridge)
  double* r;            // [nc][npad] CG residual
  const double* v0;     // [npad] power-iteration start vector, internal order
  double* red;          // [nc][slots][TRF_NRED]
  int gn, gm, slots;
  int max_iter;
  double gap_factor;
};

enum {
  // n-space passes
  MN_XBAR = 0,  // xbar = xs / m
  MN_V0,        // z = v0 (power iteration)
  MN_LOADZ,     // xs = f32(z); partial xbar.z
  MN_LOADW,     // xs = f32(w); partial xbar.w (duality gap)
  MN_POW,       // wn = X_c^T(X_c v); partial |wn|^2
  MN_POWNORM,   // z = wn / lam
  MN_ZERO,      // w = z = 0
  MN_RHS,       // rhs = X_c^T y_c (CG: r = p = rhs); partial |rhs|^2
  MN_GRAD,      // FISTA: w_new, partial restart dot; CG: A p, partial p.Ap
  MN_UPD,       // FISTA: z, w; partials |w_new - w|^2, |w_new|^2, nnz(w_new); CG: w, r; partial |r|^2
  MN_CGP,       // CG: p = r + beta p
  MN_GAP,       // partials of the duality gap: max |X^T R - beta_s w|, w.w, |w|_1
  MN_FINAL,     // xs = f32(w)
  // m-space passes
  MM_SETUP,     // partials sum(real*y), sum(real)
  MM_YY,        // partial |y_c|^2
  MM_MASK,      // u = real
  MM_YC,        // u = f32(y_c); partial sum(y_c)
  MM_ROW,       // u = f32(r), r = mask*(A q - s) (ridge, power) or mask*(y_c - (A q - s)) (elastic net); partial sum(r)
  MM_GAPROW,    // R = mask*(y_c - (A w - s)); u = f32(R); partials sum R, R.R, R.y_c
};
enum {
  MS_SETUP = 0, MS_YY, MS_S, MS_SR, MS_RHS, MS_POW, MS_LIP, MS_BEGIN, MS_GRAD, MS_UPD, MS_GAP,
};

// Which candidates a pass or a decision touches.  it_global: the batch's iteration (1-based) for MS_BEGIN.
__device__ __forceinline__ bool mdl_iterating(const ModelState& S) { return S.active && !S.stop; }
__device__ __forceinline__ bool mdl_gap_due(const ModelState& S) {
  return mdl_iterating(S) && S.kind == MDL_FISTA_ENET && S.it % 10 == 0;
}
__device__ __forceinline__ bool mdl_pass_active(const ModelState& S, int op) {
  switch (op) {
    case MN_POW: case MN_POWNORM: return !S.lip_zero;
    case MN_LOADZ: case MM_ROW: return S.in_power ? !S.lip_zero : mdl_iterating(S);
    case MN_GRAD: case MN_UPD: return mdl_iterating(S);
    case MN_CGP: return mdl_iterating(S) && S.kind == MDL_CG_RIDGE;
    case MN_LOADW: case MN_GAP: case MM_GAPROW: return mdl_gap_due(S);
    case MN_RHS: case MM_YC: return S.kind != MDL_FISTA_ENET;
    default: return true;
  }
}

__device__ __forceinline__ bool mdl_real_voxel(const BD& B, int i) { return i < B.npad && (i % B.L3P) < B.L3; }

template <int OP>
__device__ __forceinline__ void mdl_n_elem(const BD& B, const MD& M, const ModelState& S, size_t o, double (&red)[TRF_NRED]) {
  double* W = B.x;
  double* Z = B.hbar;
  if (OP == MN_XBAR) M.xbar[o] = (double)B.xs[o] / S.m;
  else if (OP == MN_V0) Z[o] = M.v0[o % B.npad];
  else if (OP == MN_LOADZ || OP == MN_LOADW) {
    if (OP == MN_LOADZ && S.zero_now) { W[o] = 0.0; Z[o] = 0.0; }  // a refit starts from w = z = 0
    const double q = OP == MN_LOADZ ? Z[o] : W[o];
    B.xs[o] = (float)q;
    red[0] += M.xbar[o] * q;
  } else if (OP == MN_POW) {
    const double g = (double)B.xs[o] - M.xbar[o] * S.sr;
    M.wn[o] = g;
    red[0] += g * g;
  } else if (OP == MN_POWNORM) Z[o] = M.wn[o] / S.lam;
  else if (OP == MN_ZERO) { W[o] = 0.0; Z[o] = 0.0; }
  else if (OP == MN_RHS) {
    const double g = (double)B.xs[o] - M.xbar[o] * S.sr;
    M.rhs[o] = g;
    if (S.kind == MDL_CG_RIDGE) { M.r[o] = g; Z[o] = g; }
    red[0] += g * g;
  } else if (OP == MN_GRAD) {
    const double g = (double)B.xs[o] - M.xbar[o] * S.sr;  // X_c^T of the row vector
    const double z = Z[o];
    if (S.kind == MDL_CG_RIDGE) {
      const double ap = g + S.alpha * z;
      M.wn[o] = ap;
      red[0] += z * ap;
    } else {
      double wn;
      if (S.kind == MDL_FISTA_ENET) {  // row vector = y_c - X_c z: grad = -g + beta_s z; soft threshold
        wn = z - S.step * (-g + S.beta_s * z);
        const double th = S.step * S.alpha_s;
        wn = wn > 0.0 ? fmax(wn - th, 0.0) : (wn < 0.0 ? -fmax(-wn - th, 0.0) : 0.0);
        if (S.positive) wn = fmax(wn, 0.0);
      } else {                          // row vector = X_c z: grad = g + alpha z - rhs; projection on w >= 0
        wn = fmax(z - S.step * (g + S.alpha * z - M.rhs[o]), 0.0);
      }
      M.wn[o] = wn;
      red[0] += (z - wn) * (wn - W[o]);
    }
  } else if (OP == MN_UPD) {
    if (S.kind == MDL_CG_RIDGE) {
      W[o] += S.a * Z[o];
      const double r = M.r[o] - S.a * M.wn[o];
      M.r[o] = r;
      red[0] += r * r;
    } else {
      const double wn = M.wn[o], w = W[o];
      Z[o] = S.restart != 0.0 ? wn : wn + ((S.t - 1.0) / S.t_new) * (wn - w);
      red[0] += (wn - w) * (wn - w);
      red[1] += wn * wn;
      red[2] += wn != 0.0 ? 1.0 : 0.0;
      W[o] = wn;
    }
  } else if (OP == MN_CGP) Z[o] = M.r[o] + S.beta * Z[o];
  else if (OP == MN_GAP) {
    const double w = W[o];
    const double xta = ((double)B.xs[o] - M.xbar[o] * S.sr) - S.beta_s * w;
    red[7] = fmax(red[7], S.positive ? xta : fabs(xta));
    red[0] += w * w;
    red[1] += fabs(w);
  } else if (OP == MN_FINAL) B.xs[o] = (float)W[o];
}

template <int OP>
__device__ __forceinline__ void mdl_m_elem(const BD& B, const MD& M, const ModelState& S, int c, long long r, size_t o,
                                           double (&red)[TRF_NRED]) {
  const bool real = M.real[o] != 0;
  const double y = r < B.cand_mdata[c] ? (double)B.b[o] : 0.0;  // the symmetry rows' right-hand side is 0
  const double yc = real ? y - S.ybar : 0.0;
  if (OP == MM_SETUP) { if (real) { red[0] += y; red[1] += 1.0; } }
  else if (OP == MM_YY) red[0] += yc * yc;
  else if (OP == MM_MASK) B.u[o] = real ? 1.f : 0.f;
  else if (OP == MM_YC) { B.u[o] = (float)yc; red[0] += yc; }
  else if (OP == MM_ROW) {
    const double xq = (double)B.u[o] - S.s;
    const double v = real ? (S.kind == MDL_FISTA_ENET && !S.in_power ? yc - xq : xq) : 0.0;
    B.u[o] = (float)v;
    red[0] += v;
  } else if (OP == MM_GAPROW) {
    const double R = real ? yc - ((double)B.u[o] - S.s) : 0.0;
    B.u[o] = (float)R;
    red[0] += R; red[1] += R * R; red[2] += R * yc;
  }
}

__host__ __device__ constexpr unsigned mdl_mask(int op) {
  return op == MN_GAP ? 0x83u : (op == MN_UPD || op == MM_GAPROW ? 0x7u : (op == MM_SETUP ? 0x3u : 0x1u));
}

template <int OP>
__global__ void __launch_bounds__(HB2_BLOCK) k_mdl_n(BD B, MD M) {
  const int c = blockIdx.y;
  const ModelState& S = M.st[c];
  if (!mdl_pass_active(S, OP)) return;
  double red[TRF_NRED];
#pragma unroll
  for (int k = 0; k < TRF_NRED; ++k) red[k] = trf_identity(k);
  const size_t base = (size_t)c * B.npad;
  const int i0 = blockIdx.x * MDL_SPAN + threadIdx.x;
#pragma unroll 4
  for (int k = 0; k < MDL_EPT; ++k) {
    const int i = i0 + k * HB2_BLOCK;
    if (!mdl_real_voxel(B, i)) continue;  // padded slices are not unknowns: they stay 0 in every vector
    mdl_n_elem<OP>(B, M, S, base + i, red);
  }
  __shared__ double shd[TRF_NRED][HB2_BLOCK / 32];
  trf_block_reduce(red, mdl_mask(OP), shd);
  if (threadIdx.x == 0) {
    double* dst = M.red + ((size_t)c * M.slots + blockIdx.x) * TRF_NRED;
#pragma unroll
    for (int k = 0; k < TRF_NRED; ++k)
      if (mdl_mask(OP) >> k & 1u) dst[k] = red[k];
  }
}

template <int OP>
__global__ void __launch_bounds__(HB2_BLOCK) k_mdl_m(BD B, MD M) {
  const int c = blockIdx.y;
  const ModelState& S = M.st[c];
  if (!mdl_pass_active(S, OP)) return;
  double red[TRF_NRED];
#pragma unroll
  for (int k = 0; k < TRF_NRED; ++k) red[k] = trf_identity(k);
  const long long m = (long long)B.cand_mdata[c] + B.cand_msym[c];  // the candidate's own rows only
  const size_t base = (size_t)B.cand_uoff[c];
  const long long r0 = (long long)blockIdx.x * MDL_SPAN + threadIdx.x;
#pragma unroll 4
  for (int k = 0; k < MDL_EPT; ++k) {
    const long long r = r0 + (long long)k * HB2_BLOCK;
    if (r >= m) continue;
    mdl_m_elem<OP>(B, M, S, c, r, base + r, red);
  }
  __shared__ double shd[TRF_NRED][HB2_BLOCK / 32];
  trf_block_reduce(red, mdl_mask(OP), shd);
  if (threadIdx.x == 0) {
    double* dst = M.red + ((size_t)c * M.slots + blockIdx.x) * TRF_NRED;
#pragma unroll
    for (int k = 0; k < TRF_NRED; ++k)
      if (mdl_mask(OP) >> k & 1u) dst[k] = red[k];
  }
}

// end of one fit: an all-zero elastic-net / lasso solution is fitted again with alpha x 0.1 (SLR:331-335); it waits
// for the next block of 10 batch iterations so that its gap checks fall on the batch's gap products
__device__ __forceinline__ void mdl_finish(ModelState& S, bool converged, bool all_zero) {
  S.active = 0;
  if (S.kind == MDL_FISTA_ENET && all_zero && S.refits < MDL_MAX_REFITS) {
    S.refits += 1;
    S.alpha *= 0.1;
    S.alpha_s = S.alpha * S.l1_ratio * S.m;
    S.beta_s = S.alpha * (1 - S.l1_ratio) * S.m;
    S.L = S.lip + S.beta_s;
    S.step = 1.0 / S.L;
    S.wait = 1;
    return;
  }
  S.not_conv = converged ? 0 : 1;
  S.stop = 1;
}

// thread 0: the candidate's scalar decision after its partials are combined into acc[0..4], acc[7]
__device__ __forceinline__ void mdl_scalar(const MD& M, ModelState& S, int op, int it_global) {
  const double* a = S.acc;
  switch (op) {
    case MS_SETUP:
      S.m = a[1];
      S.ybar = S.m > 0 ? a[0] / S.m : 0.0;
      S.alpha_s = S.alpha * S.l1_ratio * S.m;  // scikit-learn's un-normalised elastic net
      S.beta_s = S.alpha * (1 - S.l1_ratio) * S.m;
      break;
    case MS_YY: S.yy = a[0]; S.tol_gap = M.gap_factor * 1e-2 * a[0]; break;
    case MS_S: S.s = a[0]; break;
    case MS_SR: S.sr = a[0]; break;
    case MS_RHS: S.rs = S.rs0 = a[0]; break;
    case MS_POW:
      S.lam = sqrt(a[0]);
      if (S.lam == 0.0) S.lip_zero = 1;
      break;
    case MS_LIP:
      S.in_power = 0;
      S.lip = S.lip_zero ? 1.0 : S.lam * 1.05;
      S.L = S.lip + (S.kind == MDL_FISTA_ENET ? S.beta_s : S.alpha);
      S.step = 1.0 / S.L;
      break;
    case MS_BEGIN:  // a pending refit starts at the first iteration of a block of 10
      S.zero_now = 0;
      if (S.wait && (it_global - 1) % 10 == 0) {
        S.wait = 0; S.active = 1; S.it = 0; S.t = 1.0; S.zero_now = 1;
      }
      if (mdl_iterating(S)) S.it += 1;
      break;
    case MS_GRAD:
      if (S.kind == MDL_CG_RIDGE) S.a = S.rs / a[0];
      else {
        S.restart = a[0] > 0.0 ? 1.0 : 0.0;  // O'Donoghue-Candes gradient restart
        S.t_new = S.restart != 0.0 ? 1.0 : 0.5 * (1 + sqrt(1 + 4 * S.t * S.t));
      }
      break;
    case MS_UPD:
      S.zero_now = 0;
      if (S.kind == MDL_CG_RIDGE) {
        const double rs_new = a[0];
        S.gap = sqrt(rs_new / fmax(S.rs0, 1e-300));  // reported: relative CG residual
        if (rs_new <= 1e-12 * S.rs0) { mdl_finish(S, true, false); break; }
        if (S.it >= M.max_iter) { mdl_finish(S, false, false); break; }
        S.beta = rs_new / S.rs;
        S.rs = rs_new;
      } else {
        S.t = S.t_new;
        S.dw = sqrt(a[0]) / fmax(sqrt(a[1]), 1e-300);
        if (S.kind == MDL_FISTA_RIDGE) {
          S.gap = S.dw;  // reported: last relative update
          if (S.dw <= 1e-7 && S.it > 10) mdl_finish(S, true, false);
          else if (S.it >= M.max_iter) mdl_finish(S, false, false);
        } else if (S.it >= M.max_iter && S.it % 10 != 0) mdl_finish(S, false, a[2] == 0.0);
      }
      break;
    case MS_GAP: {  // scikit-learn's duality gap (_enet_gap): a[7] dual norm, a[0] w.w, a[1] |w|_1, acc[2..4] of the rows
      const double dual = a[7], w2 = a[0], l1 = a[1];
      const double R2 = S.acc[3], Ry = S.acc[4];
      double cst, gap;
      if (dual > S.alpha_s) { cst = S.alpha_s / dual; gap = 0.5 * (R2 + R2 * cst * cst); }
      else { cst = 1.0; gap = R2; }
      gap += S.alpha_s * l1 - cst * Ry + 0.5 * S.beta_s * (1 + cst * cst) * w2;
      S.gap = gap;
      if (gap <= S.tol_gap) mdl_finish(S, true, l1 == 0.0);
      else if (S.it >= M.max_iter) mdl_finish(S, false, l1 == 0.0);
      break;
    }
  }
}

// one CTA per candidate: combine the nslots partials of the slots in mask in a fixed order, then decide.  keep_rows:
// the gap's row partials (R.R, R.y_c) are kept in acc[3], acc[4] for the n-space half of the gap.
__global__ void __launch_bounds__(HB2_BLOCK) k_mdl_reduce(MD M, int nslots, unsigned mask, int op, int it_global, int gate) {
  const int c = blockIdx.x;
  __shared__ double shd[TRF_NRED][HB2_BLOCK / 32];
  ModelState& S = M.st[c];
  if (!mdl_pass_active(S, gate)) return;
  double v[TRF_NRED];
#pragma unroll
  for (int k = 0; k < TRF_NRED; ++k) v[k] = trf_identity(k);
  for (int s2 = threadIdx.x; s2 < nslots; s2 += HB2_BLOCK) {
    const double* p = M.red + ((size_t)c * M.slots + s2) * TRF_NRED;
#pragma unroll
    for (int k = 0; k < TRF_NRED; ++k)
      if (mask >> k & 1u) v[k] = trf_combine(k, v[k], p[k]);
  }
  trf_block_reduce(v, mask, shd);
  if (threadIdx.x == 0) {
    if (gate == MM_GAPROW) {  // keep sum R, R.R, R.y_c for MS_GAP
      S.sr = v[0]; S.acc[3] = v[1]; S.acc[4] = v[2];
      return;
    }
#pragma unroll
    for (int k = 0; k < 5; ++k)
      if (mask >> k & 1u) S.acc[k] = v[k];
    if (mask >> 7 & 1u) S.acc[7] = v[7];
    mdl_scalar(M, S, op, it_global);
  }
}

// candidates still iterating or waiting for a refit
__global__ void k_mdl_count(const ModelState* __restrict__ st, int nc, int* __restrict__ nactive) {
  __shared__ int n;
  if (threadIdx.x == 0) n = 0;
  __syncthreads();
  for (int c = threadIdx.x; c < nc; c += blockDim.x)
    if (!st[c].stop) atomicAdd(&n, 1);
  __syncthreads();
  if (threadIdx.x == 0) *nactive = n;
}

// the model's iteration count where the score map and the results read LSMR's
__global__ void k_mdl_publish(BD B, const ModelState* __restrict__ st) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < B.nc) { B.st[c].itn = st[c].it; B.st[c].istop = 0; }
}
