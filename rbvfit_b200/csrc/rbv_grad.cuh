// rbvfit_b200 -- analytic gradient of lnprob / lnlike: one forward pass + one adjoint pass per walker (sm_100a).
//
// Notation of rbv_device.cuh: u_p = 1/lambda_p, x_lp = A_l u_p - B_l, S_l = ((N f) K) the line's optical-depth scale
// (LC_COEF), tau_p = sum_l S_l H(a_l, x_lp), F = exp(-tau), M = taps * F (true convolution, edges replicated),
// lnL = -1/2 sum_p [(D_p - M_p)^2 w_p - log w_p].  Adjoint (DESIGN.md section 14):
//   r_p = (D_p - M_p) w_p,   s_q = sum_p r_p dM_p/dF_q (transposed convolution: clamped taps pile up on 0 and P-1),
//   g_q = -F_q s_q = dlnL/dtau_q,
//   per line: T_N = sum_q g_q H,  T_b = sum_q g_q (H + x H_x + a H_a),  T_v = sum_q g_q u_q H_x
//   dlnL/dlogN_c += ln(10) S_l T_N,  dlnL/db_c += -(S_l / b_c) T_b,  dlnL/dv_c += S_l A_l T_v / (c_kms + v_c).
// H + x H_x + a H_a vanishes at leading order in the far wing (tau there does not depend on b); every tier forms it
// per pixel from its own expansion, so nothing cancels in the sums.
//
// Launches per call (all FP64, every (line, pixel) pair evaluated directly -- no far-field interpolant):
//   grad_prep_kernel     (walker, 128 lines)   prior flag + the line-constant record of prep_kernel
//   grad_flux_kernel     (256 px, walker)      tau -> F
//   grad_resid_kernel    (256 px, walker)      M = taps * F, r, chi^2 partial of the block
//   grad_adjoint_kernel  (256 px, walker)      s = taps^T r, g = -F s
//   grad_line_kernel     (1024 px, walker)     H, H_x, H + x H_x + a H_a per (line, pixel) -> per-tile line sums
//   grad_finalize_kernel (warp per walker)     fixed-order sums over blocks, tiles, lines and instruments
// Every reduction runs in an order fixed by the instrument geometry alone: a row's value and gradient do not depend
// on the batch size or on the position of the row in the batch.
// The launches with the walker in grid y (flux, resid, adjoint, line) go over the batch in slices of at most 65 535
// rows, the CUDA limit of gridDim.y / gridDim.z: row GradParams::w0 + blockIdx.y of the full-size buffers.
#pragma once

namespace rbv {

constexpr double kLn10 = 2.3025850929940456840;
constexpr int kGradBlock = 256;                 // pixels per block of the per-pixel passes
constexpr int kGradPPT = 4;                     // pixels per thread of the line pass
constexpr int kGradTile = kGradBlock * kGradPPT;
constexpr int kGradLineChunk = 32;              // lines whose series coefficients sit in shared memory at once
// terms of the rho-series derivatives beyond kDFar.  E = H + x H_x + a H_a starts at rho^2 (its p = 1 terms cancel),
// so its truncation after NQ terms is ~rho^(NQ - 1) relative: kNQFar = 3 (enough for H, 2e-13) leaves E off by up to
// 1.6e-8 at |z|^2 = 4e4, 5 terms by 4e-16
constexpr int kNQFarGrad = 5;

struct GradInst {
  int blk_off;        // first 256-pixel block of the instrument (pixel buffers are padded to whole blocks)
  int n_blk;
  int tile_off;       // first 1024-pixel tile of the line pass
  int n_tiles;
  long long part_off; // first double of the instrument in a walker's line partials [tile][line][3]
  const double* cum_lo;   // [K] cum_lo[j] = sum_{m <= j} taps_rev[m]
  const double* cum_hi;   // [K] cum_hi[j] = sum_{m >= j} taps_rev[m]
};

struct GradParams {
  const InstDev* inst;
  GradInst gi[kMaxInst];
  const double* theta;
  const double* lb;       // NULL: no prior (lnlike)
  const double* ub;
  const double* core_tab;
  double* value;          // [W]
  double* grad;           // [W, ndim]
  int* oob;               // [W]
  double* lc;             // [W, n_lines_total, LC_STRIDE]
  double* F;              // [W, n_blk_total * 256]
  double* r;
  double* g;
  double* pval;           // [W, n_blk_total]
  double* pline;          // [W, part_stride]
  double* linegrad;       // [W, n_lines_total, 3]
  long long part_stride;
  int W, ndim, n_inst, n_lines_total, n_blk_total, n_tiles_total;
  int w0;                 // first row of a launch with the row in grid y / z (a slice of at most 65 535 rows)
};

// Survey mode of the forward and Fisher kernels (template parameter SL): row w is evaluated against instrument
// inst0 + w / wps alone, with the geometry of one instrument (gi[0], n_inst = 1, its lines at lc offset 0), so every
// buffer and grid is sized for one sightline whatever the number of sightlines.  The per-instrument tables that the
// joint fit passes as kernel parameters (at most kMaxInst) come from device arrays indexed by instrument.
struct SlRows {
  int wps;                  // rows per sightline
  int inst0;                // instrument of row 0
  const int* active;        // [W] or NULL: a row with active[w] == 0 returns at kernel entry
  const int* const* order;  // [n_inst] FisherParams::order of each instrument
  const int* has_lsf;       // [n_inst] FisherParams::has_lsf of each instrument
};

template <bool SL>
__device__ __forceinline__ bool sl_skip(const SlRows& sl, int w) {
  return SL && sl.active != nullptr && !sl.active[w];
}
// instrument of row w; k is the joint fit's instrument (from the block / tile / line index)
template <bool SL>
__device__ __forceinline__ int sl_inst(const SlRows& sl, int w, int k) {
  return SL ? sl.inst0 + w / sl.wps : k;
}

// ------------------------------------------------------------------------------------------ H and its derivatives
// q_p(a^2) and dq_p/d(a^2), p = 1..kNQNear, unscaled (kappa = 1)
__device__ __forceinline__ void asym_coef_grad(double a2, double* q, double* qd) {
#pragma unroll
  for (int p = 1; p <= kNQNear; ++p) {
    const double* row = c_ctab + p * (RBV_ASYM_MMAX + 1);
    double v = row[RBV_ASYM_MMAX], dv = RBV_ASYM_MMAX * row[RBV_ASYM_MMAX];
#pragma unroll
    for (int m = RBV_ASYM_MMAX - 1; m >= 0; --m) {
      v = fma(v, a2, row[m]);
      if (m > 0) dv = fma(dv, a2, m * row[m]);
    }
    q[p - 1] = v;
    qd[p - 1] = dv;
  }
}

struct HGrad {
  double H, Hx, Ha, E;   // E = H + x H_x + a H_a
};

// rho-series tier (a <= kABig, |z|^2 >= 64): H = (a/sqrt(pi)) sum_p q_p rho^p, differentiated term by term:
//   H_x = -2 x rho (a/sqrt(pi)) sum_p p q_p rho^p
//   H_a = (1/sqrt(pi)) sum_p q_p rho^p + (2 a^2/sqrt(pi)) sum_p (q_p' rho^p - p q_p rho^(p+1))
//   E   = (2a/sqrt(pi)) [sum_{p>=2} (1 - p) q_p rho^p + a^2 sum_p q_p' rho^p]       (the p = 1 terms cancel exactly)
template <int NQ>
__device__ __forceinline__ HGrad series_grad(double x, double a, double a2, double d, const double* q,
                                             const double* qd) {
  const double rho = rcp_pos(d);
  double s0 = q[NQ - 1], s1 = NQ * q[NQ - 1], sE = (1 - NQ) * q[NQ - 1], sd = qd[NQ - 1];
#pragma unroll
  for (int p = NQ - 1; p >= 1; --p) {
    s0 = fma(s0, rho, q[p - 1]);
    s1 = fma(s1, rho, p * q[p - 1]);
    sE = fma(sE, rho, (1 - p) * q[p - 1]);
    sd = fma(sd, rho, qd[p - 1]);
  }
  s0 *= rho;
  s1 *= rho;
  sE *= rho;
  sd *= rho;
  const double k = a * kInvSqrtPi;
  HGrad h;
  h.H = k * s0;
  h.Hx = -2.0 * x * rho * k * s1;
  h.Ha = kInvSqrtPi * fma(2.0 * a2, fma(-rho, s1, sd), s0);
  h.E = 2.0 * k * fma(a2, sd, sE);
  return h;
}

// complex asymptotic tier (a > kABig, |z|^2 >= 64): w = (i/sqrt(pi)) sum_k c_k zeta^(2k+1), zeta = 1/z;
//   w' = -(i/sqrt(pi)) zeta^2 sum_k (2k+1) c_k zeta^(2k),   w + z w' = (i/sqrt(pi)) zeta sum_k (-2k) c_k zeta^(2k)
__device__ __noinline__ HGrad asym_complex_grad(double x, double a, double d) {
  const double rho = 1.0 / d;
  const double rr = x * rho, ri = -a * rho;                    // zeta
  const double sr = fma(rr, rr, -ri * ri), si = 2.0 * rr * ri; // zeta^2
  double c[13];
  c[0] = 1.0;
#pragma unroll
  for (int k = 1; k <= 12; ++k) c[k] = c[k - 1] * (2 * k - 1) * 0.5;
  double S0r = c[12], S0i = 0.0, S1r = 25.0 * c[12], S1i = 0.0, S2r = -24.0 * c[12], S2i = 0.0;
#pragma unroll
  for (int k = 11; k >= 0; --k) {
    double tr = fma(S0r, sr, fma(-S0i, si, c[k])), ti = fma(S0r, si, S0i * sr);
    S0r = tr;
    S0i = ti;
    tr = fma(S1r, sr, fma(-S1i, si, (2 * k + 1) * c[k]));
    ti = fma(S1r, si, S1i * sr);
    S1r = tr;
    S1i = ti;
    tr = fma(S2r, sr, fma(-S2i, si, (-2 * k) * c[k]));
    ti = fma(S2r, si, S2i * sr);
    S2r = tr;
    S2i = ti;
  }
  const double P1r = fma(sr, S1r, -si * S1i), P1i = fma(sr, S1i, si * S1r);   // zeta^2 S1
  HGrad h;
  h.H = -kInvSqrtPi * fma(rr, S0i, ri * S0r);
  h.Hx = kInvSqrtPi * P1i;
  h.Ha = kInvSqrtPi * P1r;
  h.E = -kInvSqrtPi * fma(rr, S2i, ri * S2r);
  return h;
}

// Weideman N = 40 in complex form (a > kAFast, |z|^2 < 64): w, then w' = -2 z w + 2i/sqrt(pi) (|z| < 8: no
// cancellation worth the name)
__device__ __noinline__ HGrad weideman_grad(double x, double a) {
  const double L = RBV_WEID_L;
  const double dr = L + a, di = -x;   // L - i z
  const double nr = L - a, ni = x;    // L + i z
  const double inv = 1.0 / fma(dr, dr, di * di);
  const double Zr = fma(nr, dr, ni * di) * inv;
  const double Zi = fma(ni, dr, -nr * di) * inv;
  double pr = c_weid[0], pi = 0.0;
#pragma unroll 4
  for (int k = 1; k < RBV_WEID_N; ++k) {
    const double tr = fma(pr, Zr, fma(-pi, Zi, c_weid[k]));
    const double ti = fma(pr, Zi, pi * Zr);
    pr = tr;
    pi = ti;
  }
  const double ir = dr * inv, ii = -di * inv;                 // 1/(L - i z)
  const double i2r = fma(ir, ir, -ii * ii), i2i = 2.0 * ir * ii;
  const double wr = fma(2.0, fma(pr, i2r, -pi * i2i), kInvSqrtPi * ir);
  const double wi = fma(2.0, fma(pr, i2i, pi * i2r), kInvSqrtPi * ii);
  const double dwr = -2.0 * fma(x, wr, -a * wi);
  const double dwi = fma(-2.0, fma(x, wi, a * wr), 2.0 * kInvSqrtPi);
  HGrad h;
  h.H = wr;
  h.Hx = dwr;
  h.Ha = -dwi;
  h.E = wr + fma(x, dwr, -a * dwi);
  return h;
}

// piecewise polynomial of the g_k table and its derivative in t
template <int DEG>
__device__ __forceinline__ void table_poly(const double* __restrict__ p, double t, double& v, double& dv) {
  v = __ldg(p + DEG * RBV_CORE_NINT);
  dv = 0.0;
#pragma unroll
  for (int k = DEG - 1; k >= 0; --k) {
    dv = fma(dv, t, v);
    v = fma(v, t, __ldg(p + k * RBV_CORE_NINT));
  }
}

// table tier (a <= kAFast, |z|^2 < 64): H = exp(a^2 - x^2) cos(2ax) + a G,  G = sum_k a^(2k) g_k(|x|)
__device__ __noinline__ HGrad table_grad(double x, double a, double a2, const double* __restrict__ tab) {
  const double ax = fabs(x);
  int j = (int)(ax * RBV_CORE_INV_H);
  j = max(0, min(j, RBV_CORE_NINT - 1));
  const double t = fma(ax, 2.0 * RBV_CORE_INV_H, -(double)(2 * j + 1));
  double g0, g1, g2, g3, d0, d1, d2, d3;
  table_poly<RBV_CORE_DEG0>(tab + RBV_CORE_OFF0 + j, t, g0, d0);
  table_poly<RBV_CORE_DEG1>(tab + RBV_CORE_OFF1 + j, t, g1, d1);
  table_poly<RBV_CORE_DEG2>(tab + RBV_CORE_OFF2 + j, t, g2, d2);
  table_poly<RBV_CORE_DEG3>(tab + RBV_CORE_OFF3 + j, t, g3, d3);
  const double G = fma(fma(fma(g3, a2, g2), a2, g1), a2, g0);
  const double dGdt = fma(fma(fma(d3, a2, d2), a2, d1), a2, d0);
  const double Gx = copysign(2.0 * RBV_CORE_INV_H, x) * dGdt;
  const double Ga2 = fma(fma(3.0 * g3, a2, 2.0 * g2), a2, g1);   // dG/d(a^2)
  const double E0 = exp_flux(fma(-x, x, a2));
  double sn, cs;
  sincos(2.0 * a * x, &sn, &cs);
  HGrad h;
  h.H = fma(E0, cs, a * G);
  h.Hx = fma(E0, -2.0 * fma(x, cs, a * sn), a * Gx);
  h.Ha = fma(E0, 2.0 * fma(a, cs, -x * sn), fma(2.0 * a2, Ga2, G));
  h.E = h.H + fma(x, h.Hx, a * h.Ha);
  return h;
}

// H, H_x, H_a, H + x H_x + a H_a with the tier chosen from |z|^2 = d as the lnprob kernels choose it.
// q, qd: q_p(a^2), q_p'(a^2) (asym_coef_grad) -- read only in the rho-series tier.
__device__ __forceinline__ HGrad voigt_hgrad(double x, double a, double a2, double d, const double* q,
                                             const double* qd, const double* __restrict__ tab) {
  if (a > kABig) return (d < kDCore) ? weideman_grad(x, a) : asym_complex_grad(x, a, d);
  if (d < kDCore) return (a <= kAFast) ? table_grad(x, a, a2, tab) : weideman_grad(x, a);
  if (d >= kDFar) return series_grad<kNQFarGrad>(x, a, a2, d, q, qd);
  if (d >= kDNear) return series_grad<kNQMid>(x, a, a2, d, q, qd);
  return series_grad<kNQNear>(x, a, a2, d, q, qd);
}

// ------------------------------------------------------------------------------------------ kernels
__device__ __forceinline__ int grad_inst_of_blk(const GradParams& prm, int blk) {
  int k = 0;
  while (k + 1 < prm.n_inst && blk >= prm.gi[k + 1].blk_off) ++k;
  return k;
}

// prior flag + per-line constants (the record prep_kernel writes: A, B, a^2, a, S, kappa-scaled series)
template <bool SL>
__global__ void __launch_bounds__(128) grad_prep_kernel(const GradParams prm, const SlRows sl) {
  const int w = blockIdx.x;
  if (sl_skip<SL>(sl, w)) return;
  const double* th = prm.theta + (size_t)w * prm.ndim;
  if (blockIdx.y == 0) {
    int bad = 0;
    if (prm.lb != nullptr)
      for (int i = threadIdx.x; i < prm.ndim; i += blockDim.x) bad |= (th[i] < prm.lb[i]) || (th[i] > prm.ub[i]);
    bad = __syncthreads_or(bad);
    if (threadIdx.x == 0) prm.oob[w] = bad;
  }
  const int gl = blockIdx.y * blockDim.x + threadIdx.x;
  if (gl >= prm.n_lines_total) return;
  int k = 0;
  if (SL) k = sl_inst<SL>(sl, w, 0);
  else while (k + 1 < prm.n_inst && gl >= prm.inst[k + 1].line_base) ++k;
  const InstDev& I = prm.inst[k];
  double lc[LC_STRIDE];
  prep_line_wofz(I, SL ? gl : gl - I.line_base, th, lc);
#pragma unroll
  for (int p = 0; p < kNQNear; ++p) lc[LC_Q + p] = asym_coef(p + 1, lc[LC_A2], lc[LC_AUX]);
  double* dst = prm.lc + ((size_t)w * prm.n_lines_total + gl) * LC_STRIDE;
#pragma unroll
  for (int i = 0; i < LC_STRIDE; ++i) dst[i] = lc[i];
}

// tau over every line, directly, then F = exp(-tau)
template <bool SL>
__global__ void __launch_bounds__(kGradBlock) grad_flux_kernel(const GradParams prm, const SlRows sl) {
  const int w = prm.w0 + blockIdx.y;
  if (sl_skip<SL>(sl, w)) return;
  if (prm.oob[w]) return;
  const int k = SL ? 0 : grad_inst_of_blk(prm, blockIdx.x);
  const InstDev& I = prm.inst[sl_inst<SL>(sl, w, k)];
  const int p = (blockIdx.x - prm.gi[k].blk_off) * kGradBlock + threadIdx.x;
  if (p >= I.P) return;
  const double u = __ldg(I.inv_wave + p);
  const double* lcw = prm.lc + ((size_t)w * prm.n_lines_total + (SL ? 0 : I.line_base)) * LC_STRIDE;
  double tau = 0.0;
  for (int l = 0; l < I.L; ++l) {
    const double* lc = lcw + l * LC_STRIDE;
    const double A = lc[LC_A], B = lc[LC_B], a2 = lc[LC_A2], a = lc[LC_a];
    const double x = fma(A, u, -B);
    const double d = fma(x, x, a2);
    if (a > kABig) tau = fma(lc[LC_COEF], general_H(x, a, d), tau);
    else if (d < kDCore) tau = fma(lc[LC_COEF], core_H(x, a, a2, prm.core_tab), tau);
    else if (d >= kDFar) tau += asym_series<kNQFar>(lc + LC_Q, d);
    else if (d >= kDNear) tau += asym_series<kNQMid>(lc + LC_Q, d);
    else tau += asym_series<kNQNear>(lc + LC_Q, d);
  }
  prm.F[(size_t)w * prm.n_blk_total * kGradBlock + (size_t)blockIdx.x * kGradBlock + threadIdx.x] = exp_flux(-tau);
}

// M_p = sum_m taps_rev[m] F[clamp(p - h + m)], r_p = (D_p - M_p) w_p, chi^2 partial of the block
template <bool SL>
__global__ void __launch_bounds__(kGradBlock) grad_resid_kernel(const GradParams prm, const SlRows sl) {
  __shared__ double s_red[kGradBlock / 32];
  const int w = prm.w0 + blockIdx.y;
  if (sl_skip<SL>(sl, w)) return;
  if (prm.oob[w]) return;
  const int k = SL ? 0 : grad_inst_of_blk(prm, blockIdx.x);
  const InstDev& I = prm.inst[sl_inst<SL>(sl, w, k)];
  const int p = (blockIdx.x - prm.gi[k].blk_off) * kGradBlock + threadIdx.x;
  const size_t base = (size_t)w * prm.n_blk_total * kGradBlock + (size_t)prm.gi[k].blk_off * kGradBlock;
  double part = 0.0;
  if (p < I.P) {
    const double* F = prm.F + base;
    const int h = I.K >> 1;
    double M = 0.0;
    for (int m = 0; m < I.K; ++m) M = fma(__ldg(I.taps_rev + m), F[min(max(p - h + m, 0), I.P - 1)], M);
    const double wgt = __ldg(I.inv_sigma2 + p);
    const double resid = __ldg(I.flux + p) - M;
    prm.r[base + p] = resid * wgt;
    part = resid * resid * wgt;
  }
  part = warp_sum(part);
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = part;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < kGradBlock / 32; ++i) s += s_red[i];
    prm.pval[(size_t)w * prm.n_blk_total + blockIdx.x] = s;
  }
}

// s_q = sum_p r_p dM_p/dF_q, g_q = -F_q s_q.  Interior q: the taps that land on q exactly; q = 0 and q = P - 1 also
// collect every tap that the edge replication clamps onto them (prefix / suffix sums of the taps).
__global__ void __launch_bounds__(kGradBlock) grad_adjoint_kernel(const GradParams prm) {
  const int w = prm.w0 + blockIdx.y;
  if (prm.oob[w]) return;
  const int k = grad_inst_of_blk(prm, blockIdx.x);
  const InstDev& I = prm.inst[k];
  const GradInst& gi = prm.gi[k];
  const int q = (blockIdx.x - gi.blk_off) * kGradBlock + threadIdx.x;
  if (q >= I.P) return;
  const size_t base = (size_t)w * prm.n_blk_total * kGradBlock + (size_t)gi.blk_off * kGradBlock;
  const double* r = prm.r + base;
  const int P = I.P, K = I.K, h = K >> 1;
  double s = 0.0;
  if (P == 1) {
    s = r[0] * gi.cum_lo[K - 1];
  } else if (q == 0) {
    for (int p = 0; p <= min(h, P - 1); ++p) s = fma(r[p], gi.cum_lo[h - p], s);
  } else if (q == P - 1) {
    for (int p = max(0, P - 1 - h); p <= P - 1; ++p) s = fma(r[p], gi.cum_hi[P - 1 - p + h], s);
  } else {
    const int m_lo = max(0, q + h - (P - 1)), m_hi = min(K - 1, q + h);
    for (int m = m_lo; m <= m_hi; ++m) s = fma(__ldg(I.taps_rev + m), r[q + h - m], s);
  }
  prm.g[base + q] = -prm.F[base + q] * s;
}

// per (line, tile): T_N, T_b, T_v over the tile's pixels -> pline[w, part_off + (tile * L + line) * 3 + c]
__global__ void __launch_bounds__(kGradBlock) grad_line_kernel(const GradParams prm) {
  __shared__ double s_q[kGradLineChunk][2][kNQNear];
  __shared__ double s_part[kGradLineChunk][kGradBlock / 32][3];
  const int w = prm.w0 + blockIdx.y;
  if (prm.oob[w]) return;
  int k = 0;
  while (k + 1 < prm.n_inst && (int)blockIdx.x >= prm.gi[k + 1].tile_off) ++k;
  const InstDev& I = prm.inst[k];
  const GradInst& gi = prm.gi[k];
  const int tile = blockIdx.x - gi.tile_off;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t base = (size_t)w * prm.n_blk_total * kGradBlock + (size_t)gi.blk_off * kGradBlock;
  double u[kGradPPT], gq[kGradPPT];
  bool valid[kGradPPT];
#pragma unroll
  for (int j = 0; j < kGradPPT; ++j) {
    const int p = tile * kGradTile + j * kGradBlock + tid;
    valid[j] = p < I.P;
    u[j] = valid[j] ? __ldg(I.inv_wave + p) : 0.0;
    gq[j] = valid[j] ? prm.g[base + p] : 0.0;
  }
  const double* lcw = prm.lc + ((size_t)w * prm.n_lines_total + I.line_base) * LC_STRIDE;
  double* out = prm.pline + (size_t)w * prm.part_stride + gi.part_off + (size_t)tile * I.L * 3;
  for (int l0 = 0; l0 < I.L; l0 += kGradLineChunk) {
    const int nl = min(kGradLineChunk, I.L - l0);
    for (int ll = tid; ll < nl; ll += kGradBlock) asym_coef_grad(lcw[(l0 + ll) * LC_STRIDE + LC_A2], s_q[ll][0], s_q[ll][1]);
    __syncthreads();
    for (int ll = 0; ll < nl; ++ll) {
      const double* lc = lcw + (l0 + ll) * LC_STRIDE;
      const double A = lc[LC_A], B = lc[LC_B], a2 = lc[LC_A2], a = lc[LC_a];
      double tN = 0.0, tb = 0.0, tv = 0.0;
#pragma unroll
      for (int j = 0; j < kGradPPT; ++j) {
        if (!valid[j]) continue;
        const double x = fma(A, u[j], -B);
        const HGrad hg = voigt_hgrad(x, a, a2, fma(x, x, a2), s_q[ll][0], s_q[ll][1], prm.core_tab);
        tN = fma(gq[j], hg.H, tN);
        tb = fma(gq[j], hg.E, tb);
        tv = fma(gq[j] * u[j], hg.Hx, tv);
      }
      tN = warp_sum(tN);
      tb = warp_sum(tb);
      tv = warp_sum(tv);
      if (lane == 0) {
        s_part[ll][warp][0] = tN;
        s_part[ll][warp][1] = tb;
        s_part[ll][warp][2] = tv;
      }
    }
    __syncthreads();
    for (int i = tid; i < nl * 3; i += kGradBlock) {
      const int ll = i / 3, c = i - 3 * ll;
      double s = 0.0;
#pragma unroll
      for (int wp = 0; wp < kGradBlock / 32; ++wp) s += s_part[ll][wp][c];
      out[(l0 + ll) * 3 + c] = s;
    }
    __syncthreads();
  }
}

// one warp per walker: value = sum over instruments of -1/2 (chi^2 - sum log w), gradient folded line -> component
__global__ void __launch_bounds__(128) grad_finalize_kernel(const GradParams prm) {
  const int w = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (w >= prm.W) return;
  double* row = prm.grad + (size_t)w * prm.ndim;
  for (int i = lane; i < prm.ndim; i += 32) row[i] = 0.0;
  if (prm.oob[w]) {
    if (lane == 0) prm.value[w] = -CUDART_INF;                   // vfit_mcmc.py:350-352; flat prior: zero gradient
    return;
  }
  const double* th = prm.theta + (size_t)w * prm.ndim;
  double total = 0.0;
  for (int k = 0; k < prm.n_inst; ++k) {
    const InstDev& I = prm.inst[k];
    const GradInst& gi = prm.gi[k];
    double s = 0.0;
    const double* pv = prm.pval + (size_t)w * prm.n_blk_total + gi.blk_off;
    for (int t0 = 0; t0 < gi.n_blk; t0 += 32) {
      const double v = (t0 + lane < gi.n_blk) ? pv[t0 + lane] : 0.0;
      const int m = min(32, gi.n_blk - t0);
      for (int t = 0; t < m; ++t) s += __shfl_sync(0xffffffffu, v, t);
    }
    total += -0.5 * (s - I.sum_log_inv_sigma2);
    const double* pl = prm.pline + (size_t)w * prm.part_stride + gi.part_off;
    const double* lcw = prm.lc + ((size_t)w * prm.n_lines_total + I.line_base) * LC_STRIDE;
    double* lg = prm.linegrad + ((size_t)w * prm.n_lines_total + I.line_base) * 3;
    __syncwarp();
    for (int l = lane; l < I.L; l += 32) {
      double T0 = 0.0, T1 = 0.0, T2 = 0.0;
      for (int t = 0; t < gi.n_tiles; ++t) {
        const double* e = pl + ((size_t)t * I.L + l) * 3;
        T0 += e[0];
        T1 += e[1];
        T2 += e[2];
      }
      const int c = I.comp[l];
      const double S = lcw[l * LC_STRIDE + LC_COEF], A = lcw[l * LC_STRIDE + LC_A];
      const double b = th[I.C + c], v = th[2 * I.C + c];
      lg[l * 3 + 0] = kLn10 * S * T0;
      lg[l * 3 + 1] = -(S / b) * T1;
      lg[l * 3 + 2] = S * A * T2 / (kCkms + v);
    }
    __syncwarp();
    for (int c = lane; c < I.C; c += 32) {
      double gN = 0.0, gb = 0.0, gv = 0.0;
      for (int l = 0; l < I.L; ++l) {
        if (I.comp[l] != c) continue;
        gN += lg[l * 3 + 0];
        gb += lg[l * 3 + 1];
        gv += lg[l * 3 + 2];
      }
      row[c] += gN;
      row[I.C + c] += gb;
      row[2 * I.C + c] += gv;
    }
    __syncwarp();
  }
  if (lane == 0) prm.value[w] = total;
}

// test hook: H, H_x, H_a on a lattice through voigt_hgrad
__global__ void voigt_h_grad_kernel(const double* __restrict__ x, const double* __restrict__ a, double* __restrict__ H,
                                    double* __restrict__ Hx, double* __restrict__ Ha, int n,
                                    const double* __restrict__ core_tab) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double xv = x[i], av = a[i], a2 = av * av;
  double q[kNQNear], qd[kNQNear];
  asym_coef_grad(a2, q, qd);
  const HGrad h = voigt_hgrad(xv, av, a2, fma(xv, xv, a2), q, qd, core_tab);
  H[i] = h.H;
  Hx[i] = h.Hx;
  Ha[i] = h.Ha;
}

}  // namespace rbv
