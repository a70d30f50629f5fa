// rbvfit_b200 -- model Jacobian and Gauss-Newton (Fisher) matrix of lnlike, forward mode per parameter column
// (sm_100a).
//
// Notation of rbv_grad.cuh (DESIGN.md sections 14, 15).  For instrument k and one walker:
//   dtau_q/dlogN_c = ln(10) sum_{l in c} S_l H,   dtau_q/db_c = -(1/b_c) sum_{l in c} S_l E,
//   dtau_q/dv_c    = u_q sum_{l in c} S_l A_l H_x / (c_kms + v_c),     E = H + x H_x + a H_a (voigt_hgrad)
//   JF[col, q] = dF_q/dtheta_col = -F_q dtau_q/dtheta_col
//   JM[col, p] = sum_m taps_rev[m] JF[col, clamp(p - h + m)]    (the M = taps * F of grad_resid_kernel)
//   fisher_ij = sum_k sum_p w_p JM_ip JM_jp,   grad_i = sum_k sum_p r_p JM_ip,   r_p = (D_p - M_p) w_p
// The value is -1/2 (sum chi^2 - sum log w), formed exactly as grad_finalize_kernel forms it.
//
// Launches per call (all FP64, every (line, pixel) pair evaluated directly -- no far-field interpolant):
//   grad_prep_kernel, grad_flux_kernel, grad_resid_kernel   (rbv_grad.cuh, unchanged; resid only for lnlike)
//   fisher_col_kernel      (256 px, walker)        JF: every column once, lines walked in component order
//   fisher_lsf_kernel      (256 px, column, walker) JM; launched only when some instrument has an LSF
//   fisher_gram_kernel     (1024 px, walker)       per-tile partials of the upper triangle and of J^T r
//   fisher_finalize_kernel (warp per walker)       fixed-order sums over tiles and instruments, mirrored triangle
//   fisher_jac_out_kernel  (256 px, row, walker)   rbv_model_jacobian_batch only: [W, ndim, P] out of JM / JF
// Every reduction runs in an order fixed by the instrument geometry alone (no atomics): a row's results do not
// depend on the batch size or on the position of the row in the batch.
// The launches with the walker in grid y or z go over the batch in slices of at most 65 535 rows (the CUDA limit of
// gridDim.y / gridDim.z): row gp.w0 + blockIdx.y (.z) of the full-size buffers, as in rbv_grad.cuh.
// Survey mode (SL = true, SlRows of rbv_grad.cuh): the same kernels with the geometry of one sightline and the
// row's own instrument, so a row gives bit for bit what a one-instrument context of that sightline gives.
#pragma once

namespace rbv {

constexpr int kFisherChunk = 32;   // pixels of the Gram pass staged in shared memory at once

struct FisherParams {
  GradParams gp;                 // the forward pass and its buffers (lc, F, r, pval)
  const int* order[kMaxInst];    // [L] lines of instrument k sorted by component (stable)
  int has_lsf[kMaxInst];         // 0: the instrument has no LSF (JM is JF)
  int ncol;                      // 3 * n_components: columns of J; theta indices beyond are 0
  int npart;                     // ncol (ncol + 1) / 2 triangle entries + ncol entries of J^T r
  long long col_stride;          // doubles per column: n_blk_total * 256
  double* JF;                    // [W, ncol, col_stride]
  double* JM;                    // [W, ncol, col_stride]
  double* pgram;                 // [W, n_tiles_total, npart]
  double* fisher;                // [W, ndim, ndim]
  double* jac;                   // rbv_model_jacobian_batch: [W, ndim, P of jac_inst]
  int jac_inst;
};

// instrument of a 1024-pixel tile (the Gram pass); grad_inst_of_blk is its 256-pixel-block twin
__device__ __forceinline__ int grad_inst_of_tile(const GradParams& prm, int tile) {
  int k = 0;
  while (k + 1 < prm.n_inst && tile >= prm.gi[k + 1].tile_off) ++k;
  return k;
}

// JF (or JM) column `col` of walker w, at the first pixel of instrument k
__device__ __forceinline__ size_t fisher_col_base(const FisherParams& fp, int w, int col, int k) {
  return ((size_t)w * fp.ncol + col) * fp.col_stride + (size_t)fp.gp.gi[k].blk_off * kGradBlock;
}

// upper-triangle entry e (row-major, i <= j) -> (i, j)
__device__ __forceinline__ void fisher_tri(int e, int n, int& i, int& j) {
  i = 0;
  while (e >= n - i) {
    e -= n - i;
    ++i;
  }
  j = i + e;
}

// the three columns of component c at one pixel from the line sums sN = sum S H, sE = sum S E, sX = sum S A H_x
__device__ __forceinline__ void fisher_store(double* jf, long long stride, int C, int c, const double* th, double mF,
                                             double u, double sN, double sE, double sX) {
  jf[(size_t)c * stride] = mF * (kLn10 * sN);
  jf[(size_t)(C + c) * stride] = mF * (-sE / th[C + c]);
  jf[(size_t)(2 * C + c) * stride] = mF * (u * sX / (kCkms + th[2 * C + c]));
}

template <bool SL>
__global__ void __launch_bounds__(kGradBlock) fisher_col_kernel(const FisherParams fp, const SlRows sl) {
  __shared__ double s_q[kGradLineChunk][2][kNQNear];
  const GradParams& prm = fp.gp;
  const int w = prm.w0 + blockIdx.y, tid = threadIdx.x;
  if (sl_skip<SL>(sl, w)) return;
  const int k = SL ? 0 : grad_inst_of_blk(prm, blockIdx.x);
  const int ki = sl_inst<SL>(sl, w, k);
  const InstDev& I = prm.inst[ki];
  const int p = (blockIdx.x - prm.gi[k].blk_off) * kGradBlock + tid;
  const bool valid = p < I.P;
  const size_t pix = (size_t)blockIdx.x * kGradBlock + tid;
  const double u = valid ? __ldg(I.inv_wave + p) : 0.0;
  const double mF = valid ? -prm.F[(size_t)w * fp.col_stride + pix] : 0.0;
  double* jf = fp.JF + (size_t)w * fp.ncol * fp.col_stride + pix;
  const double* th = prm.theta + (size_t)w * prm.ndim;
  const double* lcw = prm.lc + ((size_t)w * prm.n_lines_total + (SL ? 0 : I.line_base)) * LC_STRIDE;
  const int* ord = SL ? sl.order[ki] : fp.order[k];
  int c = 0;
  double sN = 0.0, sE = 0.0, sX = 0.0;
  for (int l0 = 0; l0 < I.L; l0 += kGradLineChunk) {
    const int nl = min(kGradLineChunk, I.L - l0);
    for (int ll = tid; ll < nl; ll += kGradBlock)
      asym_coef_grad(lcw[ord[l0 + ll] * LC_STRIDE + LC_A2], s_q[ll][0], s_q[ll][1]);
    __syncthreads();
    for (int ll = 0; ll < nl; ++ll) {
      const int l = ord[l0 + ll], cl = I.comp[l];
      for (; c < cl; ++c) {   // lines are in component order: component c is complete
        if (valid) fisher_store(jf, fp.col_stride, I.C, c, th, mF, u, sN, sE, sX);
        sN = sE = sX = 0.0;
      }
      if (!valid) continue;
      const double* lc = lcw + l * LC_STRIDE;
      const double A = lc[LC_A], B = lc[LC_B], a2 = lc[LC_A2], a = lc[LC_a], S = lc[LC_COEF];
      const double x = fma(A, u, -B);
      const HGrad hg = voigt_hgrad(x, a, a2, fma(x, x, a2), s_q[ll][0], s_q[ll][1], prm.core_tab);
      sN = fma(S, hg.H, sN);
      sE = fma(S, hg.E, sE);
      sX = fma(S * A, hg.Hx, sX);
    }
    __syncthreads();
  }
  if (!valid) return;
  for (; c < I.C; ++c) {
    fisher_store(jf, fp.col_stride, I.C, c, th, mF, u, sN, sE, sX);
    sN = sE = sX = 0.0;
  }
  for (int col = 3 * I.C; col < fp.ncol; ++col) jf[(size_t)col * fp.col_stride] = 0.0;
}

// JM = taps * JF per column, the expression grad_resid_kernel forms M with
template <bool SL>
__global__ void __launch_bounds__(kGradBlock) fisher_lsf_kernel(const FisherParams fp, const SlRows sl) {
  const GradParams& prm = fp.gp;
  const int w = prm.w0 + blockIdx.z, col = blockIdx.y;
  if (sl_skip<SL>(sl, w)) return;
  const int k = SL ? 0 : grad_inst_of_blk(prm, blockIdx.x);
  const int ki = sl_inst<SL>(sl, w, k);
  if (!(SL ? sl.has_lsf[ki] : fp.has_lsf[k])) return;
  const InstDev& I = prm.inst[ki];
  const int p = (blockIdx.x - prm.gi[k].blk_off) * kGradBlock + threadIdx.x;
  if (p >= I.P) return;
  const size_t base = fisher_col_base(fp, w, col, k);
  const double* J = fp.JF + base;
  const int h = I.K >> 1;
  double M = 0.0;
  for (int m = 0; m < I.K; ++m) M = fma(__ldg(I.taps_rev + m), J[min(max(p - h + m, 0), I.P - 1)], M);
  fp.JM[base + p] = M;
}

// per 1024-pixel tile: sum_p w_p J_i J_j (i <= j) and sum_p r_p J_i, pixels in ascending order
template <bool SL>
__global__ void __launch_bounds__(kGradBlock) fisher_gram_kernel(const FisherParams fp, const SlRows sl) {
  extern __shared__ double s_j[];   // [ncol][kFisherChunk] columns, then weights, then residuals
  const GradParams& prm = fp.gp;
  const int w = prm.w0 + blockIdx.y, tid = threadIdx.x;
  if (sl_skip<SL>(sl, w)) return;
  const int k = SL ? 0 : grad_inst_of_tile(prm, blockIdx.x);
  const int ki = sl_inst<SL>(sl, w, k);
  const InstDev& I = prm.inst[ki];
  const int p0 = (blockIdx.x - prm.gi[k].tile_off) * kGradTile;
  const int np = min(kGradTile, I.P - p0);
  const int ncol = fp.ncol, ntri = ncol * (ncol + 1) / 2;
  const double* J = ((SL ? sl.has_lsf[ki] : fp.has_lsf[k]) ? fp.JM : fp.JF) + fisher_col_base(fp, w, 0, k) + p0;
  const double* r = prm.r + (size_t)w * fp.col_stride + (size_t)prm.gi[k].blk_off * kGradBlock + p0;
  double* s_w = s_j + ncol * kFisherChunk;
  double* s_r = s_w + kFisherChunk;
  for (int e0 = 0; e0 < fp.npart; e0 += kGradBlock) {
    const int e = e0 + tid;
    int i = 0, j = -1;
    if (e < ntri) fisher_tri(e, ncol, i, j);
    else if (e < fp.npart) i = e - ntri;
    double acc = 0.0;
    for (int c0 = 0; c0 < np; c0 += kFisherChunk) {
      const int n = min(kFisherChunk, np - c0);
      for (int x = tid; x < ncol * kFisherChunk; x += kGradBlock) {
        const int col = x / kFisherChunk, pp = x - col * kFisherChunk;
        s_j[x] = pp < n ? J[(size_t)col * fp.col_stride + c0 + pp] : 0.0;
      }
      if (tid < kFisherChunk) {
        s_w[tid] = tid < n ? __ldg(I.inv_sigma2 + p0 + c0 + tid) : 0.0;
        s_r[tid] = tid < n ? r[c0 + tid] : 0.0;
      }
      __syncthreads();
      if (e < fp.npart) {
        const double* ci = s_j + i * kFisherChunk;
        if (j >= 0) {
          const double* cj = s_j + j * kFisherChunk;
          for (int pp = 0; pp < n; ++pp) acc = fma(s_w[pp] * ci[pp], cj[pp], acc);
        } else {
          for (int pp = 0; pp < n; ++pp) acc = fma(s_r[pp], ci[pp], acc);
        }
      }
      __syncthreads();
    }
    if (e < fp.npart) fp.pgram[((size_t)w * prm.n_tiles_total + blockIdx.x) * fp.npart + e] = acc;
  }
}

// one warp per walker: value as grad_finalize_kernel; gradient and the mirrored matrix from the tile partials
template <bool SL>
__global__ void __launch_bounds__(128) fisher_finalize_kernel(const FisherParams fp, const SlRows sl) {
  const GradParams& prm = fp.gp;
  const int w = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (w >= prm.W || sl_skip<SL>(sl, w)) return;
  const int ndim = prm.ndim, ncol = fp.ncol, ntri = ncol * (ncol + 1) / 2;
  double* row = prm.grad + (size_t)w * ndim;
  double* F = fp.fisher + (size_t)w * ndim * ndim;
  for (int i = ncol + lane; i < ndim; i += 32) row[i] = 0.0;
  for (int x = lane; x < ndim * ndim; x += 32)
    if (x / ndim >= ncol || x % ndim >= ncol) F[x] = 0.0;
  double total = 0.0;
  for (int k = 0; k < prm.n_inst; ++k) {
    const InstDev& I = prm.inst[sl_inst<SL>(sl, w, k)];
    const GradInst& gi = prm.gi[k];
    double s = 0.0;
    const double* pv = prm.pval + (size_t)w * prm.n_blk_total + gi.blk_off;
    for (int t0 = 0; t0 < gi.n_blk; t0 += 32) {
      const double v = (t0 + lane < gi.n_blk) ? pv[t0 + lane] : 0.0;
      const int m = min(32, gi.n_blk - t0);
      for (int t = 0; t < m; ++t) s += __shfl_sync(0xffffffffu, v, t);
    }
    total += -0.5 * (s - I.sum_log_inv_sigma2);
  }
  if (lane == 0) prm.value[w] = total;
  const double* pg = fp.pgram + (size_t)w * prm.n_tiles_total * fp.npart;
  for (int e = lane; e < fp.npart; e += 32) {
    double s = 0.0;
    for (int t = 0; t < prm.n_tiles_total; ++t) s += pg[(size_t)t * fp.npart + e];   // instruments in order
    if (e < ntri) {
      int i, j;
      fisher_tri(e, ncol, i, j);
      F[(size_t)i * ndim + j] = s;
      F[(size_t)j * ndim + i] = s;
    } else {
      row[e - ntri] = s;
    }
  }
}

// rbv_model_jacobian_batch: out[w, i, p] = dM_p/dtheta_i of instrument jac_inst, rows beyond ncol zero
__global__ void __launch_bounds__(kGradBlock) fisher_jac_out_kernel(const FisherParams fp) {
  const GradParams& prm = fp.gp;
  const int k = fp.jac_inst, w = prm.w0 + blockIdx.z, i = blockIdx.y;
  const InstDev& I = prm.inst[k];
  const int p = blockIdx.x * kGradBlock + threadIdx.x;
  if (p >= I.P) return;
  double v = 0.0;
  if (i < fp.ncol) v = (fp.has_lsf[k] ? fp.JM : fp.JF)[fisher_col_base(fp, w, i, k) + p];
  fp.jac[((size_t)w * prm.ndim + i) * I.P + p] = v;
}

}  // namespace rbv
