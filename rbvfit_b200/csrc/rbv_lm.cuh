// rbvfit_b200 -- survey-mode Levenberg-Marquardt: the step, accept / reject and damping update of every sightline on
// the device (sm_100a), one warp per sightline (DESIGN.md section 16).
//
// The decision rules are those of rbvfit_b200/lm.py.  One iteration of rbv_lm_run_sightlines is
//   survey-mode Fisher over the candidate rows xc of the active sightlines  ->  lm_update_kernel  ->  active count,
// and lm_update_kernel takes a sightline from "candidate evaluated" to "next candidate written" or to finished.
//
// Replay contract (oracle/lm_replay.py restates this file in scalar numpy): every floating-point operation is an
// explicitly rounded __dadd_rn / __dsub_rn / __dmul_rn / __ddiv_rn / __dsqrt_rn (nothing is contracted into an FMA),
// in these orders, indices ascending unless stated:
//   chi2        -2 * value
//   A           F_ff with A_ii = F_ii + lambda F_ii (the covariance: lambda absent, A_ii = F_ii)
//   Cholesky    for j: s = A_jj - sum_{k<j} L_jk L_jk, fail unless s > 0, L_jj = sqrt(s);
//               for i > j: L_ij = (A_ij - sum_{k<j} L_ik L_jk) / L_jj       (A_ij read from the lower triangle of F)
//   solve       y_i = (g_i - sum_{k<i} L_ik y_k) / L_ii;  d_i = (y_i - sum_{k>i} L_ki d_k) / L_ii   (i descending)
//   candidate   xc_i = min(max(x_i + d_i, lb_i), ub_i)  (d_i = 0 off the free set);  delta_i = xc_i - x_i
//   norms       |delta| = sqrt(sum delta_i delta_i), |x| likewise;  small: |delta| <= xtol (|x| + xtol)
//   pred        2 (sum g_i delta_i) - sum_i delta_i (sum_j F_ij delta_j)
//   damping     t = 2 rho - 1; lambda *= max(1/3, 1 - t t t)
//   covariance  Li = L^-1 by columns: Li_ic = ((i == c) - sum_{k=c}^{i-1} L_ik Li_kc) / L_ii;
//               cov_ij = sum_{k >= max(i, j)} Li_ki Li_kj
// Each sightline's numbers depend on its own rows only: not on n, on the block [first, first + n) or on the order.
#pragma once

namespace rbv {

constexpr int kLMWarps = 4;   // sightlines per 128-thread block
constexpr int kLMFailed = -1, kLMMaxEvals = 0, kLMFtol = 1, kLMXtol = 2;   // lm.STATUS_*

struct LMParams {
  int n, ndim, max_evals;
  double ftol, xtol;
  const double* lb;     // [ndim]
  const double* ub;
  double* x;            // [n, ndim] current point (the caller's theta: start in, best point out)
  double* g;            // [n, ndim] gradient at x
  double* F;            // [n, ndim, ndim] Gauss-Newton matrix at x
  double* xc;           // [n, ndim] candidate: the rows of the Fisher launch
  const double* vc;     // [n] lnlike, gradient and matrix at the candidate
  const double* gc;
  const double* Fc;
  double* L;            // [n, ndim, ndim] Cholesky factor (scratch)
  double* Li;           // [n, ndim, ndim] its inverse (scratch)
  double* y;            // [n, ndim] triangular solves (scratch)
  int* idx;             // [n, ndim] free parameters (scratch)
  double* lam;          // [n] damping
  double* nu;           // [n]
  int* started;         // [n] 0 until the start has been evaluated
  int* active;          // [n] the survey-mode Fisher skips rows with 0
  int* count;           // active sightlines after the update (zeroed before it)
  double* chi2;         // [n] outputs
  double* cov;          // [n, ndim, ndim]
  int* n_evals;         // [n]
  int* status;          // [n]
  int* flags;           // [n] bit 0: F_ff not positive definite at the end (cov left NaN)
};

constexpr unsigned kFull = 0xffffffffu;

// free set of lm.free_set into idx (lane 0 writes); every lane returns its size
__device__ int lm_free_set(const double* x, const double* g, const double* F, const double* lb, const double* ub,
                           int ndim, int* idx, int lane) {
  int m = 0;
  for (int i = 0; i < ndim; ++i) {
    const bool pinned = (x[i] <= lb[i] && g[i] < 0.0) || (x[i] >= ub[i] && g[i] > 0.0);
    if (F[(size_t)i * ndim + i] > 0.0 && !pinned) {
      if (lane == 0) idx[m] = i;
      ++m;
    }
  }
  __syncwarp();
  return m;
}

// Cholesky factor of F_ff (+ lambda diag F_ff when damped) into L (row stride ndim); false when not positive definite
__device__ bool lm_cholesky(const double* F, int ndim, const int* idx, int m, bool damped, double lam, double* L,
                            int lane) {
  for (int j = 0; j < m; ++j) {
    const double f = F[(size_t)idx[j] * ndim + idx[j]];
    double s = damped ? __dadd_rn(f, __dmul_rn(lam, f)) : f;
    for (int k = 0; k < j; ++k) s = __dsub_rn(s, __dmul_rn(L[j * ndim + k], L[j * ndim + k]));
    if (!(s > 0.0)) return false;   // every lane holds the same s
    const double d = __dsqrt_rn(s);
    if (lane == 0) L[j * ndim + j] = d;
    for (int i = j + 1 + lane; i < m; i += 32) {
      double t = F[(size_t)idx[i] * ndim + idx[j]];
      for (int k = 0; k < j; ++k) t = __dsub_rn(t, __dmul_rn(L[i * ndim + k], L[j * ndim + k]));
      L[i * ndim + j] = __ddiv_rn(t, d);
    }
    __syncwarp();
  }
  return true;
}

__device__ bool lm_finite(const double* v, int n, int lane) {
  bool ok = true;
  for (int i = lane; i < n; i += 32) ok = ok && isfinite(v[i]);
  return __all_sync(kFull, ok);
}

// finish sightline s: status, inv(F_ff) at x over the free set (NaN elsewhere), inactive
__device__ void lm_finish(const LMParams& p, int s, int st, bool with_cov, int lane) {
  const int nd = p.ndim;
  double* cov = p.cov + (size_t)s * nd * nd;
  for (int e = lane; e < nd * nd; e += 32) cov[e] = CUDART_NAN;
  __syncwarp();
  int flag = 0;
  if (with_cov) {
    const double* x = p.x + (size_t)s * nd;
    const double* F = p.F + (size_t)s * nd * nd;
    int* idx = p.idx + (size_t)s * nd;
    double* L = p.L + (size_t)s * nd * nd;
    double* Li = p.Li + (size_t)s * nd * nd;
    const int m = lm_free_set(x, p.g + (size_t)s * nd, F, p.lb, p.ub, nd, idx, lane);
    if (m > 0) {
      if (!lm_cholesky(F, nd, idx, m, false, 0.0, L, lane)) {
        flag = 1;
      } else {
        for (int c = lane; c < m; c += 32)
          for (int i = c; i < m; ++i) {
            double t = (i == c) ? 1.0 : 0.0;
            for (int k = c; k < i; ++k) t = __dsub_rn(t, __dmul_rn(L[i * nd + k], Li[k * nd + c]));
            Li[i * nd + c] = __ddiv_rn(t, L[i * nd + i]);
          }
        __syncwarp();
        for (int e = lane; e < m * m; e += 32) {
          const int i = e / m, j = e - i * m;
          double t = 0.0;
          for (int k = max(i, j); k < m; ++k) t = __dadd_rn(t, __dmul_rn(Li[k * nd + i], Li[k * nd + j]));
          cov[(size_t)idx[i] * nd + idx[j]] = t;
        }
      }
    }
  }
  if (lane == 0) {
    p.status[s] = st;
    p.flags[s] = flag;
    p.active[s] = 0;
  }
}

__global__ void __launch_bounds__(32 * kLMWarps) lm_init_kernel(const LMParams p) {
  const int s = blockIdx.x * kLMWarps + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (s >= p.n) return;
  for (int i = lane; i < p.ndim; i += 32) {
    const double v = p.x[(size_t)s * p.ndim + i];
    p.xc[(size_t)s * p.ndim + i] = fmin(fmax(v, p.lb[i]), p.ub[i]);
  }
  if (lane == 0) {
    p.lam[s] = 0.1;   // lm.py: 1e-3 lets the first Gauss-Newton step of C4 clip a b onto its bound
    p.nu[s] = 2.0;
    p.started[s] = 0;
    p.active[s] = 1;
    p.n_evals[s] = 0;
    p.status[s] = kLMMaxEvals;
    p.flags[s] = 0;
  }
}

// one warp per sightline: take the evaluated candidate, then propose the next one or finish
__global__ void __launch_bounds__(32 * kLMWarps) lm_update_kernel(const LMParams p) {
  const int s = blockIdx.x * kLMWarps + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (s >= p.n || !p.active[s]) return;
  const int nd = p.ndim;
  double* x = p.x + (size_t)s * nd;
  double* g = p.g + (size_t)s * nd;
  double* F = p.F + (size_t)s * nd * nd;
  double* xc = p.xc + (size_t)s * nd;
  const double* gc = p.gc + (size_t)s * nd;
  const double* Fc = p.Fc + (size_t)s * nd * nd;
  double* L = p.L + (size_t)s * nd * nd;
  double* y = p.y + (size_t)s * nd;
  int* idx = p.idx + (size_t)s * nd;
  double lam = p.lam[s], nu = p.nu[s], chi2 = p.chi2[s];
  const int n_ev = p.n_evals[s] + 1;
  const double chi2_n = __dmul_rn(-2.0, p.vc[s]);
  const bool fin = isfinite(chi2_n) && lm_finite(gc, nd, lane) && lm_finite(Fc, nd * nd, lane);
  const bool first = !p.started[s];
  bool accept;
  double actual = 0.0;
  if (first) {   // the start, clipped into the box
    accept = true;
    if (!fin) {
      for (int i = lane; i < nd; i += 32) x[i] = xc[i];
      if (lane == 0) {
        p.chi2[s] = chi2_n;
        p.n_evals[s] = n_ev;
      }
      lm_finish(p, s, kLMFailed, false, lane);
      return;
    }
  } else {
    double gd = 0.0, q = 0.0;
    for (int i = 0; i < nd; ++i) {
      const double di = __dsub_rn(xc[i], x[i]);
      gd = __dadd_rn(gd, __dmul_rn(g[i], di));
      double t = 0.0;
      for (int j = 0; j < nd; ++j) t = __dadd_rn(t, __dmul_rn(F[(size_t)i * nd + j], __dsub_rn(xc[j], x[j])));
      q = __dadd_rn(q, __dmul_rn(di, t));
    }
    const double pred = __dsub_rn(__dmul_rn(2.0, gd), q);
    actual = __dsub_rn(chi2, chi2_n);
    const double rho = (fin && pred > 0.0) ? __ddiv_rn(actual, pred) : -1.0;
    accept = rho > 0.0;
    if (accept) {
      const double t = __dsub_rn(__dmul_rn(2.0, rho), 1.0);
      lam = __dmul_rn(lam, fmax(1.0 / 3.0, __dsub_rn(1.0, __dmul_rn(__dmul_rn(t, t), t))));
      nu = 2.0;
    } else {
      lam = __dmul_rn(lam, nu);
      nu = __dmul_rn(nu, 2.0);
    }
  }
  __syncwarp();   // every lane has read x, g, F before they are replaced
  const double chi2_old = chi2;
  if (accept) {
    for (int i = lane; i < nd; i += 32) {
      x[i] = xc[i];
      g[i] = gc[i];
    }
    for (int e = lane; e < nd * nd; e += 32) F[e] = Fc[e];
    chi2 = chi2_n;
  }
  if (lane == 0) {
    p.chi2[s] = chi2;
    p.n_evals[s] = n_ev;
    p.started[s] = 1;
  }
  __syncwarp();
  if (!first && accept && actual <= __dmul_rn(p.ftol, fabs(chi2_old))) {
    lm_finish(p, s, kLMFtol, true, lane);
    return;
  }
  while (true) {
    const int m = lm_free_set(x, g, F, p.lb, p.ub, nd, idx, lane);
    if (m == 0) {
      lm_finish(p, s, kLMXtol, true, lane);
      return;
    }
    if (!lm_cholesky(F, nd, idx, m, true, lam, L, lane)) {
      __syncwarp();
      lam = __dmul_rn(lam, nu);
      nu = __dmul_rn(nu, 2.0);
      if (lam > 1e30) {
        lm_finish(p, s, kLMFailed, true, lane);
        return;
      }
      continue;
    }
    int small = 0;
    if (lane == 0) {
      for (int i = 0; i < m; ++i) {
        double t = g[idx[i]];
        for (int k = 0; k < i; ++k) t = __dsub_rn(t, __dmul_rn(L[i * nd + k], y[k]));
        y[i] = __ddiv_rn(t, L[i * nd + i]);
      }
      for (int i = m - 1; i >= 0; --i) {
        double t = y[i];
        for (int k = i + 1; k < m; ++k) t = __dsub_rn(t, __dmul_rn(L[k * nd + i], y[k]));
        y[i] = __ddiv_rn(t, L[i * nd + i]);
      }
      double sd = 0.0, sx = 0.0;
      for (int i = 0, f = 0; i < nd; ++i) {
        double di = 0.0;
        if (f < m && idx[f] == i) di = y[f++];
        const double v = fmin(fmax(__dadd_rn(x[i], di), p.lb[i]), p.ub[i]);
        xc[i] = v;
        const double dd = __dsub_rn(v, x[i]);
        sd = __dadd_rn(sd, __dmul_rn(dd, dd));
        sx = __dadd_rn(sx, __dmul_rn(x[i], x[i]));
      }
      small = __dsqrt_rn(sd) <= __dmul_rn(p.xtol, __dadd_rn(__dsqrt_rn(sx), p.xtol));
    }
    small = __shfl_sync(kFull, small, 0);
    __syncwarp();
    if (small) {
      lm_finish(p, s, kLMXtol, true, lane);
      return;
    }
    if (n_ev >= p.max_evals) {
      lm_finish(p, s, kLMMaxEvals, true, lane);
      return;
    }
    break;
  }
  if (lane == 0) {
    p.lam[s] = lam;
    p.nu[s] = nu;
    atomicAdd(p.count, 1);
  }
}

}  // namespace rbv
