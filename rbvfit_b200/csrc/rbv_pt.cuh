// rbvfit_b200 -- parallel tempering on the device (rbv_pt_run), sm_100a.
//
// The algorithm is ptemcee's (Vousden, Farr & Mandel 2016, MNRAS 455, 1919): T ensembles of W walkers sample the
// tempered targets prior x L^beta_t on a ladder 1 = beta_0 > beta_1 > ... >= 0 and exchange states between adjacent
// temperatures once per step.  The state is coords [T, W, ndim] and lnprob [T, W]; every walker keeps its UNTEMPERED
// lnprob (ln L inside the box prior of rbv_set_bounds, -inf outside).  One step:
//
//   half-step 0, half-step 1   the stretch move of rbv_sampler.cuh with S = T ensembles (partners from the same
//                              temperature's complementary half, random streams of a single ensemble with the walker
//                              counter offset by t W), accepted against the tempered target (tempered_accept); the
//                              lnprob batch of a half-step is ONE joint-mode launch over the T ceil(W/2) proposal rows
//   swap stage                 for i = T-1 down to 1 (hottest pair first, sequentially): walker p_i(k) of temperature
//                              i and walker q_i(k) of temperature i-1 (k = 0 .. W-1) exchange coords and lnprob when
//                                  ln u < (beta_{i-1} - beta_i) (lnL_{i, p_i(k)} - lnL_{i-1, q_i(k)})
//                              (NaN or -inf on the right rejects); p_i, q_i are random affine permutations like the
//                              step's split.  pt_swap_plan_kernel (ONE CTA) runs the levels on lnprob and a slot map,
//                              pt_gather_record_kernel then moves the coordinates once: two launches and one copy
//                              per step whatever T is
//   ladder adaptation          optional (burn-in only: it breaks detailed balance), ptemcee's rule after every step
//                              with A_i the step's swap acceptance of pair (i, i+1) and t the adaptation steps done:
//                                  kappa = (lag / (t + lag)) / tau,  dS = kappa (A[:-1] - A[1:]),
//                                  dT = diff(1 / beta[:-1]) exp(dS),  beta[1:-1] = 1 / (cumsum(dT) + 1 / beta_0)
//   record                     the state AFTER the swaps (ptemcee's order): coordinates of the n_record coldest
//                              temperatures and lnprob of all T; the same kernel advances the device step counter
//
// Random purposes (Philox counter (step, walker, purpose), key = seed; 0-4 are the stretch move's, 8.. the slice
// sampler's):
//   5   swap permutations: walker counter 2 i -> p_i, 2 i + 1 -> q_i (affine_perm of the draw)
//   6   swap decisions: walker counter i W + k -> u of pair k of level i (x, y)
//
// Survey mode (rbv_pt_run_sightlines): S sightlines of T temperatures each, ensemble e = s T + t (sightline-major),
// coords [S, T, W, ndim], lnprob [S, T, W], ladders [S, T].  Every walker counter of sightline s, purposes 1-6, is
// offset by s T W, so sightline s runs the streams of a one-sightline rbv_pt_run shifted by s T W (with T = 1: those
// of rbv_stretch_run_sightlines).  The plan kernel runs one CTA per sightline; rbv_pt_run is the case S = 1.
//
// Thermodynamic-integration moments (survey mode, optional): ti [S, T, 3] = (n, mean, M2) of the post-swap lnprob of
// every step, accumulated on the device in the plan kernel.  A step's W values of one temperature are reduced in
// walker order k = 0 .. W-1 to m = (sum x_k) / W and q = sum (x_k - m)^2, then merged by Chan's formula
//     n' = n + W,  d = m - mean,  mean' = mean + d (W / n'),  M2' = M2 + q + d^2 (n W / n')
// in explicitly rounded operations (at n = 0 this gives (W, m, q) exactly; a non-finite value makes the result
// non-finite).  Var = M2 / n is numpy's var of the same values.
#pragma once

#include "rbv_sampler.cuh"

namespace rbv {

struct PtParams {
  double* coords;          // [S, T, W, ndim] (the stretch move's coords)
  double* lnp;             // [S, T, W] untempered lnprob, permuted in place by the plan kernel
  double* betas;           // [S, T] the ladders (in/out: adapted in place)
  double* coords_tmp;      // [S, T, W, ndim] copy of coords taken before the swap stage
  int* src;                // [S, T, W] slot -> slot whose state it holds after the swaps (global slot indices)
  unsigned long long* n_swaps;   // [S, T - 1] accumulated accepted swaps of pair (i, i + 1), or NULL (T = 1)
  double* chain;           // [steps, S, n_record, W, ndim] (a ring of ring_steps steps with the sink) or NULL
  double* lnp_chain;       // [steps, S, T, W] (ring likewise) or NULL
  double* beta_history;    // [n_steps, S, T] or NULL: the ladder each step ran with
  double* ti;              // [S, T, 3] (n, mean, M2) of the post-swap lnprob, accumulated, or NULL (no accumulation)
  unsigned long long* step_ctr;   // steps done in this run (advanced by pt_gather_record_kernel)
  unsigned int* ticket;    // CTAs of pt_gather_record_kernel done with the current step
  unsigned long long first_step, seed;
  unsigned long long adapt_t0;    // adaptation steps done before this run
  double adapt_lag, adapt_time;
  int adapt;
  int S, T, W, ndim, n_record;   // S sightlines (1 in rbv_pt_run)
  int survey;              // lnprob in sightline mode (row r belongs to sightline r / (T n_S)); 0: one joint context
  int ring_steps;          // 0: chain / lnp_chain hold every step; > 0: rings of that many steps
};

constexpr int kPtPlanThreads = 256;

// ONE CTA per sightline (blockIdx.x): the swap levels in ptemcee's order on lnprob and the slot map, the
// thermodynamic-integration moments, the swap counters and the ladder update.  Dynamic shared memory: T unsigned
// counters.  Levels are sequential (__syncthreads between them); the W pairs of a level are disjoint, so its threads
// swap without atomics.
__global__ void __launch_bounds__(kPtPlanThreads) pt_swap_plan_kernel(const PtParams P) {
  extern __shared__ unsigned int n_acc[];            // [T]: this step's accepted swaps of pair (i, i + 1)
  const int T = P.T, W = P.W, tid = threadIdx.x, sl = blockIdx.x;
  const int base = sl * T * W;                       // the sightline's first slot and its walker-counter offset
  double* __restrict__ lnp = P.lnp + base;
  int* __restrict__ src = P.src + base;
  double* __restrict__ betas = P.betas + (size_t)sl * T;
  const unsigned long long s = __ldcg(P.step_ctr), step = P.first_step + s;
  for (int x = tid; x < T * W; x += blockDim.x) src[x] = base + x;
  for (int i = tid; i < T; i += blockDim.x) {
    n_acc[i] = 0u;
    if (P.beta_history) P.beta_history[(s * (unsigned long long)P.S + sl) * T + i] = betas[i];
  }
  __syncthreads();
  for (int i = T - 1; i >= 1; --i) {
    uint32_t pa, pb, qa, qb;
    affine_perm(sampler_rand(P.seed, step, (uint32_t)base + 2u * (uint32_t)i, 5u), W, pa, pb);
    affine_perm(sampler_rand(P.seed, step, (uint32_t)base + 2u * (uint32_t)i + 1u, 5u), W, qa, qb);
    const double dbeta = __dsub_rn(betas[i - 1], betas[i]);
    unsigned int n = 0u;
    for (int k = tid; k < W; k += blockDim.x) {
      const int x = i * W + walker_at(pa, pb, W, k), y = (i - 1) * W + walker_at(qa, qb, W, k);
      const uint4 r = sampler_rand(P.seed, step, (uint32_t)(base + i * W + k), 6u);
      const double lx = lnp[x], ly = lnp[y];
      if (log(u01(r.x, r.y)) < __dmul_rn(dbeta, __dsub_rn(lx, ly))) {
        lnp[x] = ly;
        lnp[y] = lx;
        const int t = src[x];
        src[x] = src[y];
        src[y] = t;
        ++n;
      }
    }
    if (n) atomicAdd(&n_acc[i - 1], n);
    __syncthreads();                                 // level i - 1 reads what level i wrote
  }
  if (P.ti) {                                        // thread per temperature, walker order (see the file comment)
    for (int t = tid; t < T; t += blockDim.x) {
      const double* __restrict__ v = lnp + t * W;
      double sum = 0.0, q = 0.0;
      for (int k = 0; k < W; ++k) sum = __dadd_rn(sum, v[k]);
      const double m = __ddiv_rn(sum, (double)W);
      for (int k = 0; k < W; ++k) {
        const double d = __dsub_rn(v[k], m);
        q = __dadd_rn(q, __dmul_rn(d, d));
      }
      double* __restrict__ M = P.ti + ((size_t)sl * T + t) * 3;
      const double n = M[0], n1 = __dadd_rn(n, (double)W), d = __dsub_rn(m, M[1]);
      M[0] = n1;
      M[1] = __dadd_rn(M[1], __dmul_rn(d, __ddiv_rn((double)W, n1)));
      M[2] = __dadd_rn(__dadd_rn(M[2], q), __dmul_rn(__dmul_rn(d, d), __ddiv_rn(__dmul_rn(n, (double)W), n1)));
    }
  }
  if (tid != 0) return;
  for (int i = 0; i + 1 < T; ++i) P.n_swaps[(size_t)sl * (T - 1) + i] += n_acc[i];
  if (!P.adapt || T < 3) return;
  // ptemcee's ladder adjustment; the coldest and hottest beta stay, the new interior values use the OLD ladder's
  // inverse temperatures, kept in `inv` as the loop overwrites beta.  Explicitly rounded (no FMA contraction).
  const double kappa = __ddiv_rn(__ddiv_rn(P.adapt_lag, __dadd_rn((double)(P.adapt_t0 + s), P.adapt_lag)),
                                 P.adapt_time);
  const double inv0 = __ddiv_rn(1.0, betas[0]);
  double inv = inv0, cs = 0.0;
  for (int j = 0; j + 2 < T; ++j) {
    const double inv_next = __ddiv_rn(1.0, betas[j + 1]);
    const double dS = __dmul_rn(kappa, __dsub_rn(__ddiv_rn((double)n_acc[j], (double)W),
                                                 __ddiv_rn((double)n_acc[j + 1], (double)W)));
    cs = __dadd_rn(cs, __dmul_rn(__dsub_rn(inv_next, inv), exp(dS)));
    inv = inv_next;
    betas[j + 1] = __ddiv_rn(1.0, __dadd_rn(cs, inv0));
  }
}

// Warp per slot (S T W slots): coords[x] = the state the plan moved into slot x, and the step's record (coordinates
// of each sightline's n_record coldest temperatures, lnprob of all).  The last CTA to finish advances the step counter.
__global__ void __launch_bounds__(128) pt_gather_record_kernel(const PtParams P) {
  const int x = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  const unsigned long long s = __ldcg(P.step_ctr);
  const unsigned long long srow = P.ring_steps ? s % (unsigned long long)P.ring_steps : s;
  const int TW = P.T * P.W;
  if (x < P.S * TW) {
    const int sl = x / TW, xs = x - sl * TW;         // sightline, slot within it
    const int from = P.src[x];
    const double* __restrict__ a = P.coords_tmp + (size_t)from * P.ndim;
    double* __restrict__ b = P.coords + (size_t)x * P.ndim;
    double* __restrict__ row =
        (P.chain && xs < P.n_record * P.W)
            ? P.chain + ((srow * P.S + sl) * P.n_record * P.W + xs) * (size_t)P.ndim : nullptr;
    for (int d = lane; d < P.ndim; d += 32) {
      const double v = a[d];
      if (from != x) b[d] = v;
      if (row) row[d] = v;
    }
    if (lane == 0 && P.lnp_chain) P.lnp_chain[srow * P.S * TW + x] = P.lnp[x];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(P.ticket, 1u) == gridDim.x - 1u) {     // every CTA has read the counter
      *P.ticket = 0u;
      *P.step_ctr = s + 1;
      __threadfence();
    }
  }
}

}  // namespace rbv
