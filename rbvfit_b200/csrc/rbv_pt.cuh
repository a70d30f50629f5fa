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
#pragma once

#include "rbv_sampler.cuh"

namespace rbv {

struct PtParams {
  double* coords;          // [T, W, ndim] (the stretch move's coords)
  double* lnp;             // [T, W] untempered lnprob, permuted in place by the plan kernel
  double* betas;           // [T] the ladder (in/out: adapted in place)
  double* coords_tmp;      // [T, W, ndim] copy of coords taken before the swap stage
  int* src;                // [T, W] slot -> slot whose state it holds after the swaps
  unsigned long long* n_swaps;   // [T - 1] accumulated accepted swaps of pair (i, i + 1), or NULL (T = 1)
  double* chain;           // [steps, n_record, W, ndim] (a ring of ring_steps steps with the sink) or NULL
  double* lnp_chain;       // [steps, T, W] (ring likewise) or NULL
  double* beta_history;    // [n_steps, T] or NULL: the ladder each step ran with
  unsigned long long* step_ctr;   // steps done in this run (advanced by pt_gather_record_kernel)
  unsigned int* ticket;    // CTAs of pt_gather_record_kernel done with the current step
  unsigned long long first_step, seed;
  unsigned long long adapt_t0;    // adaptation steps done before this run
  double adapt_lag, adapt_time;
  int adapt;
  int T, W, ndim, n_record;
  int ring_steps;          // 0: chain / lnp_chain hold every step; > 0: rings of that many steps
};

constexpr int kPtPlanThreads = 256;

// ONE CTA: the swap levels in ptemcee's order on lnprob and the slot map, the swap counters and the ladder update.
// Dynamic shared memory: T unsigned counters.  Levels are sequential (__syncthreads between them); the W pairs of a
// level are disjoint, so its threads swap without atomics.
__global__ void __launch_bounds__(kPtPlanThreads) pt_swap_plan_kernel(const PtParams P) {
  extern __shared__ unsigned int n_acc[];            // [T]: this step's accepted swaps of pair (i, i + 1)
  const int T = P.T, W = P.W, tid = threadIdx.x;
  const unsigned long long s = __ldcg(P.step_ctr), step = P.first_step + s;
  for (int x = tid; x < T * W; x += blockDim.x) P.src[x] = x;
  for (int i = tid; i < T; i += blockDim.x) {
    n_acc[i] = 0u;
    if (P.beta_history) P.beta_history[s * (unsigned long long)T + i] = P.betas[i];
  }
  __syncthreads();
  for (int i = T - 1; i >= 1; --i) {
    uint32_t pa, pb, qa, qb;
    affine_perm(sampler_rand(P.seed, step, 2u * (uint32_t)i, 5u), W, pa, pb);
    affine_perm(sampler_rand(P.seed, step, 2u * (uint32_t)i + 1u, 5u), W, qa, qb);
    const double dbeta = __dsub_rn(P.betas[i - 1], P.betas[i]);
    unsigned int n = 0u;
    for (int k = tid; k < W; k += blockDim.x) {
      const int x = i * W + walker_at(pa, pb, W, k), y = (i - 1) * W + walker_at(qa, qb, W, k);
      const uint4 r = sampler_rand(P.seed, step, (uint32_t)(i * W + k), 6u);
      const double lx = P.lnp[x], ly = P.lnp[y];
      if (log(u01(r.x, r.y)) < __dmul_rn(dbeta, __dsub_rn(lx, ly))) {
        P.lnp[x] = ly;
        P.lnp[y] = lx;
        const int t = P.src[x];
        P.src[x] = P.src[y];
        P.src[y] = t;
        ++n;
      }
    }
    if (n) atomicAdd(&n_acc[i - 1], n);
    __syncthreads();                                 // level i - 1 reads what level i wrote
  }
  if (tid != 0) return;
  for (int i = 0; i + 1 < T; ++i) P.n_swaps[i] += n_acc[i];
  if (!P.adapt || T < 3) return;
  // ptemcee's ladder adjustment; the coldest and hottest beta stay, the new interior values use the OLD ladder's
  // inverse temperatures, kept in `inv` as the loop overwrites beta.  Explicitly rounded (no FMA contraction).
  const double kappa = __ddiv_rn(__ddiv_rn(P.adapt_lag, __dadd_rn((double)(P.adapt_t0 + s), P.adapt_lag)),
                                 P.adapt_time);
  const double inv0 = __ddiv_rn(1.0, P.betas[0]);
  double inv = inv0, cs = 0.0;
  for (int j = 0; j + 2 < T; ++j) {
    const double inv_next = __ddiv_rn(1.0, P.betas[j + 1]);
    const double dS = __dmul_rn(kappa, __dsub_rn(__ddiv_rn((double)n_acc[j], (double)W),
                                                 __ddiv_rn((double)n_acc[j + 1], (double)W)));
    cs = __dadd_rn(cs, __dmul_rn(__dsub_rn(inv_next, inv), exp(dS)));
    inv = inv_next;
    P.betas[j + 1] = __ddiv_rn(1.0, __dadd_rn(cs, inv0));
  }
}

// Warp per slot: coords[x] = the state the plan moved into slot x, and the step's record (coordinates of the
// n_record coldest temperatures, lnprob of all).  The last CTA to finish advances the step counter.
__global__ void __launch_bounds__(128) pt_gather_record_kernel(const PtParams P) {
  const int x = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  const unsigned long long s = __ldcg(P.step_ctr);
  const unsigned long long srow = P.ring_steps ? s % (unsigned long long)P.ring_steps : s;
  if (x < P.T * P.W) {
    const int from = P.src[x];
    const double* __restrict__ a = P.coords_tmp + (size_t)from * P.ndim;
    double* __restrict__ b = P.coords + (size_t)x * P.ndim;
    double* __restrict__ row =
        (P.chain && x < P.n_record * P.W) ? P.chain + (srow * P.n_record * P.W + x) * (size_t)P.ndim : nullptr;
    for (int d = lane; d < P.ndim; d += 32) {
      const double v = a[d];
      if (from != x) b[d] = v;
      if (row) row[d] = v;
    }
    if (lane == 0 && P.lnp_chain) P.lnp_chain[srow * P.T * P.W + x] = P.lnp[x];
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
