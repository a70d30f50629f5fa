// rbvfit_b200 -- device-resident affine-invariant ensemble sampler (stretch move), sm_100a.
//
// The reference runs emcee.EnsembleSampler(nwalkers, ndim, vfit.lnprob).run_mcmc(...) (vfit_mcmc.py:408-423,
// 536-540).  emcee is a third-party dependency that is not vendored in the reference; its algorithm is restated
// from the published description (Goodman & Weare 2010; Foreman-Mackey et al. 2013, emcee 3 RedBlueMove +
// StretchMove), exactly as rbvfit_b200/sampler.py does on the host:
//
//   per step: split the walkers at random into two halves; for each half S with complement C
//       z_k   = ((a - 1) u_k + 1)^2 / a,  u_k ~ U(0,1)
//       Y_k   = C_j(k) - (C_j(k) - S_k) z_k,             j(k) uniform over the complement
//       ln q  = (ndim - 1) ln z_k + lnp(Y_k) - lnp(S_k);  accept when ln U < ln q
//
// Here the whole loop lives on the device: three small kernels around the likelihood launch per half-step, no host
// round trip, every random number from a counter-based generator (Philox4x32-10 keyed by the seed, counter =
// (step, walker, split, purpose)) so that a run is reproducible whatever the launch geometry.  The random split of
// emcee (shuffle of 0/1 labels) becomes a random affine permutation pos -> (a pos + b) mod W, gcd(a, W) = 1, whose
// first half is S; like emcee's it is drawn independently of the walker positions, which is all detailed balance
// needs.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace rbv {

struct StretchParams {
  double* coords;        // [W, ndim] current ensemble (in/out)
  double* lnp;           // [W]       its log-probabilities (in/out)
  double* prop;          // [ceil(W/2), ndim] proposals of the active half
  double* lnp_prop;      // [ceil(W/2)]
  double* factors;       // [ceil(W/2)] (ndim - 1) ln z
  int* walker_of;        // [ceil(W/2)] walker index of the k-th row of the active half
  double* chain;         // [n_steps, W, ndim] or NULL
  double* lnp_chain;     // [n_steps, W] or NULL
  int* n_accepted;       // [W] accumulates
  int* flag;             // bit 0: a proposal's lnprob was NaN
  unsigned long long* step_ctr;   // [0] steps done in this run (device counter, advanced by the last accept of a step);
                                  // NULL = the host drives the steps (multi-GPU form): step = first_step, chain row 0
  unsigned int* ticket;  // walkers of the current half-step whose accept/record is done
  unsigned long long first_step;  // global index of the run's first step (continues the random streams)
  unsigned long long seed;
  double a;
  int W, ndim;
  int ring_steps;        // 0: chain / lnp_chain hold every step of the run; > 0: they are rings of that many steps
                         // (rbv_stretch_run_sink: blocks of the ring are copied to the host while the run goes on)
  int S;                 // independent ensembles of W walkers each that advance in lockstep (survey mode: one per
                         // sightline, rbv_stretch_run_sightlines); 1 everywhere else.  Ensemble e owns walkers
                         // e W .. e W + W - 1 of coords / lnp / n_accepted and rows e n_S .. of the half-step buffers;
                         // its random streams are those of a single ensemble with the walker counter offset by e W
  const double* beta;    // [S] or NULL: ensemble e accepts against prior x L^beta[e] (parallel tempering, rbv_pt.cuh;
                         // lnp stays the untempered lnprob).  NULL: the untempered test of every other path
};

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}

// uniform in (0, 1): 53 random bits, never 0 or 1
__device__ __forceinline__ double u01(uint32_t hi, uint32_t lo) {
  const unsigned long long m = (((unsigned long long)hi << 32) | lo) >> 11;
  return ((double)m + 0.5) * 1.1102230246251565e-16;
}

// the sampler's random stream: counter = (step lo, step hi, walker, purpose), key = seed
__device__ __forceinline__ uint4 sampler_rand(unsigned long long seed, unsigned long long step, uint32_t walker,
                                              uint32_t purpose) {
  return philox4x32_10(make_uint4((uint32_t)step, (uint32_t)(step >> 32), walker, purpose),
                       make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
}

__device__ __forceinline__ uint4 stretch_rand(const StretchParams& P, unsigned long long step, uint32_t walker,
                                              uint32_t purpose) {
  return sampler_rand(P.seed, step, walker, purpose);
}

// an affine permutation of W positions from one random draw r: pos -> (a pos + b) mod W, a advanced until gcd(a, W) = 1
__device__ __forceinline__ void affine_perm(uint4 r, int n_walkers, uint32_t& a, uint32_t& b) {
  const uint32_t W = (uint32_t)n_walkers;
  a = r.x % W;
  b = r.y % W;
  for (;;) {
    uint32_t x = a, y = W;
    while (y) {
      const uint32_t t = x % y;
      x = y;
      y = t;
    }
    if (x == 1u || W == 1u) break;
    a = (a + 1u) % W;
  }
}

// the step's affine permutation of walker positions: walker(pos) = (a pos + b) mod W
__device__ __forceinline__ void sampler_perm(unsigned long long seed, int n_walkers, unsigned long long step,
                                             uint32_t& a, uint32_t& b) {
  affine_perm(sampler_rand(seed, step, 0xffffffffu, 0u), n_walkers, a, b);
}

__device__ __forceinline__ void stretch_perm(const StretchParams& P, unsigned long long step, uint32_t& a, uint32_t& b) {
  sampler_perm(P.seed, P.W, step, a, b);
}

__device__ __forceinline__ int walker_at(uint32_t a, uint32_t b, int W, int pos) {
  return (int)(((unsigned long long)a * (unsigned)pos + b) % (unsigned)W);
}

// sizes/offsets of the active half and its complement for split s (first half = ceil(W/2) walkers)
__device__ __forceinline__ void split_geometry(int W, int split, int& offS, int& nS, int& offC, int& nC) {
  const int h = (W + 1) / 2;
  if (split == 0) { offS = 0; nS = h; offC = h; nC = W - h; }
  else            { offS = h; nS = W - h; offC = 0; nC = h; }
}

// The tempered accept test of parallel tempering, case by case on the untempered lnprob values: beta (new - old)
// would be 0 x (-inf) = NaN at beta = 0, and a walker that starts outside the bounds would never move.  Explicitly
// rounded operations: the numpy replay evaluates the same expression.
__device__ __forceinline__ bool tempered_accept(double beta, double factor, double new_lp, double old_lp, double lnu) {
  if (!(new_lp > -INFINITY)) return false;                  // -inf (or NaN) proposal: always rejected
  if (old_lp == -INFINITY) return true;
  return lnu < __dsub_rn(__dadd_rn(factor, __dmul_rn(beta, new_lp)), __dmul_rn(beta, old_lp));
}

// Accept / reject for row k of the active half once its lnprob is known, by the WARP that finalised it (last CTA of
// the walker in the tile kernel, or finalize_kernel).  Every lane takes the same decision; the lanes copy the
// parameter columns in parallel (a single thread would pay one L2 round trip per column: proposal -> walker ->
// chain row).  The walker's row of the chain is written here too: after its own half-step a walker does not change
// again within the step.  The last walker of the second half advances the step counter.
__device__ __forceinline__ void stretch_accept_record(const StretchParams& P, int split, int k, double new_lp,
                                                      int lane, int e = 0) {
  int offS, nS, offC, nC;
  split_geometry(P.W, split, offS, nS, offC, nC);
  const unsigned long long s = P.step_ctr ? __ldcg(P.step_ctr) : 0ull, step = P.first_step + s;   // L2: see below
  const int i = e * P.W + P.walker_of[k];              // k: row of the half-step buffers, i: global walker
  const uint4 r = stretch_rand(P, step, (uint32_t)i, 3u + (uint32_t)split);
  const double old_lp = P.lnp[i];
  bool accept;
  if (!P.beta) {
    const double lnpdiff = P.factors[k] + new_lp - old_lp;
    accept = log(u01(r.x, r.y)) < lnpdiff;
  } else {
    accept = tempered_accept(P.beta[e], P.factors[k], new_lp, old_lp, log(u01(r.x, r.y)));
  }
  const double* __restrict__ src = accept ? P.prop + (size_t)k * P.ndim : P.coords + (size_t)i * P.ndim;
  double* __restrict__ x = P.coords + (size_t)i * P.ndim;
  const unsigned long long srow = P.ring_steps ? s % (unsigned long long)P.ring_steps : s;   // row of the chain buffers
  double* __restrict__ row = P.chain ? P.chain + (srow * P.S * P.W + i) * (size_t)P.ndim : nullptr;
  for (int d = lane; d < P.ndim; d += 32) {
    const double v = src[d];
    if (accept) x[d] = v;
    if (row) row[d] = v;
  }
  __syncwarp();
  if (lane == 0) {
    if (new_lp != new_lp) atomicOr(P.flag, 1);               // emcee: "Probability function returned NaN"
    if (accept) {
      P.lnp[i] = new_lp;
      P.n_accepted[i] += 1;
    }
    if (P.lnp_chain) P.lnp_chain[srow * P.S * P.W + i] = accept ? new_lp : old_lp;
    if (!P.ticket) return;        // host-driven steps, or the step ends later (parallel tempering's swap stage)
    __threadfence();
    if (atomicAdd(P.ticket, 1u) == (unsigned)nS - 1u) {      // last walker of this half-step
      *P.ticket = 0u;
      if (split == 1) *P.step_ctr = s + 1;
      __threadfence();
    }
  }
}

// ---- multi-GPU form: the half-step is split around the caller's all-gather of lnprob -------------------------
// Every rank builds ALL proposals of the active half (the state is replicated and the random streams are counter
// based, so the rows are identical on every rank), evaluates only its own rows, and after the all-gather applies
// the same accept/reject to every walker.
__device__ __forceinline__ void stretch_propose_row(const StretchParams& P, int split, int k, int& i_out,
                                                    int& j_out, double& zz_out, int e = 0) {
  int offS, nS, offC, nC;
  split_geometry(P.W, split, offS, nS, offC, nC);
  // (the counter is advanced by another CTA of the SAME launch in voigt_mcmc_kernel: read it from L2)
  const unsigned long long step = P.first_step + (P.step_ctr ? __ldcg(P.step_ctr) : 0ull);
  uint32_t pa, pb;
  stretch_perm(P, step, pa, pb);
  const int i = walker_at(pa, pb, P.W, offS + k);
  const uint4 r = stretch_rand(P, step, (uint32_t)(e * P.W + i), 1u + (uint32_t)split);
  const double u = u01(r.x, r.y);
  // explicitly rounded operations (no FMA contraction): the proposal is bit-identical to the numpy expression
  const double t = __dadd_rn(__dmul_rn(P.a - 1.0, u), 1.0);
  i_out = i;
  j_out = walker_at(pa, pb, P.W, offC + (int)(r.z % (uint32_t)nC));
  zz_out = __ddiv_rn(__dmul_rn(t, t), P.a);
}

__global__ void __launch_bounds__(128) stretch_propose_kernel(const StretchParams P, int split) {
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;   // warp per row
  int offS, nS, offC, nC;
  split_geometry(P.W, split, offS, nS, offC, nC);
  if (r >= P.S * nS) return;
  const int e = r / nS, k = r - e * nS;                // ensemble, row within its half
  int i, j;
  double zz;
  stretch_propose_row(P, split, k, i, j, zz, e);
  if (lane == 0) {
    P.factors[r] = (P.ndim - 1.0) * log(zz);
    P.walker_of[r] = i;
  }
  const double* s = P.coords + ((size_t)e * P.W + i) * P.ndim;
  const double* c = P.coords + ((size_t)e * P.W + j) * P.ndim;
  for (int d = lane; d < P.ndim; d += 32)
    P.prop[(size_t)r * P.ndim + d] = __dsub_rn(c[d], __dmul_rn(__dsub_rn(c[d], s[d]), zz));
}

__global__ void __launch_bounds__(128) stretch_accept_kernel(const StretchParams P, int split) {
  const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;   // warp per row
  int offS, nS, offC, nC;
  split_geometry(P.W, split, offS, nS, offC, nC);
  if (r >= P.S * nS) return;
  stretch_accept_record(P, split, r, P.lnp_prop[r], lane, r / nS);
}

}  // namespace rbv
