// rbvfit_b200 -- device-resident ensemble slice sampler (zeus's differential move), sm_100a.
//
// The reference runs zeus.EnsembleSampler(nwalkers, ndim, vfit.lnprob).run_mcmc(...) when sampler='zeus'
// (vfit_mcmc.py:425-440, 536-540).  zeus-mcmc is a third-party dependency that is not vendored in the reference
// (requirements.txt:11); its algorithm is restated from the published description (Karamanis & Beutler 2021,
// "Ensemble slice sampling", Algorithms 2-3; zeus 2.x defaults), exactly as rbvfit_b200/slice_sampler.py does on
// the host:
//
//   per step, for each half S of the ensemble (split as in rbv_sampler.cuh) with complement C, per walker k of S:
//       direction  eta_k = 2 mu (C_j - C_l),  j != l drawn from C                     (differential move)
//       slice level  y_k = lnp(X_k) - Exp(1)
//       stepping out: [L, R] = [-U, 1 - U]; L -= 1 while lnp(X_k + L eta_k) >= y_k (budget J), then the same for R
//       shrinking:    t ~ U(L, R); accept X_k + t eta_k when lnp >= y_k, else L = t (t < 0) or R = t
//   after the step: mu <- mu * 2 n_exp / (n_exp + n_con) while tuning is on (slice_record_kernel)
//
// Here every walker of the half is a small state machine (widening: either end of the bracket still open;
// shrinking; finished) and one ITERATION advances every unfinished walker by one step of it:
//   the lnprob launch over the half (masked rows are skipped through row_skip)
//                           ->  slice_update_kernel (state machines, then the candidates of the next launch;
//                               slice_candidate_kernel writes the first candidates of a half-step)
// While a walker widens, BOTH ends of its bracket are evaluated in the same iteration (row k = X + L eta, row
// n_S + k = X + R eta; the two sides have independent budgets, so this is zeus's left-then-right loop run
// concurrently); while it shrinks only row k is live.  The number of device batches per half-step is therefore the
// longest chain  max(n_L, n_R) + 1 + n_shrink  over the walkers, where the host sampler pays the sum of the longest
// chains of its three loops.  Random numbers come from the same counter-based Philox streams as the stretch move:
// purpose 8 + split (partners, budget), 10 + split (slice level, bracket), 16 + 2 it + split (the shrink draw of
// iteration it).  All floating-point steps that decide the chain are written with explicitly rounded operations so
// that oracle/slice_replay.py reproduces them bit for bit in numpy.
//
// Speculation (depth 2, the default).  One launch can serve TWO logical iterations of a walker, because the second
// one's candidates do not depend on the first one's lnprob values, only on WHICH case they select: while widening,
// the next test point of an open end is one unit further out (rows 2 n_S + k and 3 n_S + k hold X + (L - 1) eta and
// X + (R + 1) eta; used only if the first test succeeds); while shrinking, a rejected draw t_1 moves the end on its
// own side, whatever lnprob was, so t_2 is drawn from the bracket that rejection would leave (row 2 n_S + k; used
// only if t_1 is rejected).  slice_update_kernel then replays the two logical iterations in order with exactly the
// rules of the sequential algorithm; rows it does not reach are dropped (not counted, not flagged).  Every walker
// keeps its own logical iteration index (lit), which keys the shrink draws -- in the sequential run every unfinished
// walker's index IS the iteration number -- so chains, mu, and the expansion / contraction / call counters are
// bit-identical for depth 1 and 2; only the number of launches per step drops (C2: 17.4 -> see DESIGN.md).  The
// extra rows cost next to nothing: the batch is far below one wave of CTAs either way.
//
// Who drives the loop.  Everything the loop needs -- step, iteration index, mu and its adaptation state, the count of
// unfinished walkers -- lives in one device struct (SliceCounters).  Graph mode: the iteration is the body of a CUDA
// graph WHILE node and the last warp of slice_update_kernel sets the loop condition (cudaGraphSetConditional), so a
// half-step is ONE graph launch and a whole run is enqueued without a single host synchronisation.  Polling mode
// (no graph): the host enqueues iterations one ahead of an asynchronous read-back of the counters.
//
// Survey mode (rbv_slice_run_sightlines): S independent ensembles of W walkers, one per sightline, advance in
// lockstep; rbv_slice_run is the case S = 1.  Ensemble e owns walkers e W .. e W + W - 1 of coords / lnp, rows
// e n_S .. e n_S + n_S - 1 of the per-walker half-step buffers (dir, z0, lo, hi, lit, budgets, phase, walker_of),
// rows e 2 n_S .. of tcur, and the contiguous block of 2 depth n_S candidate rows starting at e 2 depth n_S (cand,
// lnp_cand, skip; inside it the single-ensemble order k, n_S + k, 2 n_S + k, 3 n_S + k), so an iteration is ONE
// sightline-mode lnprob launch.  Its random streams are those of one ensemble with the walker counter offset by
// e W (walker_of holds that global index); the step's split is shared.  mu, its adaptation state and the counters are
// per ensemble (SliceParams::mu / adapt / totals / nstep); the loop state (SliceCounters) is shared: a half-step
// iterates until no walker of any ensemble is unfinished, and an ensemble whose walkers have all finished masks its
// rows, so its chain does not depend on how long the others take.
#pragma once

#include "rbv_sampler.cuh"

namespace rbv {

struct SliceCounters {          // device; the loop state of a run, shared by every ensemble
  unsigned int remaining;       // walkers of the half-step that are not finished after the last update
  unsigned int it;              // iteration index within the half-step
  unsigned int ticket;          // warps of slice_update_kernel that have finished the current iteration
  unsigned int guard;           // iterations started in this half-step (second, independent loop bound)
  unsigned int over;            // unfinished walkers whose logical iteration index has passed maxiter
  unsigned int pending;         // `remaining` of the last finished iteration (what the host-polled loop reads:
                                // `remaining` itself is re-armed by the warp that closes an iteration)
  int error;                    // 1 = a half-step needed more than maxiter iterations
  unsigned long long step;      // global index of the step being sampled
  unsigned long long batches;   // lnprob launches in this run
};

// mu, adaptation state and counters of ONE ensemble: rbv_slice_run keeps it in its workspace, next to the counters
// (SliceParams::mu / adapt / totals / nstep point into it); survey mode passes arrays of S of each instead
struct SliceEnsemble {
  double mu;                    // length scale of the directions
  int adapt[2];                 // tune, good (zeus: tune, count of steps inside the tolerance)
  unsigned long long totals[3]; // expansions, contractions (finished steps), likelihood rows
  unsigned int nstep[2];        // expansions / contractions of the current step
};

struct SliceState {             // the workspace block of rbv_slice_run (and its page-locked host image)
  SliceCounters c;
  SliceEnsemble solo;
};

// walker state: bit 0 = left end still open, bit 1 = right end still open (widening while either is set)
constexpr int kSliceLeft = 1, kSliceRight = 2, kSliceShrink = 4, kSliceDone = 8;

struct SliceParams {
  double* coords;        // [S W, ndim] current ensembles (in/out)
  double* lnp;           // [S W]       their log-probabilities (in/out)
  double* cand;          // [S 2 depth h, ndim] candidates of the active half, h = ceil(W/2)
  double* lnp_cand;      // [S 2 depth h]
  double* dir;           // [S h, ndim] directions
  double* z0;            // [S h] slice levels
  double* lo;            // [S h] bracket
  double* hi;            // [S h]
  double* tcur;          // [S 2 h] the shrink draws that produced the current candidates (second: speculative)
  int* lit;              // [S h] logical iterations the walker has consumed in this half-step
  int* jbudget;          // [S h] expansions left on the left / right side
  int* kbudget;          // [S h]
  int* phase;            // [S h] kSlice* state
  int* skip;             // [S 2 depth h] row_skip of the lnprob launch (1 = no candidate in this row)
  int* walker_of;        // [S h] global walker index (e W + i) of each row
  int* flag;             // bit 0: a candidate's lnprob was NaN
  SliceCounters* ctr;
  double* mu;                  // [S] (in/out)
  int* adapt;                  // [S, 2] tune, good (in/out)
  unsigned long long* totals;  // [S, 3] expansions, contractions, likelihood rows (accumulated)
  unsigned int* nstep;         // [S, 2] expansions / contractions of the current step
  unsigned long long seed;
  double tolerance;
  int W, ndim, maxsteps, maxiter, patience;
  int depth;             // logical iterations per launch: 1 or 2 (rows per launch: 2 depth n_S per ensemble)
  int S;                 // ensembles (1: rbv_slice_run)
};

// Start of a half-step: direction, slice level, bracket and budgets of every walker of the half (warp per row).
__global__ void __launch_bounds__(128) slice_begin_kernel(const SliceParams P, unsigned long long step, int split) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  int offS, nS, offC, nC;
  split_geometry(P.W, split, offS, nS, offC, nC);
  if (row >= P.S * nS) return;
  const int e = row / nS, k = row - e * nS;
  if (lane == 0) {                 // loop state of this half-step; the iteration kernels are later launches
    if (k == 0 && split == 0) {
      P.nstep[2 * e] = 0u;
      P.nstep[2 * e + 1] = 0u;
    }
    if (row == 0) {
      P.ctr->step = step;
      P.ctr->it = 0u;
      P.ctr->ticket = 0u;
      P.ctr->guard = 0u;
    }
  }
  uint32_t pa, pb;
  sampler_perm(P.seed, P.W, step, pa, pb);
  const int base = e * P.W;
  const int i = base + walker_at(pa, pb, P.W, offS + k);
  const uint4 r = sampler_rand(P.seed, step, (uint32_t)i, 8u + (uint32_t)split);
  const int j = (int)(r.x % (uint32_t)nC);
  const int l = (int)(((uint32_t)j + 1u + r.y % (uint32_t)(nC - 1)) % (uint32_t)nC);   // l != j
  const double* cj = P.coords + (size_t)(base + walker_at(pa, pb, P.W, offC + j)) * P.ndim;
  const double* cl = P.coords + (size_t)(base + walker_at(pa, pb, P.W, offC + l)) * P.ndim;
  const double two_mu = 2.0 * P.mu[e];                  // written by the previous step's slice_record_kernel
  for (int d = lane; d < P.ndim; d += 32) P.dir[(size_t)row * P.ndim + d] = __dmul_rn(two_mu, __dsub_rn(cj[d], cl[d]));
  if (lane == 0) {
    const uint4 q = sampler_rand(P.seed, step, (uint32_t)i, 10u + (uint32_t)split);
    const int J = (int)__dmul_rn((double)P.maxsteps, u01(r.z, r.w));     // floor: the product is >= 0
    const double left = -u01(q.z, q.w);
    P.z0[row] = P.lnp[i] + log(u01(q.x, q.y));                           // lnp - Exp(1)
    P.lo[row] = left;
    P.hi[row] = __dadd_rn(left, 1.0);
    P.jbudget[row] = J;
    P.kbudget[row] = P.maxsteps - 1 - J;
    P.phase[row] = kSliceLeft | kSliceRight;
    P.lit[row] = 0;
    P.walker_of[row] = i;
  }
}

// Candidates of walker-row `row` (= e n_S + k) for the next launch (a whole warp): widening walkers put X + L eta
// into candidate row c = e 2 depth n_S + k and X + R eta into row n_S + c (open ends only), shrinking walkers X + t
// eta with t drawn from (L, R) into row c, the speculative second iteration goes into rows 2 n_S + c and 3 n_S + c;
// every other row is masked.
__device__ __forceinline__ void slice_candidates(const SliceParams& P, int split, int nS, int row, int c, int t,
                                                 int lane, unsigned long long step) {
  const int ph = P.phase[row];
  const bool rowA = (ph & (kSliceLeft | kSliceShrink)) != 0, rowB = (ph & kSliceRight) != 0;
  // second logical iteration (speculative): shrinking -- always; widening -- an end that still has budget
  const bool rowA2 = P.depth > 1 && rowA && ((ph & kSliceShrink) || P.jbudget[row] >= 1);
  const bool rowB2 = P.depth > 1 && rowB && P.kbudget[row] >= 1;
  if (lane == 0) {
    P.skip[c] = !rowA;
    P.skip[nS + c] = !rowB;
    if (P.depth > 1) {
      P.skip[2 * nS + c] = !rowA2;
      P.skip[3 * nS + c] = !rowB2;
    }
  }
  if (!rowA && !rowB) return;
  const int i = P.walker_of[row];
  const double* x = P.coords + (size_t)i * P.ndim;
  const double* e = P.dir + (size_t)row * P.ndim;
  if (rowA) {
    double s = P.lo[row], s2;
    if (ph & kSliceShrink) {
      const unsigned int lit = (unsigned int)P.lit[row];
      const double left = s, right = P.hi[row];
      const uint4 r = sampler_rand(P.seed, step, (uint32_t)i, 16u + 2u * lit + (uint32_t)split);
      s = __dadd_rn(left, __dmul_rn(u01(r.x, r.y), __dsub_rn(right, left)));
      // the draw that follows if s is rejected: the end on s's side moves to s
      const double left2 = (s < 0.0) ? s : left, right2 = (s < 0.0) ? right : s;
      const uint4 r2 = sampler_rand(P.seed, step, (uint32_t)i, 16u + 2u * (lit + 1u) + (uint32_t)split);
      s2 = __dadd_rn(left2, __dmul_rn(u01(r2.x, r2.y), __dsub_rn(right2, left2)));
      if (lane == 0) {
        P.tcur[t] = s;
        P.tcur[nS + t] = s2;
      }
    } else {
      s2 = __dsub_rn(s, 1.0);
    }
    for (int d = lane; d < P.ndim; d += 32) P.cand[(size_t)c * P.ndim + d] = __dadd_rn(x[d], __dmul_rn(s, e[d]));
    if (rowA2)
      for (int d = lane; d < P.ndim; d += 32)
        P.cand[(size_t)(2 * nS + c) * P.ndim + d] = __dadd_rn(x[d], __dmul_rn(s2, e[d]));
  }
  if (rowB) {
    const double s = P.hi[row];
    for (int d = lane; d < P.ndim; d += 32) P.cand[(size_t)(nS + c) * P.ndim + d] = __dadd_rn(x[d], __dmul_rn(s, e[d]));
    if (rowB2) {
      const double s2 = __dadd_rn(s, 1.0);
      for (int d = lane; d < P.ndim; d += 32)
        P.cand[(size_t)(3 * nS + c) * P.ndim + d] = __dadd_rn(x[d], __dmul_rn(s2, e[d]));
    }
  }
}

// First candidates of a half-step (launched once, after slice_begin_kernel; every later iteration gets its candidates
// from slice_update_kernel itself).
__global__ void __launch_bounds__(128) slice_candidate_kernel(const SliceParams P, int split) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  int offS, nS, offC, nC;
  split_geometry(P.W, split, offS, nS, offC, nC);
  if (row >= P.S * nS) return;
  const int e = row / nS, k = row - e * nS;
  if (row == 0 && lane == 0) {    // every warp of the first update kernel runs later
    P.ctr->pending = (unsigned)(P.S * nS);
    P.ctr->remaining = 0u;
    P.ctr->over = 0u;
    P.ctr->guard = 1u;
  }
  slice_candidates(P, split, nS, row, e * 2 * P.depth * nS + k, e * 2 * nS + k, lane, P.ctr->step);
}

// Advance every unfinished walker's state machine with the lnprob of its candidate(s), then write its candidates for
// the next launch (one kernel less per iteration than a separate candidate launch).  The last warp of all S n_S to
// finish closes the iteration: iteration index, batch count, the counters of the next iteration and -- in graph
// mode -- the WHILE node's condition (`loop`, use_loop != 0).  (Minimum of 8 CTAs per SM: without it ptxas aims at 16
// and caps the kernel at 32 registers, which spills once the rows of several ensembles are indexed.)
__global__ void __launch_bounds__(128, 8) slice_update_kernel(const SliceParams P, int split,
                                                           cudaGraphConditionalHandle loop, int use_loop) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  int offS, nS, offC, nC;
  split_geometry(P.W, split, offS, nS, offC, nC);
  if (row >= P.S * nS) return;
  const int e = row / nS, k = row - e * nS;
  const int c = e * 2 * P.depth * nS + k, t = e * 2 * nS + k;    // candidate row, shrink-draw row
  const unsigned long long step = P.ctr->step;     // written by an earlier launch
  int ph = P.phase[row];
  if (!(ph & kSliceDone)) {
    const double z0 = P.z0[row];
    int lit = P.lit[row];
    if (ph & kSliceShrink) {
      // up to `depth` logical iterations: draw d is looked at only if every earlier one was rejected
      unsigned int ncon = 0u, ncall = 0u;
      bool nan = false;
      for (int d = 0; d < P.depth; ++d) {
        const int cr = 2 * d * nS + c;
        const double zs = P.lnp_cand[cr];
        ++ncall;
        ++lit;
        nan |= (zs != zs);
        if (zs >= z0) {                                  // accepted: the candidate becomes the walker
          const int i = P.walker_of[row];
          for (int q = lane; q < P.ndim; q += 32) P.coords[(size_t)i * P.ndim + q] = P.cand[(size_t)cr * P.ndim + q];
          if (lane == 0) P.lnp[i] = zs;
          ph = kSliceDone;
          break;
        }
        if (lane == 0) {                                 // NaN: outside (and flagged)
          const double tt = P.tcur[d * nS + t];
          if (tt < 0.0) P.lo[row] = tt;
          else P.hi[row] = tt;
        }
        ++ncon;
      }
      if (lane == 0) {
        if (nan) atomicOr(P.flag, 1);                    // zeus / emcee: "Probability function returned NaN"
        if (ncon) atomicAdd(&P.nstep[2 * e + 1], ncon);
        atomicAdd(&P.totals[3 * e + 2], (unsigned long long)ncall);
      }
    } else if (lane == 0) {
      unsigned int widened = 0u, evaluated = 0u;
      for (int d = 0; d < P.depth && ph != kSliceShrink; ++d) {
        if (ph & kSliceLeft) {
          const double zs = P.lnp_cand[2 * d * nS + c];
          const int b = P.jbudget[row];
          if (zs != zs) atomicOr(P.flag, 1);
          if (zs >= z0 && b >= 1) {
            P.lo[row] = __dsub_rn(P.lo[row], 1.0);
            P.jbudget[row] = b - 1;
            ++widened;
          } else {
            ph &= ~kSliceLeft;
          }
          ++evaluated;
        }
        if (ph & kSliceRight) {
          const double zs = P.lnp_cand[(2 * d + 1) * nS + c];
          const int b = P.kbudget[row];
          if (zs != zs) atomicOr(P.flag, 1);
          if (zs >= z0 && b >= 1) {
            P.hi[row] = __dadd_rn(P.hi[row], 1.0);
            P.kbudget[row] = b - 1;
            ++widened;
          } else {
            ph &= ~kSliceRight;
          }
          ++evaluated;
        }
        ++lit;
        if (ph == 0) ph = kSliceShrink;
      }
      if (widened) atomicAdd(&P.nstep[2 * e], widened);
      atomicAdd(&P.totals[3 * e + 2], (unsigned long long)evaluated);
    }
    if (lane == 0) {
      P.phase[row] = ph;
      P.lit[row] = lit;
      if (!(ph & kSliceDone)) {
        atomicAdd(&P.ctr->remaining, 1u);
        if (lit > P.maxiter) atomicAdd(&P.ctr->over, 1u);
      }
    }
  }
  __syncwarp();                       // lane 0's state of this walker -> the whole warp
  slice_candidates(P, split, nS, row, c, t, lane, step);      // (a finished walker masks all its rows)
  __syncwarp();
  if (lane == 0) {
    __threadfence();
    if (atomicAdd(&P.ctr->ticket, 1u) == (unsigned)(P.S * nS) - 1u) {   // every row of the half has been updated
      P.ctr->ticket = 0u;
      const unsigned int rem = atomicAdd(&P.ctr->remaining, 0u);
      const unsigned int over = atomicAdd(&P.ctr->over, 0u);
      P.ctr->pending = rem;
      P.ctr->remaining = 0u;                                        // counters of the next iteration: its update
      P.ctr->over = 0u;                                             // kernel is a later launch
      const unsigned int it = P.ctr->it + 1u;
      P.ctr->it = it;
      P.ctr->batches += 1ull;
      bool go = rem > 0u;
      if (go && over > 0u) {                                        // zeus: "Number of contractions exceeded ..."
        P.ctr->error = 1;
        go = false;
      }
      if (go) {                                                     // second, independent loop bound
        const unsigned int g = P.ctr->guard + 1u;
        P.ctr->guard = g;
        if (g > (unsigned)P.maxiter + 8u) {
          P.ctr->error = 1;
          go = false;
        }
      }
      if (use_loop) cudaGraphSetConditional(loop, go ? 1u : 0u);
      __threadfence();
    }
  }
}

// End of a step: the ensembles and their lnprob become row s of the chain (warp per walker); the first thread of
// each ensemble adapts its mu (zeus: stochastic approximation towards an expansion fraction of 1/2) for the next step.
__global__ void __launch_bounds__(128) slice_record_kernel(const SliceParams P, double* __restrict__ chain_row,
                                                           double* __restrict__ lnp_row, double* __restrict__ mu_out) {
  const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (w >= P.S * P.W) return;
  if (chain_row)
    for (int d = lane; d < P.ndim; d += 32) chain_row[(size_t)w * P.ndim + d] = P.coords[(size_t)w * P.ndim + d];
  if (lnp_row && lane == 0) lnp_row[w] = P.lnp[w];
  const int e = w / P.W;
  if (w == e * P.W && lane == 0) {
    const unsigned int nexp = P.nstep[2 * e], ncon = P.nstep[2 * e + 1];
    P.totals[3 * e] += nexp;
    P.totals[3 * e + 1] += ncon;
    double mu = P.mu[e];
    if (P.adapt[2 * e]) {
      const double ne = (double)max(nexp, 1u), tot = ne + (double)ncon;
      mu = __dmul_rn(mu, __ddiv_rn(__dmul_rn(2.0, ne), tot));
      P.mu[e] = mu;
      int good = P.adapt[2 * e + 1];
      if (fabs(__ddiv_rn(ne, tot) - 0.5) < P.tolerance) P.adapt[2 * e + 1] = ++good;
      if (good > P.patience) P.adapt[2 * e] = 0;
    }
    if (mu_out) mu_out[e] = mu;
  }
}

}  // namespace rbv
