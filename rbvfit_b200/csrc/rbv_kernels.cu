// rbvfit_b200 -- fused Voigt forward model + likelihood kernels for sm_100a, and their C ABI.
//
// One CTA = one (walker, pixel tile).  Per CTA:
//   prep    (prep_kernel, once per walker) theta row -> per-line constants (A, B, a^2, kappa-scaled series
//           coefficients; _evaluate_compiled_model :192-200 and _vectorized_voigt_tau :142-150) + prior flag
//   phase 0 per 1024-pixel super-chunk: tier of every line from the chunk's range of 1/lambda, and the far-field
//           record: the summed far wings at 8 Chebyshev nodes -> 8 polynomial coefficients (DESIGN.md 4c)
//   phase 1 tau_p = far-field polynomial + sum over the remaining lines coef_l H(a_l, x_lp) for the tile's pixels
//           + LSF halo, flux = exp(-tau) into shared memory (edge pixels replicated = ndimage 'nearest' /
//           astropy 'extend')
//   phase 2 LSF convolution from shared memory with R outputs per thread (register-blocked sliding
//           window), then either the chi^2 partial of vfit.lnlike (vfit_mcmc.py:309-311) reduced with
//           warp shuffles, or the model flux written out
//   final   the last CTA of a walker (atomic ticket) adds the tile partials in fixed order, applies
//           -0.5 per instrument, and writes lnprob; rows outside [lb, ub] get -inf without evaluation
//           (vfit.lnprior :291-295, lnprob :348-353).
//
// Data layout in HBM (all float64): per instrument 1/wave, flux, inv_sigma2, log_inv_sigma2 [P] shared by
// every walker (L2-resident) + derived block tables; theta [W, ndim] row-major; lnprob [W]; workspace = tickets,
// prior flags, tile partials [W, n_tiles], line constants [W, L, 22].  No per-line optical depth is ever
// materialised.
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/rbvfit_b200.h"
#include "rbv_device.cuh"
#include "rbv_sampler.cuh"   // StretchParams + Philox streams (embedded in LaunchParams for the fused sampler step)
#include "rbv_pt.cuh"        // parallel tempering: swap stage and record (rbv_pt_run)
#include "rbv_slice.cuh"     // device-resident ensemble slice sampler (kernels around the lnprob launch)

namespace rbv {

// ------------------------------------------------------------------------------------------ device structs
struct InstDev {
  const double* inv_wave;
  const double* flux;
  const double* inv_sigma2;
  const double* log_inv_sigma2;
  const double* lambda0;   // [L]
  const double* gamma;     // [L]
  const double* f;         // [L]
  const double* zfac;      // [L]
  const int* comp;         // [L]
  const double2* ublk;     // [ceil(P / 256)] (min, max) of 1/wave over aligned 256-pixel blocks
  const double2* useg;     // [ceil(P / 1024)] (min, max) of 1/wave over pixels K/2 + 1024 s .. + 1023 (clamped): the
                           // super-chunks of the streaming kernel
  const double* taps_rev;  // [Kpad] flipped taps, zero padded to a multiple of R
  double sum_log_inv_sigma2;   // sum_p log_inv_sigma2[p] (theta-independent part of lnlike), fixed order
  const double2* obs_w;        // (flux, inv_sigma2) pairs re-ordered per 256-pixel block so that phase 2 loads them
                               // coalesced: element (lane, r) = pixel 256 J + 8 lane + r sits at 256 J + 32 r + lane
  int P, K, Kpad, L, C, method;
  int R;                   // register blocking of the LSF stage (context-wide)
  int line_base;           // first row of this instrument in the per-walker line-constant block
};

// Tile geometry of one instrument for ONE launch (chosen per launch from the batch size: big tiles when
// there are plenty of walkers, small ones when the grid would otherwise not fill the GPU).
struct TileGeom {
  int tile;        // output pixels per CTA
  int ext_alloc;   // flux slots per CTA in shared memory (tile + halo + slack)
  int first_tile;  // index of this instrument's first tile in the launch's tile list
  int n_tiles;
  int n_super;     // super-chunks (kSuperPix flux slots) per CTA
};
constexpr int kMaxInst = 16;
constexpr int kMaxStreamRanges = 128;   // slots (ranges of all instruments) of one streaming launch

struct LaunchParams {
  const InstDev* inst;
  TileGeom geom[kMaxInst];
  const double* theta;   // [W, ndim]
  const double* lb;
  const double* ub;
  const double* core_tab;
  double* lnprob;        // [W]
  double* partials;      // [W, n_tiles]
  unsigned int* tickets; // [W]
  int* oob;              // [W] 1 = row violates the prior bounds (written by prep_kernel)
  const int* row_skip;   // [W] or NULL: rows with a non-zero entry are not evaluated at all (their lnprob is -inf);
                         // the slice sampler masks the walkers that have finished their half-step this way
  double* lc;            // [W, n_lines_total, LC_STRIDE] per-walker line constants (written by prep_kernel)
  double* out_flux;      // flux mode: [W, P]
  int ndim, n_tiles, n_inst, W, n_lines_total;
  int tile_base;         // flux mode: first tile of the instrument
  int precision;
  int farfield;          // 1 = far wings of a chunk through the Chebyshev far-field interpolant (section 4c)
  double ff_budget;      // far-field error budget in optical depth per pixel, summed over lines (kFFEps)
  int wps;               // sightline mode: walkers per sightline (walker w belongs to instrument w / wps); 0 = off
  // device-resident sampler (rbv_stretch_run): when sampler_split >= 0 the prep kernel first builds the stretch
  // proposal of row w, and the CTA that finalises lnprob[w] also applies accept/reject and records the chain
  int sampler_split;
  int separate_finalize; // 1 = lnprob is formed by finalize_kernel (big grids), 0 = by the walker's last CTA
  int inst_in_params;    // 1 = inst_v holds the instruments (joint fits: no global round trip in the CTA prologue)
  StretchParams sp;
  InstDev inst_v[kMaxInst];
  // streaming kernel: slot s (a range of one instrument, see TileGeom::first_tile) covers the 1024-pixel segments
  // [range_lo[s], range_hi[s]) of its instrument
  unsigned short range_lo[kMaxStreamRanges], range_hi[kMaxStreamRanges];
  // streaming kernel: boundary records [W, n_tiles, bnd_stride]: record (w, s) = the 2 (K - 1) flux values around the
  // first output of range s -- the K - 1 in front written by range s - 1 (its last carry), the K - 1 behind by range
  // s (the head of its first row); finalize adds the K - 1 outputs that straddle the boundary.  NULL otherwise.
  double* bnd;
  int bnd_stride;
};

__device__ __forceinline__ int smem_pos(int i, int logR) { return i + (i >> logR); }

// ticket = (*counter)++ on a shared-memory counter: one ATOMS instruction (atomicAdd on the generic address costs
// an address-space check and a dozen instructions per draw)
__device__ __forceinline__ int smem_ticket(int* counter) {
  int t;
  asm volatile("atom.shared.add.u32 %0, [%1], 1;"
               : "=r"(t) : "r"((unsigned)__cvta_generic_to_shared(counter)) : "memory");
  return t;
}

// ------------------------------------------------------------------------------------------ prep
// per-line constants for the wofz method
__device__ __forceinline__ void prep_line_wofz(const InstDev& I, int l, const double* __restrict__ th,
                                               double* __restrict__ lc) {
  int c = I.comp[l];
  double logN = th[c], b = th[I.C + c], v = th[2 * I.C + c];
  double lam0 = I.lambda0[l], gam = I.gamma[l], f = I.f[l], zf = I.zfac[l];
  double N = pow(10.0, logN);                       // 10**theta[N_indices], voigt_model.py:192
  double b_f = b / lam0 * 1e13;                     // :142
  double nu0 = kCFreq / lam0;                       // :143
  double konst = kAtomicConst / (nu0 * b);          // :146
  double a = gam / (kFourPi * b_f);                 // :149
  double zt = zf * (1.0 + v / kCkms) - 1.0;         // :200
  double opz = 1.0 + zt;                            // :204
  double coef = N * f * konst;                      // :158  ((N*f)*constant)
  double A = kCFreq * opz / b_f;                    // x = (c/(lambda/(1+zt)) - nu0)/b_f = A/lambda - B
  double B = nu0 / b_f;
  if (!(b > 0.0)) {  // b <= 0 or NaN: outside the model's domain (documented: NaN)
    A = B = a = coef = CUDART_NAN;
  }
  double a2 = a * a;
  lc[LC_A] = A;
  lc[LC_B] = B;
  lc[LC_A2] = a2;
  lc[LC_a] = a;
  lc[LC_COEF] = coef;
  lc[LC_F32B] = 0.0;
  lc[LC_F32A] = lc[LC_F32A + 1] = 0.0;
  lc[LC_AUX] = coef * a * kInvSqrtPi;  // kappa
}

// FP32 copies of the far-tier constants (A, a^2, Q1..Q3) for the gated FP32 path
// ... and the far-field gate of the streaming kernel's phase 0 solved for the distance: the a-priori bound
// 8 (m + 1) kappa (hw / (2 xm))^m / xm^2 <= eps with hw = |A| du / 2 (classify_lines) holds exactly when
// xm >= G du^(m / (m + 2)),  G = [8 (m + 1) |kappa| (|A| / 4)^m / eps]^(1 / (m + 2))  -- one number per (walker, line).
__device__ __forceinline__ void fill_fp32_constants(double* __restrict__ lc, double ff_eps) {
  float4 fa = make_float4((float)lc[LC_A], (float)lc[LC_A2], (float)lc[LC_Q], (float)lc[LC_Q + 1]);
  const double G = (ff_eps > 0.0)
      ? exp2((log2(8.0 * (RBV_FF_M + 1) * 1.001 * fabs(lc[LC_AUX]) / ff_eps) + RBV_FF_M * log2(0.25 * fabs(lc[LC_A]))) /
             (RBV_FF_M + 2))
      : CUDART_INF;
  float2 fb = make_float2((float)lc[LC_Q + 2], (float)G * 1.0001f);       // rounded to the conservative side
  *reinterpret_cast<float4*>(lc + LC_F32A) = fa;
  *reinterpret_cast<float2*>(lc + LC_F32B) = fb;
}

// per-line constants for the Tepper-Garcia method (voigt_approx.py:69-86)
__device__ __forceinline__ void prep_line_fast(const InstDev& I, int l, const double* __restrict__ th,
                                               double* __restrict__ lc) {
  prep_line_wofz(I, l, th, lc);
  double a = lc[LC_a];
  lc[LC_A2] = fmax(1e-2, 100.0 * fabs(a) / kSqrtPi);  // eps
  lc[LC_a] = a / kSqrtPi;                             // a / sqrt_pi
  lc[LC_AUX] = 1.0 - 2.0 * a / kSqrtPi;               // core factor
}

// ------------------------------------------------------------------------------------------ phase 1
extern __shared__ double smem[];   // every hot-loop access indexes this array directly (shared-space addressing)

// Tier codes of a (warp chunk, line) pair
constexpr int kTierFar = 0, kTierMid = 1, kTierNear = 2, kTierCore = 3, kTierGeneral = 4, kTierFar32 = 5,
              kTierFF = 6;
// Far-field budget: the interpolation errors of all lines of one pixel sum to <= kFFEps in optical depth
// (flux error <= 1e-12, two decades inside the 1e-10 parity tolerance; the bound is conservative -- measured against
// the direct evaluation on the C1..C5a workloads the flux differs by <= 2e-14, profiles/r02_notes.md).
constexpr double kFFEps = 1e-12;

// Classify every line once per warp chunk from the chunk's range of 1/lambda (lane l handles line l):
// far lines go to the front of the warp's list, everything else to the back with its tier in the top bits.
// Returns (n_far, n_other).  Conservative: uses the smallest |z|^2 any pixel of the chunk can reach; the
// comparisons run on the high words of the doubles (integer pipe, thresholds have zero low words).
// A NaN line lands in the far list and its NaN propagates through the arithmetic.
// With gate32 > 0, far lines whose largest possible contribution over the chunk, kappa / min|z|^2, is at most
// gate32 go to a second list (list32) and are evaluated on the FP32 pipe; returns their count in .z.
// With ff_eps > 0, far lines whose wing is smooth enough over the chunk go to listff (count in .w): the chunk
// then evaluates their SUM at RBV_FF_M Chebyshev nodes and interpolates it.  A-priori error bound of the
// degree-(m-1) Chebyshev interpolant of kappa/x^2 on [xm, xm + 2 hw] (m-th derivative (m+1)!/x^(m+2)):
//     |err| <= 2 (m+1) kappa (hw / (2 xm))^m / xm^2;
// the gate uses 8 (m+1): the 4x margin covers the a^2 and rho^2, rho^3, ... corrections, whose m-th derivatives
// add <= 6 % at the smallest admitted distance (|z|^2 >= 576, a <= 1: the mid and far tiers, evaluated at the
// nodes with the 6-term series); it runs in FP32 with every rounding pushed to the conservative side.
__device__ __forceinline__ int4 classify_lines(int lc_off, int L, unsigned short* __restrict__ list,
                                               unsigned short* __restrict__ list32,
                                               unsigned short* __restrict__ listff, double gate32, float ff_eps,
                                               double umin, double umax, int lane) {
  int n_far = 0, n_oth = 0, n_32 = 0, n_ff = 0;
  const double du = umax - umin;
  const unsigned lt = (1u << lane) - 1u;
  for (int l0 = 0; l0 < L; l0 += 32) {
    const int l = l0 + lane;
    const bool valid = l < L;
    int tier = kTierCore;
    if (valid) {
      const int off = lc_off + l * LC_STRIDE;
      const double A = smem[off + LC_A], B = smem[off + LC_B], a2 = smem[off + LC_A2];
      const double x1 = fma(A, umin, -B), x2 = fma(A, umax, -B);
      const int h1 = __double2hiint(fma(x1, x1, a2)), h2 = __double2hiint(fma(x2, x2, a2));
      const int ha = __double2hiint(a2);
      const bool crosses = ((__double2hiint(x1) ^ __double2hiint(x2)) < 0);   // line centre inside the chunk
      const int hmin = crosses ? ha : min(h1, h2);
      tier = (ha >= 0x3ff00000) ? kTierGeneral      // a >= 1
             : (hmin >= kHiFar) ? kTierFar
             : (hmin >= kHiNear) ? kTierMid
             : (hmin >= kHiCore) ? kTierNear
                                 : kTierCore;
      if (ff_eps > 0.f && (tier == kTierFar || tier == kTierMid)) {   // |z|^2 >= 576: the 6-term series is exact
        const float xm = fminf(fabsf((float)x1), fabsf((float)x2)) * 0.99999f;     // rounded towards the line
        const float hw = (float)(0.5 * fabs(A) * du) * 1.00001f;
        const float r = __fdividef(hw, 2.f * xm) * 1.00001f;
        const float r2 = r * r, r4 = r2 * r2;
        const float bound = (8.f * (RBV_FF_M + 1) * 1.001f) * fabsf((float)smem[off + LC_AUX]) *
                            __fdividef(r4 * r4, xm * xm);
        if (bound <= ff_eps) tier = kTierFF;       // NaN fails the comparison and stays on the direct path
      }
      if (gate32 > 0.0 && tier == kTierFar) {
        // kappa / dmin with dmin rounded DOWN to its high word: an upper bound of the line's contribution
        const double tmax = fabs(smem[off + LC_AUX]) / __hiloint2double(hmin, 0);
        if (tmax <= gate32) tier = kTierFar32;     // NaN fails the comparison and stays on the FP64 path
      }
    }
    const unsigned far_mask = __ballot_sync(0xffffffffu, valid && tier == kTierFar);
    const unsigned f32_mask = __ballot_sync(0xffffffffu, valid && tier == kTierFar32);
    const unsigned ff_mask = __ballot_sync(0xffffffffu, valid && tier == kTierFF);
    const unsigned oth_mask = __ballot_sync(0xffffffffu, valid && tier != kTierFar && tier != kTierFar32 &&
                                                             tier != kTierFF);
    if (valid) {
      if (tier == kTierFar) list[n_far + __popc(far_mask & lt)] = (unsigned short)l;
      else if (tier == kTierFar32) list32[n_32 + __popc(f32_mask & lt)] = (unsigned short)l;
      else if (tier == kTierFF) listff[n_ff + __popc(ff_mask & lt)] = (unsigned short)l;
      else list[L - 1 - (n_oth + __popc(oth_mask & lt))] = (unsigned short)(l | (tier << 12));
    }
    n_far += __popc(far_mask);
    n_32 += __popc(f32_mask);
    n_ff += __popc(ff_mask);
    n_oth += __popc(oth_mask);
  }
  __syncwarp();
  return make_int4(n_far, n_oth, n_32, n_ff);
}

// FP32 far-wing accumulation for the gated lines.  x = X0 + A du with X0 = A u_ref - B formed in FP64 once per
// (line, chunk) and du = u - u_ref exact in FP64, both then rounded to FP32 (no cancellation left in FP32);
// two pixels share one MUFU.RCP through 1/(d1 d2).  Error model (DESIGN.md section 4b): relative 3e-7 per
// contribution + 6e-8 per FP32 accumulation step; the gate bounds the gated sum by 4e-6, i.e. |dtau| <= 1e-11.
template <int PPT>
__device__ __forceinline__ void accum_far32(int lc_off, const unsigned short* __restrict__ list32, int n32,
                                            const double (&u)[PPT], double (&tau)[PPT]) {
  static_assert(PPT % 2 == 0, "pairs of pixels share one reciprocal");
  const double u_ref = __shfl_sync(0xffffffffu, u[0], 0);
  float du[PPT], acc[PPT];
#pragma unroll
  for (int j = 0; j < PPT; ++j) {
    du[j] = (float)(u[j] - u_ref);
    acc[j] = 0.f;
  }
#pragma unroll 2
  for (int k = 0; k < n32; ++k) {
    const int off = lc_off + (int)list32[k] * LC_STRIDE;
    const float X0 = (float)fma(smem[off + LC_A], u_ref, -smem[off + LC_B]);
    const float4 c = *reinterpret_cast<const float4*>(smem + off + LC_F32A);   // A, a^2, Q1, Q2
    const float q3 = reinterpret_cast<const float2*>(smem + off + LC_F32B)->x;
#pragma unroll
    for (int j = 0; j < PPT; j += 2) {
      const float x0 = fmaf(c.x, du[j], X0), x1 = fmaf(c.x, du[j + 1], X0);
      const float d0 = fmaf(x0, x0, c.y), d1 = fmaf(x1, x1, c.y);
      float r;
      asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(d0 * d1));
      const float r0 = r * d1, r1 = r * d0;
      acc[j] = fmaf(fmaf(fmaf(q3, r0, c.w), r0, c.z), r0, acc[j]);
      acc[j + 1] = fmaf(fmaf(fmaf(q3, r1, c.w), r1, c.z), r1, acc[j + 1]);
    }
  }
#pragma unroll
  for (int j = 0; j < PPT; ++j) tau[j] += (double)acc[j];
}

template <int NQ, int PPT>
__device__ __forceinline__ void accum_asym_line(int off, const double (&u)[PPT], double (&tau)[PPT]) {
  const double A = smem[off + LC_A], B = smem[off + LC_B], a2 = smem[off + LC_A2];
  double Q[NQ];
#pragma unroll
  for (int p = 0; p < NQ; ++p) Q[p] = smem[off + LC_Q + p];
#pragma unroll
  for (int j = 0; j < PPT; ++j) {
    const double x = fma(A, u[j], -B);
    const double rho = rcp_pos(fma(x, x, a2));
    double s = Q[NQ - 1];
#pragma unroll
    for (int p = NQ - 2; p >= 0; --p) s = fma(s, rho, Q[p]);
    tau[j] = fma(s, rho, tau[j]);
  }
}

// Far field of one super-chunk (DESIGN.md section 4c).  The listed lines are all >= 200 Doppler widths away from
// every pixel of the super-chunk, where their summed optical depth
//     g(u) = sum_l kappa_l rho_l (q1 + q2 rho_l + q3 rho_l^2)
// is an analytic, slowly varying function of u = 1/lambda.  Instead of n_ff series evaluations per pixel:
//   phase 0, once per super-chunk (one warp):
//   1. lane = line: evaluate the line at the RBV_FF_M Chebyshev nodes of [umin, umax] (same 8-FMA body as the
//      direct far tier, ILP 8 over the nodes);
//   2. transpose-reduce over the lanes (through shared memory, fixed order) -> node sums S_k;
//   3. lanes 0..7: monomial coefficients c_j = sum_k MINV[j][k] S_k (constant matrix, generated in 60-digit
//      arithmetic) -> the super-chunk's record in shared memory, with the affine map u -> t in [-1, 1];
//   phase 1, every pixel: t = u * scale + offset (one FMA), tau = Horner_7(t): 8 FMAs whatever the number of lines.
// Fixed evaluation order -> bit-reproducible for a given tile geometry.
constexpr int SC_COEF = 0, SC_SCALE = 8, SC_OFFSET = 9, SC_COUNTS = 10 /* 4 ints */, SC_STRIDE = 12;

__device__ __forceinline__ void farfield_coefficients(int lc_off, const unsigned short* __restrict__ listff,
                                                      int n_ff, double umin, double umax, int rec_off,
                                                      int scratch_off, int lane) {
  static_assert(RBV_FF_M == 8, "far-field code is written for 8 nodes");
  const double um = 0.5 * (umin + umax), uh = 0.5 * (umax - umin);
  double S[8];
  {
    double un[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      un[k] = fma(uh, c_ff_nodes[k], um);
      S[k] = 0.0;
    }
    if (lane < n_ff) accum_asym_line<kNQMid, 8>(lc_off + (int)listff[lane] * LC_STRIDE, un, S);
    // lines beyond the first 32 (L = 33 is a common case: one line would cost a whole second round of 8 node
    // evaluations per lane): one (line, node) pair per lane -- node = lane & 7, lines 32 + (lane >> 3) + 4 i --
    // summed over the four lane groups in fixed order into column 32 of the transpose scratch
    double rest = 0.0;
    if (n_ff > 32) {
      double un1[1], v[1];
      un1[0] = fma(uh, c_ff_nodes[lane & 7], um);
      v[0] = 0.0;
      for (int i = 32 + (lane >> 3); i < n_ff; i += 4) accum_asym_line<kNQMid, 1>(lc_off + (int)listff[i] * LC_STRIDE, un1, v);
      rest = v[0];
      rest += __shfl_xor_sync(0xffffffffu, rest, 8);
      rest += __shfl_xor_sync(0xffffffffu, rest, 16);
    }
    if (lane < 8) smem[scratch_off + lane * 33 + 32] = rest;
  }
  // transpose-reduce through shared memory (the flux tile is still unused in phase 0): lane writes its 8 node
  // values, then lane (k = lane >> 2, q = lane & 3) adds the values of lanes 8q .. 8q+7 for node k in lane order and
  // two shuffle-adds finish the sum -- fixed order, 8 STS + 8 LDS + 10 adds instead of a 3-level select/shuffle tree
  double T1 = 0.0;
  {
    const int base = scratch_off;                   // [8 nodes][33] doubles of this warp
#pragma unroll
    for (int k = 0; k < 8; ++k) smem[base + k * 33 + lane] = S[k];
    __syncwarp();
    const int rd = base + (lane >> 2) * 33 + (lane & 3) * 8;
#pragma unroll
    for (int i = 0; i < 8; ++i) T1 += smem[rd + i];
    if ((lane & 3) == 0) T1 += smem[base + (lane >> 2) * 33 + 32];      // the lines beyond the first 32
    T1 += __shfl_xor_sync(0xffffffffu, T1, 1);
    T1 += __shfl_xor_sync(0xffffffffu, T1, 2);     // every lane: S_k of node k = lane >> 2
    __syncwarp();
  }
  double c = 0.0;                                   // lane j < 8: c_j = sum_k MINV[j][k] S_k
#pragma unroll
  for (int k = 0; k < 8; ++k) c = fma(c_ff_minv[(lane & 7) * 8 + k], __shfl_sync(0xffffffffu, T1, 4 * k), c);
  const double sc = rcp_pos(uh);                      // uh > 0 (umax carries an all-ones low word)
  if (lane < 8) smem[rec_off + SC_COEF + lane] = c;
  if (lane == 8) smem[rec_off + SC_SCALE] = sc;
  if (lane == 9) smem[rec_off + SC_OFFSET] = -um * sc;
}

// same series from precomputed |z|^2
template <int NQ, int PPT>
__device__ __forceinline__ void accum_asym_from_d(int off, const double (&d)[PPT], double (&tau)[PPT]) {
  double Q[NQ];
#pragma unroll
  for (int p = 0; p < NQ; ++p) Q[p] = smem[off + LC_Q + p];
#pragma unroll
  for (int j = 0; j < PPT; ++j) {
    const double rho = rcp_pos(d[j]);
    double s = Q[NQ - 1];
#pragma unroll
    for (int p = NQ - 2; p >= 0; --p) s = fma(s, rho, Q[p]);
    tau[j] = fma(s, rho, tau[j]);
  }
}

template <int PPT>
__device__ __forceinline__ void farfield_eval(int rec_off, const double (&u)[PPT], double (&tau)[PPT]) {
  double c[8];
#pragma unroll
  for (int j = 0; j < 8; j += 2) {
    const double2 v = *reinterpret_cast<const double2*>(smem + rec_off + SC_COEF + j);
    c[j] = v.x;
    c[j + 1] = v.y;
  }
  const double2 so = *reinterpret_cast<const double2*>(smem + rec_off + SC_SCALE);
#pragma unroll
  for (int j = 0; j < PPT; ++j) {
    const double t = fma(u[j], so.x, so.y);
    double p = c[7];
#pragma unroll
    for (int q = 6; q >= 0; --q) p = fma(p, t, c[q]);
    tau[j] = p;                                        // tau starts from the far field
  }
}

// Phase 0 for one super-chunk (one warp): range of 1/lambda over the aligned 256-pixel blocks that cover its
// pixels [plo, phi] (from the per-instrument block table: no monotonicity assumed), tier lists, far-field record.
__device__ __forceinline__ void prepare_super_chunk(const InstDev& I, int lc_off, int rec_off,
                                                    unsigned short* __restrict__ list,
                                                    unsigned short* __restrict__ list32,
                                                    unsigned short* __restrict__ listff, double gate32,
                                                    float ff_eps, int plo, int phi, int scratch_off, int lane) {
  int hlo = 0x7fffffff, hhi = 0;
  for (int b = (plo >> 8) + lane; b <= (phi >> 8); b += 32) {
    const double2 mm = I.ublk[b];
    hlo = min(hlo, __double2hiint(mm.x));
    hhi = max(hhi, __double2hiint(mm.y));
  }
  hlo = __reduce_min_sync(0xffffffffu, hlo);       // 1/lambda > 0: the high words order like the values
  hhi = __reduce_max_sync(0xffffffffu, hhi);
  const double umin = __hiloint2double(hlo, 0), umax = __hiloint2double(hhi, (int)0xffffffff);
  const int4 n = classify_lines(lc_off, I.L, list, list32, listff, gate32, ff_eps, umin, umax, lane);
  if (n.w > 0) farfield_coefficients(lc_off, listff, n.w, umin, umax, rec_off, scratch_off, lane);
  else if (lane < SC_COUNTS) smem[rec_off + lane] = 0.0;          // zero polynomial, t = 0
  if (lane == 0) *reinterpret_cast<int4*>(smem + rec_off + SC_COUNTS) = n;
}

template <int PPT>
__device__ __forceinline__ void tau_wofz(int lc_off, int L, const unsigned short* __restrict__ list,
                                         const unsigned short* __restrict__ list32, int rec_off,
                                         const double (&u)[PPT], double (&tau)[PPT],
                                         const double* __restrict__ core_tab) {
  const int4 n = *reinterpret_cast<const int4*>(smem + rec_off + SC_COUNTS);   // n_far, n_other, n_fp32, n_farfield
  // big tiles: the record always holds a polynomial (all-zero coefficients when no line qualified), so tau needs
  // no separate zeroing and no branch; small tiles often have no far field at all and keep the test
  if (PPT == 8 || n.w > 0) {
    farfield_eval(rec_off, u, tau);
  } else {
#pragma unroll
    for (int j = 0; j < PPT; ++j) tau[j] = 0.0;
  }
  if (n.z > 0) accum_far32(lc_off, list32, n.z, u, tau);

  // far lines: branch-free body, 8 FP64 instructions per (line, pixel)
#pragma unroll 2
  for (int k = 0; k < n.x; ++k) accum_asym_line<kNQFar, PPT>(lc_off + (int)list[k] * LC_STRIDE, u, tau);

  // everything else (a few lines per chunk at most)
  for (int k = 0; k < n.y; ++k) {
    const int e = list[L - 1 - k];
    const int off = lc_off + (e & 0xfff) * LC_STRIDE;
    const int tier = e >> 12;
    if (tier == kTierMid) {
      accum_asym_line<kNQMid, PPT>(off, u, tau);
    } else if (tier == kTierNear) {
      accum_asym_line<kNQNear, PPT>(off, u, tau);
    } else {
      const double A = smem[off + LC_A], B = smem[off + LC_B], a2 = smem[off + LC_A2], a = smem[off + LC_a],
                   coef = smem[off + LC_COEF];
      if (tier == kTierGeneral) {
#pragma unroll
        for (int j = 0; j < PPT; ++j) {   // unrolled: tau/u must stay in registers
          const double x = fma(A, u[j], -B);
          tau[j] = fma(coef, general_H(x, a, fma(x, x, a2)), tau[j]);
        }
      } else {
        if (PPT == 2) {
          // small tiles (64-pixel chunks): the tier was taken over the whole super-chunk, refine it for this chunk
          // from the pixels themselves -- a super-chunk that holds a line core is mostly wing.  (Measured: +4 %
          // on the sightline workload; with 8 pixels per lane the extra warp reduction costs more than it saves.)
          double x[PPT], d[PPT];
          int hmin = 0x7fffffff;
#pragma unroll
          for (int j = 0; j < PPT; ++j) {
            x[j] = fma(A, u[j], -B);
            d[j] = fma(x[j], x[j], a2);
            hmin = min(hmin, __double2hiint(d[j]));
          }
          hmin = __reduce_min_sync(0xffffffffu, hmin);
          if (hmin >= kHiNear) {
            accum_asym_from_d<kNQMid, PPT>(off, d, tau);
          } else if (hmin >= kHiCore) {
            accum_asym_from_d<kNQNear, PPT>(off, d, tau);
          } else {
#pragma unroll
            for (int j = 0; j < PPT; ++j) {
              if (d[j] < kDCore) tau[j] = fma(coef, core_H(x[j], a, a2, core_tab), tau[j]);
              else tau[j] += asym_series<kNQNear>(smem + off + LC_Q, d[j]);
            }
          }
        } else {
#pragma unroll
          for (int j = 0; j < PPT; ++j) {
            const double x = fma(A, u[j], -B);
            const double d = fma(x, x, a2);
            if (d < kDCore) tau[j] = fma(coef, core_H(x, a, a2, core_tab), tau[j]);
            else tau[j] += asym_series<kNQNear>(smem + off + LC_Q, d);
          }
        }
      }
    }
  }
}

template <int PPT>
__device__ __forceinline__ void tau_fast(int lc_off, int L, const double (&u)[PPT], double (&tau)[PPT]) {
#pragma unroll
  for (int j = 0; j < PPT; ++j) tau[j] = 0.0;
  for (int l = 0; l < L; ++l) {
    const int off = lc_off + l * LC_STRIDE;
    const double A = smem[off + LC_A], B = smem[off + LC_B], eps = smem[off + LC_A2], aos = smem[off + LC_a],
                 cf = smem[off + LC_AUX], coef = smem[off + LC_COEF];
#pragma unroll
    for (int j = 0; j < PPT; ++j) {
      double x = fma(A, u[j], -B);
      tau[j] = fma(coef, tg_H(x, aos, eps, cf), tau[j]);
    }
  }
}

// ------------------------------------------------------------------------------------------ prep kernel
// One thread per (walker, line of any instrument): theta row -> the 20-double line-constant record, once per
// walker instead of once per tile (pow, five divisions and the 13 series coefficients are ~400 dependent
// FP64 instructions -- as long as a tile's whole phase 1 when done by 33 threads of every CTA).
// The walker's first block also evaluates the uniform prior (vfit.lnprior, vfit_mcmc.py:291-295), one parameter per
// thread + a block-wide OR (a single thread walking 36 parameters was a 3 us chain of dependent L2 round trips).
__device__ __forceinline__ void prep_walker_lines(const LaunchParams& prm, int w, int g, const double* __restrict__ th) {
  const bool skipped = prm.row_skip != nullptr && prm.row_skip[w] != 0;
  if (blockIdx.y == 0) {   // the walker's first block (every thread of it gets here): one parameter per thread
    int bad = skipped;
    if (prm.lb != nullptr) {     // the flux entry point has no prior
      for (int i = threadIdx.x; i < prm.ndim; i += blockDim.x) {
        const double t = th[i];
        bad |= (t < prm.lb[i]) || (t > prm.ub[i]);
      }
    }
    bad = __syncthreads_or(bad);
    if (threadIdx.x == 0) {
      prm.oob[w] = bad;
      prm.tickets[w] = 0u;   // the workspace layout depends on W: never trust ticket state from an earlier call
      if (w == 0) prm.tickets[prm.W] = 0u;     // work-queue counter of the streaming kernel
    }
  }
  if (g >= prm.n_lines_total || skipped) return;
  int k = 0, l = g;
  if (prm.wps > 0) {
    k = w / prm.wps;                       // sightline mode: the walker's own instrument, all L lines
  } else {
    const InstDev* tab = prm.inst_in_params ? prm.inst_v : prm.inst;
    while (k + 1 < prm.n_inst && g >= tab[k + 1].line_base) ++k;
    l = g - tab[k].line_base;
  }
  const InstDev& I = prm.inst_in_params ? prm.inst_v[k] : prm.inst[k];
  __align__(16) double lc[LC_STRIDE];
  if (I.method == RBV_VOIGT_FAST) {
    prep_line_fast(I, l, th, lc);
  } else {
    prep_line_wofz(I, l, th, lc);
#pragma unroll
    for (int p = 0; p < kNQNear; ++p) lc[LC_Q + p] = asym_coef(p + 1, lc[LC_A2], lc[LC_AUX]);
    fill_fp32_constants(lc, prm.farfield ? prm.ff_budget / (double)I.L : 0.0);
  }
  double2* dst = reinterpret_cast<double2*>(prm.lc + ((size_t)w * prm.n_lines_total + g) * LC_STRIDE);
#pragma unroll
  for (int i = 0; i < LC_STRIDE / 2; ++i) dst[i] = make_double2(lc[2 * i], lc[2 * i + 1]);
}

__global__ void __launch_bounds__(128) prep_kernel(const LaunchParams prm) {
  const int w = blockIdx.x;
  prep_walker_lines(prm, w, blockIdx.y * blockDim.x + threadIdx.x, prm.theta + (size_t)w * prm.ndim);
}

// Sampler variant: row w of the batch is the stretch proposal of the w-th walker of the active half, built here
// (every block of the walker rebuilds it in shared memory; block y = 0 also writes it to prm.theta for the accept
// step) and then lowered to line constants exactly as above.
__global__ void __launch_bounds__(128) prep_propose_kernel(const LaunchParams prm) {
  extern __shared__ double s_row[];           // [ndim]
  __shared__ int s_ij[2];
  __shared__ double s_zz;
  const StretchParams& P = prm.sp;
  const int k = blockIdx.x, split = prm.sampler_split;
  if (threadIdx.x == 0) {
    int i, j;
    double zz;
    stretch_propose_row(P, split, k, i, j, zz);
    s_ij[0] = i;
    s_ij[1] = j;
    s_zz = zz;
    if (blockIdx.y == 0) {
      P.factors[k] = (P.ndim - 1.0) * log(zz);
      P.walker_of[k] = i;
    }
  }
  __syncthreads();
  {
    const double* s = P.coords + (size_t)s_ij[0] * P.ndim;
    const double* c = P.coords + (size_t)s_ij[1] * P.ndim;
    const double zz = s_zz;
    for (int d = threadIdx.x; d < P.ndim; d += blockDim.x) {
      const double q = __dsub_rn(c[d], __dmul_rn(__dsub_rn(c[d], s[d]), zz));
      s_row[d] = q;
      if (blockIdx.y == 0) P.prop[(size_t)k * P.ndim + d] = q;
    }
  }
  __syncthreads();
  prep_walker_lines(prm, k, blockIdx.y * blockDim.x + threadIdx.x, s_row);
}

// Sum of a walker's tile partials in fixed order -> lnprob (and, for the device-resident sampler, accept/reject).
// Called by a whole warp: the partials are loaded lane-parallel and added by lane 0 in tile order (the same
// order whatever path or geometry calls it), the sampler step uses all lanes.
// BND (finalize_kernel after the streaming kernel): E = the calling warp's shared memory, cap doubles of it for
// boundary records + 72 for the taps behind them.
constexpr int kFinalizeBndDoubles = 1024;
template <bool BND>
__device__ __forceinline__ void finalize_walker(const LaunchParams& prm, int w, int inst_id, int oob, int lane,
                                                int split, double* E = nullptr, int cap = 0) {
  double total;
  if (oob) {
    total = -CUDART_INF;                                          // vfit_mcmc.py:350-352
  } else {
    total = 0.0;
    const double* pp = prm.partials + (size_t)w * prm.n_tiles;
    const int n_sum = (prm.wps > 0) ? 1 : prm.n_inst;   // a sightline walker sees one instrument only
    for (int k = 0; k < n_sum; ++k) {
      double s = 0.0;
      const int first = prm.geom[k].first_tile, n = prm.geom[k].n_tiles;
      for (int t0 = 0; t0 < n; t0 += 32) {
        const double v = (t0 + lane < n) ? __ldcg(pp + first + t0 + lane) : 0.0;     // L2: written by other CTAs
        const int m = min(32, n - t0);
        for (int t = 0; t < m; ++t) s += __shfl_sync(0xffffffffu, v, t);
      }
      const int ki = (prm.wps > 0) ? inst_id : k;
      if (BND && prm.bnd != nullptr && n > 1) {
        // streaming kernel: the K - 1 outputs behind every range boundary, from the flux values the two ranges left
        // in the boundary records (same tap order as the kernel's LSF).  Records of consecutive slots are contiguous:
        // chunks of them go through the warp's shared memory with one coalesced pass; (boundary, output) pairs are
        // dealt to the lanes in index order, one fixed-order sum per instrument.
        double* tp = E + cap;
        const InstDev& I = prm.inst_in_params ? prm.inst_v[ki] : prm.inst[ki];
        const int K = I.K, halo = K - 1, stride = prm.bnd_stride;
        // asynchronous copies (every 8-byte piece in flight at once; records are only 8-byte aligned in general)
        __syncwarp();
        const unsigned tdst = (unsigned)__cvta_generic_to_shared(tp);
        for (int m = lane; m < K; m += 32)
          asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(tdst + 8u * (unsigned)m), "l"(I.taps_rev + m) : "memory");
        const int per_chunk = max(1, cap / stride);
        double part = 0.0;
        for (int t0 = 1; t0 < n; t0 += per_chunk) {
          const int nt = min(per_chunk, n - t0);
          const double* src = prm.bnd + ((size_t)w * prm.n_tiles + first + t0) * stride;
          __syncwarp();
          const unsigned edst = (unsigned)__cvta_generic_to_shared(E);
          for (int i = lane; i < nt * stride; i += 32)
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(edst + 8u * (unsigned)i), "l"(src + i) : "memory");
          asm volatile("cp.async.wait_all;" ::: "memory");
          __syncwarp();
          for (int idx = lane; idx < nt * halo; idx += 32) {
            const int t = idx / halo, q = idx - t * halo;
            const int slot = first + t0 + t;
            const int o = (int)prm.range_lo[slot] * kSuperPix + q;
            if (o < min((int)prm.range_hi[slot] * kSuperPix, I.P)) {
              const double* e = E + t * stride + q;
              double acc = 0.0;
              for (int m = 0; m < K; ++m) acc = fma(tp[m], e[m], acc);
              const double resid = __ldg(I.flux + o) - acc;
              part = fma(resid * resid, __ldg(I.inv_sigma2 + o), part);
            }
          }
        }
        s += __shfl_sync(0xffffffffu, warp_sum(part), 0);
      }
      const double slog = prm.inst_in_params ? prm.inst_v[ki].sum_log_inv_sigma2 : prm.inst[ki].sum_log_inv_sigma2;
      total += -0.5 * (s - slog);                                   // vfit_mcmc.py:309-313
    }
  }
  if (lane == 0) prm.lnprob[w] = total;
  if (split >= 0) stretch_accept_record(prm.sp, split, w, total, lane);
}

// ------------------------------------------------------------------------------------------ main kernel
// MODE 0: lnprob (chi^2 partial + ticket finalisation); MODE 1: model flux out.
// PPT = pixels per lane in phase 1: 8 for big tiles (ILP), 2 when a tile has only a few chunks per warp, so that
// the chunks that hold line cores (several times the cost of a far-wing chunk) can be balanced over the warps.
// The work of one CTA on one (walker w, tile) -- the body of voigt_tile_kernel, and of every half-step of
// voigt_mcmc_kernel.  split: -1, or the half of the stretch move whose proposal row w is (fused sampler).
template <int LOGR, int MODE, int PPT>
__device__ __forceinline__ void tile_body(const LaunchParams& prm, const int w, const int tile_blk, const int split) {
  constexpr int R = 1 << LOGR;
  constexpr int kWarpPix = 32 * PPT;                  // pixels per chunk
  constexpr int kSuperChunks = kSuperPix / kWarpPix;  // chunks per super-chunk
  __shared__ double s_red[kThreads / 32];
  __shared__ int s_next;   // dynamic chunk counter of phase 1

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tile_id = (MODE == 0) ? tile_blk : prm.tile_base + tile_blk;
  int inst_id = 0;
  if (prm.wps > 0) {
    inst_id = w / prm.wps;                 // sightline mode: every instrument shares geom[0]
  } else {
    while (inst_id + 1 < prm.n_inst && tile_id >= prm.geom[inst_id + 1].first_tile) ++inst_id;
  }
  const TileGeom G = prm.geom[prm.wps > 0 ? 0 : inst_id];
  const InstDev I = prm.inst_in_params ? prm.inst_v[inst_id] : prm.inst[inst_id];
  const int ndim = prm.ndim;
  if (tid == 0) s_next = 0;

  const int lc_off = (ndim + 1) & ~1;                  // smem layout (doubles): theta | line consts | taps |
  const int taps_off = lc_off + I.L * LC_STRIDE;       //   flux tile | super-chunk records | line lists (u16)
  const int flux_off = taps_off + I.Kpad;
  const int rec_off = flux_off + ((smem_pos(G.ext_alloc, LOGR) + 1) & ~1);              // super-chunk records
  const int list_off = rec_off + G.n_super * SC_STRIDE;
  double* s_theta = smem;
  double* s_lc = smem + lc_off;
  double* s_taps = smem + taps_off;
  double* s_flux = smem + flux_off;
  const int list_stride = (I.L + 3) & ~3;
  // u16 lists: [n_super][2][list_stride] (direct tiers, FP32-gated), then one far-field scratch list per warp
  unsigned short* s_lists = reinterpret_cast<unsigned short*>(smem + list_off);
  unsigned short* s_listff = s_lists + (G.n_super * 2 + warp) * list_stride;
  // FP32 gate: the gated contributions of one pixel sum to <= 4e-6 (=> |dtau| <= 1e-11, DESIGN.md section 4b)
  const double gate32 = (prm.precision == RBV_PRECISION_FP32_GATED) ? 4e-6 / (double)I.L : 0.0;
  const float ff_eps = prm.farfield ? (float)(prm.ff_budget / (double)I.L) : 0.f;

  for (int i = tid; i < I.Kpad; i += kThreads) s_taps[i] = I.taps_rev[i];
  int oob = 0;
  const bool fast = (I.method == RBV_VOIGT_FAST);
  if (prm.lc != nullptr) {
    // ---- per-line constants and the prior flag were computed once per walker by prep_kernel; the copy does not
    // wait for the flag (an out-of-bounds row's constants are finite or NaN, never read)
    {
      const double2* src =
          reinterpret_cast<const double2*>(
              prm.lc + ((size_t)w * prm.n_lines_total + (prm.wps > 0 ? 0 : I.line_base)) * LC_STRIDE);
      double2* dst = reinterpret_cast<double2*>(s_lc);
      for (int i = tid; i < I.L * (LC_STRIDE / 2); i += kThreads) dst[i] = src[i];
    }
    if (MODE == 0) oob = prm.oob[w];
    __syncthreads();
  } else {
    // ---- the CTA prepares its own constants: flux mode without a workspace, and the lnprob launch of a small
    // batch (prm.lc == NULL: no prep_kernel in front -- one launch less on the latency path; every CTA of the walker
    // repeats the ~400 dependent FP64 instructions per line, which costs nothing while the GPU is mostly empty)
    __shared__ int s_ij[2];
    __shared__ double s_zz;
    if (MODE == 0 && split >= 0) {
      // device-resident sampler: row w of the batch is the stretch proposal of the w-th walker of the active half
      // (what prep_propose_kernel builds); the walker's first CTA also stores it for the accept step
      const StretchParams& P = prm.sp;
      if (tid == 0) {
        int i, j;
        double zz;
        stretch_propose_row(P, split, w, i, j, zz);
        s_ij[0] = i;
        s_ij[1] = j;
        s_zz = zz;
        if (tile_id == 0) {
          P.factors[w] = (P.ndim - 1.0) * log(zz);
          P.walker_of[w] = i;
        }
      }
      __syncthreads();
      const double* sp = P.coords + (size_t)s_ij[0] * P.ndim;
      const double* cp = P.coords + (size_t)s_ij[1] * P.ndim;
      const double zz = s_zz;
      for (int d = tid; d < ndim; d += kThreads) {
        const double cd = __ldcg(cp + d), sd = __ldcg(sp + d);       // L2: written by other CTAs (persistent launch)
        const double q = __dsub_rn(cd, __dmul_rn(__dsub_rn(cd, sd), zz));
        s_theta[d] = q;
        if (tile_id == 0) P.prop[(size_t)w * ndim + d] = q;
      }
    } else {
      const double* th_g = prm.theta + (size_t)w * ndim;
      for (int i = tid; i < ndim; i += kThreads) s_theta[i] = th_g[i];
    }
    __syncthreads();
    if (MODE == 0) {   // uniform prior (vfit.lnprior, vfit_mcmc.py:291-295) and the slice sampler's row mask
      int bad = (prm.row_skip != nullptr && prm.row_skip[w] != 0);
      if (prm.lb != nullptr)
        for (int i = tid; i < ndim; i += kThreads) bad |= (s_theta[i] < prm.lb[i]) || (s_theta[i] > prm.ub[i]);
      oob = __syncthreads_or(bad);
    }
    if (!oob) {
      for (int l = tid; l < I.L; l += kThreads) {
        if (fast) prep_line_fast(I, l, s_theta, s_lc + l * LC_STRIDE);
        else prep_line_wofz(I, l, s_theta, s_lc + l * LC_STRIDE);
      }
      __syncthreads();
      if (!fast) {
        for (int t = tid; t < I.L * kNQNear; t += kThreads) {
          int l = t / kNQNear, p = t - l * kNQNear;
          const double* lc = s_lc + l * LC_STRIDE;
          s_lc[l * LC_STRIDE + LC_Q + p] = asym_coef(p + 1, lc[LC_A2], lc[LC_AUX]);
        }
        __syncthreads();
        for (int l = tid; l < I.L; l += kThreads)
          fill_fp32_constants(s_lc + l * LC_STRIDE, prm.farfield ? prm.ff_budget / (double)I.L : 0.0);
        __syncthreads();
      }
    }
  }

  double part = 0.0;
  if (!oob) {
    // ---- phase 1: flux for the tile + halo into shared memory
    const int h = I.K >> 1;
    const int p0 = (tile_id - G.first_tile) * G.tile;
    const int n_out = min(G.tile, I.P - p0);
    const int ext = n_out + I.K - 1;
    const int n_chunks = (ext + kWarpPix - 1) / kWarpPix;
    // ---- phase 0: tier lists + far-field record of every super-chunk (one warp each)
    if (!fast) {
      const int n_sc = (ext + kSuperPix - 1) / kSuperPix;
      for (int sc = warp; sc < n_sc; sc += kThreads / 32) {
        const int plo = min(max(p0 - h + sc * kSuperPix, 0), I.P - 1);
        const int phi = min(max(p0 - h + min((sc + 1) * kSuperPix, ext) - 1, 0), I.P - 1);
        prepare_super_chunk(I, lc_off, rec_off + sc * SC_STRIDE, s_lists + sc * 2 * list_stride,
                            s_lists + (sc * 2 + 1) * list_stride, s_listff, gate32, ff_eps, plo, phi,
                            flux_off + min(warp, n_sc - 1) * (8 * 33), lane);   // scratch: the idle flux tile
      }
      __syncthreads();
    }
    // warps pull 32*PPT-pixel chunks from a CTA-wide counter: chunks that contain a line core cost
    // several times a far-wing chunk, and static assignment would leave the other warps waiting at the barrier
    // (the ticket for the NEXT chunk is drawn one iteration ahead: the shared-memory atomic's latency overlaps the
    // current chunk)
    int c = 0;
    if (lane == 0) c = smem_ticket(&s_next);
    c = __shfl_sync(0xffffffffu, c, 0);
    while (c < n_chunks) {
      int c_next = 0;
      if (lane == 0) c_next = smem_ticket(&s_next);
      const int i0 = c * kWarpPix;
      double u[PPT], tau[PPT];
      const int pc = p0 - h + i0;                     // first pixel of the chunk
      if (pc >= 0 && pc + kWarpPix <= I.P) {          // interior chunk: base pointer + compile-time offsets
        const double* up = I.inv_wave + pc + lane;
#pragma unroll
        for (int j = 0; j < PPT; ++j) u[j] = __ldg(up + j * 32);
      } else {
#pragma unroll
        for (int j = 0; j < PPT; ++j) {
          const int p = min(max(pc + j * 32 + lane, 0), I.P - 1);   // edge replication
          u[j] = __ldg(I.inv_wave + p);
        }
      }
      c_next = __shfl_sync(0xffffffffu, c_next, 0);
      if (fast) tau_fast(lc_off, I.L, u, tau);
      else {
        const int sc = c / kSuperChunks;
        tau_wofz(lc_off, I.L, s_lists + sc * 2 * list_stride, s_lists + (sc * 2 + 1) * list_stride,
                 rec_off + sc * SC_STRIDE, u, tau, prm.core_tab);
      }
      // flux = exp(-tau), voigt_model.py:217.  Away from line cores every pixel of the chunk has |tau| < 2^-6,
      // where the degree-6 Taylor polynomial is exact to 4.5e-17 (under half an ulp) and needs no range reduction.
      unsigned hmax = 0u;
#pragma unroll
      for (int j = 0; j < PPT; ++j) hmax = max(hmax, (unsigned)__double2hiint(tau[j]));   // negative or NaN: huge
      // slot(i0 + 32 j + lane) = slot(i0) + (R + 1) * (32 / R) * j + lane + lane / R   (i0 and 32 are multiples of R)
      static_assert(32 % (1 << LOGR) == 0, "chunk rows must be whole groups of R");
      double* fo = s_flux + smem_pos(i0, LOGR) + lane + (lane >> LOGR);
      constexpr int kRow = (R + 1) * (32 / R);
      const bool small = __reduce_max_sync(0xffffffffu, hmax) < 0x3F900000u;   // NaN has a larger high word
      if (i0 + kWarpPix <= ext) {               // full chunk: no per-pixel predicate
        if (small) {
#pragma unroll
          for (int j = 0; j < PPT; ++j) fo[j * kRow] = exp_small(-tau[j]);
        } else {
#pragma unroll
          for (int j = 0; j < PPT; ++j) fo[j * kRow] = exp_flux(-tau[j]);
        }
      } else {
#pragma unroll
        for (int j = 0; j < PPT; ++j)
          if (i0 + j * 32 + lane < ext) fo[j * kRow] = small ? exp_small(-tau[j]) : exp_flux(-tau[j]);
      }
      c = c_next;
    }
    // observed spectrum of a group of R outputs from the block-transposed (flux, inv_sigma2) copy: lane-contiguous
    // 16-byte loads (tiles start on 256-pixel boundaries); the first group's loads are issued BEFORE the barrier
    // so that their latency overlaps the wait
    static_assert(R == 8, "the packed observed-spectrum layout assumes 8 outputs per lane");
    const int n_groups = (n_out + R - 1) >> LOGR;
    double obs[R], wgt[R];
    auto load_group = [&](int g) {
      const double2* src = I.obs_w + ((size_t)(p0 >> 8) + (g >> 5)) * 256 + lane;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const double2 v = __ldg(src + 32 * r);
        obs[r] = v.x;
        wgt[r] = v.y;
      }
    };
    if (MODE == 0 && tid < n_groups) load_group(tid);
    // zero the slack the register-blocked window may touch (taps there are zero, values must be finite)
    for (int i = ext + tid; i < G.ext_alloc; i += kThreads) s_flux[smem_pos(i, LOGR)] = 0.0;
    __syncthreads();

    // ---- phase 2: LSF + chi^2 (or flux out).  M_p = sum_m taps_rev[m] * E[o + m]
    for (int g = tid; g < n_groups; g += kThreads) {
      double acc[R], win[2 * R - 1];
#pragma unroll
      for (int r = 0; r < R; ++r) acc[r] = 0.0;
      const int e0 = g << LOGR;
      if (MODE == 0 && g != tid) load_group(g);
      // padded layout: slot(R g + j) = (R + 1) g + j for j < R, so every window position is the group's base
      // plus a compile-time offset (block b of R taps starts (R + 1) b further on)
      int fw = flux_off + (R + 1) * g;
#pragma unroll
      for (int q = 0; q < R - 1; ++q) win[q] = smem[fw + q];
      const int n_blocks = I.Kpad >> LOGR;              // >= 1: Kpad is a positive multiple of R
      __builtin_assume(n_blocks >= 1);
#pragma unroll 3
      for (int blk = 0; blk < n_blocks; ++blk, fw += R + 1) {
        const int m0 = blk << LOGR;
        win[R - 1] = smem[fw + R - 1];
#pragma unroll
        for (int q = 1; q < R; ++q) win[R - 1 + q] = smem[fw + R + q];
#pragma unroll
        for (int mm = 0; mm < R; mm += 2) {
          const double2 tap = *reinterpret_cast<const double2*>(smem + taps_off + m0 + mm);
#pragma unroll
          for (int r = 0; r < R; ++r) acc[r] = fma(tap.x, win[mm + r], acc[r]);
#pragma unroll
          for (int r = 0; r < R; ++r) acc[r] = fma(tap.y, win[mm + 1 + r], acc[r]);
        }
#pragma unroll
        for (int q = 0; q < R - 1; ++q) win[q] = win[R + q];
      }
      const int pbase = p0 + e0;
      if (MODE == 0) {
        // vfit_mcmc.py:310; the log_inv_sigma2 term is summed once per instrument at set-up
        // (InstDev::sum_log_inv_sigma2).  Same order of additions in both branches.
        if (e0 + R <= n_out) {
#pragma unroll
          for (int r = 0; r < R; ++r) {
            const double resid = obs[r] - acc[r];
            part = fma(resid * resid, wgt[r], part);
          }
        } else {
#pragma unroll
          for (int r = 0; r < R; ++r) {
            if (e0 + r < n_out) {
              const double resid = obs[r] - acc[r];
              part = fma(resid * resid, wgt[r], part);
            }
          }
        }
      } else {
        double* out = prm.out_flux + (size_t)w * I.P;
#pragma unroll
        for (int r = 0; r < R; ++r)
          if (e0 + r < n_out) out[pbase + r] = acc[r];
      }
    }
  }

  if (MODE == 0) {
    // ---- CTA reduction of the chi^2 partial (fixed order -> reproducible)
    part = warp_sum(part);
    if (lane == 0) s_red[warp] = part;
    __syncthreads();
    if (warp == 0) {
      unsigned int prev = 0u;
      if (lane == 0) {
        double s = 0.0;
#pragma unroll
        for (int k = 0; k < kThreads / 32; ++k) s += s_red[k];
        prm.partials[(size_t)w * prm.n_tiles + tile_id] = s;
        // big grids: finalize_kernel adds the partials (no tail in this CTA); otherwise release our partial /
        // acquire the others' with ONE acq_rel ticket atomic: the walker's last CTA finalises
        if (!prm.separate_finalize)
          asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], 1;" : "=r"(prev) : "l"(prm.tickets + w) : "memory");
      }
      if (prm.separate_finalize) return;
      prev = __shfl_sync(0xffffffffu, prev, 0);
      if (prev != (unsigned int)(prm.n_tiles - 1)) return;
      finalize_walker<false>(prm, w, inst_id, oob, lane, split);
      if (lane == 0) prm.tickets[w] = 0u;     // re-armed for a launch without prep_kernel (harmless otherwise)
    }
  }
}

template <int LOGR, int MODE, int PPT>
__global__ void __launch_bounds__(kThreads, RBV_MIN_CTAS) voigt_tile_kernel(const LaunchParams prm) {
  tile_body<LOGR, MODE, PPT>(prm, blockIdx.x, blockIdx.y, prm.sampler_split);
}

// Grid-wide barrier of a cooperative launch: one counter that only grows (target = generation x CTAs).  A bounded
// spin: if the grid were ever not co-resident the launch ends with flag bit 2 set instead of hanging the device.
__device__ __forceinline__ void grid_barrier(unsigned int* bar, unsigned int target, int* flag) {
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int v;
    asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], 1;" : "=r"(v) : "l"(bar) : "memory");
    const long long t0 = clock64();
    for (;;) {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(bar) : "memory");
      if (v >= target) break;
      if (clock64() - t0 > (4LL << 30)) {       // ~2 s at 2 GHz
        atomicOr(flag, 4);
        break;
      }
    }
  }
  __syncthreads();
}

// The whole stretch-move loop of a SMALL ensemble as ONE cooperative launch: grid = (walkers of a half, tiles), every
// CTA runs the tile body of its (proposal row, tile) -- proposal and line constants in the prologue, accept/reject
// by the walker's last CTA -- then all CTAs meet at a grid barrier, half-step after half-step.  Per half-step this
// replaces two kernel launches of a CUDA graph (~19 us on the README problem) by the body plus one barrier.
template <int LOGR, int PPT>
__global__ void __launch_bounds__(kThreads, RBV_MIN_CTAS) voigt_mcmc_kernel(const __grid_constant__ LaunchParams prm,
                                                                           const int n_steps, unsigned int* bar) {
  const int n_ctas = gridDim.x * gridDim.y, h = (prm.sp.W + 1) / 2;
  unsigned int gen = 0u;
  for (int s = 0; s < n_steps; ++s) {
    for (int split = 0; split < 2; ++split) {
      const int nS = split == 0 ? h : prm.sp.W - h;
      if ((int)blockIdx.x < nS) tile_body<LOGR, 0, PPT>(prm, blockIdx.x, blockIdx.y, split);
      grid_barrier(bar, ++gen * (unsigned int)n_ctas, prm.sp.flag);
    }
  }
}

// lnprob of every walker from its tile partials, as a separate launch.  Used for big grids: the in-kernel
// finalisation keeps one thread of every CTA (and with it the CTA's registers and shared memory) alive for the
// round trip of the ticket atomic -- about 15 % of a CTA's lifetime at C5a.
__global__ void __launch_bounds__(128) finalize_kernel(const LaunchParams prm) {
  const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);       // one warp per walker
  if (w >= prm.W) return;
  finalize_walker<false>(prm, w, prm.wps > 0 ? w / prm.wps : 0, prm.oob[w], threadIdx.x & 31, prm.sampler_split);
}

// ... after the streaming kernel: + the outputs behind the range boundaries (records through shared memory)
__global__ void __launch_bounds__(128) finalize_stream_kernel(const LaunchParams prm) {
  __shared__ double s_bnd[4][kFinalizeBndDoubles + 72];
  const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (w >= prm.W) return;
  finalize_walker<true>(prm, w, prm.wps > 0 ? w / prm.wps : 0, prm.oob[w], threadIdx.x & 31, prm.sampler_split,
                        s_bnd[threadIdx.x >> 5], kFinalizeBndDoubles);
}

}  // namespace rbv
#include "rbv_stream.cuh"   // warp-autonomous streaming form of the lnprob kernel (big batches)
#include "rbv_grad.cuh"     // analytic gradient of lnprob / lnlike (forward + adjoint pass)
#include "rbv_fisher.cuh"   // model Jacobian and Gauss-Newton matrix of lnlike (forward mode per column)
#include "rbv_lm.cuh"       // survey-mode Levenberg-Marquardt update (one warp per sightline)
namespace rbv {

// ------------------------------------------------------------------------------------------ small kernels
__global__ void reciprocal_kernel(const double* __restrict__ in, double* __restrict__ out, int n) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = 1.0 / in[i];
}

// (min, max) of 1/wave over aligned 256-pixel blocks: the tile kernel's phase 0 takes the range of a super-chunk
// from this table instead of re-reading its pixels (no monotonicity of the wavelength grid is assumed).
__global__ void __launch_bounds__(256) block_range_kernel(const double* __restrict__ inv_wave,
                                                          double2* __restrict__ out, int n) {
  __shared__ double s_lo[8], s_hi[8];
  const int i = blockIdx.x * 256 + threadIdx.x;
  double v = inv_wave[min(i, n - 1)];
  double lo = v, hi = v;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o));
  }
  if ((threadIdx.x & 31) == 0) {
    s_lo[threadIdx.x >> 5] = lo;
    s_hi[threadIdx.x >> 5] = hi;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int k = 1; k < 8; ++k) {
      lo = fmin(lo, s_lo[k]);
      hi = fmax(hi, s_hi[k]);
    }
    out[blockIdx.x] = make_double2(lo, hi);
  }
}

// (min, max) of 1/wave over the streaming kernel's super-chunks: pixels first + 1024 s .. first + 1024 s + 1023,
// indices clamped to the spectrum (edge replication)
__global__ void __launch_bounds__(256) segment_range_kernel(const double* __restrict__ inv_wave,
                                                            double2* __restrict__ out, int n, int first) {
  __shared__ double s_lo[8], s_hi[8];
  double lo = CUDART_INF, hi = -CUDART_INF;
  for (int i = threadIdx.x; i < kSuperPix; i += 256) {
    const double v = inv_wave[min(max(first + blockIdx.x * kSuperPix + i, 0), n - 1)];
    lo = fmin(lo, v);
    hi = fmax(hi, v);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o));
  }
  if ((threadIdx.x & 31) == 0) {
    s_lo[threadIdx.x >> 5] = lo;
    s_hi[threadIdx.x >> 5] = hi;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int k = 1; k < 8; ++k) {
      lo = fmin(lo, s_lo[k]);
      hi = fmax(hi, s_hi[k]);
    }
    out[blockIdx.x] = make_double2(lo, hi);
  }
}

// (flux, inv_sigma2) -> block-transposed pairs (InstDev::obs_w); pixels beyond the spectrum are zero-filled
__global__ void __launch_bounds__(256) pack_observed_kernel(const double* __restrict__ flux,
                                                            const double* __restrict__ inv_sigma2,
                                                            double2* __restrict__ out, int n) {
  const int t = threadIdx.x, lane = t & 31, r = t >> 5;
  const int p = blockIdx.x * 256 + 8 * lane + r;
  out[(size_t)blockIdx.x * 256 + t] = (p < n) ? make_double2(flux[p], inv_sigma2[p]) : make_double2(0.0, 0.0);
}

// sum_p v[p] in a fixed order (one CTA; set-up only)
__global__ void __launch_bounds__(256) fixed_order_sum_kernel(const double* __restrict__ v, int n, double* out) {
  __shared__ double s[256];
  double acc = 0.0;
  for (int i = threadIdx.x; i < n; i += 256) acc += v[i];
  s[threadIdx.x] = acc;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) *out = s[0];
}

// H(a,x) on a lattice through the same device functions the tile kernel uses (test hook).
__global__ void voigt_h_kernel(const double* __restrict__ x, const double* __restrict__ a, double* __restrict__ out,
                               int n, int method, const double* __restrict__ core_tab) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double xv = x[i], av = a[i];
  if (method == RBV_VOIGT_FAST) {
    out[i] = tg_H(xv, av / kSqrtPi, fmax(1e-2, 100.0 * fabs(av) / kSqrtPi), 1.0 - 2.0 * av / kSqrtPi);
    return;
  }
  double a2 = av * av;
  double d = fma(xv, xv, a2);
  double H;
  if (av > kABig) {
    H = general_H(xv, av, d);
  } else if (d < kDCore) {
    H = core_H(xv, av, a2, core_tab);
  } else {
    double Q[kNQNear];
    double kappa = av * kInvSqrtPi;
    for (int p = 0; p < kNQNear; ++p) Q[p] = asym_coef(p + 1, a2, kappa);
    if (d >= kDFar) H = asym_series<kNQFar>(Q, d);
    else if (d >= kDNear) H = asym_series<kNQMid>(Q, d);
    else H = asym_series<kNQNear>(Q, d);
  }
  out[i] = H;
}

// max relative error of rcp_pos over a sweep of positive doubles (self-test of the MUFU seed accuracy)
__global__ void rcp_selftest_kernel(double* out_max) {
  double worst = 0.0;
  for (int k = threadIdx.x; k < (1 << 16); k += blockDim.x) {
    double d = 64.0 * exp2(k * (40.0 / 65536.0)) * (1.0 + 1e-3 * (k % 7));
    double r = rcp_pos(d);
    double err = fabs(fma(r, d, -1.0));
    worst = fmax(worst, err);
  }
  worst = fmax(worst, __shfl_xor_sync(0xffffffffu, worst, 16));
  worst = fmax(worst, __shfl_xor_sync(0xffffffffu, worst, 8));
  worst = fmax(worst, __shfl_xor_sync(0xffffffffu, worst, 4));
  worst = fmax(worst, __shfl_xor_sync(0xffffffffu, worst, 2));
  worst = fmax(worst, __shfl_xor_sync(0xffffffffu, worst, 1));
  if ((threadIdx.x & 31) == 0) atomicMax((unsigned long long*)out_max, (unsigned long long)__double_as_longlong(worst));
}

// dependent-chain DFMA throughput probe: 8 chains per thread
__global__ void __launch_bounds__(256) dfma_peak_kernel(double* out, int iters, double seed) {
  double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6,
         a7 = a0 + 7;
  const double m = 0.999999, c = 1e-7;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
      a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
  }
  double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
  if (s == 123.456) out[0] = s;
}

}  // namespace rbv

// =============================================================================================== host / C ABI
using namespace rbv;

constexpr int kGeomLevels = 6;   // tile sizes, see compute_geometry
static thread_local std::string g_last_error;

// Tuning / test hooks, read from the environment when a context is created and kept in that context
struct Tuning {
  int force_ppt = 0;        // RBVFIT_B200_PPT=2|8: pixels per lane in phase 1 of the tile kernel
  int force_level = -1;     // RBVFIT_B200_GEOM=0..5: tile size of the tile kernel
  int force_finalize = -1;  // RBVFIT_B200_FINALIZE=0|1: lnprob by a separate launch
  int stream = -1;          // RBVFIT_B200_STREAM=0|1: streaming kernel never / whenever eligible (-1: by batch size)
  int stream_segs = 0;      // RBVFIT_B200_STREAM_SEGS=n: 1024-pixel segments per work item of the streaming kernel
  int stream_ctas = 0;      // RBVFIT_B200_STREAM_CTAS=n: CTAs per SM of the streaming kernel (0: occupancy)
  int stream_cap = 16;      // RBVFIT_B200_STREAM_CAP=n: longest range of the streaming kernel's schedule (segments)
  int stream_div = 3;       // RBVFIT_B200_STREAM_DIV=n: a range is 1/n of what is left of the spectrum
  double ff_budget = kFFEps;   // RBVFIT_B200_FF_EPS=x: far-field error budget (experiments only)
  int slice_dist_graph = 0;    // RBVFIT_B200_SLICE_DIST_GRAPH=1: multi-GPU slice sampler as a CUDA-graph WHILE loop
  int slice_depth = 0;         // RBVFIT_B200_SLICE_DEPTH=1|2: logical iterations per launch of the slice sampler
  int inline_prep = -1;        // RBVFIT_B200_INLINE_PREP=0|1: line constants prepared by prep_kernel / in the CTA prologue
  int mcmc_persistent = -1;    // RBVFIT_B200_MCMC_PERSISTENT=0|1: small-ensemble stretch move as one cooperative launch
};

// Every entry point runs on the context's device and leaves the caller's current device as it found it.
struct DeviceGuard {
  int prev = -1;
  cudaError_t err = cudaSuccess;
  explicit DeviceGuard(int device) {
    err = cudaGetDevice(&prev);
    if (err == cudaSuccess && prev != device) err = cudaSetDevice(device);
    else if (err == cudaSuccess) prev = -1;   // nothing to restore
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};
#define RBV_ON_DEVICE(ctx)                    \
  DeviceGuard _guard((ctx)->device);          \
  RBV_CUDA(_guard.err)

#define RBV_CHECK(expr)                   \
  do {                                    \
    const int _rc = (expr);               \
    if (_rc != RBV_OK) return _rc;        \
  } while (0)

static int fail(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}

#define RBV_CUDA(expr)                                                                                   \
  do {                                                                                                   \
    cudaError_t _e = (expr);                                                                             \
    if (_e != cudaSuccess)                                                                               \
      return fail(RBV_ECUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));                        \
  } while (0)


// ------------------------------------------------------------------------------------------ NCCL (multi-GPU)
// The collective of the path is one tiny all-gather of lnprob values per half-step (SURVEY 8e).  It is issued from
// inside the library, on the library's stream, so that a whole multi-GPU MCMC step is one CUDA graph per rank and no
// Python runs between its kernels.  libnccl is resolved at run time (the copy PyTorch has already loaded, else the
// system one): a single-GPU process never needs it and the library has no link-time dependency on it.  The handful
// of declarations below restate NCCL's public C API (nccl.h, stable since 2.x).
typedef struct ncclComm* RbvNcclComm;
typedef struct { char internal[128]; } RbvNcclUniqueId;
struct NcclApi {
  void* handle = nullptr;
  int (*GetUniqueId)(RbvNcclUniqueId*) = nullptr;
  int (*CommInitRank)(RbvNcclComm*, int, RbvNcclUniqueId, int) = nullptr;
  int (*CommDestroy)(RbvNcclComm) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, RbvNcclComm, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  int (*GetVersion)(int*) = nullptr;
};
constexpr int kNcclFloat64 = 8;    // ncclDouble / ncclFloat64 in ncclDataType_t
static NcclApi g_nccl;

static int load_nccl() {
  if (g_nccl.handle) return RBV_OK;
  void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);     // the copy torch has loaded
  if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!h) return fail(RBV_ESTATE, std::string("NCCL not available: ") + dlerror());
  NcclApi api;
  api.handle = h;
  api.GetUniqueId = (int (*)(RbvNcclUniqueId*))dlsym(h, "ncclGetUniqueId");
  api.CommInitRank = (int (*)(RbvNcclComm*, int, RbvNcclUniqueId, int))dlsym(h, "ncclCommInitRank");
  api.CommDestroy = (int (*)(RbvNcclComm))dlsym(h, "ncclCommDestroy");
  api.AllGather = (int (*)(const void*, void*, size_t, int, RbvNcclComm, cudaStream_t))dlsym(h, "ncclAllGather");
  api.GetErrorString = (const char* (*)(int))dlsym(h, "ncclGetErrorString");
  api.GetVersion = (int (*)(int*))dlsym(h, "ncclGetVersion");
  if (!api.GetUniqueId || !api.CommInitRank || !api.CommDestroy || !api.AllGather || !api.GetErrorString)
    return fail(RBV_ESTATE, "NCCL library lacks a required symbol");
  g_nccl = api;
  return RBV_OK;
}

#define RBV_NCCL(expr)                                                                                    \
  do {                                                                                                    \
    int _r = (expr);                                                                                      \
    if (_r != 0) return fail(RBV_ECUDA, std::string(#expr) + ": " + g_nccl.GetErrorString(_r));           \
  } while (0)

struct HostInst {
  InstDev dev;
  std::vector<double> taps;  // LSF taps as applied by the reference (normalised if requested), length K
  double* d_taps = nullptr;  // flipped + zero-padded copy on the device (rebuilt when R changes)
  double* d_grad_cum = nullptr;   // [2K] prefix / suffix sums of the flipped taps (gradient path, built on first use)
  int* d_fisher_order = nullptr;  // [L] line indices sorted by component, stable (Jacobian path; in owned)
  std::vector<void*> owned;  // device allocations owned by the library for this instrument
};

struct RbvContext {
  Tuning tune;
  std::vector<std::pair<int, int>> stream_ctas_cache;   // (smem bytes, resident CTAs per SM) of voigt_stream_kernel
  int device = 0;
  int sm_count = 148;
  int ndim = 0;
  int n_tiles = 0;
  int n_lines_total = 0;
  int precision = RBV_PRECISION_FP64;
  int farfield = RBV_FARFIELD_CHEBYSHEV;
  long long launches = 0;
  int last_kernel = -1;
  RbvNcclComm comm = nullptr;   // rbv_comm_init: one rank per context
  // rbv_peer_export / rbv_peer_attach: the all-gather as ONE kernel over NVLink peer memory (push + flags)
  void* peer_block = nullptr;            // this rank's exchange block (call counter | 2 x kPeerCap slots)
  void* peer_open[16] = {nullptr};       // the other ranks' blocks, opened through CUDA IPC
  int peer_world = 0;                    // > 0: attached
  cudaStream_t sink_stream = nullptr;                        // rbv_stretch_run_sink: D2H copies of the chain ring
  cudaEvent_t sink_done[2] = {nullptr, nullptr}, sink_copied[2] = {nullptr, nullptr};
  int comm_rank = 0, comm_world = 1;
  std::vector<HostInst> inst;
  InstDev* d_inst = nullptr;
  size_t d_inst_capacity = 0;
  int max_dyn_smem = 0;
  double* d_lb = nullptr;
  double* d_ub = nullptr;
  double* d_core_tab = nullptr;
  double* d_unit_taps = nullptr;        // {1, 0 x 7}: the 'no convolution' LSF of rbv_model_flux_batch(convolve = 0)
  unsigned int* d_grid_bar = nullptr;   // grid-barrier counter of voigt_mcmc_kernel
  size_t max_smem_lnprob[2] = {0, 0};  // per LOGR in {2,3}
  // rbv_slice_run: pinned landing slots + events for the per-iteration read-back of the counters
  SliceState* h_poll = nullptr;        // [2], page-locked
  cudaEvent_t poll_ev[2] = {nullptr, nullptr};
  // survey-mode Fisher: per-instrument order / has_lsf as device tables (host copies to detect a change)
  std::vector<const int*> sl_order;
  std::vector<int> sl_has_lsf;
  const int** d_sl_order = nullptr;
  int* d_sl_has_lsf = nullptr;
  int* h_lm_count = nullptr;           // rbv_lm_run_sightlines: page-locked landing slot of the active count
};

template <typename T>
static cudaError_t upload(T** dst, const T* src, size_t n) {
  cudaError_t e = cudaMalloc((void**)dst, std::max<size_t>(n, 1) * sizeof(T));
  if (e != cudaSuccess) return e;
  if (n) e = cudaMemcpy(*dst, src, n * sizeof(T), cudaMemcpyHostToDevice);
  return e;
}

static size_t smem_bytes_for(const InstDev& I, const TileGeom& G, int ndim) {
  int logR = (I.R == 8) ? 3 : 2;
  size_t n = ((ndim + 1) & ~1) + (size_t)I.L * LC_STRIDE + I.Kpad + (G.ext_alloc + (G.ext_alloc >> logR)) + 4 +
             (size_t)G.n_super * SC_STRIDE;
  size_t lists = (size_t)(G.n_super * 2 + kThreads / 32) * ((I.L + 3) & ~3) * sizeof(unsigned short);
  return n * sizeof(double) + ((lists + 15) & ~(size_t)15);
}

extern "C" {

const char* rbv_last_error(void) { return g_last_error.c_str(); }
const char* rbv_version(void) { return "rbvfit_b200 0.1 (sm_100a)"; }

int rbv_create(int device, RbvContext** out) {
  if (!out) return fail(RBV_EINVAL, "rbv_create: out is NULL");
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return fail(RBV_ECUDA, std::string("rbv_create: no CUDA device (") + cudaGetErrorString(e) +
                               "); this library has no CPU fallback");
  if (device < 0 || device >= count) return fail(RBV_EINVAL, "rbv_create: bad device index");
  DeviceGuard _guard(device);
  RBV_CUDA(_guard.err);
  RbvContext* ctx = new RbvContext();
  ctx->device = device;
  struct Guard {   // a failed set-up must not leak the half-built context
    RbvContext* c;
    ~Guard() { if (c) rbv_destroy(c); }
  } guard{ctx};
  {   // tuning / test hooks
    const char* e = getenv("RBVFIT_B200_PPT");
    ctx->tune.force_ppt = e ? atoi(e) : 0;
    e = getenv("RBVFIT_B200_FINALIZE");
    ctx->tune.force_finalize = e ? atoi(e) : -1;
    e = getenv("RBVFIT_B200_GEOM");
    ctx->tune.force_level = e ? std::min(std::max(atoi(e), 0), kGeomLevels - 1) : -1;
    e = getenv("RBVFIT_B200_STREAM");
    ctx->tune.stream = e ? atoi(e) : -1;
    e = getenv("RBVFIT_B200_STREAM_SEGS");
    ctx->tune.stream_segs = e ? std::max(atoi(e), 0) : 0;
    e = getenv("RBVFIT_B200_STREAM_CAP");
    if (e && atoi(e) > 0) ctx->tune.stream_cap = atoi(e);
    e = getenv("RBVFIT_B200_STREAM_DIV");
    if (e && atoi(e) > 0) ctx->tune.stream_div = atoi(e);
    e = getenv("RBVFIT_B200_STREAM_CTAS");
    ctx->tune.stream_ctas = e ? std::max(atoi(e), 0) : 0;
    e = getenv("RBVFIT_B200_MCMC_PERSISTENT");
    ctx->tune.mcmc_persistent = e ? atoi(e) : -1;
    e = getenv("RBVFIT_B200_INLINE_PREP");
    ctx->tune.inline_prep = e ? atoi(e) : -1;
    e = getenv("RBVFIT_B200_SLICE_DIST_GRAPH");
    ctx->tune.slice_dist_graph = e ? atoi(e) : 0;
    e = getenv("RBVFIT_B200_SLICE_DEPTH");
    ctx->tune.slice_depth = e ? atoi(e) : 0;
    e = getenv("RBVFIT_B200_FF_EPS");
    if (e && atof(e) > 0.0) ctx->tune.ff_budget = atof(e);
  }
  cudaDeviceProp prop;
  RBV_CUDA(cudaGetDeviceProperties(&prop, device));
  ctx->sm_count = prop.multiProcessorCount;
  RBV_CUDA(cudaMemcpyToSymbol(c_ctab, RBV_ASYM_CTAB_HOST, sizeof(RBV_ASYM_CTAB_HOST)));
  RBV_CUDA(cudaMemcpyToSymbol(c_weid, RBV_WEID_COEF_HOST, sizeof(RBV_WEID_COEF_HOST)));
  RBV_CUDA(cudaMemcpyToSymbol(c_ff_nodes, RBV_FF_NODES_HOST, sizeof(RBV_FF_NODES_HOST)));
  RBV_CUDA(cudaMemcpyToSymbol(c_ff_minv, RBV_FF_MINV_HOST, sizeof(RBV_FF_MINV_HOST)));
  RBV_CUDA(upload(&ctx->d_core_tab, RBV_CORE_TABLE_HOST, (size_t)RBV_CORE_TABLE_LEN));
  {
    const double unit[8] = {1.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    RBV_CUDA(upload(&ctx->d_unit_taps, unit, (size_t)8));
  }
  const int max_dyn = (int)prop.sharedMemPerBlockOptin - 2048;
  ctx->max_dyn_smem = max_dyn;
  RBV_CUDA(cudaFuncSetAttribute(voigt_tile_kernel<3, 0, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_dyn));
  RBV_CUDA(cudaFuncSetAttribute(voigt_tile_kernel<3, 0, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_dyn));
  RBV_CUDA(cudaFuncSetAttribute(voigt_tile_kernel<3, 1, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_dyn));
  RBV_CUDA(cudaFuncSetAttribute(voigt_tile_kernel<3, 1, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_dyn));
  RBV_CUDA(cudaFuncSetAttribute(voigt_stream_kernel<3, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_dyn));
  RBV_CUDA(cudaFuncSetAttribute(voigt_stream_kernel<3, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_dyn));
  RBV_CUDA(cudaFuncSetAttribute(voigt_mcmc_kernel<3, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_dyn));
  RBV_CUDA(cudaFuncSetAttribute(voigt_mcmc_kernel<3, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_dyn));
  RBV_CUDA(cudaMalloc((void**)&ctx->d_grid_bar, 256));
  RBV_CUDA(cudaMallocHost((void**)&ctx->h_poll, 2 * sizeof(SliceState)));
  for (int k = 0; k < 2; ++k) RBV_CUDA(cudaEventCreateWithFlags(&ctx->poll_ev[k], cudaEventDisableTiming));
  guard.c = nullptr;
  *out = ctx;
  return RBV_OK;
}

void rbv_destroy(RbvContext* ctx) {
  if (!ctx) return;
  DeviceGuard _guard(ctx->device);
  for (auto& hi : ctx->inst) {
    for (void* p : hi.owned) cudaFree(p);
    cudaFree(hi.d_taps);
    cudaFree(hi.d_grad_cum);
  }
  if (ctx->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(ctx->comm);
  for (int r = 0; r < 16; ++r)
    if (ctx->peer_open[r]) cudaIpcCloseMemHandle(ctx->peer_open[r]);
  cudaFree(ctx->peer_block);
  for (int k = 0; k < 2; ++k) {
    if (ctx->sink_done[k]) cudaEventDestroy(ctx->sink_done[k]);
    if (ctx->sink_copied[k]) cudaEventDestroy(ctx->sink_copied[k]);
  }
  if (ctx->sink_stream) cudaStreamDestroy(ctx->sink_stream);
  cudaFree(ctx->d_inst);
  cudaFree(ctx->d_lb);
  cudaFree(ctx->d_ub);
  cudaFree(ctx->d_core_tab);
  cudaFree(ctx->d_unit_taps);
  cudaFree(ctx->d_grid_bar);
  if (ctx->h_poll) cudaFreeHost(ctx->h_poll);
  if (ctx->h_lm_count) cudaFreeHost(ctx->h_lm_count);
  cudaFree(ctx->d_sl_order);
  cudaFree(ctx->d_sl_has_lsf);
  for (int k = 0; k < 2; ++k)
    if (ctx->poll_ev[k]) cudaEventDestroy(ctx->poll_ev[k]);
  delete ctx;
}

int rbv_set_precision(RbvContext* ctx, int precision) {
  if (!ctx) return fail(RBV_EINVAL, "null context");
  if (precision != RBV_PRECISION_FP64 && precision != RBV_PRECISION_FP32_GATED)
    return fail(RBV_EINVAL, "rbv_set_precision: unknown precision");
  ctx->precision = precision;
  return RBV_OK;
}

int rbv_set_farfield(RbvContext* ctx, int mode) {
  if (!ctx) return fail(RBV_EINVAL, "null context");
  if (mode != RBV_FARFIELD_DIRECT && mode != RBV_FARFIELD_CHEBYSHEV)
    return fail(RBV_EINVAL, "rbv_set_farfield: unknown mode");
  ctx->farfield = mode;
  return RBV_OK;
}

// Tile geometry of every instrument for one launch; returns the total tile count and the dynamic smem.
// Tile geometry in units of 256 flux slots: level 0..kGeomLevels-1 -> 2, 3, 4, 8, 16, 32 units for an LSF with a
// short halo (tile = units * 256 - (K - 1), rounded down to whole 256-pixel blocks); wide LSFs start from the
// size that keeps the halo below ~8 % of the slots.  Small tiles = many CTAs per walker (latency of small
// batches), big tiles = less halo and per-CTA preamble (throughput of big batches).
static const int kGeomUnits[kGeomLevels] = {2, 3, 4, 8, 16, 32};

static TileGeom geometry_for(const InstDev& I, int level, int first_tile) {
  int units = kGeomUnits[level];
  if (I.K - 1 > 20) {                                     // halo <= ~8 % of the slots, at least one whole block out
    const int min_units = std::max((int)std::ceil((I.K - 1) / (0.08 * 256)), (I.K - 1 + 255) / 256 + 1);
    if (units < 8) units = std::max(units, std::min(min_units, 8 * 8));
    else units = std::max(units, std::min(min_units, 8 * 8) * (units / 8));
    units = std::min(units, 8 * 32);
  }
  const int need = (I.P + I.K - 1 + 255) / 256;           // no bigger than the spectrum
  units = std::max(std::min(units, need), (I.K - 1 + 255) / 256 + 1);
  TileGeom g;
  g.tile = (units * 256 - (I.K - 1)) & ~255;              // tiles start on the 256-pixel blocks of InstDev::obs_w
  g.ext_alloc = units * 256 + 2 * I.R;
  g.n_super = (units * 256 + kSuperPix - 1) / kSuperPix;
  g.first_tile = first_tile;
  g.n_tiles = (I.P + g.tile - 1) / g.tile;
  return g;
}

static int compute_geometry(const RbvContext* ctx, int level, TileGeom* geom, size_t* smem_out,
                            size_t n_inst_used = (size_t)-1) {
  int total = 0;
  size_t smem = 0;
  int ndim = ctx->ndim;
  for (size_t k = 0; k < std::min(ctx->inst.size(), n_inst_used); ++k) {
    const InstDev& I = ctx->inst[k].dev;
    const TileGeom g = geometry_for(I, level, total);
    total += g.n_tiles;
    geom[k] = g;
    smem = std::max(smem, smem_bytes_for(I, g, ndim ? ndim : 3 * I.C));
  }
  if (smem_out) *smem_out = smem;
  return total;
}

// Chunk size of phase 1: 64-pixel chunks (2 px per lane) when the biggest tile of the launch has fewer than
// kSmallChunkLimit 256-pixel chunks (<= 2 per warp: no room to balance line-core chunks), else 256-pixel chunks.
static bool small_chunks(const RbvContext* ctx, const TileGeom* geom, int n) {
  if (ctx->tune.force_ppt) return ctx->tune.force_ppt == 2;
  int big = 0;
  for (int k = 0; k < n; ++k) big = std::max(big, geom[k].ext_alloc);
  return big < kSmallChunkLimit * 256;
}

// Picks the largest tiles that still give every SM several CTAs (and fit RBV_MIN_CTAS CTAs per SM); a batch too
// small for that gets the smallest tiles, i.e. the most CTAs per walker.
static int choose_geometry(const RbvContext* ctx, int W, TileGeom* geom, size_t* smem_out,
                           size_t n_inst_used = (size_t)-1) {
  const long long want = (long long)kWantWaves * RBV_MIN_CTAS * ctx->sm_count;
  int total = 0;
  for (int level = kGeomLevels - 1; level >= 0; --level) {
    if (ctx->tune.force_level >= 0) level = ctx->tune.force_level;
    size_t smem = 0;
    total = compute_geometry(ctx, level, geom, &smem, n_inst_used);
    bool fits = smem <= (size_t)std::min(ctx->max_dyn_smem, (227 * 1024) / RBV_MIN_CTAS - 2048);
    if (level == 0 || ctx->tune.force_level >= 0 || (fits && (long long)W * total >= want)) {
      if (smem_out) *smem_out = smem;
      return total;
    }
  }
  return total;
}

// ---- streaming kernel (rbv_stream.cuh): work items = (walker, range of whole 1024-pixel segments of one instrument)
constexpr int kStreamBndMinLines = 8;   // fewer lines: a range evaluates its K-1 leading flux values itself (cheap)
constexpr int kStreamMaxHalo = 64;      // wider LSFs stay on the tile kernel (its LSF loop is unrolled 3 x 8 taps)
constexpr int kStreamWarps = kStreamThreads / 32;

// Shared memory per warp (doubles) for the instruments of a launch; 0 = not eligible.
static int stream_warp_doubles(const RbvContext* ctx, size_t n_inst_used) {
  int need = 0;
  for (size_t k = 0; k < std::min(ctx->inst.size(), n_inst_used); ++k) {
    const InstDev& I = ctx->inst[k].dev;
    if (I.K - 1 > kStreamMaxHalo) return 0;
    need = std::max(need, stream_smem_layout(I.L, I.K, I.Kpad).total);
  }
  return need;
}

// Ranges of every instrument of a launch (lo/hi/geom may be NULL: count only); 0 = the spectra do not fit the
// streaming kernel.  Longest first (the counter hands items out in slot order, so the launch ends on short items:
// guided self-scheduling): 16 segments while more than 48 are left, then a third of the remainder, down to single
// segments (C5a: 16 16 16 16 11 7 5 3 2 2 1 1 1 1).  An item start costs the line constants, the taps and ~750
// scalar instructions -- 5 us of warp time, measured through the schedule (14 / 22 / 26 / 31 items per walker:
// 5.38 / 5.51 / 5.56 / 5.67 ms at C5a) -- so finer schedules lose more in item starts than they win at the end of
// the launch, even on a 1024-row share (0.75 ms with this schedule, 0.79 ms with 22 items per walker whose idle
// tail is 4 % instead of 10 %).  The schedule depends on the spectra ONLY: a walker's lnprob is bit-identical in
// every batch that takes this kernel, on any number of ranks.  RBVFIT_B200_STREAM_SEGS=n: uniform ranges of n
// segments; RBVFIT_B200_STREAM_CAP / _DIV: longest range / divisor of the remainder (experiments).
static int stream_schedule(const RbvContext* ctx, size_t n_inst_used, TileGeom* geom, unsigned short* range_lo,
                           unsigned short* range_hi) {
  const size_t n_used = std::min(ctx->inst.size(), n_inst_used);
  if (n_used == 0 || n_used > (size_t)kMaxInst) return 0;
  TileGeom g0[kMaxInst];
  compute_geometry(ctx, 0, g0, nullptr, n_used);     // the workspace holds one partial per level-0 tile
  for (int cap = ctx->tune.stream_cap; cap <= 512; cap *= 2) {
    int total = 0;
    bool fits = true;
    for (size_t k = 0; k < n_used && fits; ++k) {
      const InstDev& I = ctx->inst[k].dev;
      const int n_seg = (I.P + kSuperPix - 1) / kSuperPix;
      const int min_seg = (g0[k].tile + kSuperPix - 1) / kSuperPix;   // never more ranges than level-0 tiles
      const int first = total;
      int at = 0;
      while (at < n_seg) {
        const int rem = n_seg - at;
        int len = ctx->tune.stream_segs > 0 ? ctx->tune.stream_segs
                                            : (n_seg <= 2 ? n_seg : std::min(cap, std::max(1, rem / ctx->tune.stream_div)));
        len = std::min(std::max(len, min_seg), rem);
        if (total >= kMaxStreamRanges) { fits = false; break; }
        if (range_lo) {
          range_lo[total] = (unsigned short)at;
          range_hi[total] = (unsigned short)(at + len);
        }
        at += len;
        ++total;
      }
      if (geom) {
        TileGeom g;
        g.tile = 0;
        g.ext_alloc = 0;
        g.n_super = 0;
        g.first_tile = first;
        g.n_tiles = total - first;
        geom[k] = g;
      }
    }
    if (fits) return total;
  }
  return 0;
}

// doubles per boundary record of a streaming launch: 2 (K - 1), K the widest LSF of the instruments used
static int stream_bnd_stride(const RbvContext* ctx, size_t n_inst_used) {
  int halo = 0;
  for (size_t k = 0; k < std::min(ctx->inst.size(), n_inst_used); ++k) halo = std::max(halo, ctx->inst[k].dev.K - 1);
  return 2 * std::max(halo, 1);
}

// Streaming kernel for a batch of W walkers?  Returns the number of ranges (0 = use the tile kernel).
static int stream_geometry(RbvContext* ctx, int W, TileGeom* geom, unsigned short* range_lo, unsigned short* range_hi,
                           int* warp_doubles, int* ctas_per_sm, size_t n_inst_used) {
  if (ctx->tune.stream == 0 || ctx->precision != RBV_PRECISION_FP64) return 0;
  const int wd = stream_warp_doubles(ctx, n_inst_used);
  const size_t smem = (size_t)wd * kStreamWarps * sizeof(double);
  if (wd == 0 || smem > (size_t)ctx->max_dyn_smem) return 0;
  int ctas = -1;
  for (auto& e : ctx->stream_ctas_cache)
    if (e.first == (int)smem) ctas = e.second;
  if (ctas < 0) {   // first use of this size (rebuild_tables warms the cache: no query while a stream is capturing)
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas, voigt_stream_kernel<3, true>, kStreamThreads, smem) != cudaSuccess)
      ctas = 0;
    ctx->stream_ctas_cache.emplace_back((int)smem, ctas);
  }
  if (ctas <= 0) return 0;
  if (ctx->tune.stream_ctas > 0) ctas = std::min(ctas, ctx->tune.stream_ctas);
  const long long warps = (long long)ctas * kStreamWarps * ctx->sm_count;
  const size_t n_used = std::min(ctx->inst.size(), n_inst_used);
  long long segs = 0, seg_max = 0;
  for (size_t k = 0; k < n_used; ++k) {
    const long long n_seg = (ctx->inst[k].dev.P + kSuperPix - 1) / kSuperPix;
    segs += n_seg;
    seg_max = std::max(seg_max, n_seg);
  }
  // too little work per resident warp: the tile kernel wins (measured crossovers: 28 segments per warp on a long
  // spectrum, where the tile kernel runs its biggest tiles; 6 on short ones -- C2's 20 000 px, a sightline batch)
  if (ctx->tune.stream < 0 && (long long)W * segs < (seg_max > 32 ? 28 : 6) * warps) return 0;
  const int total = stream_schedule(ctx, n_inst_used, geom, range_lo, range_hi);
  if (total == 0 || (long long)W * total >= 0x7fffffffLL) return 0;
  *warp_doubles = wd;
  *ctas_per_sm = ctas;
  return total;
}

// Tap upload + line bases for every instrument.  The register blocking R is context-wide (8 as soon as one
// instrument has a wide LSF) so that all instruments run in ONE launch.
static int rebuild_tables(RbvContext* ctx) {
  const int R = 8;   // outputs per thread in the LSF stage (64 FMAs per 8 flux + 8 tap loads)
  // only what the newest instrument changes: its taps, its line base, one more slot of the device table (a survey
  // context holds a thousand instruments -- rebuilding everything per add would be quadratic)
  for (size_t k = 0; k < ctx->inst.size(); ++k) {
    HostInst& hi = ctx->inst[k];
    InstDev& I = hi.dev;
    if (hi.d_taps) continue;
    I.K = (int)hi.taps.size();
    I.R = R;
    I.Kpad = (I.K + R - 1) / R * R;
    std::vector<double> rev(I.Kpad, 0.0);
    for (int m = 0; m < I.K; ++m) rev[m] = hi.taps[I.K - 1 - m];   // true convolution -> correlation
    RBV_CUDA(upload(&hi.d_taps, rev.data(), rev.size()));
    I.taps_rev = hi.d_taps;
    I.line_base = (k == 0) ? 0 : ctx->inst[k - 1].dev.line_base + ctx->inst[k - 1].dev.L;
    {
      const int n_seg = (I.P + kSuperPix - 1) / kSuperPix;
      double2* d_seg = nullptr;
      RBV_CUDA(cudaMalloc((void**)&d_seg, (size_t)n_seg * sizeof(double2)));
      hi.owned.push_back(d_seg);
      segment_range_kernel<<<n_seg, 256>>>(I.inv_wave, d_seg, I.P, I.K >> 1);
      RBV_CUDA(cudaGetLastError());
      RBV_CUDA(cudaDeviceSynchronize());     // set-up runs on the default stream, the batches on the caller's
      I.useg = d_seg;
      ctx->launches++;
    }
  }
  TileGeom geom[kMaxInst];
  // smallest tiles = most tiles: sizes the workspace (joint fits use <= 16 instruments; larger contexts are
  // sightline batches, which size their workspace from one instrument)
  ctx->n_tiles = compute_geometry(ctx, 0, geom, nullptr, kMaxInst);
  ctx->n_lines_total = 0;
  for (auto& hi : ctx->inst) ctx->n_lines_total += hi.dev.L;
  const size_t n = ctx->inst.size();
  if (n > ctx->d_inst_capacity) {
    const size_t cap = std::max<size_t>(16, 2 * n);
    InstDev* grown = nullptr;
    RBV_CUDA(cudaMalloc((void**)&grown, cap * sizeof(InstDev)));
    std::vector<InstDev> flat;
    for (auto& hi : ctx->inst) flat.push_back(hi.dev);
    RBV_CUDA(cudaMemcpy(grown, flat.data(), n * sizeof(InstDev), cudaMemcpyHostToDevice));
    cudaFree(ctx->d_inst);
    ctx->d_inst = grown;
    ctx->d_inst_capacity = cap;
  } else if (n > 0) {
    RBV_CUDA(cudaMemcpy(ctx->d_inst + (n - 1), &ctx->inst[n - 1].dev, sizeof(InstDev), cudaMemcpyHostToDevice));
  }
  if (n <= (size_t)kMaxInst) {   // occupancy of the streaming kernel for a joint launch and for a sightline launch
    TileGeom g[kMaxInst];
    unsigned short lo[kMaxStreamRanges], hi[kMaxStreamRanges];
    int wd = 0, nb = 0;
    stream_geometry(ctx, 1 << 20, g, lo, hi, &wd, &nb, kMaxInst);
    stream_geometry(ctx, 1 << 20, g, lo, hi, &wd, &nb, 1);
  }
  return RBV_OK;
}

int rbv_add_instrument(RbvContext* ctx, const RbvLineTable* lt, const RbvSpectrum* sp, int* out_index) {
  if (!ctx || !lt || !sp) return fail(RBV_EINVAL, "rbv_add_instrument: null argument");
  if (lt->n_lines <= 0 || lt->n_components <= 0) return fail(RBV_EINVAL, "rbv_add_instrument: empty line table");
  if (lt->n_lines > 4095) return fail(RBV_EINVAL, "rbv_add_instrument: more than 4095 lines per instrument");
  if (sp->n_pixels <= 0 || !sp->wave || !sp->inv_wave)
    return fail(RBV_EINVAL, "rbv_add_instrument: empty spectrum (n_pixels, wave and inv_wave are required)");
  if (lt->voigt_method != RBV_VOIGT_WOFZ && lt->voigt_method != RBV_VOIGT_FAST)
    return fail(RBV_EINVAL, "rbv_add_instrument: voigt_method must be RBV_VOIGT_WOFZ or RBV_VOIGT_FAST");
  if (sp->n_taps < 0 || (sp->n_taps > 0 && (sp->n_taps % 2 == 0 || !sp->taps)))
    return fail(RBV_EINVAL, "rbv_add_instrument: the LSF needs an odd number of taps");
  for (int l = 0; l < lt->n_lines; ++l)
    if (lt->comp[l] < 0 || lt->comp[l] >= lt->n_components)
      return fail(RBV_EINVAL, "rbv_add_instrument: component index out of range");
  RBV_ON_DEVICE(ctx);

  HostInst hi;
  struct Rollback {   // a failure half-way must not leak what was already uploaded
    HostInst* h;
    ~Rollback() {
      if (!h) return;
      for (void* p : h->owned) cudaFree(p);
      cudaFree(h->d_taps);
    }
  } rollback{&hi};
  InstDev& I = hi.dev;
  memset(&I, 0, sizeof(I));
  I.P = sp->n_pixels;
  I.L = lt->n_lines;
  I.C = lt->n_components;
  I.method = lt->voigt_method;
  I.inv_wave = sp->inv_wave;
  I.flux = sp->flux;
  I.inv_sigma2 = sp->inv_sigma2;
  I.log_inv_sigma2 = sp->log_inv_sigma2;

  // LSF taps as the reference applies them; "no kernel" = the single tap 1.0
  hi.taps.assign(sp->n_taps > 0 ? sp->n_taps : 1, 1.0);
  if (sp->n_taps > 0) {
    std::copy(sp->taps, sp->taps + sp->n_taps, hi.taps.begin());
    if (sp->normalize_taps) {
      double s = 0.0;
      for (double t : hi.taps) s += t;
      for (double& t : hi.taps) t /= s;
    }
  }
  if ((int)hi.taps.size() - 1 > kMaxHalo) return fail(RBV_EINVAL, "rbv_add_instrument: LSF too wide (max 8193 taps)");

  double *d_l0, *d_g, *d_f, *d_z;
  int* d_c;
  RBV_CUDA(upload(&d_l0, lt->lambda0, (size_t)I.L)); hi.owned.push_back(d_l0);
  RBV_CUDA(upload(&d_g, lt->gamma, (size_t)I.L));    hi.owned.push_back(d_g);
  RBV_CUDA(upload(&d_f, lt->f, (size_t)I.L));        hi.owned.push_back(d_f);
  RBV_CUDA(upload(&d_z, lt->zfac, (size_t)I.L));     hi.owned.push_back(d_z);
  RBV_CUDA(upload(&d_c, lt->comp, (size_t)I.L));     hi.owned.push_back(d_c);
  I.lambda0 = d_l0; I.gamma = d_g; I.f = d_f; I.zfac = d_z; I.comp = d_c;
  {
    std::vector<int> order(I.L);
    for (int l = 0; l < I.L; ++l) order[l] = l;
    std::stable_sort(order.begin(), order.end(), [lt](int x, int y) { return lt->comp[x] < lt->comp[y]; });
    RBV_CUDA(upload(&hi.d_fisher_order, order.data(), order.size())); hi.owned.push_back(hi.d_fisher_order);
  }

  reciprocal_kernel<<<(I.P + 255) / 256, 256>>>(sp->wave, sp->inv_wave, I.P);
  RBV_CUDA(cudaGetLastError());
  const int n_blk = (I.P + 255) / 256;
  double2* d_blk;
  RBV_CUDA(cudaMalloc((void**)&d_blk, (size_t)n_blk * sizeof(double2)));
  hi.owned.push_back(d_blk);
  block_range_kernel<<<n_blk, 256>>>(sp->inv_wave, d_blk, I.P);
  RBV_CUDA(cudaGetLastError());
  RBV_CUDA(cudaDeviceSynchronize());
  I.ublk = d_blk;
  ctx->launches += 2;
  if (I.flux && I.inv_sigma2) {
    double2* d_ow;
    RBV_CUDA(cudaMalloc((void**)&d_ow, (size_t)n_blk * 256 * sizeof(double2)));
    hi.owned.push_back(d_ow);
    pack_observed_kernel<<<n_blk, 256>>>(I.flux, I.inv_sigma2, d_ow, I.P);
    RBV_CUDA(cudaGetLastError());
    I.obs_w = d_ow;
    ctx->launches++;
  }
  if (I.log_inv_sigma2) {
    double* d_sum;
    RBV_CUDA(cudaMalloc((void**)&d_sum, sizeof(double)));
    hi.owned.push_back(d_sum);          // freed with the instrument (or by the rollback)
    fixed_order_sum_kernel<<<1, 256>>>(I.log_inv_sigma2, I.P, d_sum);
    RBV_CUDA(cudaGetLastError());
    RBV_CUDA(cudaMemcpy(&I.sum_log_inv_sigma2, d_sum, sizeof(double), cudaMemcpyDeviceToHost));
    ctx->launches++;
  }

  ctx->inst.push_back(hi);
  rollback.h = nullptr;                 // the context owns the arrays from here on (rbv_destroy frees them)
  int rc = rebuild_tables(ctx);
  if (rc != RBV_OK) return rc;
  if (out_index) *out_index = (int)ctx->inst.size() - 1;
  return RBV_OK;
}

int rbv_set_bounds(RbvContext* ctx, const double* lb, const double* ub, int ndim) {
  if (!ctx || !lb || !ub || ndim <= 0) return fail(RBV_EINVAL, "rbv_set_bounds: bad argument");
  for (auto& hi : ctx->inst)
    if (3 * hi.dev.C > ndim) return fail(RBV_EINVAL, "rbv_set_bounds: ndim smaller than 3 * n_components");
  RBV_ON_DEVICE(ctx);
  cudaFree(ctx->d_lb);
  cudaFree(ctx->d_ub);
  ctx->d_lb = ctx->d_ub = nullptr;
  RBV_CUDA(upload(&ctx->d_lb, lb, (size_t)ndim));
  RBV_CUDA(upload(&ctx->d_ub, ub, (size_t)ndim));
  ctx->ndim = ndim;
  return RBV_OK;
}

struct WorkspaceLayout {
  size_t tickets, oob, partials, lc, bnd, total;   // byte offsets
};

// [tickets u32 x W][oob i32 x W][partials f64 x W x n_tiles][line constants f64 x W x n_lines x LC_STRIDE]
// [boundary records f64 x W x bnd_doubles (streaming kernel: ranges x 2 (K - 1))]
static WorkspaceLayout workspace_layout_raw(int W, int tiles_per_walker, int lines_per_walker, size_t bnd_doubles = 0) {
  auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
  WorkspaceLayout lay;
  lay.tickets = 0;
  lay.oob = up(((size_t)W + 1) * sizeof(unsigned int));   // + the streaming kernel's work-queue counter
  lay.partials = lay.oob + up((size_t)W * sizeof(int));
  lay.lc = lay.partials + up((size_t)W * std::max(tiles_per_walker, 1) * sizeof(double));
  lay.bnd = lay.lc + up((size_t)W * std::max(lines_per_walker, 1) * LC_STRIDE * sizeof(double));
  lay.total = lay.bnd + up((size_t)W * bnd_doubles * sizeof(double));
  return lay;
}
static size_t stream_bnd_doubles(const RbvContext* ctx, size_t n_inst_used) {
  if (ctx->inst.empty() || stream_warp_doubles(ctx, n_inst_used) == 0) return 0;
  return (size_t)stream_schedule(ctx, n_inst_used, nullptr, nullptr, nullptr) * stream_bnd_stride(ctx, n_inst_used);
}
static WorkspaceLayout workspace_layout(const RbvContext* ctx, int W, bool sightlines) {
  if (!sightlines)
    return workspace_layout_raw(W, ctx->n_tiles, ctx->n_lines_total,
                                ctx->inst.size() <= (size_t)kMaxInst ? stream_bnd_doubles(ctx, (size_t)-1) : 0);
  TileGeom g[1];
  int tiles = compute_geometry(ctx, 0, g, nullptr, 1);
  return workspace_layout_raw(W, tiles, ctx->inst.empty() ? 1 : ctx->inst[0].dev.L, stream_bnd_doubles(ctx, 1));
}

int rbv_workspace_bytes(const RbvContext* ctx, int n_walkers, size_t* bytes) {
  if (!ctx || !bytes || n_walkers < 0) return fail(RBV_EINVAL, "rbv_workspace_bytes: bad argument");
  WorkspaceLayout lay = workspace_layout(ctx, n_walkers, false);
  *bytes = lay.total;
  return RBV_OK;
}

int rbv_workspace_bytes_sightlines(const RbvContext* ctx, int n_walkers, size_t* bytes) {
  if (!ctx || !bytes || n_walkers < 0) return fail(RBV_EINVAL, "rbv_workspace_bytes_sightlines: bad argument");
  *bytes = workspace_layout(ctx, n_walkers, true).total;
  return RBV_OK;
}

// What rbv_stretch_run needs to run the sampler's half-steps as ONE cooperative launch (voigt_mcmc_kernel): the
// parameters launch_lnprob would hand to the tile kernel with the constants prepared in the CTA prologue, and the
// launch shape.  launch_lnprob(plan != NULL) fills it and launches nothing; ok = false when the batch does not
// qualify (stream kernel, separate finalisation, too many lines).
struct LaunchPlan {
  LaunchParams prm;
  dim3 grid;
  size_t smem = 0;
  bool small = false;    // 2 pixels per lane in phase 1 (voigt_tile_kernel<3, 0, 2>)
  bool ok = false;
};

// W_hint (0 = W): the launch geometry (kernel, tile size / ranges) is chosen as for a batch of W_hint rows.
// The multi-GPU entry points pass the size of the WHOLE batch here, so that a rank evaluating 1/N of the rows uses
// the partition -- far-field super-chunks, order of the chi^2 additions -- the single-GPU launch uses, and every
// row's lnprob is bit-identical whatever the number of ranks.
static int launch_lnprob(RbvContext* ctx, const double* theta, int W, int wps, double* lnprob, void* workspace,
                         size_t workspace_bytes, void* stream, const char* who,
                         const StretchParams* sampler = nullptr, int sampler_split = -1,
                         const int* row_skip = nullptr, int W_hint = 0, bool with_prior = true,
                         LaunchPlan* plan = nullptr) {
  if (!ctx || !theta || !lnprob) return fail(RBV_EINVAL, std::string(who) + ": null argument");
  if (W < 0) return fail(RBV_EINVAL, std::string(who) + ": negative n_walkers");
  if (W == 0) return RBV_OK;
  if (ctx->inst.empty()) return fail(RBV_ESTATE, std::string(who) + ": no instrument added");
  if (ctx->ndim == 0) return fail(RBV_ESTATE, std::string(who) + ": bounds not set (rbv_set_bounds)");
  for (auto& hi : ctx->inst) {
    if (!hi.dev.flux || !hi.dev.inv_sigma2 || !hi.dev.log_inv_sigma2)
      return fail(RBV_ESTATE, std::string(who) + ": an instrument has no observed spectrum (flux-only instrument)");
    if (3 * hi.dev.C > ctx->ndim) return fail(RBV_EINVAL, std::string(who) + ": ndim smaller than 3 * n_components");
  }
  const bool sl = wps > 0;
  if (sl) {
    if ((long long)wps * (long long)ctx->inst.size() != (long long)W)
      return fail(RBV_EINVAL, std::string(who) + ": n_walkers must equal n_sightlines * walkers_per_sightline");
    const InstDev& A = ctx->inst[0].dev;
    for (auto& hi : ctx->inst)
      if (hi.dev.P != A.P || hi.dev.K != A.K || hi.dev.L != A.L || hi.dev.C != A.C)
        return fail(RBV_EINVAL, std::string(who) + ": sightlines must share n_pixels, n_taps, n_lines, n_components");
  } else if (ctx->inst.size() > (size_t)kMaxInst) {
    return fail(RBV_EINVAL, std::string(who) + ": at most 16 instruments in a joint fit (use the sightline entry "
                            "point for batches of independent spectra)");
  }
  WorkspaceLayout lay = workspace_layout(ctx, W, sl);
  if (!workspace || workspace_bytes < lay.total) return fail(RBV_ENOMEM, std::string(who) + ": workspace too small");
  RBV_ON_DEVICE(ctx);

  LaunchParams prm;
  memset(&prm, 0, sizeof(prm));
  prm.inst = ctx->d_inst;
  prm.theta = theta;
  prm.lb = with_prior ? ctx->d_lb : nullptr;      // no bounds: prep_kernel flags no row (vfit.lnlike, :297-319)
  prm.ub = with_prior ? ctx->d_ub : nullptr;
  prm.core_tab = ctx->d_core_tab;
  prm.lnprob = lnprob;
  prm.tickets = (unsigned int*)((char*)workspace + lay.tickets);
  prm.oob = (int*)((char*)workspace + lay.oob);
  prm.row_skip = row_skip;
  prm.partials = (double*)((char*)workspace + lay.partials);
  prm.lc = (double*)((char*)workspace + lay.lc);
  prm.n_lines_total = sl ? ctx->inst[0].dev.L : ctx->n_lines_total;
  prm.ndim = ctx->ndim;
  prm.n_inst = (int)ctx->inst.size();
  prm.W = W;
  prm.precision = ctx->precision;
  prm.farfield = ctx->farfield;
  prm.ff_budget = ctx->tune.ff_budget;
  prm.wps = wps;
  prm.sampler_split = -1;
  if (sampler) {
    prm.sampler_split = sampler_split;
    prm.sp = *sampler;
  }
  cudaStream_t st = (cudaStream_t)stream;

  // ONE launch covers every instrument: grid = (walkers, tiles per walker); the tile size is chosen per launch
  // from the batch size.  Sightline mode: each walker sees only its own instrument (identical geometry).
  size_t smem = 0;
  int stream_wd = 0, stream_ctas = 0;
  const int Wg = W_hint > 0 ? W_hint : W;
  const int stream_ranges = plan ? 0 : stream_geometry(ctx, Wg, prm.geom, prm.range_lo, prm.range_hi, &stream_wd,
                                                       &stream_ctas, sl ? 1 : (size_t)-1);
  bool stream_bnd = false;
  if (stream_ranges > 0) {
    prm.n_tiles = stream_ranges;
    // boundary records where a spectrum has several ranges AND evaluating the K-1 leading flux values per range
    // would be expensive (kStreamBndMinLines lines or more); else every range evaluates them itself
    int max_lines = 0;
    for (size_t k = 0; k < (sl ? (size_t)1 : ctx->inst.size()); ++k) max_lines = std::max(max_lines, ctx->inst[k].dev.L);
    stream_bnd = stream_ranges > (sl ? 1 : (int)ctx->inst.size()) && max_lines >= kStreamBndMinLines;
    if (stream_bnd) {
      prm.bnd = (double*)((char*)workspace + lay.bnd);
      prm.bnd_stride = stream_bnd_stride(ctx, sl ? 1 : (size_t)-1);
    }
  } else prm.n_tiles = choose_geometry(ctx, Wg, prm.geom, &smem, sl ? 1 : (size_t)-1);
  dim3 grid((unsigned)W, (unsigned)prm.n_tiles);
  if (prm.n_tiles > 65535) return fail(RBV_EINVAL, std::string(who) + ": more than 65535 tiles per walker");
  // the walker's last CTA finalises in-kernel when the grid is small (one launch less on the latency path); big
  // grids use a separate tiny launch instead, so that no CTA waits for the ticket round trip
  prm.inst_in_params = !sl && ctx->inst.size() <= (size_t)kMaxInst;
  if (prm.inst_in_params)
    for (size_t k = 0; k < ctx->inst.size(); ++k) prm.inst_v[k] = ctx->inst[k].dev;
  prm.separate_finalize = (long long)Wg * prm.n_tiles >= 8LL * RBV_MIN_CTAS * ctx->sm_count;
  if (ctx->tune.force_finalize >= 0) prm.separate_finalize = ctx->tune.force_finalize;
  // Small grids (the 25-walker half-steps of an MCMC run, the slice sampler's iterations): no prep launch at all --
  // every CTA prepares the walker's line constants (and, for the fused sampler, its proposal row) in its prologue.
  // The tickets then have to be zero on entry: a memset node instead of a kernel.
  int max_lines = 0;
  for (size_t k = 0; k < (sl ? (size_t)1 : ctx->inst.size()); ++k) max_lines = std::max(max_lines, ctx->inst[k].dev.L);
  // (opt-in, RBVFIT_B200_INLINE_PREP=1: measured neutral on the C1 stretch move -- 25.6k steps/s either way, the
  // prologue's dependent chain replaces the prep launch one for one -- and 3 % slower on the C2 slice move)
  const bool inline_prep = ctx->tune.inline_prep > 0 && stream_ranges == 0 && !prm.separate_finalize &&
                           max_lines <= 256 && (long long)Wg * prm.n_tiles <= 2LL * RBV_MIN_CTAS * ctx->sm_count;
  if (plan) {
    plan->ok = !prm.separate_finalize && max_lines <= 256;
    prm.lc = nullptr;                    // constants (and the proposal) in the CTA prologue
    plan->prm = prm;
    plan->grid = grid;
    plan->smem = smem;
    plan->small = small_chunks(ctx, prm.geom, sl ? 1 : prm.n_inst);
    return RBV_OK;
  }
  if (inline_prep) {
    prm.lc = nullptr;
    RBV_CUDA(cudaMemsetAsync(prm.tickets, 0, (size_t)W * sizeof(unsigned int), st));
  } else {
    dim3 pgrid((unsigned)W, (unsigned)((prm.n_lines_total + 127) / 128));
    if (sampler) prep_propose_kernel<<<pgrid, 128, (size_t)prm.ndim * sizeof(double), st>>>(prm);
    else prep_kernel<<<pgrid, 128, 0, st>>>(prm);
    RBV_CUDA(cudaGetLastError());
    ctx->launches++;
  }
  if (stream_ranges > 0) {
    // persistent warps pull (walker, range) items from a global counter; lnprob always by finalize_kernel (a
    // per-walker ticket + in-kernel finalisation by the last range to finish was measured 5 % slower at C5a)
    prm.separate_finalize = 1;
    const long long items = (long long)W * stream_ranges;
    const unsigned ctas = (unsigned)std::min<long long>((long long)stream_ctas * ctx->sm_count,
                                                        (items + kStreamWarps - 1) / kStreamWarps);
    const size_t stream_smem = (size_t)stream_wd * kStreamWarps * sizeof(double);
    if (stream_bnd) voigt_stream_kernel<3, true><<<ctas, kStreamThreads, stream_smem, st>>>(prm, stream_wd);
    else voigt_stream_kernel<3, false><<<ctas, kStreamThreads, stream_smem, st>>>(prm, stream_wd);
    ctx->last_kernel = RBV_KERNEL_STREAM;
  } else if (small_chunks(ctx, prm.geom, sl ? 1 : prm.n_inst)) {
    voigt_tile_kernel<3, 0, 2><<<grid, kThreads, smem, st>>>(prm);
    ctx->last_kernel = RBV_KERNEL_TILE;
  } else {
    voigt_tile_kernel<3, 0, 8><<<grid, kThreads, smem, st>>>(prm);
    ctx->last_kernel = RBV_KERNEL_TILE;
  }
  RBV_CUDA(cudaGetLastError());
  ctx->launches++;
  if (prm.separate_finalize) {
    if (stream_bnd) finalize_stream_kernel<<<(W + 3) / 4, 128, 0, st>>>(prm);
    else finalize_kernel<<<(W + 3) / 4, 128, 0, st>>>(prm);
    RBV_CUDA(cudaGetLastError());
    ctx->launches++;
  }
  return RBV_OK;
}

int rbv_lnprob_batch(RbvContext* ctx, const double* theta, int W, double* lnprob, void* workspace,
                     size_t workspace_bytes, void* stream) {
  return launch_lnprob(ctx, theta, W, 0, lnprob, workspace, workspace_bytes, stream, "rbv_lnprob_batch");
}

int rbv_lnlike_batch(RbvContext* ctx, const double* theta, int W, double* lnlike, void* workspace,
                     size_t workspace_bytes, void* stream) {
  return launch_lnprob(ctx, theta, W, 0, lnlike, workspace, workspace_bytes, stream, "rbv_lnlike_batch", nullptr, -1,
                       nullptr, 0, false);
}

int rbv_lnprob_batch_sightlines(RbvContext* ctx, const double* theta, int W, int walkers_per_sightline,
                                double* lnprob, void* workspace, size_t workspace_bytes, void* stream) {
  if (walkers_per_sightline <= 0) return fail(RBV_EINVAL, "rbv_lnprob_batch_sightlines: walkers_per_sightline <= 0");
  return launch_lnprob(ctx, theta, W, walkers_per_sightline, lnprob, workspace, workspace_bytes, stream,
                       "rbv_lnprob_batch_sightlines");
}

// 1 = p points into page-locked host memory (cudaMallocHost / cudaHostRegister / a pinned torch tensor): an
// asynchronous H2D copy can read it in place, no staging copy needed
int rbv_host_pinned(const void* p) {
  if (!p) return 0;
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return a.type == cudaMemoryTypeHost ? 1 : 0;
}

int rbv_lnprob_batch_host(RbvContext* ctx, const double* theta_host, int W, double* lnprob_host,
                          double* theta_dev, double* lnprob_dev, void* workspace, size_t workspace_bytes,
                          void* stream) {
  if (!ctx || !theta_host || !lnprob_host || !theta_dev || !lnprob_dev)
    return fail(RBV_EINVAL, "rbv_lnprob_batch_host: null argument");
  if (W <= 0) return W == 0 ? RBV_OK : fail(RBV_EINVAL, "negative n_walkers");
  RBV_ON_DEVICE(ctx);
  cudaStream_t st = (cudaStream_t)stream;
  RBV_CUDA(cudaMemcpyAsync(theta_dev, theta_host, (size_t)W * ctx->ndim * sizeof(double), cudaMemcpyHostToDevice, st));
  int rc = rbv_lnprob_batch(ctx, theta_dev, W, lnprob_dev, workspace, workspace_bytes, stream);
  if (rc != RBV_OK) return rc;
  RBV_CUDA(cudaMemcpyAsync(lnprob_host, lnprob_dev, (size_t)W * sizeof(double), cudaMemcpyDeviceToHost, st));
  RBV_CUDA(cudaStreamSynchronize(st));
  return RBV_OK;
}

// ------------------------------------------------------------------------------------------ device-resident sampler
constexpr int kMaxRanks = 64;   // ranks of one communicator (rows of a half-step are padded to world x chunk)
constexpr int kPtMaxTemps = 4096;   // temperatures of rbv_pt_run (one shared-memory counter each in the plan kernel)
struct StretchLayout {
  size_t prop, lnp_prop, factors, walker_of, ctr, lnprob_ws, total;
  size_t pt_tmp = 0, pt_src = 0;   // rbv_pt_run only: coordinates before the swap stage, slot map
};
static StretchLayout stretch_layout(const RbvContext* ctx, int W) {
  auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
  const size_t h = (size_t)(W + 1) / 2;
  StretchLayout lay;
  lay.prop = 0;
  lay.lnp_prop = up(h * std::max(ctx->ndim, 1) * sizeof(double));
  lay.factors = lay.lnp_prop + up((h + kMaxRanks) * sizeof(double));   // padded to world x chunk rows: the in-place
  lay.walker_of = lay.factors + up(h * sizeof(double));                //   all-gather of the multi-GPU form
  lay.ctr = lay.walker_of + up(h * sizeof(int));
  lay.lnprob_ws = lay.ctr + 256;
  lay.total = lay.lnprob_ws + workspace_layout(ctx, (int)h, false).total;
  return lay;
}

int rbv_stretch_workspace_bytes(const RbvContext* ctx, int n_walkers, size_t* bytes) {
  if (!ctx || !bytes || n_walkers < 2) return fail(RBV_EINVAL, "rbv_stretch_workspace_bytes: bad argument");
  *bytes = stretch_layout(ctx, n_walkers).total;
  return RBV_OK;
}

// forward declarations (multi-GPU helpers, defined with the communicator entry points below)
static void rank_rows(int n, int rank, int world, int* lo, int* hi, int* chunk);
static int allgather_rows(RbvContext* ctx, double* buf, int chunk, cudaStream_t st);

// The run loop shared by rbv_stretch_run / rbv_stretch_run_dist / rbv_stretch_run_sink / rbv_pt_run.  One step is
// captured in a CUDA graph (the step index lives in device memory) and replayed.
//   dist   rows of every half-step split over the ranks of the context's communicator, in-place NCCL all-gather of
//          their lnprob inside the captured step (separate propose / accept kernels); otherwise the fused single-GPU
//          step (proposal in the prep kernel, accept/reject in the finalisation)
//   sink   chain hand-off to the host while the run goes on: P.chain / P.lnp_chain are device RINGS of
//          2 x block_steps steps; after every block the finished half is copied to page-locked staging on a second
//          stream and from there by this thread into the caller's arrays, while the device runs the next block
//   pt     parallel tempering (rbv_pt.cuh): P holds the S T = P.S tempered ensembles of S sightlines (S = 1: one
//          joint context); a half-step is the separate propose kernel, ONE lnprob launch over all ensembles' rows (in
//          sightline mode with T n_S rows per sightline when pt->survey) and the accept kernel, then the swap stage
//          records the step and advances the counter.  A recorded step is row_c chain and row_l lnprob doubles (the
//          sink's ring; row_l = 0 when no lnprob chain is recorded)
static int stretch_run_impl(RbvContext* ctx, StretchParams& P, const StretchLayout& lay, char* ws,
                            size_t workspace_bytes, int n_walkers, int n_steps, bool dist, const RbvChainSink* sink,
                            int use_graph, cudaStream_t st, const char* who, const PtParams* pt = nullptr) {
  RBV_CUDA(cudaMemsetAsync(ws + lay.ctr, 0, 256, st));
  const size_t row_c = pt ? (size_t)pt->S * pt->n_record * n_walkers * ctx->ndim : (size_t)n_walkers * ctx->ndim;
  const size_t row_l = pt ? (pt->lnp_chain ? (size_t)pt->S * pt->T * n_walkers : 0) : (size_t)n_walkers;
  const size_t lnprob_ws_bytes = workspace_bytes - lay.lnprob_ws;
  const int h = (n_walkers + 1) / 2;
  const int rank = (dist && ctx->comm) ? ctx->comm_rank : 0, world = (dist && ctx->comm) ? ctx->comm_world : 1;
  void* stream = (void*)st;

  auto one_step = [&]() -> int {
    if (pt) {
      for (int split = 0; split < 2; ++split) {
        const int nS = split == 0 ? h : n_walkers - h, rows = P.S * nS;
        stretch_propose_kernel<<<(unsigned)((rows + 3) / 4), 128, 0, st>>>(P, split);
        RBV_CUDA(cudaGetLastError());
        ctx->launches++;
        int rc = launch_lnprob(ctx, P.prop, rows, pt->survey ? pt->T * nS : 0, P.lnp_prop, ws + lay.lnprob_ws,
                               lnprob_ws_bytes, stream, who);
        if (rc != RBV_OK) return rc;
        stretch_accept_kernel<<<(unsigned)((rows + 3) / 4), 128, 0, st>>>(P, split);
        RBV_CUDA(cudaGetLastError());
        ctx->launches++;
      }
      const int slots = pt->S * pt->T * n_walkers;
      RBV_CUDA(cudaMemcpyAsync(pt->coords_tmp, pt->coords, (size_t)slots * ctx->ndim * sizeof(double),
                               cudaMemcpyDeviceToDevice, st));
      pt_swap_plan_kernel<<<(unsigned)pt->S, kPtPlanThreads, (size_t)pt->T * sizeof(unsigned int), st>>>(*pt);
      RBV_CUDA(cudaGetLastError());
      pt_gather_record_kernel<<<(unsigned)((slots + 3) / 4), 128, 0, st>>>(*pt);
      RBV_CUDA(cudaGetLastError());
      ctx->launches += 2;
      return RBV_OK;
    }
    for (int split = 0; split < 2; ++split) {
      const int nS = split == 0 ? h : n_walkers - h;
      if (!dist) {
        // two launches per half-step: prep_propose_kernel (proposal + line constants) and the lnprob kernel, whose
        // per-walker finalisation also applies accept/reject and appends the walker's row to the chain
        int rc = launch_lnprob(ctx, P.prop, nS, 0, P.lnp_prop, ws + lay.lnprob_ws, lnprob_ws_bytes, stream, who, &P,
                               split);
        if (rc != RBV_OK) return rc;
        continue;
      }
      // every rank builds all proposals (replicated state, counter-based streams), evaluates its rows, the ranks
      // all-gather the 8-byte lnprob values in place over NCCL, every rank applies the same accept/reject
      int lo, hi, chunk;
      rank_rows(nS, rank, world, &lo, &hi, &chunk);
      stretch_propose_kernel<<<(nS + 3) / 4, 128, 0, st>>>(P, split);
      RBV_CUDA(cudaGetLastError());
      ctx->launches++;
      if (hi > lo) {
        int rc = launch_lnprob(ctx, P.prop + (size_t)lo * ctx->ndim, hi - lo, 0, P.lnp_prop + lo, ws + lay.lnprob_ws,
                               lnprob_ws_bytes, stream, who, nullptr, -1, nullptr, nS);
        if (rc != RBV_OK) return rc;
      }
      int rc = allgather_rows(ctx, P.lnp_prop, chunk, st);
      if (rc != RBV_OK) return rc;
      stretch_accept_kernel<<<(nS + 3) / 4, 128, 0, st>>>(P, split);
      RBV_CUDA(cudaGetLastError());
      ctx->launches++;
    }
    return RBV_OK;
  };

  const bool graph_ok = use_graph && st != nullptr && n_steps >= 4;
  if (sink && !graph_ok) return fail(RBV_EINVAL, std::string(who) + ": the chain sink needs use_graph, a non-default "
                                                                    "stream and at least 4 steps");
  // ---- small ensembles: the whole loop as cooperative launches of voigt_mcmc_kernel (one per block of steps)
  LaunchPlan plan;
  bool persistent = false;
  if (graph_ok && !dist && !pt && ctx->tune.mcmc_persistent != 0 && ctx->tune.stream != 1) {   // (STREAM=1: tests
                                                                                       // force the stream kernel everywhere)
    int rc0 = launch_lnprob(ctx, P.prop, h, 0, P.lnp_prop, ws + lay.lnprob_ws, lnprob_ws_bytes, stream, who, &P, 0,
                            nullptr, 0, true, &plan);
    if (rc0 != RBV_OK) return rc0;
    if (plan.ok) {
      int per_sm = 0;      // resident CTAs per SM at this launch's shared-memory size (a query, not a stream call)
      cudaError_t eo = plan.small
          ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, voigt_mcmc_kernel<3, 2>, kThreads, plan.smem)
          : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, voigt_mcmc_kernel<3, 8>, kThreads, plan.smem);
      if (eo != cudaSuccess) per_sm = 0;
      persistent = (long long)plan.grid.x * plan.grid.y <= (long long)per_sm * ctx->sm_count;
    }
  }
  auto run_persistent = [&](int ns) -> cudaError_t {      // ns steps, enqueued on st
    int n = ns;
    unsigned int* bar = ctx->d_grid_bar;
    void* args[] = {(void*)&plan.prm, (void*)&n, (void*)&bar};
    cudaError_t e2 = cudaMemsetAsync(ctx->d_grid_bar, 0, sizeof(unsigned int), st);
    if (e2 == cudaSuccess) e2 = cudaMemsetAsync(plan.prm.tickets, 0, (size_t)h * sizeof(unsigned int), st);
    if (e2 != cudaSuccess) return e2;
    ctx->launches++;
    ctx->last_kernel = RBV_KERNEL_TILE;
    return plan.small ? cudaLaunchCooperativeKernel((void*)voigt_mcmc_kernel<3, 2>, plan.grid, dim3(kThreads), args,
                                                    plan.smem, st)
                      : cudaLaunchCooperativeKernel((void*)voigt_mcmc_kernel<3, 8>, plan.grid, dim3(kThreads), args,
                                                    plan.smem, st);
  };
  if (persistent && !sink) {
    cudaError_t e2 = cudaSuccess;
    for (int done = 0; done < n_steps && e2 == cudaSuccess; done += 1024) e2 = run_persistent(std::min(1024, n_steps - done));
    if (e2 == cudaSuccess) e2 = cudaStreamSynchronize(st);
    if (e2 != cudaSuccess) return fail(RBV_ECUDA, std::string(who) + " (cooperative launch): " + cudaGetErrorString(e2));
    return RBV_OK;
  }
  if (!graph_ok) {
    for (int s2 = 0; s2 < n_steps; ++s2) {
      int rc = one_step();
      if (rc != RBV_OK) return rc;
    }
    if (dist) RBV_CUDA(cudaStreamSynchronize(st));
    return RBV_OK;
  }
  if (dist && world > 1) {
    for (int split = 0; split < 2; ++split) {   // NCCL sets up its buffers on the first collective of a size: not
      int lo, hi, chunk;                        // inside a capture (lnp_prop is scratch here)
      rank_rows(split == 0 ? h : n_walkers - h, rank, world, &lo, &hi, &chunk);
      int rc = allgather_rows(ctx, P.lnp_prop, chunk, st);
      if (rc != RBV_OK) return rc;
    }
    RBV_CUDA(cudaStreamSynchronize(st));
  }
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  cudaError_t e = cudaSuccess;
  if (!persistent) {
    const long long launches_before = ctx->launches;
    RBV_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    int rc = one_step();
    e = cudaStreamEndCapture(st, &graph);
    if (rc != RBV_OK) {
      if (graph) cudaGraphDestroy(graph);
      return rc;
    }
    if (e != cudaSuccess) return fail(RBV_ECUDA, std::string("cudaStreamEndCapture: ") + cudaGetErrorString(e));
    const long long per_step = ctx->launches - launches_before;
    e = cudaGraphInstantiate(&exec, graph, 0);
    if (e != cudaSuccess) {
      cudaGraphDestroy(graph);
      return fail(RBV_ECUDA, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e));
    }
    ctx->launches = launches_before + per_step * n_steps;
  }
  if (!sink) {
    for (int s2 = 0; s2 < n_steps && e == cudaSuccess; ++s2) e = cudaGraphLaunch(exec, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  } else {
    // ---- pipelined hand-off: block b runs on the device while block b - 1 travels device ring -> pinned staging
    // (copy stream) -> the caller's host arrays (this thread)
    const int K = sink->block_steps;
    const int n_blocks = (n_steps + K - 1) / K;
    auto steps_of = [&](int b) { return std::min(K, n_steps - b * K); };
    auto drain = [&](int b) -> cudaError_t {       // pinned half of block b -> host arrays
      cudaError_t e2 = cudaEventSynchronize(ctx->sink_copied[b & 1]);
      if (e2 != cudaSuccess) return e2;
      const int half = b & 1, ns = steps_of(b);
      if (sink->chain_host)
        memcpy(sink->chain_host + (size_t)b * K * row_c, sink->ring_pinned + (size_t)half * K * row_c,
               (size_t)ns * row_c * sizeof(double));
      if (sink->lnprob_chain_host)
        memcpy(sink->lnprob_chain_host + (size_t)b * K * row_l,
               sink->ring_pinned + 2 * (size_t)K * row_c + (size_t)half * K * row_l, (size_t)ns * row_l * sizeof(double));
      return cudaSuccess;
    };
    for (int b = 0; b < n_blocks && e == cudaSuccess; ++b) {
      const int half = b & 1, ns = steps_of(b);
      if (b >= 2) e = cudaStreamWaitEvent(st, ctx->sink_copied[half], 0);      // the ring half is free again
      if (persistent) e = (e == cudaSuccess) ? run_persistent(ns) : e;
      else for (int k = 0; k < ns && e == cudaSuccess; ++k) e = cudaGraphLaunch(exec, st);
      if (e == cudaSuccess) e = cudaEventRecord(ctx->sink_done[half], st);
      if (e == cudaSuccess && b >= 1) e = drain(b - 1);      // frees pinned half (b - 1) & 1 for block b + 1's copy
      if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->sink_stream, ctx->sink_done[half], 0);
      if (e == cudaSuccess)
        e = cudaMemcpyAsync(sink->ring_pinned + (size_t)half * K * row_c, sink->ring_dev + (size_t)half * K * row_c,
                            (size_t)ns * row_c * sizeof(double), cudaMemcpyDeviceToHost, ctx->sink_stream);
      if (e == cudaSuccess)
        e = cudaMemcpyAsync(sink->ring_pinned + 2 * (size_t)K * row_c + (size_t)half * K * row_l,
                            sink->ring_dev + 2 * (size_t)K * row_c + (size_t)half * K * row_l,
                            (size_t)ns * row_l * sizeof(double), cudaMemcpyDeviceToHost, ctx->sink_stream);
      if (e == cudaSuccess) e = cudaEventRecord(ctx->sink_copied[half], ctx->sink_stream);
    }
    if (e == cudaSuccess) e = drain(n_blocks - 1);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  }
  if (exec) cudaGraphExecDestroy(exec);
  if (graph) cudaGraphDestroy(graph);
  if (e != cudaSuccess) return fail(RBV_ECUDA, std::string(who) + " (graph): " + cudaGetErrorString(e));
  return RBV_OK;
}

// the copy stream and events of the chain sink (created on first use, owned by the context)
static int sink_stream_setup(RbvContext* ctx) {
  if (!ctx->sink_stream) {
    RBV_CUDA(cudaStreamCreateWithFlags(&ctx->sink_stream, cudaStreamNonBlocking));
    for (int k = 0; k < 2; ++k) {
      RBV_CUDA(cudaEventCreateWithFlags(&ctx->sink_done[k], cudaEventDisableTiming));
      RBV_CUDA(cudaEventCreateWithFlags(&ctx->sink_copied[k], cudaEventDisableTiming));
    }
  }
  return RBV_OK;
}

static int stretch_run_entry(RbvContext* ctx, double* coords, double* lnprob, int n_walkers, int n_steps, double a,
                             unsigned long long seed, unsigned long long first_step, double* chain,
                             double* lnprob_chain, const RbvChainSink* sink, int* n_accepted, int* flag,
                             void* workspace, size_t workspace_bytes, bool dist, int use_graph, void* stream,
                             const char* who) {
  if (!ctx || !coords || !lnprob || !n_accepted || !flag) return fail(RBV_EINVAL, std::string(who) + ": null argument");
  if (n_walkers < 2) return fail(RBV_EINVAL, std::string(who) + ": need at least two walkers");
  if (n_steps < 0 || !(a > 1.0)) return fail(RBV_EINVAL, std::string(who) + ": n_steps < 0 or stretch scale a <= 1");
  if (ctx->inst.empty() || ctx->ndim == 0) return fail(RBV_ESTATE, std::string(who) + ": context not set up");
  if (sink && (sink->block_steps < 1 || !sink->ring_dev || !sink->ring_pinned))
    return fail(RBV_EINVAL, std::string(who) + ": incomplete chain sink");
  if (n_steps == 0) return RBV_OK;
  const StretchLayout lay = stretch_layout(ctx, n_walkers);
  if (!workspace || workspace_bytes < lay.total) return fail(RBV_ENOMEM, std::string(who) + ": workspace too small");
  RBV_ON_DEVICE(ctx);
  cudaStream_t st = (cudaStream_t)stream;
  char* ws = (char*)workspace;
  StretchParams P;
  memset(&P, 0, sizeof(P));
  P.coords = coords;
  P.lnp = lnprob;
  P.prop = (double*)(ws + lay.prop);
  P.lnp_prop = (double*)(ws + lay.lnp_prop);
  P.factors = (double*)(ws + lay.factors);
  P.walker_of = (int*)(ws + lay.walker_of);
  P.chain = chain;
  P.lnp_chain = lnprob_chain;
  if (sink) {
    P.ring_steps = 2 * sink->block_steps;
    P.chain = sink->ring_dev;
    P.lnp_chain = sink->ring_dev + (size_t)P.ring_steps * n_walkers * ctx->ndim;
    int rc = sink_stream_setup(ctx);
    if (rc != RBV_OK) return rc;
  }
  P.n_accepted = n_accepted;
  P.flag = flag;
  P.step_ctr = (unsigned long long*)(ws + lay.ctr);
  P.ticket = (unsigned int*)(ws + lay.ctr + 64);
  P.first_step = first_step;
  P.seed = seed;
  P.a = a;
  P.W = n_walkers;
  P.ndim = ctx->ndim;
  P.S = 1;
  return stretch_run_impl(ctx, P, lay, ws, workspace_bytes, n_walkers, n_steps, dist, sink, use_graph, st, who);
}

int rbv_stretch_run(RbvContext* ctx, double* coords, double* lnprob, int n_walkers, int n_steps, double a,
                    unsigned long long seed, unsigned long long first_step, double* chain, double* lnprob_chain,
                    int* n_accepted, int* flag, void* workspace, size_t workspace_bytes, int use_graph,
                    void* stream) {
  return stretch_run_entry(ctx, coords, lnprob, n_walkers, n_steps, a, seed, first_step, chain, lnprob_chain, nullptr,
                           n_accepted, flag, workspace, workspace_bytes, false, use_graph, stream, "rbv_stretch_run");
}

int rbv_stretch_run_dist(RbvContext* ctx, double* coords, double* lnprob, int n_walkers, int n_steps, double a,
                         unsigned long long seed, unsigned long long first_step, double* chain, double* lnprob_chain,
                         int* n_accepted, int* flag, void* workspace, size_t workspace_bytes, int use_graph,
                         void* stream) {
  return stretch_run_entry(ctx, coords, lnprob, n_walkers, n_steps, a, seed, first_step, chain, lnprob_chain, nullptr,
                           n_accepted, flag, workspace, workspace_bytes, true, use_graph, stream,
                           "rbv_stretch_run_dist");
}

int rbv_stretch_run_sink(RbvContext* ctx, double* coords, double* lnprob, int n_walkers, int n_steps, double a,
                         unsigned long long seed, unsigned long long first_step, const RbvChainSink* sink,
                         int* n_accepted, int* flag, void* workspace, size_t workspace_bytes, int distributed,
                         void* stream) {
  if (!sink) return fail(RBV_EINVAL, "rbv_stretch_run_sink: null sink");
  return stretch_run_entry(ctx, coords, lnprob, n_walkers, n_steps, a, seed, first_step, nullptr, nullptr, sink,
                           n_accepted, flag, workspace, workspace_bytes, distributed != 0, 1, stream,
                           "rbv_stretch_run_sink");
}

// ---- parallel tempering (rbv_pt.cuh): T tempered stretch-move ensembles and ptemcee's swap stage --------------
// S sightlines of T temperatures (survey mode), or S = 1 and one joint context (rbv_pt_run)
static StretchLayout pt_layout(const RbvContext* ctx, int S, int T, int W, bool survey) {
  auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
  const size_t rows = (size_t)((W + 1) / 2) * T * S, slots = (size_t)S * T * W, nd = std::max(ctx->ndim, 1);
  StretchLayout lay;
  lay.prop = 0;
  lay.lnp_prop = up(rows * nd * sizeof(double));
  lay.factors = lay.lnp_prop + up(rows * sizeof(double));
  lay.walker_of = lay.factors + up(rows * sizeof(double));
  lay.ctr = lay.walker_of + up(rows * sizeof(int));
  lay.pt_tmp = lay.ctr + 256;
  lay.pt_src = lay.pt_tmp + up(slots * nd * sizeof(double));
  lay.lnprob_ws = lay.pt_src + up(slots * sizeof(int));
  lay.total = lay.lnprob_ws + workspace_layout(ctx, (int)rows, survey).total;
  return lay;
}

static int pt_shape_ok(int T, int W) {
  return T >= 1 && T <= kPtMaxTemps && W >= 2 && (long long)T * W <= 0x7fffffffLL;
}

// S T W slots and S T ceil(W / 2) half-step rows in int range
static int pt_sightlines_shape_ok(long long S, int T, int W) {
  return S >= 1 && pt_shape_ok(T, W) && S * T * W <= 0x7fffffffLL;
}

int rbv_pt_workspace_bytes(const RbvContext* ctx, int n_temps, int n_walkers, size_t* bytes) {
  if (!ctx || !bytes || !pt_shape_ok(n_temps, n_walkers)) return fail(RBV_EINVAL, "rbv_pt_workspace_bytes: bad argument");
  *bytes = pt_layout(ctx, 1, n_temps, n_walkers, false).total;
  return RBV_OK;
}

int rbv_pt_workspace_bytes_sightlines(const RbvContext* ctx, int n_temps, int walkers_per_sightline, size_t* bytes) {
  if (!ctx || !bytes || ctx->inst.empty() ||
      !pt_sightlines_shape_ok((long long)ctx->inst.size(), n_temps, walkers_per_sightline))
    return fail(RBV_EINVAL, "rbv_pt_workspace_bytes_sightlines: bad argument");
  *bytes = pt_layout(ctx, (int)ctx->inst.size(), n_temps, walkers_per_sightline, true).total;
  return RBV_OK;
}

// The two entry points: S = 1 and a joint context (rbv_pt_run), or one sightline per instrument of the context
// (rbv_pt_run_sightlines, survey = true).  Arguments are checked by the callers except the ladder, which is copied to
// the host and checked here.
static int pt_run_entry(RbvContext* ctx, int S, bool survey, double* coords, double* lnprob, double* betas, int T,
                        int W, int n_steps, const RbvPtControl* control, unsigned long long seed,
                        unsigned long long first_step, double* chain, double* lnprob_chain, const RbvChainSink* sink,
                        double* beta_history, double* ti_moments, int* n_accepted,
                        unsigned long long* n_swaps_accepted, int* flag, void* workspace, size_t workspace_bytes,
                        int use_graph, void* stream, const char* who) {
  const std::string w(who);
  if (n_steps < 0 || !(control->a > 1.0)) return fail(RBV_EINVAL, w + ": n_steps < 0 or stretch scale a <= 1");
  if (control->n_record < 1 || control->n_record > T) return fail(RBV_EINVAL, w + ": n_record outside 1 .. n_temps");
  if (control->adapt && !(control->adaptation_lag > 0.0 && control->adaptation_time > 0.0))
    return fail(RBV_EINVAL, w + ": adaptation_lag and adaptation_time must be > 0");
  if (sink && (chain || lnprob_chain)) return fail(RBV_EINVAL, w + ": pass device chains or a sink, not both");
  if (sink && (sink->block_steps < 1 || !sink->ring_dev || !sink->ring_pinned))
    return fail(RBV_EINVAL, w + ": incomplete chain sink");
  if (ctx->inst.empty() || ctx->ndim == 0) return fail(RBV_ESTATE, w + ": context not set up");
  const StretchLayout lay = pt_layout(ctx, S, T, W, survey);
  if (!workspace || workspace_bytes < lay.total) return fail(RBV_ENOMEM, w + ": workspace too small");
  RBV_ON_DEVICE(ctx);
  cudaStream_t st = (cudaStream_t)stream;
  std::vector<double> b((size_t)S * T);      // the ladders are checked on the host: a 8 S T-byte copy before the run
  RBV_CUDA(cudaMemcpyAsync(b.data(), betas, b.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
  RBV_CUDA(cudaStreamSynchronize(st));
  for (int sl = 0; sl < S; ++sl) {
    const double* bs = b.data() + (size_t)sl * T;
    const std::string where = survey ? w + ": sightline " + std::to_string(sl) + ": " : w + ": ";
    if (bs[0] != 1.0) return fail(RBV_EINVAL, where + "betas[0] must be 1");
    for (int t = 1; t < T; ++t)
      if (!(bs[t] < bs[t - 1]) || !(bs[t] >= 0.0))
        return fail(RBV_EINVAL, where + "betas must be strictly decreasing and >= 0");
  }
  if (n_steps == 0) return RBV_OK;
  char* ws = (char*)workspace;
  StretchParams P;
  memset(&P, 0, sizeof(P));
  P.coords = coords;
  P.lnp = lnprob;
  P.prop = (double*)(ws + lay.prop);
  P.lnp_prop = (double*)(ws + lay.lnp_prop);
  P.factors = (double*)(ws + lay.factors);
  P.walker_of = (int*)(ws + lay.walker_of);
  P.n_accepted = n_accepted;
  P.flag = flag;
  P.step_ctr = (unsigned long long*)(ws + lay.ctr);
  P.ticket = nullptr;            // the accept kernels neither record nor advance the step: the swap stage does
  P.first_step = first_step;
  P.seed = seed;
  P.a = control->a;
  P.W = W;
  P.ndim = ctx->ndim;
  P.S = S * T;                   // ensemble e = s T + t: its stretch streams are offset by e W = s T W + t W
  P.beta = betas;
  PtParams Q;
  memset(&Q, 0, sizeof(Q));
  Q.coords = coords;
  Q.lnp = lnprob;
  Q.betas = betas;
  Q.coords_tmp = (double*)(ws + lay.pt_tmp);
  Q.src = (int*)(ws + lay.pt_src);
  Q.n_swaps = n_swaps_accepted;
  Q.chain = chain;
  Q.lnp_chain = lnprob_chain;
  Q.beta_history = beta_history;
  Q.ti = ti_moments;
  Q.step_ctr = P.step_ctr;
  Q.ticket = (unsigned int*)(ws + lay.ctr + 64);
  Q.first_step = first_step;
  Q.seed = seed;
  Q.adapt_t0 = control->adapt_steps_done;
  Q.adapt_lag = control->adaptation_lag;
  Q.adapt_time = control->adaptation_time;
  Q.adapt = control->adapt != 0;
  Q.S = S;
  Q.T = T;
  Q.W = W;
  Q.ndim = ctx->ndim;
  Q.n_record = control->n_record;
  Q.survey = survey ? 1 : 0;
  if (sink) {
    Q.ring_steps = 2 * sink->block_steps;
    Q.chain = sink->ring_dev;
    // survey mode without a host lnprob array: the ring holds chain rows only
    Q.lnp_chain = (survey && !sink->lnprob_chain_host)
                      ? nullptr : sink->ring_dev + (size_t)Q.ring_steps * S * Q.n_record * W * ctx->ndim;
    int rc = sink_stream_setup(ctx);
    if (rc != RBV_OK) return rc;
  }
  return stretch_run_impl(ctx, P, lay, ws, workspace_bytes, W, n_steps, false, sink, use_graph, st, who, &Q);
}

int rbv_pt_run(RbvContext* ctx, double* coords, double* lnprob, double* betas, int n_temps, int n_walkers,
               int n_steps, const RbvPtControl* control, unsigned long long seed, unsigned long long first_step,
               double* chain, double* lnprob_chain, const RbvChainSink* sink, double* beta_history, int* n_accepted,
               unsigned long long* n_swaps_accepted, int* flag, void* workspace, size_t workspace_bytes,
               int use_graph, void* stream) {
  const int T = n_temps, W = n_walkers;
  if (!ctx || !coords || !lnprob || !betas || !control || !n_accepted || !flag || (T > 1 && !n_swaps_accepted))
    return fail(RBV_EINVAL, "rbv_pt_run: null argument");
  if (!pt_shape_ok(T, W))
    return fail(RBV_EINVAL, "rbv_pt_run: need 1 <= n_temps <= 4096, n_walkers >= 2 and n_temps * n_walkers in int range");
  return pt_run_entry(ctx, 1, false, coords, lnprob, betas, T, W, n_steps, control, seed, first_step, chain,
                      lnprob_chain, sink, beta_history, nullptr, n_accepted, n_swaps_accepted, flag, workspace,
                      workspace_bytes, use_graph, stream, "rbv_pt_run");
}

int rbv_pt_run_sightlines(RbvContext* ctx, double* coords, double* lnprob, double* betas, int n_temps,
                          int walkers_per_sightline, int n_steps, const RbvPtControl* control, unsigned long long seed,
                          unsigned long long first_step, double* chain, double* lnprob_chain,
                          const RbvChainSink* sink, double* beta_history, double* ti_moments, int* n_accepted,
                          unsigned long long* n_swaps_accepted, int* flag, void* workspace, size_t workspace_bytes,
                          int use_graph, void* stream) {
  const int T = n_temps, W = walkers_per_sightline;
  if (!ctx || !coords || !lnprob || !betas || !control || !n_accepted || !flag || (T > 1 && !n_swaps_accepted))
    return fail(RBV_EINVAL, "rbv_pt_run_sightlines: null argument");
  if (ctx->inst.empty() || ctx->ndim == 0) return fail(RBV_ESTATE, "rbv_pt_run_sightlines: context not set up");
  if (!pt_sightlines_shape_ok((long long)ctx->inst.size(), T, W))
    return fail(RBV_EINVAL, "rbv_pt_run_sightlines: need 1 <= n_temps <= 4096, walkers_per_sightline >= 2 and "
                            "n_sightlines * n_temps * walkers_per_sightline in int range");
  if (control->adapt && ti_moments)
    return fail(RBV_EINVAL, "rbv_pt_run_sightlines: ti_moments with adapt: adaptation breaks detailed balance, "
                            "its steps must not enter the evidence");
  return pt_run_entry(ctx, (int)ctx->inst.size(), true, coords, lnprob, betas, T, W, n_steps, control, seed,
                      first_step, chain, lnprob_chain, sink, beta_history, ti_moments, n_accepted, n_swaps_accepted,
                      flag, workspace, workspace_bytes, use_graph, stream, "rbv_pt_run_sightlines");
}

// ---- multi-GPU form of the sampler: half-step = propose_eval | caller's all-gather of lnprob | accept ----------
static int stretch_params(RbvContext* ctx, int n_walkers, void* workspace, size_t workspace_bytes, const char* who,
                          StretchParams* P, StretchLayout* lay_out) {
  if (!ctx) return fail(RBV_EINVAL, std::string(who) + ": null context");
  if (n_walkers < 2) return fail(RBV_EINVAL, std::string(who) + ": need at least two walkers");
  if (ctx->inst.empty() || ctx->ndim == 0) return fail(RBV_ESTATE, std::string(who) + ": context not set up");
  const StretchLayout lay = stretch_layout(ctx, n_walkers);
  if (!workspace || workspace_bytes < lay.total) return fail(RBV_ENOMEM, std::string(who) + ": workspace too small");
  char* ws = (char*)workspace;
  memset(P, 0, sizeof(*P));
  P->prop = (double*)(ws + lay.prop);
  P->lnp_prop = (double*)(ws + lay.lnp_prop);
  P->factors = (double*)(ws + lay.factors);
  P->walker_of = (int*)(ws + lay.walker_of);
  P->step_ctr = nullptr;      // host-driven steps
  P->ticket = nullptr;
  P->W = n_walkers;
  P->ndim = ctx->ndim;
  P->S = 1;
  *lay_out = lay;
  return RBV_OK;
}

int rbv_stretch_propose_eval(RbvContext* ctx, const double* coords, int n_walkers, double a, unsigned long long seed,
                             unsigned long long step, int split, int row_lo, int row_hi, double* lnprob_rows,
                             void* workspace, size_t workspace_bytes, void* stream) {
  StretchParams P;
  StretchLayout lay;
  int rc = stretch_params(ctx, n_walkers, workspace, workspace_bytes, "rbv_stretch_propose_eval", &P, &lay);
  if (rc != RBV_OK) return rc;
  const int h = (n_walkers + 1) / 2, nS = split == 0 ? h : n_walkers - h;
  if (!coords || !lnprob_rows || (split != 0 && split != 1) || row_lo < 0 || row_hi < row_lo || row_hi > nS || !(a > 1.0))
    return fail(RBV_EINVAL, "rbv_stretch_propose_eval: bad argument");
  RBV_ON_DEVICE(ctx);
  cudaStream_t st = (cudaStream_t)stream;
  P.coords = const_cast<double*>(coords);
  P.first_step = step;
  P.seed = seed;
  P.a = a;
  stretch_propose_kernel<<<(nS + 3) / 4, 128, 0, st>>>(P, split);
  RBV_CUDA(cudaGetLastError());
  ctx->launches++;
  if (row_hi == row_lo) return RBV_OK;
  return launch_lnprob(ctx, P.prop + (size_t)row_lo * ctx->ndim, row_hi - row_lo, 0, lnprob_rows + row_lo,
                       (char*)workspace + lay.lnprob_ws, workspace_bytes - lay.lnprob_ws, stream,
                       "rbv_stretch_propose_eval", nullptr, -1, nullptr, nS);   // geometry of the whole half-step
}

int rbv_stretch_accept(RbvContext* ctx, double* coords, double* lnprob, int n_walkers, double a,
                       unsigned long long seed, unsigned long long step, int split, const double* lnprob_rows,
                       double* chain_row, double* lnprob_chain_row, int* n_accepted, int* flag, void* workspace,
                       size_t workspace_bytes, void* stream) {
  StretchParams P;
  StretchLayout lay;
  int rc = stretch_params(ctx, n_walkers, workspace, workspace_bytes, "rbv_stretch_accept", &P, &lay);
  if (rc != RBV_OK) return rc;
  if (!coords || !lnprob || !lnprob_rows || !n_accepted || !flag || (split != 0 && split != 1))
    return fail(RBV_EINVAL, "rbv_stretch_accept: bad argument");
  RBV_ON_DEVICE(ctx);
  const int h = (n_walkers + 1) / 2, nS = split == 0 ? h : n_walkers - h;
  P.coords = coords;
  P.lnp = lnprob;
  P.lnp_prop = const_cast<double*>(lnprob_rows);
  P.chain = chain_row;
  P.lnp_chain = lnprob_chain_row;
  P.n_accepted = n_accepted;
  P.flag = flag;
  P.first_step = step;
  P.seed = seed;
  P.a = a;
  stretch_accept_kernel<<<(nS + 3) / 4, 128, 0, (cudaStream_t)stream>>>(P, split);
  RBV_CUDA(cudaGetLastError());
  ctx->launches++;
  return RBV_OK;
}


// ---- multi-GPU entry points: the lnprob all-gather is issued by the library on its own stream ---------------------
int rbv_comm_unique_id(unsigned char* out_id128) {
  if (!out_id128) return fail(RBV_EINVAL, "rbv_comm_unique_id: null argument");
  int rc = load_nccl();
  if (rc != RBV_OK) return rc;
  RbvNcclUniqueId id;
  RBV_NCCL(g_nccl.GetUniqueId(&id));
  memcpy(out_id128, id.internal, sizeof(id.internal));
  return RBV_OK;
}

int rbv_comm_init(RbvContext* ctx, const unsigned char* id128, int rank, int world) {
  if (!ctx || !id128 || world < 1 || rank < 0 || rank >= world) return fail(RBV_EINVAL, "rbv_comm_init: bad argument");
  if (world > kMaxRanks) return fail(RBV_EINVAL, "rbv_comm_init: more than 64 ranks");
  int rc = load_nccl();
  if (rc != RBV_OK) return rc;
  RBV_ON_DEVICE(ctx);
  if (ctx->comm) {
    g_nccl.CommDestroy(ctx->comm);
    ctx->comm = nullptr;
  }
  RbvNcclUniqueId id;
  memcpy(id.internal, id128, sizeof(id.internal));
  RBV_NCCL(g_nccl.CommInitRank(&ctx->comm, world, id, rank));
  ctx->comm_rank = rank;
  ctx->comm_world = world;
  return RBV_OK;
}

int rbv_comm_info(const RbvContext* ctx, int* rank, int* world, int* nccl_version) {
  if (!ctx) return fail(RBV_EINVAL, "rbv_comm_info: null context");
  if (rank) *rank = ctx->comm ? ctx->comm_rank : 0;
  if (world) *world = ctx->comm ? ctx->comm_world : 1;
  if (nccl_version) {
    *nccl_version = 0;
    if (g_nccl.GetVersion) g_nccl.GetVersion(nccl_version);
  }
  return RBV_OK;
}

// rows [lo, hi) of n rows owned by `rank` when every rank owns `chunk` = ceil(n / world) consecutive rows
static void rank_rows(int n, int rank, int world, int* lo, int* hi, int* chunk) {
  const int c = (n + world - 1) / world;
  *chunk = c;
  *lo = std::min(rank * c, n);
  *hi = std::min(*lo + c, n);
}

// ---- the all-gather as one kernel over peer memory (NVLink / NVSwitch) ---------------------------------------------
// Every rank owns an exchange block [epoch u64 | err i32 | pad -> 256 B][2 x kPeerCap slots of 8 bytes] and maps the
// others' through CUDA IPC.  One CTA per rank and call: PUSH the rank's rows into the block of every other rank
// (8-byte stores over NVLink), then wait for every other rank's rows in the own block and copy them out.  There
// are no flags and no fences: an empty slot holds the bit pattern 0xFFFF...F (a NaN no arithmetic produces; a value
// with exactly these bits is sent as the default NaN), an 8-byte store is indivisible, so the arrival of a value IS
// its signal (the idea of NCCL's low-latency protocol); the receiver puts the empty pattern back once it has read a
// slot.  The two halves of the block alternate from call to call: a rank can be at most one call ahead of a peer
// (to finish a call it needs that peer's rows of the same call), so the half it writes next is never one the peer
// still reads or has not yet emptied.  The call counter lives in device memory: the kernel replays inside a CUDA
// graph.  A lnprob all-gather is 8 B per walker -- the cost of the exchange is latency: this is one launch and one
// NVLink hop.  A wait that sees nothing for 30 s sets the block's error word, hands NaN to the caller for the rows it
// did not receive and gives up (rbv_peer_info reports it) instead of hanging the device.
constexpr int kPeerMaxWorld = 16;
constexpr size_t kPeerCap = 1u << 16;          // slots per half: world * chunk above this goes through NCCL
constexpr size_t kPeerHeader = 256;            // bytes
constexpr unsigned long long kPeerEmpty = 0xFFFFFFFFFFFFFFFFull;
struct PeerDev {
  unsigned char* block[kPeerMaxWorld];
  int rank, world;
};

__device__ __forceinline__ unsigned long long peer_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

__global__ void __launch_bounds__(1024) peer_allgather_kernel(const PeerDev d, double* __restrict__ buf, const int chunk) {
  unsigned char* mine = d.block[d.rank];
  unsigned long long* my_epoch = reinterpret_cast<unsigned long long*>(mine);
  int* my_err = reinterpret_cast<int*>(my_epoch + 1);
  const unsigned long long e = *my_epoch + 1ull;       // every thread reads it; thread 0 writes it back at the end
  const size_t half = (size_t)(e & 1ull) * kPeerCap;
  const int total = chunk * d.world;
  // push: this rank's rows into every other rank's block
  for (int i = threadIdx.x; i < total; i += blockDim.x) {
    const int r = i / chunk, j = i - r * chunk;
    if (r == d.rank) continue;
    unsigned long long v = (unsigned long long)__double_as_longlong(buf[(size_t)d.rank * chunk + j]);
    if (v == kPeerEmpty) v = 0x7ff8000000000000ull;
    unsigned long long* dst = reinterpret_cast<unsigned long long*>(d.block[r] + kPeerHeader) + half + (size_t)d.rank * chunk + j;
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(dst), "l"(v) : "memory");
  }
  // receive: the other ranks' rows out of the own block; every slot is emptied again once read
  unsigned long long* got = reinterpret_cast<unsigned long long*>(mine + kPeerHeader) + half;
  const unsigned long long t0 = peer_timer_ns();
  for (int i = threadIdx.x; i < total; i += blockDim.x) {
    if (i / chunk == d.rank) continue;
    unsigned long long v;
    for (;;) {
      asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(got + i) : "memory");
      if (v != kPeerEmpty) break;
      if (peer_timer_ns() - t0 > 30000000000ull) {
        *my_err = 1;
        break;
      }
    }
    buf[i] = __longlong_as_double((long long)v);
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(got + i), "l"(kPeerEmpty) : "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) *my_epoch = e;
}

// in-place all-gather of `chunk` doubles per rank: rank r's chunk sits at buf + r * chunk
static int allgather_rows(RbvContext* ctx, double* buf, int chunk, cudaStream_t st) {
  if (!ctx->comm || ctx->comm_world == 1 || chunk == 0) return RBV_OK;
  if (ctx->peer_world == ctx->comm_world && (size_t)chunk * ctx->comm_world <= kPeerCap) {
    PeerDev d;
    memset(&d, 0, sizeof(d));
    for (int r = 0; r < ctx->comm_world; ++r)
      d.block[r] = (unsigned char*)(r == ctx->comm_rank ? ctx->peer_block : ctx->peer_open[r]);
    d.rank = ctx->comm_rank;
    d.world = ctx->comm_world;
    peer_allgather_kernel<<<1, 1024, 0, st>>>(d, buf, chunk);
    RBV_CUDA(cudaGetLastError());
    ctx->launches++;
    return RBV_OK;
  }
  RBV_NCCL(g_nccl.AllGather(buf + (size_t)ctx->comm_rank * chunk, buf, (size_t)chunk, kNcclFloat64, ctx->comm, st));
  return RBV_OK;
}

int rbv_peer_export(RbvContext* ctx, unsigned char* out_handle64) {
  if (!ctx || !out_handle64) return fail(RBV_EINVAL, "rbv_peer_export: null argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle size");
  RBV_ON_DEVICE(ctx);
  if (!ctx->peer_block) {
    const size_t bytes = kPeerHeader + 2 * kPeerCap * sizeof(double);
    RBV_CUDA(cudaMalloc(&ctx->peer_block, bytes));
    RBV_CUDA(cudaMemset(ctx->peer_block, 0xFF, bytes));         // every slot empty
    RBV_CUDA(cudaMemset(ctx->peer_block, 0, kPeerHeader));      // call counter, error word
    RBV_CUDA(cudaDeviceSynchronize());
  }
  cudaIpcMemHandle_t h;
  RBV_CUDA(cudaIpcGetMemHandle(&h, ctx->peer_block));
  memcpy(out_handle64, &h, sizeof(h));
  return RBV_OK;
}

int rbv_peer_attach(RbvContext* ctx, const unsigned char* handles, int rank, int world) {
  if (!ctx || !handles) return fail(RBV_EINVAL, "rbv_peer_attach: null argument");
  if (!ctx->peer_block) return fail(RBV_ESTATE, "rbv_peer_attach: call rbv_peer_export first");
  if (world < 2 || world > kPeerMaxWorld || rank < 0 || rank >= world)
    return fail(RBV_EINVAL, "rbv_peer_attach: 2..16 ranks");
  if (ctx->peer_world > 0) return fail(RBV_ESTATE, "rbv_peer_attach: already attached");
  RBV_ON_DEVICE(ctx);
  for (int r = 0; r < world; ++r) {
    if (r == rank) continue;
    cudaIpcMemHandle_t h;
    memcpy(&h, handles + (size_t)r * sizeof(h), sizeof(h));
    cudaError_t e = cudaIpcOpenMemHandle(&ctx->peer_open[r], h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      for (int q = 0; q < world; ++q)
        if (ctx->peer_open[q]) {
          cudaIpcCloseMemHandle(ctx->peer_open[q]);
          ctx->peer_open[q] = nullptr;
        }
      cudaGetLastError();
      return fail(RBV_ECUDA, std::string("rbv_peer_attach: cudaIpcOpenMemHandle: ") + cudaGetErrorString(e));
    }
  }
  ctx->peer_world = world;
  return RBV_OK;
}

// 1 = the all-gather runs over peer memory; *error = the exchange block's error word (a spin that timed out)
int rbv_peer_info(RbvContext* ctx, int* attached, int* error) {
  if (!ctx) return fail(RBV_EINVAL, "rbv_peer_info: null context");
  if (attached) *attached = ctx->peer_world > 0;
  if (error) {
    *error = 0;
    if (ctx->peer_block) {
      RBV_ON_DEVICE(ctx);
      RBV_CUDA(cudaMemcpy(error, (char*)ctx->peer_block + sizeof(unsigned long long), sizeof(int),
                          cudaMemcpyDeviceToHost));
    }
  }
  return RBV_OK;
}

int rbv_lnprob_batch_allgather(RbvContext* ctx, const double* theta, int W, double* lnprob, void* workspace,
                               size_t workspace_bytes, void* stream) {
  if (!ctx || !theta || !lnprob) return fail(RBV_EINVAL, "rbv_lnprob_batch_allgather: null argument");
  if (W <= 0) return W == 0 ? RBV_OK : fail(RBV_EINVAL, "negative n_walkers");
  int lo, hi, chunk;
  rank_rows(W, ctx->comm ? ctx->comm_rank : 0, ctx->comm ? ctx->comm_world : 1, &lo, &hi, &chunk);
  if (hi > lo) {
    int rc = launch_lnprob(ctx, theta + (size_t)lo * ctx->ndim, hi - lo, 0, lnprob + lo, workspace, workspace_bytes,
                           stream, "rbv_lnprob_batch_allgather", nullptr, -1, nullptr, W);
    if (rc != RBV_OK) return rc;
  }
  RBV_ON_DEVICE(ctx);
  return allgather_rows(ctx, lnprob, chunk, (cudaStream_t)stream);
}

// ---- survey mode: one stretch-move ensemble per sightline, all advancing in lockstep -------------------------
static StretchLayout stretch_layout_sightlines(const RbvContext* ctx, int W) {
  auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
  const size_t rows = (size_t)((W + 1) / 2) * std::max<size_t>(ctx->inst.size(), 1);
  StretchLayout lay;
  lay.prop = 0;
  lay.lnp_prop = up(rows * std::max(ctx->ndim, 1) * sizeof(double));
  lay.factors = lay.lnp_prop + up(rows * sizeof(double));
  lay.walker_of = lay.factors + up(rows * sizeof(double));
  lay.ctr = lay.walker_of + up(rows * sizeof(int));
  lay.lnprob_ws = lay.ctr + 256;
  lay.total = lay.lnprob_ws + workspace_layout(ctx, (int)rows, true).total;
  return lay;
}

int rbv_stretch_workspace_bytes_sightlines(const RbvContext* ctx, int walkers_per_sightline, size_t* bytes) {
  if (!ctx || !bytes || walkers_per_sightline < 2 || ctx->inst.empty())
    return fail(RBV_EINVAL, "rbv_stretch_workspace_bytes_sightlines: bad argument");
  if ((long long)((walkers_per_sightline + 1) / 2) * (long long)ctx->inst.size() > 0x7fffffffLL)
    return fail(RBV_EINVAL, "rbv_stretch_workspace_bytes_sightlines: too many rows");
  *bytes = stretch_layout_sightlines(ctx, walkers_per_sightline).total;
  return RBV_OK;
}

int rbv_stretch_run_sightlines(RbvContext* ctx, double* coords, double* lnprob, int walkers_per_sightline, int n_steps,
                               double a, unsigned long long seed, unsigned long long first_step, double* chain,
                               double* lnprob_chain, int* n_accepted, int* flag, void* workspace,
                               size_t workspace_bytes, void* stream) {
  if (!ctx || !coords || !lnprob || !n_accepted || !flag)
    return fail(RBV_EINVAL, "rbv_stretch_run_sightlines: null argument");
  const int W = walkers_per_sightline;
  if (W < 2) return fail(RBV_EINVAL, "rbv_stretch_run_sightlines: need at least two walkers per sightline");
  if (n_steps < 0 || !(a > 1.0))
    return fail(RBV_EINVAL, "rbv_stretch_run_sightlines: n_steps < 0 or stretch scale a <= 1");
  if (ctx->inst.empty() || ctx->ndim == 0) return fail(RBV_ESTATE, "rbv_stretch_run_sightlines: context not set up");
  const long long S = (long long)ctx->inst.size();
  if (S * W > 0x7fffffffLL) return fail(RBV_EINVAL, "rbv_stretch_run_sightlines: too many walkers");
  if (n_steps == 0) return RBV_OK;
  const StretchLayout lay = stretch_layout_sightlines(ctx, W);
  if (!workspace || workspace_bytes < lay.total)
    return fail(RBV_ENOMEM, "rbv_stretch_run_sightlines: workspace too small");
  RBV_ON_DEVICE(ctx);
  cudaStream_t st = (cudaStream_t)stream;
  char* ws = (char*)workspace;
  StretchParams P;
  memset(&P, 0, sizeof(P));
  P.coords = coords;
  P.lnp = lnprob;
  P.prop = (double*)(ws + lay.prop);
  P.lnp_prop = (double*)(ws + lay.lnp_prop);
  P.factors = (double*)(ws + lay.factors);
  P.walker_of = (int*)(ws + lay.walker_of);
  P.n_accepted = n_accepted;
  P.flag = flag;
  P.step_ctr = nullptr;       // the step index is a launch argument: chain / lnp_chain point at the step's own rows
  P.ticket = nullptr;
  P.seed = seed;
  P.a = a;
  P.W = W;
  P.ndim = ctx->ndim;
  P.S = (int)S;
  const int h = (W + 1) / 2;
  const size_t step_rows = (size_t)S * W;
  for (int s = 0; s < n_steps; ++s) {
    P.first_step = first_step + (unsigned long long)s;
    P.chain = chain ? chain + (size_t)s * step_rows * ctx->ndim : nullptr;
    P.lnp_chain = lnprob_chain ? lnprob_chain + (size_t)s * step_rows : nullptr;
    for (int split = 0; split < 2; ++split) {
      const int nS = split == 0 ? h : W - h;
      const int rows = (int)S * nS;
      stretch_propose_kernel<<<(unsigned)((rows + 3) / 4), 128, 0, st>>>(P, split);
      RBV_CUDA(cudaGetLastError());
      ctx->launches++;
      int rc = launch_lnprob(ctx, P.prop, rows, nS, P.lnp_prop, ws + lay.lnprob_ws, workspace_bytes - lay.lnprob_ws,
                             stream, "rbv_stretch_run_sightlines");
      if (rc != RBV_OK) return rc;
      stretch_accept_kernel<<<(unsigned)((rows + 3) / 4), 128, 0, st>>>(P, split);
      RBV_CUDA(cudaGetLastError());
      ctx->launches++;
    }
  }
  return RBV_OK;
}

// ---- device-resident ensemble slice sampler (zeus's differential move), rbv_slice.cuh ------------------------
struct SliceLayout {
  size_t cand, lnp_cand, dir, z0, lo, hi, tcur, jbudget, kbudget, phase, lit, skip, walker_of, ctr, nstep, lnprob_ws,
      total;
};
// sl = false: rbv_slice_run (one ensemble, joint-fit lnprob workspace, its SliceEnsemble inside the SliceState
// block); sl = true: survey mode, one ensemble per sightline of the context
static SliceLayout slice_layout(const RbvContext* ctx, int W, bool sl) {
  auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
  const size_t S = sl ? std::max<size_t>(ctx->inst.size(), 1) : 1;
  const size_t h = (size_t)(W + 1) / 2 * S, row = h * std::max(ctx->ndim, 1) * sizeof(double);   // h: all ensembles
  SliceLayout lay;
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o += up(bytes); return at; };
  lay.cand = take(4 * row);                       // two rows per walker and logical iteration (depth 2)
  lay.lnp_cand = take((4 * h + kMaxRanks) * sizeof(double));   // padded for the in-place all-gather
  lay.dir = take(row);
  lay.z0 = take(h * sizeof(double));
  lay.lo = take(h * sizeof(double));
  lay.hi = take(h * sizeof(double));
  lay.tcur = take(2 * h * sizeof(double));
  lay.jbudget = take(h * sizeof(int));
  lay.kbudget = take(h * sizeof(int));
  lay.phase = take(h * sizeof(int));
  lay.lit = take(h * sizeof(int));
  lay.skip = take(4 * h * sizeof(int));
  lay.walker_of = take(h * sizeof(int));
  lay.ctr = take(sizeof(SliceState));
  lay.nstep = sl ? take(2 * S * sizeof(unsigned int)) : lay.ctr + offsetof(SliceState, solo.nstep);
  lay.lnprob_ws = o;
  lay.total = o + workspace_layout(ctx, (int)(4 * h), sl).total;
  return lay;
}

int rbv_slice_workspace_bytes(const RbvContext* ctx, int n_walkers, size_t* bytes) {
  if (!ctx || !bytes || n_walkers < 4) return fail(RBV_EINVAL, "rbv_slice_workspace_bytes: bad argument");
  *bytes = slice_layout(ctx, n_walkers, false).total;
  return RBV_OK;
}

int rbv_slice_workspace_bytes_sightlines(const RbvContext* ctx, int walkers_per_sightline, size_t* bytes) {
  if (!ctx || !bytes || walkers_per_sightline < 4 || ctx->inst.empty())
    return fail(RBV_EINVAL, "rbv_slice_workspace_bytes_sightlines: bad argument");
  if (4LL * ((walkers_per_sightline + 1) / 2) * (long long)ctx->inst.size() > 0x7fffffffLL)
    return fail(RBV_EINVAL, "rbv_slice_workspace_bytes_sightlines: too many rows");
  *bytes = slice_layout(ctx, walkers_per_sightline, true).total;
  return RBV_OK;
}

// Half-step buffers, loop state and settings of a run (P.mu / adapt / totals / nstep are the caller's).
static void slice_params(RbvContext* ctx, SliceParams& P, const SliceLayout& lay, char* ws, double* coords,
                         double* lnprob, int W, int S, const RbvSliceTuning* tuning, unsigned long long seed,
                         int* flag) {
  P.coords = coords;
  P.lnp = lnprob;
  P.cand = (double*)(ws + lay.cand);
  P.lnp_cand = (double*)(ws + lay.lnp_cand);
  P.dir = (double*)(ws + lay.dir);
  P.z0 = (double*)(ws + lay.z0);
  P.lo = (double*)(ws + lay.lo);
  P.hi = (double*)(ws + lay.hi);
  P.tcur = (double*)(ws + lay.tcur);
  P.jbudget = (int*)(ws + lay.jbudget);
  P.kbudget = (int*)(ws + lay.kbudget);
  P.phase = (int*)(ws + lay.phase);
  P.lit = (int*)(ws + lay.lit);
  P.skip = (int*)(ws + lay.skip);
  P.walker_of = (int*)(ws + lay.walker_of);
  P.flag = flag;
  P.ctr = (SliceCounters*)(ws + lay.ctr);
  P.nstep = (unsigned int*)(ws + lay.nstep);
  P.seed = seed;
  P.tolerance = tuning->tolerance;
  P.W = W;
  P.ndim = ctx->ndim;
  P.maxsteps = tuning->maxsteps;
  P.maxiter = tuning->maxiter;
  P.patience = tuning->patience;
  // logical iterations per launch (rbv_slice.cuh, "Speculation"): chains and counters do not depend on it
  P.depth = tuning->depth == 1 ? 1 : 2;
  if (ctx->tune.slice_depth > 0) P.depth = std::min(ctx->tune.slice_depth, 2);
  P.S = S;
}

// The run loop shared by rbv_slice_run (S = 1, joint lnprob, optionally over the ranks of a communicator) and
// rbv_slice_run_sightlines (sl: S ensembles, one sightline-mode lnprob launch per iteration).  `init` is the
// SliceState the run starts from; on return ctx->h_poll[0] holds the final one.  chain / lnprob_chain /
// mu_history rows are S W ndim / S W / S wide.
static int slice_run_impl(RbvContext* ctx, SliceParams& P, const SliceLayout& lay, char* ws, size_t workspace_bytes,
                          bool sl, const SliceState& init, int n_steps, unsigned long long first_step,
                          double* chain, double* lnprob_chain, double* mu_history, int use_graph,
                          cudaStream_t st, const char* who) {
  const int n_walkers = P.W, S = P.S;
  const int rows_per_walker = 2 * P.depth;
  ctx->h_poll[0] = init;         // the host slot is reused by the polls below
  RBV_CUDA(cudaMemcpyAsync(P.ctr, &ctx->h_poll[0], sizeof(SliceState), cudaMemcpyHostToDevice, st));
  RBV_CUDA(cudaStreamSynchronize(st));
  const size_t lnprob_ws_bytes = workspace_bytes - lay.lnprob_ws;
  const int h = (n_walkers + 1) / 2;
  const long long launches_before = ctx->launches;

  // one iteration of half `split`: lnprob of the S x 2 depth n_S candidate rows (masked rows skipped) -> update +
  // the candidates of the next iteration
  auto iteration = [&](int split, int rows, cudaGraphConditionalHandle loop, int use_loop) -> int {
    const int nS = split == 0 ? h : n_walkers - h;
    const unsigned rows_grid = (unsigned)((S * nS + 3) / 4);
    // multi-GPU (rbv_comm_init, single ensemble only): this rank evaluates its share of the rows, in-place
    // all-gather of their lnprob
    int lo = 0, hi = rows, chunk = rows;
    const bool dist = !sl && ctx->comm && ctx->comm_world > 1;
    if (dist) rank_rows(rows, ctx->comm_rank, ctx->comm_world, &lo, &hi, &chunk);
    if (hi > lo) {
      // geometry as for the 2 n_S rows of one logical iteration, whatever the depth: about half the rows of a launch
      // are masked, and the two depths then produce the same bits (measured at C2, depth 2: 1.70k steps/s with the
      // 4096-pixel tiles this picks, 1.58k with the 8192-pixel tiles picked for 4 n_S rows)
      int rc = launch_lnprob(ctx, P.cand + (size_t)lo * ctx->ndim, hi - lo, sl ? rows / S : 0, P.lnp_cand + lo,
                             ws + lay.lnprob_ws, lnprob_ws_bytes, st, who, nullptr, -1, P.skip + lo, 2 * nS * S);
      if (rc != RBV_OK) return rc;
    }
    if (dist) {
      int rc = allgather_rows(ctx, P.lnp_cand, chunk, st);
      if (rc != RBV_OK) return rc;
    }
    slice_update_kernel<<<rows_grid, 128, 0, st>>>(P, split, loop, use_loop);
    RBV_CUDA(cudaGetLastError());
    return RBV_OK;
  };
  auto begin = [&](unsigned long long step, int split) -> int {
    const int nS = split == 0 ? h : n_walkers - h;
    slice_begin_kernel<<<(unsigned)((S * nS + 3) / 4), 128, 0, st>>>(P, step, split);
    RBV_CUDA(cudaGetLastError());
    slice_candidate_kernel<<<(unsigned)((S * nS + 3) / 4), 128, 0, st>>>(P, split);     // the first candidates
    RBV_CUDA(cudaGetLastError());
    return RBV_OK;
  };
  auto record = [&](int s) -> int {
    const size_t step_rows = (size_t)S * n_walkers;
    slice_record_kernel<<<(unsigned)((step_rows + 3) / 4), 128, 0, st>>>(
        P, chain ? chain + (size_t)s * step_rows * ctx->ndim : nullptr,
        lnprob_chain ? lnprob_chain + (size_t)s * step_rows : nullptr,
        mu_history ? mu_history + (size_t)s * S : nullptr);
    RBV_CUDA(cudaGetLastError());
    return RBV_OK;
  };

  int rc = RBV_OK;
  long long per_iteration = 0;
  const bool dist_run = !sl && ctx->comm && ctx->comm_world > 1;
  if (dist_run) {
    // multi-GPU: NCCL sets up its buffers on the first collective of a size -- do that outside any capture
    // (lnp_cand is scratch here).  The WHILE-node loop with a collective in its body is opt-in
    // (RBVFIT_B200_SLICE_DIST_GRAPH=1); by default the host-polled loop runs: every rank reads the same replicated
    // counters and therefore enqueues the same iterations.
    for (int split = 0; split < 2; ++split) {
      int lo, hi, chunk;
      rank_rows(rows_per_walker * (split == 0 ? h : n_walkers - h), ctx->comm_rank, ctx->comm_world, &lo, &hi, &chunk);
      rc = allgather_rows(ctx, P.lnp_cand, chunk, st);
      if (rc != RBV_OK) return rc;
    }
    RBV_CUDA(cudaStreamSynchronize(st));
    if (!ctx->tune.slice_dist_graph) use_graph = 0;
  }
  if (use_graph && st != nullptr) {
    // Graph mode: per half a graph whose only node is a WHILE node; its body is one iteration, captured from the
    // stream, and slice_update_kernel sets the condition.  A step = (begin, first candidates, graph) x 2, record --
    // seven asynchronous launches whatever the number of iterations, and no host synchronisation inside the run.
    cudaGraph_t graph[2] = {nullptr, nullptr};
    cudaGraphExec_t exec[2] = {nullptr, nullptr};
    cudaError_t e = cudaSuccess;
    for (int split = 0; split < 2 && rc == RBV_OK && e == cudaSuccess; ++split) {
      const int nS = split == 0 ? h : n_walkers - h;
      e = cudaGraphCreate(&graph[split], 0);
      if (e != cudaSuccess) break;
      cudaGraphConditionalHandle loop;
      e = cudaGraphConditionalHandleCreate(&loop, graph[split], 1, cudaGraphCondAssignDefault);
      if (e != cudaSuccess) break;
      cudaGraphNodeParams np = {cudaGraphNodeTypeConditional};
      np.conditional.handle = loop;
      np.conditional.type = cudaGraphCondTypeWhile;
      np.conditional.size = 1;
      cudaGraphNode_t node;
      e = cudaGraphAddNode(&node, graph[split], nullptr, 0, &np);
      if (e != cudaSuccess) break;
      e = cudaStreamBeginCaptureToGraph(st, np.conditional.phGraph_out[0], nullptr, nullptr, 0,
                                        cudaStreamCaptureModeThreadLocal);
      if (e != cudaSuccess) break;
      const long long l0 = ctx->launches;
      rc = iteration(split, S * rows_per_walker * nS, loop, 1);
      per_iteration = ctx->launches - l0 + 1;
      cudaGraph_t captured = nullptr;
      e = cudaStreamEndCapture(st, &captured);
      if (e != cudaSuccess || rc != RBV_OK) break;
      e = cudaGraphInstantiate(&exec[split], graph[split], 0);
    }
    for (int s = 0; s < n_steps && rc == RBV_OK && e == cudaSuccess; ++s) {
      for (int split = 0; split < 2 && rc == RBV_OK && e == cudaSuccess; ++split) {
        rc = begin(first_step + (unsigned long long)s, split);
        if (rc == RBV_OK) e = cudaGraphLaunch(exec[split], st);
      }
      if (rc == RBV_OK && e == cudaSuccess) rc = record(s);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    for (int k = 0; k < 2; ++k) {
      if (exec[k]) cudaGraphExecDestroy(exec[k]);
      if (graph[k]) cudaGraphDestroy(graph[k]);
    }
    if (rc != RBV_OK) return rc;
    if (e != cudaSuccess) return fail(RBV_ECUDA, std::string(who) + " (graph): " + cudaGetErrorString(e));
  } else {
    // Polling mode: iterations are enqueued one ahead of the read-back of the counters -- while the host waits for
    // those of iteration it - 1 the device already runs iteration it; when it - 1 left nothing to do, iteration it
    // found every row masked and changed nothing.  (The batch always has 2 n_S rows, as in graph mode: masked rows
    // cost a CTA prologue each, and the two modes then produce bit-identical chains.)
    for (int s = 0; s < n_steps; ++s) {
      for (int split = 0; split < 2; ++split) {
        const int nS = split == 0 ? h : n_walkers - h;
        rc = begin(first_step + (unsigned long long)s, split);
        if (rc != RBV_OK) return rc;
        bool done = false;
        for (int it = 0; !done; ++it) {
          const long long l0 = ctx->launches;
          rc = iteration(split, S * rows_per_walker * nS, 0, 0);
          if (rc != RBV_OK) return rc;
          per_iteration = ctx->launches - l0 + 1;
          RBV_CUDA(cudaMemcpyAsync(&ctx->h_poll[it & 1].c, P.ctr, sizeof(SliceCounters), cudaMemcpyDeviceToHost,
                                   st));
          RBV_CUDA(cudaEventRecord(ctx->poll_ev[it & 1], st));
          if (it >= 1) {
            RBV_CUDA(cudaEventSynchronize(ctx->poll_ev[(it - 1) & 1]));
            const SliceCounters& c = ctx->h_poll[(it - 1) & 1].c;
            if (c.pending == 0u || c.error) done = true;
          }
        }
      }
      rc = record(s);
      if (rc != RBV_OK) return rc;
    }
  }
  RBV_CUDA(cudaMemcpyAsync(&ctx->h_poll[0], P.ctr, sizeof(SliceState), cudaMemcpyDeviceToHost, st));
  RBV_CUDA(cudaStreamSynchronize(st));
  // + begin, candidates (x 2), record
  ctx->launches = launches_before + (long long)ctx->h_poll[0].c.batches * per_iteration + 5LL * n_steps;
  return RBV_OK;
}

int rbv_slice_run(RbvContext* ctx, double* coords, double* lnprob, int n_walkers, int n_steps, RbvSliceTuning* tuning,
                  unsigned long long seed, unsigned long long first_step, double* chain, double* lnprob_chain,
                  double* mu_history, int* flag, void* workspace, size_t workspace_bytes, int use_graph,
                  void* stream) {
  if (!ctx || !coords || !lnprob || !tuning || !flag) return fail(RBV_EINVAL, "rbv_slice_run: null argument");
  if (n_walkers < 4) return fail(RBV_EINVAL, "rbv_slice_run: need at least four walkers (two per complement)");
  if (n_steps < 0 || !(tuning->mu > 0.0) || tuning->maxsteps < 1 || tuning->maxiter < 1)
    return fail(RBV_EINVAL, "rbv_slice_run: n_steps < 0, mu <= 0, maxsteps < 1 or maxiter < 1");
  if (ctx->inst.empty() || ctx->ndim == 0) return fail(RBV_ESTATE, "rbv_slice_run: context not set up");
  if (n_steps == 0) return RBV_OK;
  const SliceLayout lay = slice_layout(ctx, n_walkers, false);
  if (!workspace || workspace_bytes < lay.total) return fail(RBV_ENOMEM, "rbv_slice_run: workspace too small");
  RBV_ON_DEVICE(ctx);
  char* ws = (char*)workspace;
  SliceParams P;
  slice_params(ctx, P, lay, ws, coords, lnprob, n_walkers, 1, tuning, seed, flag);
  SliceState* dev = (SliceState*)(ws + lay.ctr);
  P.mu = &dev->solo.mu;
  P.adapt = dev->solo.adapt;
  P.totals = dev->solo.totals;
  // loop state: everything zero except mu and its adaptation state
  SliceState init;
  memset(&init, 0, sizeof(init));
  init.solo.mu = tuning->mu;
  init.solo.adapt[0] = tuning->tune != 0;
  init.solo.adapt[1] = tuning->good;
  int rc = slice_run_impl(ctx, P, lay, ws, workspace_bytes, false, init, n_steps, first_step, chain, lnprob_chain,
                          mu_history, use_graph, (cudaStream_t)stream, "rbv_slice_run");
  if (rc != RBV_OK) return rc;
  const SliceState& c = ctx->h_poll[0];
  tuning->mu = c.solo.mu;
  tuning->tune = c.solo.adapt[0];
  tuning->good = c.solo.adapt[1];
  tuning->n_expansions = c.solo.totals[0];
  tuning->n_contractions = c.solo.totals[1];
  tuning->n_calls = c.solo.totals[2];
  tuning->n_batches = c.c.batches;
  if (c.c.error) return fail(RBV_ESTATE, "rbv_slice_run: number of contractions exceeded the maximum (maxiter)");
  return RBV_OK;
}

int rbv_slice_run_sightlines(RbvContext* ctx, double* coords, double* lnprob, int walkers_per_sightline, int n_steps,
                             RbvSliceTuning* tuning, double* mu, int* tune_good, unsigned long long* totals,
                             unsigned long long seed, unsigned long long first_step, double* chain,
                             double* lnprob_chain, double* mu_history, int* flag, void* workspace,
                             size_t workspace_bytes, int use_graph, void* stream) {
  const char* who = "rbv_slice_run_sightlines";
  if (!ctx || !coords || !lnprob || !tuning || !mu || !tune_good || !totals || !flag)
    return fail(RBV_EINVAL, std::string(who) + ": null argument");
  const int W = walkers_per_sightline;
  if (W < 4) return fail(RBV_EINVAL, std::string(who) + ": need at least four walkers per sightline");
  if (n_steps < 0 || tuning->maxsteps < 1 || tuning->maxiter < 1)
    return fail(RBV_EINVAL, std::string(who) + ": n_steps < 0, maxsteps < 1 or maxiter < 1");
  if (ctx->inst.empty() || ctx->ndim == 0) return fail(RBV_ESTATE, std::string(who) + ": context not set up");
  const long long S = (long long)ctx->inst.size();
  if (S * W > 0x7fffffffLL || 4LL * ((W + 1) / 2) * S > 0x7fffffffLL)
    return fail(RBV_EINVAL, std::string(who) + ": too many walkers");
  const InstDev& A = ctx->inst[0].dev;
  for (auto& hi : ctx->inst)
    if (hi.dev.P != A.P || hi.dev.K != A.K || hi.dev.L != A.L || hi.dev.C != A.C)
      return fail(RBV_EINVAL, std::string(who) + ": sightlines must share n_pixels, n_taps, n_lines, n_components");
  if (n_steps == 0) return RBV_OK;
  const SliceLayout lay = slice_layout(ctx, W, true);
  if (!workspace || workspace_bytes < lay.total) return fail(RBV_ENOMEM, std::string(who) + ": workspace too small");
  RBV_ON_DEVICE(ctx);
  cudaStream_t st = (cudaStream_t)stream;
  {   // every sightline's mu must be positive (the one read-back before the run)
    std::vector<double> m((size_t)S);
    RBV_CUDA(cudaMemcpyAsync(m.data(), mu, (size_t)S * sizeof(double), cudaMemcpyDeviceToHost, st));
    RBV_CUDA(cudaStreamSynchronize(st));
    for (double v : m)
      if (!(v > 0.0)) return fail(RBV_EINVAL, std::string(who) + ": mu <= 0");
  }
  char* ws = (char*)workspace;
  SliceParams P;
  slice_params(ctx, P, lay, ws, coords, lnprob, W, (int)S, tuning, seed, flag);
  P.mu = mu;
  P.adapt = tune_good;
  P.totals = totals;
  SliceState init;
  memset(&init, 0, sizeof(init));
  int rc = slice_run_impl(ctx, P, lay, ws, workspace_bytes, true, init, n_steps, first_step, chain, lnprob_chain,
                          mu_history, use_graph, st, who);
  if (rc != RBV_OK) return rc;
  const SliceCounters& c = ctx->h_poll[0].c;
  tuning->n_batches = c.batches;
  if (c.error) return fail(RBV_ESTATE, std::string(who) + ": number of contractions exceeded the maximum (maxiter)");
  return RBV_OK;
}

// The instrument as the flux entry point sees it: with its LSF, or with the single tap 1.0 (convolve = 0:
// VoigtModel.evaluate(return_unconvolved=True) skips the kernel, voigt_model.py:221, 537-548).
static InstDev flux_instrument(const RbvContext* ctx, int inst, int convolve) {
  InstDev I = ctx->inst[inst].dev;
  if (!convolve) {
    I.K = 1;
    I.Kpad = I.R;
    I.taps_rev = ctx->d_unit_taps;
  }
  I.line_base = 0;
  return I;
}

int rbv_flux_workspace_bytes(const RbvContext* ctx, int inst, int n_walkers, size_t* bytes) {
  if (!ctx || !bytes || n_walkers < 0 || inst < 0 || inst >= (int)ctx->inst.size())
    return fail(RBV_EINVAL, "rbv_flux_workspace_bytes: bad argument");
  *bytes = workspace_layout_raw(n_walkers, 1, ctx->inst[inst].dev.L).total;
  return RBV_OK;
}

int rbv_model_flux_batch(RbvContext* ctx, int inst, const double* theta, int W, int convolve, double* out_flux,
                         void* workspace, size_t workspace_bytes, void* stream) {
  if (!ctx || !theta || !out_flux) return fail(RBV_EINVAL, "rbv_model_flux_batch: null argument");
  if (inst < 0 || inst >= (int)ctx->inst.size()) return fail(RBV_EINVAL, "rbv_model_flux_batch: bad instrument index");
  if (W <= 0) return W == 0 ? RBV_OK : fail(RBV_EINVAL, "negative n_walkers");
  RBV_ON_DEVICE(ctx);
  const InstDev I = flux_instrument(ctx, inst, convolve);
  int ndim = ctx->ndim ? ctx->ndim : 3 * I.C;
  LaunchParams prm;
  memset(&prm, 0, sizeof(prm));
  prm.inst = ctx->d_inst;
  prm.theta = theta;
  prm.core_tab = ctx->d_core_tab;
  prm.out_flux = out_flux;
  prm.ndim = ndim;
  prm.n_inst = 1;                     // the launch sees this one instrument (possibly without its LSF)
  prm.W = W;
  prm.precision = ctx->precision;
  prm.farfield = ctx->farfield;
  prm.ff_budget = ctx->tune.ff_budget;
  prm.sampler_split = -1;
  prm.inst_in_params = 1;
  prm.inst_v[0] = I;
  prm.n_lines_total = I.L;
  // biggest tiles that still give every CTA slot of the GPU one CTA (as choose_geometry does for lnprob)
  const long long want = (long long)kWantWaves * RBV_MIN_CTAS * ctx->sm_count;
  size_t smem = 0;
  for (int level = kGeomLevels - 1; level >= 0; --level) {
    if (ctx->tune.force_level >= 0) level = ctx->tune.force_level;
    prm.geom[0] = geometry_for(I, level, 0);
    smem = smem_bytes_for(I, prm.geom[0], ndim);
    const bool fits = smem <= (size_t)std::min(ctx->max_dyn_smem, (227 * 1024) / RBV_MIN_CTAS - 2048);
    if (level == 0 || ctx->tune.force_level >= 0 || (fits && (long long)W * prm.geom[0].n_tiles >= want)) break;
  }
  prm.n_tiles = prm.geom[0].n_tiles;
  prm.tile_base = 0;
  if (prm.n_tiles > 65535) return fail(RBV_EINVAL, "rbv_model_flux_batch: more than 65535 tiles per walker");
  cudaStream_t st = (cudaStream_t)stream;
  if (workspace) {
    // line constants once per walker (prep_kernel), as in the lnprob launch, instead of once per CTA
    const WorkspaceLayout lay = workspace_layout_raw(W, 1, I.L);
    if (workspace_bytes < lay.total) return fail(RBV_ENOMEM, "rbv_model_flux_batch: workspace too small");
    prm.tickets = (unsigned int*)((char*)workspace + lay.tickets);
    prm.oob = (int*)((char*)workspace + lay.oob);
    prm.lc = (double*)((char*)workspace + lay.lc);
    dim3 pgrid((unsigned)W, (unsigned)((I.L + 127) / 128));
    prep_kernel<<<pgrid, 128, 0, st>>>(prm);
    RBV_CUDA(cudaGetLastError());
    ctx->launches++;
  }
  dim3 grid((unsigned)W, (unsigned)prm.n_tiles);
  if (small_chunks(ctx, prm.geom, 1)) voigt_tile_kernel<3, 1, 2><<<grid, kThreads, smem, st>>>(prm);
  else voigt_tile_kernel<3, 1, 8><<<grid, kThreads, smem, st>>>(prm);
  RBV_CUDA(cudaGetLastError());
  ctx->launches++;
  return RBV_OK;
}

int rbv_num_instruments(const RbvContext* ctx) { return ctx ? (int)ctx->inst.size() : 0; }
int rbv_num_tiles(const RbvContext* ctx) { return ctx ? ctx->n_tiles : 0; }
int rbv_ndim(const RbvContext* ctx) { return ctx ? ctx->ndim : 0; }
long long rbv_launch_count(const RbvContext* ctx) { return ctx ? ctx->launches : 0; }
int rbv_last_kernel(const RbvContext* ctx) { return ctx ? ctx->last_kernel : -1; }

int rbv_voigt_h(RbvContext* ctx, const double* x, const double* a, double* out, int n, int method, void* stream) {
  if (!ctx || !x || !a || !out || n < 0) return fail(RBV_EINVAL, "rbv_voigt_h: bad argument");
  if (n == 0) return RBV_OK;
  RBV_ON_DEVICE(ctx);
  voigt_h_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(x, a, out, n, method, ctx->d_core_tab);
  RBV_CUDA(cudaGetLastError());
  ctx->launches++;
  return RBV_OK;
}

int rbv_voigt_h_grad(RbvContext* ctx, const double* x, const double* a, double* H, double* Hx, double* Ha, int n,
                     void* stream) {
  if (!ctx || !x || !a || !H || !Hx || !Ha || n < 0) return fail(RBV_EINVAL, "rbv_voigt_h_grad: bad argument");
  if (n == 0) return RBV_OK;
  RBV_ON_DEVICE(ctx);
  voigt_h_grad_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(x, a, H, Hx, Ha, n, ctx->d_core_tab);
  RBV_CUDA(cudaGetLastError());
  ctx->launches++;
  return RBV_OK;
}

// ------------------------------------------------------------------------------------------ analytic gradient
// Workspace of rbv_lnprob_grad_batch (byte offsets, 256-byte aligned); geometry per instrument is fixed by its pixel
// count alone, so every row is reduced in the same order whatever the batch.
struct GradLayout {
  size_t oob, lc, F, r, g, pval, pline, linegrad, total;
  int n_blk_total, n_tiles_total;
  long long part_stride;
};
// one_inst: the geometry of instrument 0 alone (survey mode, where every sightline shares it)
static GradLayout grad_layout(const RbvContext* ctx, int W, GradInst* gi, bool one_inst = false) {
  GradLayout L;
  memset(&L, 0, sizeof(L));
  int blk = 0, tiles = 0;
  long long part = 0;
  for (size_t k = 0; k < (one_inst ? std::min<size_t>(1, ctx->inst.size()) : ctx->inst.size()); ++k) {
    const InstDev& I = ctx->inst[k].dev;
    GradInst g;
    memset(&g, 0, sizeof(g));
    g.blk_off = blk;
    g.n_blk = (I.P + kGradBlock - 1) / kGradBlock;
    g.tile_off = tiles;
    g.n_tiles = (I.P + kGradTile - 1) / kGradTile;
    g.part_off = part;
    blk += g.n_blk;
    tiles += g.n_tiles;
    part += (long long)g.n_tiles * I.L * 3;
    if (gi && k < (size_t)kMaxInst) gi[k] = g;
  }
  L.n_blk_total = blk;
  L.n_tiles_total = tiles;
  L.part_stride = part;
  auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
  const size_t Wz = (size_t)std::max(W, 1);
  size_t off = 0;
  L.oob = off;      off = al(off + Wz * sizeof(int));
  L.lc = off;       off = al(off + Wz * ctx->n_lines_total * LC_STRIDE * sizeof(double));
  L.F = off;        off = al(off + Wz * blk * kGradBlock * sizeof(double));
  L.r = off;        off = al(off + Wz * blk * kGradBlock * sizeof(double));
  L.g = off;        off = al(off + Wz * blk * kGradBlock * sizeof(double));
  L.pval = off;     off = al(off + Wz * blk * sizeof(double));
  L.pline = off;    off = al(off + Wz * (size_t)part * sizeof(double));
  L.linegrad = off; off = al(off + Wz * ctx->n_lines_total * 3 * sizeof(double));
  L.total = off;
  return L;
}

int rbv_grad_workspace_bytes(const RbvContext* ctx, int n_walkers, size_t* bytes) {
  if (!ctx || !bytes || n_walkers < 0) return fail(RBV_EINVAL, "rbv_grad_workspace_bytes: bad argument");
  *bytes = grad_layout(ctx, n_walkers, nullptr).total;
  return RBV_OK;
}

// Launches with the row in grid y or z (gradient, Fisher, Jacobian): CUDA caps gridDim.y / gridDim.z at 65 535, so
// such a launch goes over the batch in slices [w0, w0 + n) of at most that many rows, every kernel indexing the
// full-size buffers with row w0 + blockIdx.y (.z).  Nothing is reduced across rows, so a row's results do not depend
// on the slicing; a batch of up to 65 535 rows is one launch as before.  launch(n) enqueues the kernel of one slice
// with the current prm.w0.
constexpr int kMaxGridRows = 65535;
extern "C++" {
template <class Launch>
static int launch_row_slices(RbvContext* ctx, GradParams& prm, int W, Launch launch) {
  for (int w0 = 0; w0 < W; w0 += kMaxGridRows) {
    prm.w0 = w0;
    launch((unsigned)std::min(kMaxGridRows, W - w0));
    RBV_CUDA(cudaGetLastError());
    ctx->launches++;
  }
  prm.w0 = 0;
  return RBV_OK;
}
}  // extern "C++"

int rbv_lnprob_grad_batch(RbvContext* ctx, const double* theta, int W, int apply_prior, double* value, double* grad,
                          void* workspace, size_t workspace_bytes, void* stream) {
  const char* who = "rbv_lnprob_grad_batch";
  if (!ctx || !theta || !value || !grad) return fail(RBV_EINVAL, std::string(who) + ": null argument");
  if (W < 0) return fail(RBV_EINVAL, std::string(who) + ": negative n_walkers");
  if (W == 0) return RBV_OK;
  if (ctx->inst.empty()) return fail(RBV_ESTATE, std::string(who) + ": no instrument added");
  if (ctx->ndim == 0) return fail(RBV_ESTATE, std::string(who) + ": bounds not set (rbv_set_bounds)");
  if (ctx->inst.size() > (size_t)kMaxInst)
    return fail(RBV_EINVAL, std::string(who) + ": at most 16 instruments in a joint fit");
  for (auto& hi : ctx->inst) {
    if (!hi.dev.flux || !hi.dev.inv_sigma2 || !hi.dev.log_inv_sigma2)
      return fail(RBV_ESTATE, std::string(who) + ": an instrument has no observed spectrum (flux-only instrument)");
    if (3 * hi.dev.C > ctx->ndim) return fail(RBV_EINVAL, std::string(who) + ": ndim smaller than 3 * n_components");
    if (hi.dev.method != RBV_VOIGT_WOFZ)
      return fail(RBV_EINVAL, std::string(who) + ": no gradient for voigt_method='fast' (Tepper-Garcia)");
  }
  GradParams prm;
  memset(&prm, 0, sizeof(prm));
  const GradLayout lay = grad_layout(ctx, W, prm.gi);
  if (!workspace || workspace_bytes < lay.total) return fail(RBV_ENOMEM, std::string(who) + ": workspace too small");
  RBV_ON_DEVICE(ctx);
  for (size_t k = 0; k < ctx->inst.size(); ++k) {
    HostInst& hi = ctx->inst[k];
    if (!hi.d_grad_cum) {   // prefix / suffix sums of the flipped taps: what the edge replication piles on 0 and P-1
      const int K = hi.dev.K;
      std::vector<double> cum(2 * (size_t)K);
      double s = 0.0;
      for (int m = 0; m < K; ++m) cum[m] = (s += hi.taps[K - 1 - m]);
      s = 0.0;
      for (int m = K - 1; m >= 0; --m) cum[K + m] = (s += hi.taps[K - 1 - m]);
      RBV_CUDA(upload(&hi.d_grad_cum, cum.data(), cum.size()));
    }
    prm.gi[k].cum_lo = hi.d_grad_cum;
    prm.gi[k].cum_hi = hi.d_grad_cum + hi.dev.K;
  }
  char* ws = (char*)workspace;
  prm.inst = ctx->d_inst;
  prm.theta = theta;
  prm.lb = apply_prior ? ctx->d_lb : nullptr;
  prm.ub = apply_prior ? ctx->d_ub : nullptr;
  prm.core_tab = ctx->d_core_tab;
  prm.value = value;
  prm.grad = grad;
  prm.oob = (int*)(ws + lay.oob);
  prm.lc = (double*)(ws + lay.lc);
  prm.F = (double*)(ws + lay.F);
  prm.r = (double*)(ws + lay.r);
  prm.g = (double*)(ws + lay.g);
  prm.pval = (double*)(ws + lay.pval);
  prm.pline = (double*)(ws + lay.pline);
  prm.linegrad = (double*)(ws + lay.linegrad);
  prm.part_stride = lay.part_stride;
  prm.W = W;
  prm.ndim = ctx->ndim;
  prm.n_inst = (int)ctx->inst.size();
  prm.n_lines_total = ctx->n_lines_total;
  prm.n_blk_total = lay.n_blk_total;
  prm.n_tiles_total = lay.n_tiles_total;
  cudaStream_t st = (cudaStream_t)stream;
  grad_prep_kernel<false><<<dim3(W, (ctx->n_lines_total + 127) / 128), 128, 0, st>>>(prm, SlRows{});
  RBV_CUDA(cudaGetLastError());
  ctx->launches++;
  RBV_CHECK(launch_row_slices(ctx, prm, W, [&](unsigned n) {
    grad_flux_kernel<false><<<dim3(lay.n_blk_total, n), kGradBlock, 0, st>>>(prm, SlRows{});
  }));
  RBV_CHECK(launch_row_slices(ctx, prm, W, [&](unsigned n) {
    grad_resid_kernel<false><<<dim3(lay.n_blk_total, n), kGradBlock, 0, st>>>(prm, SlRows{});
  }));
  RBV_CHECK(launch_row_slices(ctx, prm, W, [&](unsigned n) {
    grad_adjoint_kernel<<<dim3(lay.n_blk_total, n), kGradBlock, 0, st>>>(prm);
  }));
  RBV_CHECK(launch_row_slices(ctx, prm, W, [&](unsigned n) {
    grad_line_kernel<<<dim3(lay.n_tiles_total, n), kGradBlock, 0, st>>>(prm);
  }));
  grad_finalize_kernel<<<(W + 3) / 4, 128, 0, st>>>(prm);
  RBV_CUDA(cudaGetLastError());
  ctx->launches++;
  return RBV_OK;
}

// ------------------------------------------------------------------------------------------ Jacobian / Fisher
// Workspace of rbv_lnlike_fisher_batch and rbv_model_jacobian_batch (byte offsets, 256-byte aligned): the forward
// buffers of the gradient path plus the columns JF, JM and the Gram partials.  sl: survey mode, every buffer sized for
// the geometry of one sightline (instrument 0), so the workspace grows as O(W) whatever the number of sightlines.
struct FisherLayout {
  size_t oob, lc, F, r, pval, JF, JM, pgram, total;
  int n_blk_total, n_tiles_total, ncol, npart;
};
static FisherLayout fisher_layout(const RbvContext* ctx, int W, GradInst* gi, bool sl = false) {
  const GradLayout g = grad_layout(ctx, 0, gi, sl);
  FisherLayout L;
  memset(&L, 0, sizeof(L));
  L.n_blk_total = g.n_blk_total;
  L.n_tiles_total = g.n_tiles_total;
  for (auto& hi : ctx->inst) L.ncol = std::max(L.ncol, 3 * hi.dev.C);
  L.npart = L.ncol * (L.ncol + 1) / 2 + L.ncol;
  auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
  const size_t Wz = (size_t)std::max(W, 1), px = (size_t)g.n_blk_total * kGradBlock;
  const size_t n_lines = sl && !ctx->inst.empty() ? (size_t)ctx->inst[0].dev.L : (size_t)ctx->n_lines_total;
  size_t off = 0;
  L.oob = off;   off = al(off + Wz * sizeof(int));
  L.lc = off;    off = al(off + Wz * n_lines * LC_STRIDE * sizeof(double));
  L.F = off;     off = al(off + Wz * px * sizeof(double));
  L.r = off;     off = al(off + Wz * px * sizeof(double));
  L.pval = off;  off = al(off + Wz * g.n_blk_total * sizeof(double));
  L.JF = off;    off = al(off + Wz * L.ncol * px * sizeof(double));
  L.JM = off;    off = al(off + Wz * L.ncol * px * sizeof(double));
  L.pgram = off; off = al(off + Wz * g.n_tiles_total * L.npart * sizeof(double));
  L.total = off;
  return L;
}

int rbv_fisher_workspace_bytes(const RbvContext* ctx, int n_walkers, size_t* bytes) {
  if (!ctx || !bytes || n_walkers < 0) return fail(RBV_EINVAL, "rbv_fisher_workspace_bytes: bad argument");
  *bytes = fisher_layout(ctx, n_walkers, nullptr).total;
  return RBV_OK;
}

int rbv_fisher_workspace_bytes_sightlines(const RbvContext* ctx, int n_walkers, size_t* bytes) {
  if (!ctx || !bytes || n_walkers < 0) return fail(RBV_EINVAL, "rbv_fisher_workspace_bytes_sightlines: bad argument");
  *bytes = fisher_layout(ctx, n_walkers, nullptr, true).total;
  return RBV_OK;
}

static bool has_lsf(const HostInst& hi) { return !(hi.taps.size() == 1 && hi.taps[0] == 1.0); }

// Checks shared by every entry point and the parameter block of the launches.  sl: survey mode (any number of
// instruments, identical geometry, one instrument's geometry in fp.gp).
static int fisher_setup(RbvContext* ctx, const char* who, const double* theta, int W, bool with_resid, bool sl,
                        void* workspace, size_t workspace_bytes, FisherParams& fp, FisherLayout& lay, bool& any_lsf) {
  if (ctx->inst.empty()) return fail(RBV_ESTATE, std::string(who) + ": no instrument added");
  if (ctx->ndim == 0) return fail(RBV_ESTATE, std::string(who) + ": bounds not set (rbv_set_bounds)");
  if (!sl && ctx->inst.size() > (size_t)kMaxInst)
    return fail(RBV_EINVAL, std::string(who) + ": at most 16 instruments in a joint fit");
  const InstDev& A = ctx->inst[0].dev;
  for (auto& hi : ctx->inst) {
    if (sl && (hi.dev.P != A.P || hi.dev.K != A.K || hi.dev.L != A.L || hi.dev.C != A.C))
      return fail(RBV_EINVAL, std::string(who) + ": sightlines must share n_pixels, n_taps, n_lines, n_components");
    if (3 * hi.dev.C > ctx->ndim) return fail(RBV_EINVAL, std::string(who) + ": ndim smaller than 3 * n_components");
    if (hi.dev.method != RBV_VOIGT_WOFZ)
      return fail(RBV_EINVAL, std::string(who) + ": no Jacobian for voigt_method='fast' (Tepper-Garcia)");
    if (with_resid && (!hi.dev.flux || !hi.dev.inv_sigma2 || !hi.dev.log_inv_sigma2))
      return fail(RBV_ESTATE, std::string(who) + ": an instrument has no observed spectrum (flux-only instrument)");
  }
  memset(&fp, 0, sizeof(fp));
  GradParams& prm = fp.gp;
  lay = fisher_layout(ctx, W, prm.gi, sl);
  if (!workspace || workspace_bytes < lay.total) return fail(RBV_ENOMEM, std::string(who) + ": workspace too small");
  const size_t smem = (size_t)(lay.ncol + 2) * kFisherChunk * sizeof(double);
  if (smem > (size_t)ctx->max_dyn_smem) return fail(RBV_EINVAL, std::string(who) + ": too many components");
  any_lsf = false;
  for (size_t k = 0; k < ctx->inst.size(); ++k) {
    const HostInst& hi = ctx->inst[k];
    if (!sl) {
      fp.order[k] = hi.d_fisher_order;
      fp.has_lsf[k] = has_lsf(hi);
    }
    any_lsf = any_lsf || has_lsf(hi);
  }
  char* ws = (char*)workspace;
  prm.inst = ctx->d_inst;
  prm.theta = theta;
  prm.core_tab = ctx->d_core_tab;
  prm.oob = (int*)(ws + lay.oob);
  prm.lc = (double*)(ws + lay.lc);
  prm.F = (double*)(ws + lay.F);
  prm.r = (double*)(ws + lay.r);
  prm.pval = (double*)(ws + lay.pval);
  prm.W = W;
  prm.ndim = ctx->ndim;
  prm.n_inst = sl ? 1 : (int)ctx->inst.size();
  prm.n_lines_total = sl ? A.L : ctx->n_lines_total;
  prm.n_blk_total = lay.n_blk_total;
  prm.n_tiles_total = lay.n_tiles_total;
  fp.ncol = lay.ncol;
  fp.npart = lay.npart;
  fp.col_stride = (long long)lay.n_blk_total * kGradBlock;
  fp.JF = (double*)(ws + lay.JF);
  fp.JM = (double*)(ws + lay.JM);
  fp.pgram = (double*)(ws + lay.pgram);
  return RBV_OK;
}

// prep -> flux [-> resid] -> columns [-> LSF] [-> Gram -> finalize]
extern "C++" {
template <bool SL>
static int fisher_launch(RbvContext* ctx, const FisherParams& fp_in, const FisherLayout& lay, bool with_resid,
                         bool any_lsf, bool gram, const SlRows& sl, cudaStream_t st) {
  FisherParams fp = fp_in;          // fp.gp.w0 walks the row slices (launch_row_slices)
  const GradParams& prm = fp.gp;
  const int W = prm.W;
  grad_prep_kernel<SL><<<dim3(W, (prm.n_lines_total + 127) / 128), 128, 0, st>>>(prm, sl);
  RBV_CUDA(cudaGetLastError());
  ctx->launches++;
  RBV_CHECK(launch_row_slices(ctx, fp.gp, W, [&](unsigned n) {
    grad_flux_kernel<SL><<<dim3(lay.n_blk_total, n), kGradBlock, 0, st>>>(prm, sl);
  }));
  if (with_resid)
    RBV_CHECK(launch_row_slices(ctx, fp.gp, W, [&](unsigned n) {
      grad_resid_kernel<SL><<<dim3(lay.n_blk_total, n), kGradBlock, 0, st>>>(prm, sl);
    }));
  RBV_CHECK(launch_row_slices(ctx, fp.gp, W, [&](unsigned n) {
    fisher_col_kernel<SL><<<dim3(lay.n_blk_total, n), kGradBlock, 0, st>>>(fp, sl);
  }));
  if (any_lsf)
    RBV_CHECK(launch_row_slices(ctx, fp.gp, W, [&](unsigned n) {
      fisher_lsf_kernel<SL><<<dim3(lay.n_blk_total, lay.ncol, n), kGradBlock, 0, st>>>(fp, sl);
    }));
  if (!gram) return RBV_OK;
  const size_t smem = (size_t)(lay.ncol + 2) * kFisherChunk * sizeof(double);
  if (smem > 48 * 1024)
    RBV_CUDA(cudaFuncSetAttribute(fisher_gram_kernel<SL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  RBV_CHECK(launch_row_slices(ctx, fp.gp, W, [&](unsigned n) {
    fisher_gram_kernel<SL><<<dim3(lay.n_tiles_total, n), kGradBlock, smem, st>>>(fp, sl);
  }));
  fisher_finalize_kernel<SL><<<(W + 3) / 4, 128, 0, st>>>(fp, sl);
  RBV_CUDA(cudaGetLastError());
  ctx->launches++;
  return RBV_OK;
}
}  // extern "C++"

// survey mode: order / has_lsf of every instrument as device tables; uploaded again only when they changed
static int sightline_tables(RbvContext* ctx, SlRows& sl) {
  std::vector<const int*> order;
  std::vector<int> lsf;
  for (auto& hi : ctx->inst) {
    order.push_back(hi.d_fisher_order);
    lsf.push_back(has_lsf(hi) ? 1 : 0);
  }
  if (order != ctx->sl_order || lsf != ctx->sl_has_lsf || !ctx->d_sl_order) {
    cudaFree(ctx->d_sl_order);
    cudaFree(ctx->d_sl_has_lsf);
    ctx->d_sl_order = nullptr;
    ctx->d_sl_has_lsf = nullptr;
    ctx->sl_order.clear();
    RBV_CUDA(upload(&ctx->d_sl_order, order.data(), order.size()));
    RBV_CUDA(upload(&ctx->d_sl_has_lsf, lsf.data(), lsf.size()));
    ctx->sl_order = order;
    ctx->sl_has_lsf = lsf;
  }
  sl.order = ctx->d_sl_order;
  sl.has_lsf = ctx->d_sl_has_lsf;
  return RBV_OK;
}

int rbv_lnlike_fisher_batch(RbvContext* ctx, const double* theta, int W, double* value, double* grad, double* fisher,
                            void* workspace, size_t workspace_bytes, void* stream) {
  const char* who = "rbv_lnlike_fisher_batch";
  if (!ctx || !theta || !value || !grad || !fisher) return fail(RBV_EINVAL, std::string(who) + ": null argument");
  if (W < 0) return fail(RBV_EINVAL, std::string(who) + ": negative n_walkers");
  if (W == 0) return RBV_OK;
  FisherParams fp;
  FisherLayout lay;
  bool any_lsf;
  const int rc = fisher_setup(ctx, who, theta, W, true, false, workspace, workspace_bytes, fp, lay, any_lsf);
  if (rc != RBV_OK) return rc;
  RBV_ON_DEVICE(ctx);
  fp.gp.value = value;
  fp.gp.grad = grad;
  fp.fisher = fisher;
  return fisher_launch<false>(ctx, fp, lay, true, any_lsf, true, SlRows{}, (cudaStream_t)stream);
}

int rbv_lnlike_fisher_batch_sightlines(RbvContext* ctx, const double* theta, int W, int walkers_per_sightline,
                                       double* value, double* grad, double* fisher, void* workspace,
                                       size_t workspace_bytes, void* stream) {
  const char* who = "rbv_lnlike_fisher_batch_sightlines";
  if (!ctx || !theta || !value || !grad || !fisher) return fail(RBV_EINVAL, std::string(who) + ": null argument");
  if (W < 0 || walkers_per_sightline <= 0)
    return fail(RBV_EINVAL, std::string(who) + ": negative n_walkers or walkers_per_sightline <= 0");
  if ((long long)walkers_per_sightline * (long long)ctx->inst.size() != (long long)W)
    return fail(RBV_EINVAL, std::string(who) + ": n_walkers must equal n_sightlines * walkers_per_sightline");
  if (W == 0) return RBV_OK;
  FisherParams fp;
  FisherLayout lay;
  bool any_lsf;
  const int rc = fisher_setup(ctx, who, theta, W, true, true, workspace, workspace_bytes, fp, lay, any_lsf);
  if (rc != RBV_OK) return rc;
  RBV_ON_DEVICE(ctx);
  SlRows sl;
  memset(&sl, 0, sizeof(sl));
  RBV_CHECK(sightline_tables(ctx, sl));
  sl.wps = walkers_per_sightline;
  fp.gp.value = value;
  fp.gp.grad = grad;
  fp.fisher = fisher;
  return fisher_launch<true>(ctx, fp, lay, true, any_lsf, true, sl, (cudaStream_t)stream);
}

int rbv_model_jacobian_batch(RbvContext* ctx, int inst, const double* theta, int W, double* out_jac, void* workspace,
                             size_t workspace_bytes, void* stream) {
  const char* who = "rbv_model_jacobian_batch";
  if (!ctx || !theta || !out_jac) return fail(RBV_EINVAL, std::string(who) + ": null argument");
  if (inst < 0 || inst >= (int)ctx->inst.size()) return fail(RBV_EINVAL, std::string(who) + ": bad instrument index");
  if (W < 0) return fail(RBV_EINVAL, std::string(who) + ": negative n_walkers");
  if (W == 0) return RBV_OK;
  cudaStream_t st = (cudaStream_t)stream;
  FisherParams fp;
  FisherLayout lay;
  bool any_lsf;
  const int rc = fisher_setup(ctx, who, theta, W, false, false, workspace, workspace_bytes, fp, lay, any_lsf);
  if (rc != RBV_OK) return rc;
  RBV_ON_DEVICE(ctx);
  RBV_CHECK(fisher_launch<false>(ctx, fp, lay, false, any_lsf, false, SlRows{}, st));
  fp.jac = out_jac;
  fp.jac_inst = inst;
  const int P = ctx->inst[inst].dev.P;
  return launch_row_slices(ctx, fp.gp, W, [&](unsigned n) {
    fisher_jac_out_kernel<<<dim3((P + kGradBlock - 1) / kGradBlock, ctx->ndim, n), kGradBlock, 0, st>>>(fp);
  });
}

// ------------------------------------------------------------------------------------------ survey-mode LM
// Workspace of rbv_lm_run_sightlines: the survey-mode Fisher workspace of n rows, then the per-sightline state of
// LMParams (rbv_lm.cuh).
struct LMLayout {
  FisherLayout fl;
  size_t g, F, xc, vc, gc, Fc, L, Li, y, idx, lam, nu, started, active, count, total;
};
static LMLayout lm_layout(const RbvContext* ctx, int n) {
  LMLayout L;
  memset(&L, 0, sizeof(L));
  L.fl = fisher_layout(ctx, n, nullptr, true);
  auto al = [](size_t v) { return (v + 255) & ~(size_t)255; };
  const size_t nz = (size_t)std::max(n, 1), d = (size_t)ctx->ndim, dd = d * d * sizeof(double);
  size_t off = L.fl.total;
  L.g = off;       off = al(off + nz * d * sizeof(double));
  L.F = off;       off = al(off + nz * dd);
  L.xc = off;      off = al(off + nz * d * sizeof(double));
  L.vc = off;      off = al(off + nz * sizeof(double));
  L.gc = off;      off = al(off + nz * d * sizeof(double));
  L.Fc = off;      off = al(off + nz * dd);
  L.L = off;       off = al(off + nz * dd);
  L.Li = off;      off = al(off + nz * dd);
  L.y = off;       off = al(off + nz * d * sizeof(double));
  L.idx = off;     off = al(off + nz * d * sizeof(int));
  L.lam = off;     off = al(off + nz * sizeof(double));
  L.nu = off;      off = al(off + nz * sizeof(double));
  L.started = off; off = al(off + nz * sizeof(int));
  L.active = off;  off = al(off + nz * sizeof(int));
  L.count = off;   off = al(off + sizeof(int));
  L.total = off;
  return L;
}

int rbv_lm_workspace_bytes_sightlines(const RbvContext* ctx, int n_sightlines, size_t* bytes) {
  if (!ctx || !bytes || n_sightlines < 0) return fail(RBV_EINVAL, "rbv_lm_workspace_bytes_sightlines: bad argument");
  *bytes = lm_layout(ctx, n_sightlines).total;
  return RBV_OK;
}

int rbv_lm_run_sightlines(RbvContext* ctx, int first, int n, double* theta, const RbvLMControl* ctl, double* chi2,
                          double* cov, int* n_evals, int* status, int* flags, void* workspace, size_t workspace_bytes,
                          void* stream) {
  const char* who = "rbv_lm_run_sightlines";
  if (!ctx || !theta || !ctl || !chi2 || !cov || !n_evals || !status || !flags)
    return fail(RBV_EINVAL, std::string(who) + ": null argument");
  if (first < 0 || n < 0 || (long long)first + n > (long long)ctx->inst.size())
    return fail(RBV_EINVAL, std::string(who) + ": [first, first + n) is not a range of the context's sightlines");
  if (ctl->max_evals < 1 || !(ctl->ftol >= 0.0) || !(ctl->xtol >= 0.0))
    return fail(RBV_EINVAL, std::string(who) + ": max_evals < 1 or a negative tolerance");
  if (n == 0) return RBV_OK;
  const LMLayout L = lm_layout(ctx, n);
  FisherParams fp;
  FisherLayout lay;
  bool any_lsf;
  char* ws = (char*)workspace;
  double* xc = (double*)(ws + L.xc);
  int rc = fisher_setup(ctx, who, xc, n, true, true, workspace, workspace_bytes, fp, lay, any_lsf);
  if (rc != RBV_OK) return rc;
  if (workspace_bytes < L.total) return fail(RBV_ENOMEM, std::string(who) + ": workspace too small");
  RBV_ON_DEVICE(ctx);
  if (!ctx->h_lm_count) RBV_CUDA(cudaMallocHost((void**)&ctx->h_lm_count, sizeof(int)));
  SlRows sl;
  memset(&sl, 0, sizeof(sl));
  RBV_CHECK(sightline_tables(ctx, sl));
  sl.wps = 1;
  sl.inst0 = first;
  sl.active = (const int*)(ws + L.active);
  fp.gp.value = (double*)(ws + L.vc);
  fp.gp.grad = (double*)(ws + L.gc);
  fp.fisher = (double*)(ws + L.Fc);
  LMParams p;
  memset(&p, 0, sizeof(p));
  p.n = n;
  p.ndim = ctx->ndim;
  p.max_evals = ctl->max_evals;
  p.ftol = ctl->ftol;
  p.xtol = ctl->xtol;
  p.lb = ctx->d_lb;
  p.ub = ctx->d_ub;
  p.x = theta;
  p.g = (double*)(ws + L.g);
  p.F = (double*)(ws + L.F);
  p.xc = xc;
  p.vc = (const double*)(ws + L.vc);
  p.gc = (const double*)(ws + L.gc);
  p.Fc = (const double*)(ws + L.Fc);
  p.L = (double*)(ws + L.L);
  p.Li = (double*)(ws + L.Li);
  p.y = (double*)(ws + L.y);
  p.idx = (int*)(ws + L.idx);
  p.lam = (double*)(ws + L.lam);
  p.nu = (double*)(ws + L.nu);
  p.started = (int*)(ws + L.started);
  p.active = (int*)(ws + L.active);
  p.count = (int*)(ws + L.count);
  p.chi2 = chi2;
  p.cov = cov;
  p.n_evals = n_evals;
  p.status = status;
  p.flags = flags;
  cudaStream_t st = (cudaStream_t)stream;
  const int blocks = (n + kLMWarps - 1) / kLMWarps;
  lm_init_kernel<<<blocks, 32 * kLMWarps, 0, st>>>(p);
  RBV_CUDA(cudaGetLastError());
  ctx->launches++;
  // every iteration evaluates one row per active sightline and n_evals never exceeds max_evals
  for (int it = 0; it < ctl->max_evals; ++it) {
    RBV_CHECK(fisher_launch<true>(ctx, fp, lay, true, any_lsf, true, sl, st));
    RBV_CUDA(cudaMemsetAsync(p.count, 0, sizeof(int), st));
    lm_update_kernel<<<blocks, 32 * kLMWarps, 0, st>>>(p);
    RBV_CUDA(cudaGetLastError());
    ctx->launches++;
    RBV_CUDA(cudaMemcpyAsync(ctx->h_lm_count, p.count, sizeof(int), cudaMemcpyDeviceToHost, st));
    RBV_CUDA(cudaStreamSynchronize(st));
    if (*ctx->h_lm_count == 0) return RBV_OK;
  }
  return fail(RBV_ESTATE, std::string(who) + ": sightlines still active after max_evals iterations");
}

int rbv_measure_fp64_peak(RbvContext* ctx, double millis, double* tflops) {
  if (!ctx || !tflops) return fail(RBV_EINVAL, "rbv_measure_fp64_peak: bad argument");
  RBV_ON_DEVICE(ctx);
  double* d_out;
  RBV_CUDA(cudaMalloc(&d_out, sizeof(double)));
  cudaEvent_t e0, e1;
  RBV_CUDA(cudaEventCreate(&e0));
  RBV_CUDA(cudaEventCreate(&e1));
  const int blocks = ctx->sm_count * 8, threads = 256;
  int iters = 2000;
  double best = 0.0, spent = 0.0;
  dfma_peak_kernel<<<blocks, threads>>>(d_out, 200, 1.0);  // warm-up
  RBV_CUDA(cudaDeviceSynchronize());
  while (spent < millis) {
    RBV_CUDA(cudaEventRecord(e0));
    dfma_peak_kernel<<<blocks, threads>>>(d_out, iters, 1.0);
    RBV_CUDA(cudaEventRecord(e1));
    RBV_CUDA(cudaEventSynchronize(e1));
    float ms = 0.f;
    RBV_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    ctx->launches++;
    double flops = 2.0 * 64.0 * (double)iters * blocks * threads;
    best = std::max(best, flops / (ms * 1e-3) / 1e12);
    spent += ms;
    if (ms < 5.0f) iters *= 2;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d_out);
  *tflops = best;
  return RBV_OK;
}

#ifdef RBV_STREAM_TIMELINE
// experiments only: per-warp timeline of the last voigt_stream_kernel launch (4 u64 per warp)
int rbv_debug_stream_timeline(unsigned long long* out, int n_u64) {
  return cudaMemcpyFromSymbol(out, g_stream_timeline, (size_t)n_u64 * sizeof(unsigned long long)) == cudaSuccess
             ? RBV_OK : RBV_ECUDA;
}
#endif

// max relative error of the device reciprocal used in the asymptotic tiers (test hook)
int rbv_selftest_rcp(RbvContext* ctx, double* max_rel_err) {
  if (!ctx || !max_rel_err) return fail(RBV_EINVAL, "rbv_selftest_rcp: bad argument");
  RBV_ON_DEVICE(ctx);
  double* d;
  RBV_CUDA(cudaMalloc(&d, sizeof(double)));
  RBV_CUDA(cudaMemset(d, 0, sizeof(double)));
  rcp_selftest_kernel<<<1, 256>>>(d);
  RBV_CUDA(cudaGetLastError());
  RBV_CUDA(cudaMemcpy(max_rel_err, d, sizeof(double), cudaMemcpyDeviceToHost));
  cudaFree(d);
  ctx->launches++;
  return RBV_OK;
}

}  // extern "C"
