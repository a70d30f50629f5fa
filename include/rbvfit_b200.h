/* rbvfit_b200 -- C ABI of the B200-native rbvfit likelihood hot path.
 *
 * This is the drop-in boundary: everything the reference does between
 *     theta  ->  CompiledVoigtModel.model_flux  ->  vfit.lnlike / lnprior / lnprob
 * (reference: src/rbvfit/core/voigt_model.py:100-323, src/rbvfit/vfit_mcmc.py:234-259, 291-353)
 * happens behind these entry points, for a whole batch of theta rows ("walkers") per call.
 *
 * Conventions
 *   - every function returns an int status: 0 = RBV_OK, otherwise an RBV_E* code; the text of the
 *     most recent failure on the calling thread is available from rbv_last_error().
 *   - "device" pointers are CUDA device pointers owned by the CALLER (PyTorch tensors in the Python
 *     host layer) and must stay alive for as long as the context may use them; "host" pointers are
 *     only read during the call.
 *   - the library owns the opaque context and its small constant tables (line tables, LSF taps,
 *     tile map, Faddeeva coefficient tables).  No *_batch call allocates memory.
 *   - one context = one device; calls on one context must not overlap (one stream at a time).
 *   - no CPU fallback exists: without a usable CUDA device rbv_create() fails.
 */
#ifndef RBVFIT_B200_H
#define RBVFIT_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RBV_OK 0
#define RBV_EINVAL 1   /* bad argument / shape */
#define RBV_ECUDA 2    /* CUDA runtime error (text in rbv_last_error) */
#define RBV_ENOMEM 3   /* caller-provided workspace too small */
#define RBV_ESTATE 4   /* call order violated (e.g. lnprob before bounds were set) */

#define RBV_VOIGT_WOFZ 0 /* H = Re w(x + i a), voigt_model.py:156 (scipy.special.wofz) */
#define RBV_VOIGT_FAST 1 /* Tepper-Garcia 2006 variant, voigt_approx.py:35-86 */

#define RBV_PRECISION_FP64 0
#define RBV_PRECISION_FP32_GATED 1 /* FP32 far-wing arithmetic, used only when the gate passes */

#define RBV_FARFIELD_DIRECT 0    /* every (line, pixel) pair evaluated on its own                          */
#define RBV_FARFIELD_CHEBYSHEV 1 /* default: summed far wings of a 1024-pixel super-chunk interpolated from 8 nodes, */
                                 /* used per (line, chunk) only when an a-priori bound keeps |dtau| <= 1e-13  */

typedef struct RbvContext RbvContext;

/* The lowered model of one instrument.
 * Replaces CompiledModelData, voigt_model.py:265-280 (built by _cache_atomic_parameters :386-412 and
 * _setup_fast_mapping :414-442).  All arrays are HOST arrays of length n_lines.
 * gamma and f must carry the reference's float32 rounding (rb_setline.py:42,44) promoted to double. */
typedef struct RbvLineTable {
  int n_lines;         /* L = sum over ion groups of transitions x components            */
  int n_components;    /* C; theta = [logN_1..C | b_1..C | v_1..C]  (parameter_manager.py:123-126) */
  const double* lambda0; /* rest wavelength [Angstrom]                                    */
  const double* gamma;   /* damping constant [1/s]                                        */
  const double* f;       /* oscillator strength                                           */
  const double* zfac;    /* 1 + z_system  (z_factors, voigt_model.py:407)                 */
  const int* comp;       /* component slot c(l) = N_indices[l]; b and v slots are c+C, c+2C */
  int voigt_method;      /* RBV_VOIGT_WOFZ | RBV_VOIGT_FAST                                */
} RbvLineTable;

/* One instrument's spectrum and line-spread function.
 * Replaces the per-instrument dict built by vfit._compile_models, vfit_mcmc.py:249-257.
 * wave/flux/inv_sigma2/log_inv_sigma2 are DEVICE arrays of n_pixels doubles; the weights must have been
 * computed by the caller with the reference's expressions and dtype (1.0/error**2, log(1.0/error**2) in
 * error's dtype) and then promoted to double.  flux/inv_sigma2/log_inv_sigma2 may be NULL for an instrument
 * that is only used with rbv_model_flux_batch().
 * inv_wave is a DEVICE scratch array of n_pixels doubles that the library fills with 1/wave.
 * The spectrum is read ONCE, by rbv_add_instrument: the library derives its own tables from it (1/wave, the range
 * of 1/wave per 256-pixel block, a block-transposed copy of (flux, inv_sigma2) for coalesced loads, the sum of
 * log_inv_sigma2) -- changing the arrays afterwards has no effect; build a new context for new data.
 * taps is a HOST array of n_taps (odd) LSF taps exactly as the reference would apply them
 * (Gaussian1DKernel.array for ndimage.convolve1d(mode='nearest'), voigt_model.py:222-224, or the
 * CustomKernel array for astropy convolve(boundary='extend'), :225-230); NULL / 0 = no convolution.
 * normalize_taps != 0 divides the taps by their sum first (astropy convolve's normalize_kernel=True). */
typedef struct RbvSpectrum {
  int n_pixels;
  const double* wave;
  const double* flux;
  const double* inv_sigma2;
  const double* log_inv_sigma2;
  double* inv_wave;
  const double* taps;
  int n_taps;
  int normalize_taps;
} RbvSpectrum;

/* Create / destroy a likelihood context on CUDA device `device`. */
int rbv_create(int device, RbvContext** out);
void rbv_destroy(RbvContext* ctx);

/* Select the arithmetic of the far-wing tier (default RBV_PRECISION_FP64). */
int rbv_set_precision(RbvContext* ctx, int precision);

/* Select how far line wings (lines >= 24 Doppler widths away from a 1024-pixel super-chunk) are accumulated
 * (default RBV_FARFIELD_CHEBYSHEV). */
int rbv_set_farfield(RbvContext* ctx, int mode);

/* Append an instrument (model + spectrum).  *out_index receives its index (0, 1, ...).
 * Replaces one iteration of the loop in vfit._compile_models (vfit_mcmc.py:238-257). */
int rbv_add_instrument(RbvContext* ctx, const RbvLineTable* lines, const RbvSpectrum* spec, int* out_index);

/* Uniform prior bounds (HOST arrays of ndim doubles); vfit.lnprior, vfit_mcmc.py:291-295.
 * ndim must be >= 3 * n_components of every instrument. */
int rbv_set_bounds(RbvContext* ctx, const double* lb, const double* ub, int ndim);

/* Bytes of caller-owned device workspace needed by rbv_lnprob_batch for up to n_walkers rows.
 * Its contents need no initialisation and do not have to survive between calls. */
int rbv_workspace_bytes(const RbvContext* ctx, int n_walkers, size_t* bytes);

/* lnprob for a batch of walkers; vfit.lnprob, vfit_mcmc.py:348-353, vectorised over rows.
 *   theta   DEVICE [n_walkers, ndim] row-major doubles
 *   lnprob  DEVICE [n_walkers] doubles (out): -inf where a row violates the bounds, NaN where the
 *           reference's numpy arithmetic would give NaN
 *   stream  cudaStream_t (as void*), NULL = default stream.  Asynchronous. */
int rbv_lnprob_batch(RbvContext* ctx, const double* theta, int n_walkers, double* lnprob,
                     void* workspace, size_t workspace_bytes, void* stream);

/* The likelihood alone, vfit.lnlike, vfit_mcmc.py:297-319: same launch without the prior -- rows outside the bounds
 * are evaluated like any other (the reference's lnlike does not look at the bounds).  Same arguments and workspace
 * as rbv_lnprob_batch; no context state is touched, so it may be interleaved freely with rbv_lnprob_batch. */
int rbv_lnlike_batch(RbvContext* ctx, const double* theta, int n_walkers, double* lnlike,
                     void* workspace, size_t workspace_bytes, void* stream);

/* Survey mode: the context holds S independent sightlines (instruments with identical n_pixels, n_taps,
 * n_lines, n_components; their line tables -- e.g. redshifts -- and spectra differ) and theta holds
 * walkers_per_sightline consecutive rows per sightline: row w is evaluated against sightline w / walkers_per_sightline
 * only.  lnprob[w] = that sightline's lnprob (same bounds for all).  n_walkers = S * walkers_per_sightline.
 * One launch for the whole batch; no limit of 16 instruments.  Workspace: rbv_workspace_bytes_sightlines(). */
int rbv_workspace_bytes_sightlines(const RbvContext* ctx, int n_walkers, size_t* bytes);
int rbv_lnprob_batch_sightlines(RbvContext* ctx, const double* theta, int n_walkers, int walkers_per_sightline,
                                double* lnprob, void* workspace, size_t workspace_bytes, void* stream);

/* Same, from HOST buffers (pinned for full speed): copies theta in, runs, copies lnprob out and
 * synchronises the stream.  theta_dev / lnprob_dev are caller-owned device staging buffers of at least
 * n_walkers*ndim / n_walkers doubles.  This is the call the Python lnprob(theta) makes. */
int rbv_lnprob_batch_host(RbvContext* ctx, const double* theta_host, int n_walkers, double* lnprob_host,
                          double* theta_dev, double* lnprob_dev, void* workspace, size_t workspace_bytes,
                          void* stream);
/* 1 when p points into page-locked host memory (cudaMallocHost, cudaHostRegister, a pinned torch tensor), else 0.
 * rbv_lnprob_batch_host copies theta_host with cudaMemcpyAsync: from page-locked memory that is a DMA in place; the
 * Python layer stages pageable arrays through its own page-locked buffer and uses this query to skip the staging
 * copy (222 us for the 2.4 MB of a C5a ensemble) when the caller's array is page-locked already. */
int rbv_host_pinned(const void* p);


/* Device-resident affine-invariant ensemble sampler (stretch move).  Replaces the sampling loop
 * emcee.EnsembleSampler(nwalkers, ndim, self.lnprob).run_mcmc(guesses, no_of_steps), vfit_mcmc.py:408-423, 536-540
 * (emcee >= 3.0.0 is not vendored in the reference; its RedBlueMove + StretchMove is restated from the published
 * algorithm).  Proposal, likelihood and accept/reject of every half-step run on the device with no host round trip;
 * random numbers come from Philox4x32-10 keyed by `seed` with counter (first_step + s, walker, purpose), so a run
 * continued with first_step = steps already done reproduces one long run.
 *   coords      DEVICE [n_walkers, ndim]  current ensemble, updated in place
 *   lnprob      DEVICE [n_walkers]        its log-probabilities (from rbv_lnprob_batch), updated in place
 *   chain       DEVICE [n_steps, n_walkers, ndim] or NULL; lnprob_chain DEVICE [n_steps, n_walkers] or NULL
 *   n_accepted  DEVICE int[n_walkers], accumulated;  flag DEVICE int, bit 0 set if a proposal's lnprob was NaN
 *   workspace   DEVICE, rbv_stretch_workspace_bytes(); use_graph != 0 captures one step in a CUDA graph and
 *               replays it (needs a non-default stream; the call then returns after the run has finished),
 *               otherwise the launches are only enqueued (asynchronous). */
int rbv_stretch_workspace_bytes(const RbvContext* ctx, int n_walkers, size_t* bytes);
int rbv_stretch_run(RbvContext* ctx, double* coords, double* lnprob, int n_walkers, int n_steps, double a,
                    unsigned long long seed, unsigned long long first_step, double* chain, double* lnprob_chain,
                    int* n_accepted, int* flag, void* workspace, size_t workspace_bytes, int use_graph,
                    void* stream);

/* Multi-GPU form of the same sampler (one process per GPU, ensemble state replicated on every rank): a half-step
 * is split around the caller's all-gather of the proposals' lnprob (NCCL over NVLink, 8 B per walker).
 *   rbv_stretch_propose_eval: builds ALL n_S proposals of half `split` of step `step` (identical on every rank:
 *       counter-based random streams) and evaluates rows [row_lo, row_hi) -> lnprob_rows[row_lo .. row_hi)
 *       (DEVICE [n_S], n_S = ceil(W/2) for split 0, floor(W/2) for split 1).
 *   rbv_stretch_accept: with lnprob_rows complete (all-gathered), applies accept/reject to every walker of the
 *       half, updates coords / lnprob / n_accepted in place and writes the walkers' rows of this step into
 *       chain_row [W, ndim] / lnprob_chain_row [W] (DEVICE, may be NULL).
 * Both use the rbv_stretch_workspace_bytes() workspace (it carries the proposals between the two calls) and are
 * asynchronous.  The walker layout of a step is the same as in rbv_stretch_run, so a run is reproducible across
 * GPU counts. */
int rbv_stretch_propose_eval(RbvContext* ctx, const double* coords, int n_walkers, double a, unsigned long long seed,
                             unsigned long long step, int split, int row_lo, int row_hi, double* lnprob_rows,
                             void* workspace, size_t workspace_bytes, void* stream);
int rbv_stretch_accept(RbvContext* ctx, double* coords, double* lnprob, int n_walkers, double a,
                       unsigned long long seed, unsigned long long step, int split, const double* lnprob_rows,
                       double* chain_row, double* lnprob_chain_row, int* n_accepted, int* flag, void* workspace,
                       size_t workspace_bytes, void* stream);

/* ---- the collective inside the library (multi-GPU, one process and one context per GPU) --------------------------
 * SURVEY 8(e): the only exchange on the path is the all-gather of lnprob values (8 B per walker) per half-step.  The
 * library issues it itself, with NCCL, on the caller's stream between its own kernels, so that a whole MCMC step is
 * one CUDA graph per rank and no host code runs inside it.  libnccl is resolved at run time (the copy the process
 * has already loaded -- PyTorch's -- else the system one); single-GPU use never touches it.
 *   rbv_comm_unique_id  rank 0 creates the 128-byte NCCL unique id; the caller broadcasts it to every rank
 *                       (torch.distributed.broadcast in the Python layer)
 *   rbv_comm_init       collective over all ranks: attaches rank `rank` of `world` to this context
 *   rbv_comm_info       rank / world of the context (0 / 1 without a communicator) and the NCCL version in use
 * Row partition of every multi-GPU call: rank r owns rows [r c, (r + 1) c) with c = ceil(n_rows / world). */
int rbv_comm_unique_id(unsigned char* out_id128);
int rbv_comm_init(RbvContext* ctx, const unsigned char* id128, int rank, int world);
int rbv_comm_info(const RbvContext* ctx, int* rank, int* world, int* nccl_version);

/* The same all-gather as ONE kernel over NVLink peer memory (optional, after rbv_comm_init; 2..16 ranks of one node).
 * Every rank owns an exchange block and maps the others' through CUDA IPC; a call pushes the rank's rows into every
 * other block with 8-byte stores and waits for the others' rows in its own: an empty slot holds a reserved NaN
 * pattern, so the arrival of a value is its own signal (no flags, no fences) -- one launch and one NVLink hop
 * instead of a NCCL collective (the payload is 8 B per walker: the cost of the exchange is latency).  Payloads above
 * 65536 doubles keep using NCCL.
 *   rbv_peer_export  allocates the block (first call) and returns its 64-byte CUDA IPC handle; the caller
 *                    all-gathers the handles (torch.distributed in the Python layer)
 *   rbv_peer_attach  handles = world x 64 bytes in rank order; opens every peer's block
 *   rbv_peer_info    attached: 1 when the all-gather runs over peer memory; error: 1 after a wait that saw
 *                    nothing for 30 s (a rank died or skipped a call) */
int rbv_peer_export(RbvContext* ctx, unsigned char* out_handle64);
int rbv_peer_attach(RbvContext* ctx, const unsigned char* handles, int rank, int world);
int rbv_peer_info(RbvContext* ctx, int* attached, int* error);

/* rbv_lnprob_batch over all ranks of the communicator: every rank passes the SAME theta [n_walkers, ndim] (replicated
 * ensemble), evaluates its own rows and the ranks all-gather in place; lnprob must hold world * ceil(n_walkers/world)
 * doubles and ends up complete on every rank.  The launch geometry is chosen as for the whole batch, so each row's
 * value is bit-identical to the single-GPU call's.  Without a communicator this is rbv_lnprob_batch. */
int rbv_lnprob_batch_allgather(RbvContext* ctx, const double* theta, int n_walkers, double* lnprob,
                               void* workspace, size_t workspace_bytes, void* stream);

/* rbv_stretch_run over all ranks of the communicator (same arguments, same workspace size; coords / lnprob / chain /
 * n_accepted are replicated on every rank and every rank must pass the same seed and initial ensemble).  A half-step
 * = stretch_propose_kernel (all proposals, identical everywhere: counter-based random streams) -> the lnprob launch
 * over this rank's rows -> in-place NCCL all-gather of the proposals' lnprob -> stretch_accept_kernel; with
 * use_graph != 0 the whole step is captured once (collective included) and replayed, the step index lives in device
 * memory.  The chain is the one rbv_stretch_run produces on one GPU with the same seed, bit for bit, for any number
 * of ranks.  rbv_slice_run needs no separate entry point: with a communicator attached it splits the rows of every
 * iteration over the ranks in the same way.  The call returns after the run has finished. */
int rbv_stretch_run_dist(RbvContext* ctx, double* coords, double* lnprob, int n_walkers, int n_steps, double a,
                         unsigned long long seed, unsigned long long first_step, double* chain,
                         double* lnprob_chain, int* n_accepted, int* flag, void* workspace, size_t workspace_bytes,
                         int use_graph, void* stream);

/* The same runs with the chain handed to the HOST while the run goes on (what emcee's backend stores: every step,
 * every walker -- 2.3 MB per step at 8000 walkers x 36 parameters).  The device keeps a ring of 2 x block_steps
 * steps; after each block the finished half is copied to page-locked staging on a second stream and from there into
 * the caller's arrays by the calling thread, while the device already runs the next block: the hand-off costs no
 * device time and no pageable-memory copy from the device.  distributed != 0: rbv_stretch_run_dist's step.
 *   chain_host / lnprob_chain_host  HOST [n_steps, n_walkers, ndim] / [n_steps, n_walkers] (any memory), may be NULL
 *   ring_dev     DEVICE, 2 * block_steps * n_walkers * (ndim + 1) doubles
 *   ring_pinned  HOST page-locked, same size
 * Needs a non-default stream and n_steps >= 4; returns after the run has finished and every row has been delivered. */
typedef struct RbvChainSink {
  double* chain_host;
  double* lnprob_chain_host;
  double* ring_dev;
  double* ring_pinned;
  int block_steps;
} RbvChainSink;
int rbv_stretch_run_sink(RbvContext* ctx, double* coords, double* lnprob, int n_walkers, int n_steps, double a,
                         unsigned long long seed, unsigned long long first_step, const RbvChainSink* sink,
                         int* n_accepted, int* flag, void* workspace, size_t workspace_bytes, int distributed,
                         void* stream);

/* Survey mode of the same sampler: the context holds S sightlines (see rbv_lnprob_batch_sightlines) and every
 * sightline has its OWN ensemble of walkers_per_sightline walkers -- what the reference does as S separate
 * vfit(...).runmcmc() calls, one after the other (vfit_mcmc.py:492-561).  The S ensembles advance in lockstep: a
 * half-step is stretch_propose_kernel over all S * n_S rows -> ONE sightline lnprob launch -> stretch_accept_kernel,
 * with no host round trip; ensembles never mix (partners come from the same sightline's complementary half).
 * Random streams: those of rbv_stretch_run with the walker counter offset by sightline * walkers_per_sightline, so
 * sightline 0 of a survey run reproduces the single-ensemble run with the same seed.
 *   coords      DEVICE [S, walkers_per_sightline, ndim], updated in place;  lnprob DEVICE [S, walkers_per_sightline]
 *   chain       DEVICE [n_steps, S, walkers_per_sightline, ndim] or NULL; lnprob_chain [n_steps, S, wps] or NULL
 *   n_accepted  DEVICE int[S, walkers_per_sightline], accumulated;  flag as in rbv_stretch_run.  Asynchronous. */
int rbv_stretch_workspace_bytes_sightlines(const RbvContext* ctx, int walkers_per_sightline, size_t* bytes);
int rbv_stretch_run_sightlines(RbvContext* ctx, double* coords, double* lnprob, int walkers_per_sightline, int n_steps,
                               double a, unsigned long long seed, unsigned long long first_step, double* chain,
                               double* lnprob_chain, int* n_accepted, int* flag, void* workspace,
                               size_t workspace_bytes, void* stream);

/* Parallel tempering on the device (ptemcee's algorithm: Vousden, Farr & Mandel 2016): n_temps = T ensembles of
 * n_walkers = W walkers sample prior x L^beta_t on the ladder betas, 1 = beta_0 > beta_1 > ... >= 0, and exchange
 * states between adjacent temperatures once per step.  A step = two half-steps of the stretch move over all T
 * ensembles (partners from the same temperature; ONE joint-mode lnprob launch over the T ceil(W/2) proposal rows;
 * accept against the tempered target, a -inf proposal always rejected, a walker at -inf always moving) -> the swap
 * stage, hottest pair first: walker p_i(k) of temperature i and q_i(k) of i - 1 exchange coords and lnprob when
 * ln u < (beta_{i-1} - beta_i)(lnL_{i,p} - lnL_{i-1,q}) -> the record of the state after the swaps.  Every walker keeps
 * its UNTEMPERED lnprob (ln L inside the bounds of rbv_set_bounds, -inf outside).  Random streams: those of
 * rbv_stretch_run with the walker counter offset by t * W (purposes 5 and 6 for the swaps, see rbv_pt.cuh), so T = 1
 * reproduces rbv_stretch_run's chain with the same seed bit for bit, and a run continued with first_step = steps
 * already done reproduces one long run.  voigt_method, precision and far-field settings act as in rbv_lnprob_batch.
 * Rows are never split across ranks: an attached communicator is not used.
 *   coords        DEVICE [T, W, ndim], updated in place;  lnprob DEVICE [T, W] (untempered), updated in place
 *   betas         DEVICE [T], in/out: the ladder (betas[0] = 1, strictly decreasing, >= 0); adapted in place when
 *                 control->adapt is set
 *   control       HOST, see RbvPtControl
 *   chain         DEVICE [n_steps, n_record, W, ndim] or NULL: coordinates of the n_record coldest temperatures
 *   lnprob_chain  DEVICE [n_steps, T, W] or NULL: untempered lnprob of every temperature (thermodynamic integration)
 *   sink          HOST or NULL: instead of chain / lnprob_chain (which must then be NULL), the chain is handed to the
 *                 host as in rbv_stretch_run_sink, with a step of n_record * W * ndim chain and T * W lnprob doubles:
 *                 ring_dev / ring_pinned hold 2 * block_steps * (n_record * W * ndim + T * W) doubles; needs
 *                 use_graph, a non-default stream and n_steps >= 4
 *   beta_history  DEVICE [n_steps, T] or NULL: the ladder each step ran with
 *   n_accepted    DEVICE int[T, W], accumulated accepted stretch moves
 *   n_swaps_accepted  DEVICE uint64[T - 1], accumulated accepted swaps of pair (i, i + 1) (NULL allowed for T = 1)
 *   flag          DEVICE int, bit 0 set if a proposal's lnprob was NaN
 *   workspace     DEVICE, rbv_pt_workspace_bytes();  use_graph as in rbv_stretch_run.  The call copies betas to the
 *                 host to check them (a synchronisation on `stream`); with use_graph it returns after the run. */
typedef struct RbvPtControl {
  double a;                             /* stretch scale (> 1; emcee's default 2)                                 */
  int adapt;                            /* != 0: adapt the interior of the ladder after every step (burn-in only:
                                         * it breaks detailed balance)                                            */
  double adaptation_lag;                /* ptemcee: 10000                                                        */
  double adaptation_time;               /* ptemcee: 100                                                          */
  unsigned long long adapt_steps_done;  /* adaptation steps of earlier calls (continues the decay of kappa)       */
  int n_record;                         /* coldest temperatures whose coordinates are recorded, 1 .. T          */
} RbvPtControl;
int rbv_pt_workspace_bytes(const RbvContext* ctx, int n_temps, int n_walkers, size_t* bytes);
int rbv_pt_run(RbvContext* ctx, double* coords, double* lnprob, double* betas, int n_temps, int n_walkers,
               int n_steps, const RbvPtControl* control, unsigned long long seed, unsigned long long first_step,
               double* chain, double* lnprob_chain, const RbvChainSink* sink, double* beta_history, int* n_accepted,
               unsigned long long* n_swaps_accepted, int* flag, void* workspace, size_t workspace_bytes,
               int use_graph, void* stream);

/* Survey-mode parallel tempering: rbv_pt_run for every sightline of a sightline context (one spectrum per
 * instrument, as rbv_stretch_run_sightlines), all S sightlines advancing in lockstep in one device loop, and
 * optionally the moments of ln L that thermodynamic integration needs, accumulated on the device.  Ensemble
 * e = s T + t (sightline-major).  A half-step is ONE sightline-mode lnprob launch over the S T ceil(W/2) proposal
 * rows; the swap stage runs one CTA per sightline and stays two kernels and one copy per step whatever S and T are.
 * Random streams: those of a one-sightline rbv_pt_run with every walker counter offset by s T W, so sightline 0
 * reproduces rbv_pt_run on that sightline alone and T = 1 reproduces rbv_stretch_run_sightlines, bit for bit.
 *   coords        DEVICE [S, T, W, ndim], updated in place;  lnprob DEVICE [S, T, W] (untempered), updated in place
 *   betas         DEVICE [S, T], in/out: one ladder per sightline (each as in rbv_pt_run; a bad ladder is refused
 *                 with the sightline named); adapted in place, per sightline, when control->adapt is set
 *   control       HOST, see RbvPtControl
 *   chain         DEVICE [n_steps, S, n_record, W, ndim] or NULL;  lnprob_chain DEVICE [n_steps, S, T, W] or NULL
 *   sink          HOST or NULL: as in rbv_pt_run with a step of S * n_record * W * ndim chain doubles and, when
 *                 sink->lnprob_chain_host is not NULL, S * T * W lnprob doubles; with lnprob_chain_host NULL no lnprob
 *                 row is recorded or copied and the ring holds chain rows only
 *   beta_history  DEVICE [n_steps, S, T] or NULL
 *   ti_moments    DEVICE [S, T, 3] or NULL, in/out, accumulated across calls: (n, mean, M2) of the post-swap lnprob
 *                 of every temperature of every step (Chan's merge, see rbv_pt.cuh; Var = M2 / n); NULL: nothing is
 *                 accumulated.  Refused with control->adapt (adaptation breaks detailed balance)
 *   n_accepted    DEVICE int[S, T, W];  n_swaps_accepted DEVICE uint64[S, T - 1] (NULL allowed for T = 1)
 *   flag, workspace (rbv_pt_workspace_bytes_sightlines), use_graph, stream  as in rbv_pt_run.
 * RBV_EINVAL also when S * T * W is outside int range. */
int rbv_pt_workspace_bytes_sightlines(const RbvContext* ctx, int n_temps, int walkers_per_sightline, size_t* bytes);
int rbv_pt_run_sightlines(RbvContext* ctx, double* coords, double* lnprob, double* betas, int n_temps,
                          int walkers_per_sightline, int n_steps, const RbvPtControl* control,
                          unsigned long long seed, unsigned long long first_step, double* chain,
                          double* lnprob_chain, const RbvChainSink* sink, double* beta_history,
                          double* ti_moments, int* n_accepted, unsigned long long* n_swaps_accepted, int* flag,
                          void* workspace, size_t workspace_bytes, int use_graph, void* stream);

/* Device-resident ensemble slice sampler (differential move).  Replaces the sampling loop
 * zeus.EnsembleSampler(nwalkers, ndim, self.lnprob).run_mcmc(guesses, no_of_steps), vfit_mcmc.py:425-440, 536-540
 * (zeus-mcmc >= 2.3.0 is not vendored in the reference; Karamanis & Beutler 2021, Algorithms 2-3 with zeus's defaults,
 * is restated).  Every walker of the active half is a small state machine (widening, shrinking, finished) kept in
 * the workspace; one iteration = candidate kernel -> the lnprob launch over the half (masked rows skipped) -> update
 * kernel.  Both ends of a widening bracket are evaluated in the same iteration (two rows per walker), so a half-step
 * costs as many device batches as the longest chain max(n_L, n_R) + 1 + n_shrink any one walker needs.
 * The loop state (step, iteration, unfinished walkers, mu and its adaptation) lives in device memory.  use_graph != 0
 * (needs a non-default stream): the iteration is the body of a CUDA-graph WHILE node whose condition the update kernel
 * sets, so a half-step is ONE graph launch and the whole run is enqueued without a host synchronisation.
 * use_graph == 0: the host enqueues iterations one ahead of an asynchronous read-back of the counters (the device
 * never waits; one fully masked batch per half-step is the price).  Both modes produce the same chain.
 * Ensemble, directions, brackets and the chain never leave the device.  Random numbers: the Philox streams of
 * rbv_stretch_run (purposes 8.., see rbv_slice.cuh), so a run continued with first_step = steps already done
 * reproduces one long run.
 *   coords, lnprob   DEVICE [n_walkers, ndim] / [n_walkers], updated in place (n_walkers >= 4)
 *   tuning           HOST, in/out: scale mu and its adaptation state (zeus: tune, tolerance 0.05, patience 5,
 *                    maxsteps 10000, maxiter 10000), adapted on the device after every step; the totals of this run
 *                    are written to the n_* fields
 *   chain            DEVICE [n_steps, n_walkers, ndim] or NULL; lnprob_chain DEVICE [n_steps, n_walkers] or NULL
 *   mu_history       DEVICE [n_steps] or NULL: mu after each step
 *   flag             DEVICE int, bit 0 set if a candidate's lnprob was NaN
 *   workspace        DEVICE, rbv_slice_workspace_bytes().  The call returns after the run has finished. */
typedef struct RbvSliceTuning {
  double mu;        /* length scale of the directions 2 mu (C_j - C_l)                                  */
  double tolerance; /* tuning stops counting a step as good when |n_exp / (n_exp + n_con) - 1/2| >= tolerance */
  int tune;         /* != 0 while mu is still adapted (cleared after more than `patience` good steps)   */
  int good;         /* good steps so far                                                                 */
  int patience;
  int maxsteps;     /* stepping-out budget per walker and step, shared between the two sides             */
  int maxiter;      /* iterations per half-step before RBV_ESTATE is returned                            */
  int depth;        /* logical iterations evaluated per launch: 1, or 2 (also 0: the default) -- the second one's
                     * candidates are speculative; chains, mu and the counters below do not depend on it */
  unsigned long long n_expansions, n_contractions; /* out */
  unsigned long long n_calls;                      /* out: lnprob rows the sequential algorithm evaluates */
  unsigned long long n_batches;                    /* out: lnprob launches                               */
} RbvSliceTuning;
int rbv_slice_workspace_bytes(const RbvContext* ctx, int n_walkers, size_t* bytes);
int rbv_slice_run(RbvContext* ctx, double* coords, double* lnprob, int n_walkers, int n_steps, RbvSliceTuning* tuning,
                  unsigned long long seed, unsigned long long first_step, double* chain, double* lnprob_chain,
                  double* mu_history, int* flag, void* workspace, size_t workspace_bytes, int use_graph,
                  void* stream);

/* Survey mode of the slice sampler: the context holds S sightlines (see rbv_lnprob_batch_sightlines) and every
 * sightline has its OWN ensemble of walkers_per_sightline walkers -- what the reference does as S separate
 * vfit(..., sampler='zeus') runs.  The S ensembles advance in lockstep: an iteration is ONE sightline-mode lnprob
 * launch over the candidate rows of every ensemble (masked rows skipped), and a half-step iterates until no walker of
 * any sightline is unfinished; a sightline whose walkers have finished masks its rows, so its chain does not depend
 * on the others.  Ensembles never mix.  Random streams: those of rbv_slice_run with the walker counter offset by
 * sightline * walkers_per_sightline (the step's split is shared), so sightline 0 of a survey run reproduces the
 * single-ensemble run with the same seed.  Loop drivers (use_graph) and depth as in rbv_slice_run; chains, mu and
 * the counters do not depend on either.  Rows are never split across ranks: an attached communicator is not used.
 *   coords, lnprob   DEVICE [S, walkers_per_sightline, ndim] / [S, walkers_per_sightline], in place (wps >= 4)
 *   tuning           HOST: tolerance, patience, maxsteps, maxiter and depth, shared by every sightline; n_batches
 *                    (lnprob launches of this run) is written; mu, tune, good and the other n_* fields are not used
 *   mu               DEVICE double[S], in/out: each sightline's scale, adapted after every step (must be > 0)
 *   tune_good        DEVICE int[S, 2], in/out: each sightline's tune flag and count of good steps
 *   totals           DEVICE uint64[S, 3], accumulated: expansions, contractions, likelihood rows of each sightline
 *   chain            DEVICE [n_steps, S, wps, ndim] or NULL; lnprob_chain DEVICE [n_steps, S, wps] or NULL
 *   mu_history       DEVICE [n_steps, S] or NULL: every sightline's mu after each step
 *   flag             DEVICE int, bit 0 set if a candidate's lnprob was NaN
 *   workspace        DEVICE, rbv_slice_workspace_bytes_sightlines().  Returns RBV_ESTATE when a half-step of any
 *                    sightline needed more than maxiter iterations.  The call returns after the run has finished. */
int rbv_slice_workspace_bytes_sightlines(const RbvContext* ctx, int walkers_per_sightline, size_t* bytes);
int rbv_slice_run_sightlines(RbvContext* ctx, double* coords, double* lnprob, int walkers_per_sightline, int n_steps,
                             RbvSliceTuning* tuning, double* mu, int* tune_good, unsigned long long* totals,
                             unsigned long long seed, unsigned long long first_step, double* chain,
                             double* lnprob_chain, double* mu_history, int* flag, void* workspace,
                             size_t workspace_bytes, int use_graph, void* stream);

/* Model flux for a batch of walkers on instrument `inst`; CompiledVoigtModel.model_flux,
 * voigt_model.py:295-311 (convolve != 0: the instrument's LSF is applied, :221-230) or
 * VoigtModel.evaluate(return_unconvolved=True), :509-558 (convolve == 0: exp(-tau) as it is, :217).
 *   theta     DEVICE [n_walkers, ndim] row-major doubles (ndim = that of rbv_set_bounds, else 3 * n_components)
 *   out_flux  DEVICE [n_walkers, n_pixels] row-major doubles
 *   workspace DEVICE, rbv_flux_workspace_bytes(), or NULL / 0.  With a workspace the per-line constants are
 *             prepared once per walker by a small launch of their own (as rbv_lnprob_batch does); without one every
 *             CTA of the walker prepares them again (fine for a handful of rows).  Same results either way.
 * No prior is applied (rows outside the bounds are evaluated like any other).  Asynchronous. */
int rbv_flux_workspace_bytes(const RbvContext* ctx, int inst, int n_walkers, size_t* bytes);
int rbv_model_flux_batch(RbvContext* ctx, int inst, const double* theta, int n_walkers, int convolve,
                         double* out_flux, void* workspace, size_t workspace_bytes, void* stream);

/* Introspection used by the host layer and the tests. */
int rbv_num_instruments(const RbvContext* ctx);
int rbv_num_tiles(const RbvContext* ctx);          /* CTAs per walker in rbv_lnprob_batch */
int rbv_ndim(const RbvContext* ctx);
long long rbv_launch_count(const RbvContext* ctx); /* kernels launched by this context so far */
/* Which kernel the most recent lnprob launch of this context used: voigt_tile_kernel (one CTA per walker and pixel
 * tile; small batches, very wide LSFs, FP32-gated precision) or voigt_stream_kernel (persistent warps streaming
 * through (walker, pixel range) items; big batches).  -1 before the first launch. */
#define RBV_KERNEL_TILE 0
#define RBV_KERNEL_STREAM 1
int rbv_last_kernel(const RbvContext* ctx);

/* Device Voigt-Hjerting function on a lattice (test hook): out[i] = H(a[i], x[i]); all DEVICE arrays. */
int rbv_voigt_h(RbvContext* ctx, const double* x, const double* a, double* out, int n, int method,
                void* stream);

/* Analytic gradient (DESIGN.md section 14): value and d/dtheta of vfit.lnprob (apply_prior != 0) or vfit.lnlike
 * (apply_prior == 0) for a batch of walkers, from one forward pass and one adjoint pass per walker (no extra rows).
 *   theta  DEVICE [n_walkers, ndim];  value DEVICE [n_walkers];  grad DEVICE [n_walkers, ndim] (columns beyond
 *          3 * n_components are 0)
 *   apply_prior != 0: rows outside the bounds get value -inf and a zero gradient row (the flat prior has zero
 *          gradient; such rows are not evaluated).  apply_prior == 0: every row is evaluated.
 *   NaN where the forward model gives NaN (b <= 0, NaN theta).  FP64 always (ignores rbv_set_precision); every
 *   (line, pixel) pair is evaluated directly (ignores rbv_set_farfield).  Every LSF width the lnprob path accepts.
 *   RBV_EINVAL for an instrument with voigt_method = RBV_VOIGT_FAST; at most 16 instruments.  Each row's result is
 *   bit-identical whatever the batch size or the row's position in it.  Asynchronous.
 * Workspace: rbv_grad_workspace_bytes() (no initialisation needed). */
int rbv_grad_workspace_bytes(const RbvContext* ctx, int n_walkers, size_t* bytes);
int rbv_lnprob_grad_batch(RbvContext* ctx, const double* theta, int n_walkers, int apply_prior, double* value,
                          double* grad, void* workspace, size_t workspace_bytes, void* stream);

/* Model Jacobian and Gauss-Newton (Fisher) matrix of vfit.lnlike (DESIGN.md section 15), forward mode: one column
 * per parameter, the LSF applied to each column, the weighted Gram reduction J^T W J.  Same forward pass as
 * rbv_lnprob_grad_batch; FP64 always (ignores rbv_set_precision / rbv_set_farfield).  NaN where the forward model
 * gives NaN (b <= 0, NaN theta).  RBV_EINVAL for voigt_method = RBV_VOIGT_FAST, more than 16 instruments or
 * ndim < 3 * n_components; RBV_ESTATE before rbv_add_instrument / rbv_set_bounds; RBV_ENOMEM when the workspace is
 * short.  Each row's results are bit-identical whatever the batch size or the row's position in it.  Asynchronous.
 * Workspace: rbv_fisher_workspace_bytes() (about 2 * 3C * P doubles per walker; no initialisation needed). */
int rbv_fisher_workspace_bytes(const RbvContext* ctx, int n_walkers, size_t* bytes);
/* vfit.lnlike (no prior: every row evaluated, as rbv_lnlike_batch), its gradient and its Gauss-Newton matrix.
 *   value  [W]; grad [W, ndim] = sum_p r_p dM_p/dtheta; fisher [W, ndim, ndim] = sum_inst sum_p w_p dM_p/dtheta_i dM_p/dtheta_j
 *   (exactly symmetric; rows / columns beyond 3C are 0).  All DEVICE arrays.  RBV_ESTATE for a flux-only instrument. */
int rbv_lnlike_fisher_batch(RbvContext* ctx, const double* theta, int n_walkers, double* value, double* grad,
                            double* fisher, void* workspace, size_t workspace_bytes, void* stream);
/* d(rbv_model_flux_batch with convolve = 1)/dtheta on instrument inst: out_jac DEVICE [W, ndim, n_pixels], rows beyond
 * 3C = 0.  Same workspace as rbv_lnlike_fisher_batch; allowed on flux-only instruments. */
int rbv_model_jacobian_batch(RbvContext* ctx, int inst, const double* theta, int n_walkers, double* out_jac,
                             void* workspace, size_t workspace_bytes, void* stream);

/* Survey mode of rbv_lnlike_fisher_batch (DESIGN.md section 16): the context holds S sightlines with identical
 * n_pixels, n_taps, n_lines and n_components (see rbv_lnprob_batch_sightlines); row w is evaluated against sightline
 * w / walkers_per_sightline alone, and its results equal bit for bit those of rbv_lnlike_fisher_batch on a context
 * holding that sightline only.  Any number of sightlines; the workspace grows with n_walkers only.  Errors as
 * rbv_lnlike_fisher_batch, and RBV_EINVAL for mismatched sightline geometry or n_walkers != S * walkers_per_sightline.
 * Asynchronous. */
int rbv_fisher_workspace_bytes_sightlines(const RbvContext* ctx, int n_walkers, size_t* bytes);
int rbv_lnlike_fisher_batch_sightlines(RbvContext* ctx, const double* theta, int n_walkers, int walkers_per_sightline,
                                       double* value, double* grad, double* fisher, void* workspace,
                                       size_t workspace_bytes, void* stream);

/* Stopping rules of rbvfit_b200.lm.levenberg_marquardt: at most max_evals evaluations (>= 1); stop when an accepted
 * step lowers chi^2 by at most ftol |chi^2| or when a step is at most xtol (|theta| + xtol) long. */
typedef struct RbvLMControl {
  int max_evals;
  double ftol, xtol;
} RbvLMControl;

/* Bounded Levenberg-Marquardt fit of every sightline in [first, first + n) of a survey-mode context, with the rules of
 * rbvfit_b200.lm.levenberg_marquardt, the context's bounds shared by all sightlines.  Each iteration is one
 * survey-mode Fisher evaluation of the sightlines still iterating, one update kernel (a warp per sightline: step,
 * accept / reject, damping) and a 4-byte read-back of the number still iterating.
 *   theta   [n, ndim]        in: start (clipped into the bounds), out: best point
 *   chi2    [n]              -2 lnlike at theta;  n_evals [n]: evaluations;  status [n]: lm.STATUS_*
 *   cov     [n, ndim, ndim]  inv(F_ff) over the free set at theta, NaN rows / columns elsewhere
 *   flags   [n]              bit 0: F_ff not positive definite at the end (cov left NaN)
 * All DEVICE arrays.  A sightline's results depend on its own data only, not on n, first or the other sightlines.
 * Errors as rbv_lnlike_fisher_batch_sightlines, and RBV_EINVAL for a bad [first, first + n) or control.  Returns
 * after the run has finished (synchronises the stream). */
int rbv_lm_workspace_bytes_sightlines(const RbvContext* ctx, int n_sightlines, size_t* bytes);
int rbv_lm_run_sightlines(RbvContext* ctx, int first, int n, double* theta, const RbvLMControl* ctl, double* chi2,
                          double* cov, int* n_evals, int* status, int* flags, void* workspace,
                          size_t workspace_bytes, void* stream);

/* Test hook, like rbv_voigt_h: H = Re w(x + i a), dH/dx and dH/da on a lattice; all DEVICE arrays. */
int rbv_voigt_h_grad(RbvContext* ctx, const double* x, const double* a, double* H, double* Hx, double* Ha, int n,
                     void* stream);

/* FP64 FMA throughput of the device (roofline denominator measured on the box): runs a dependent-chain
 * DFMA kernel for about `millis` ms and returns TFLOP/s (2 flops per FMA). */
int rbv_measure_fp64_peak(RbvContext* ctx, double millis, double* tflops);

/* Largest relative error of the device reciprocal (MUFU seed + one cubic step) used by the asymptotic tiers, over a
 * sweep of 65 536 positive doubles (test hook; expected < 2^-52). */
int rbv_selftest_rcp(RbvContext* ctx, double* max_rel_err);

/* Text of the last error raised on this thread ("" if none). */
const char* rbv_last_error(void);

/* Library version string. */
const char* rbv_version(void);

#ifdef __cplusplus
}
#endif
#endif /* RBVFIT_B200_H */
