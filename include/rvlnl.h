/*
 * rvlnl.h — C-ABI of librvlnl.so: the B200-native batched Keplerian
 * radial-velocity log-likelihood and unit-cube prior transform.
 *
 * This is the drop-in boundary for the likelihood hot path of the `evidence`
 * package.  Each entry point cites the reference interface it replaces
 * (paths relative to the reference checkout):
 *
 *   evidence/rvmodel/trueanomaly.h:4          int trueanomaly(double*,int,double,double*,int,double)
 *   evidence/rvmodel/__init__.py:157-219      RVModel.log_likelihood(x)
 *   evidence/rvmodel/__init__.py:59-80        BaseModel.logL(residuals, var)
 *   evidence/rvmodel/__init__.py:222-273      RVModel.drift
 *   evidence/rvmodel/__init__.py:343-463      RVModel.kep_rv / modelk
 *   evidence/ultranest/__init__.py:125-146    prior(hypercube) / loglike(x) closures
 *   evidence/polychord/__init__.py:130-171    prior(hypercube) / loglike(x) closures
 *   evidence/priors.py:41-42,62-63,82-83,100-101,249-252  closed-form ppf
 *   evidence/fip_criterion.py:303-338         FIP-periodogram accumulation (next row of the path)
 *   evidence/post_processing.py:93-128        posterior planet ordering      (next row of the path)
 *
 * Conventions
 *   - plain C types only; caller owns every host buffer; the library owns all
 *     device memory.  Row-major, C-contiguous float64.
 *   - theta rows are in the model's SORTED-parnames column order
 *     (evidence/rvmodel/__init__.py:43).
 *   - return 0 on success, a negative RVL_E* code on failure; the message is
 *     available from rvl_last_error().  Nothing throws across the ABI.
 *   - an invalid Keplerian (e > 1 in the secos/sesin and ecos/esin
 *     parametrisations) is DATA, not an error: lnL = -1e30
 *     (evidence/rvmodel/__init__.py:198-203).
 *   - host-buffer calls are synchronous (stream synchronised on return), like
 *     the blocking callbacks of UltraNest / PolyChord.  The *_dev variants take
 *     device pointers and a cudaStream_t (passed as void*) and are asynchronous.
 *   - one handle per host thread.  There is no CPU fallback: every compute
 *     entry point fails with RVL_ENODEV when no sm_100 device is usable.
 */
#ifndef RVLNL_H
#define RVLNL_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RVL_ABI_VERSION 1

#define RVL_MAX_PLANETS 8
#define RVL_MAX_INST 16
#define RVL_MAX_LINPAR 8
#define RVL_MAX_DIM 128
#define RVL_MAX_PEERS 16
#define RVL_FIP_MAX_PLANETS 8
#define RVL_ORDER_MAX_PARAMS 16

/* error codes */
#define RVL_OK 0
#define RVL_EINVAL (-1)  /* bad argument / inconsistent description        */
#define RVL_ENODEV (-2)  /* no usable CUDA device                          */
#define RVL_ECUDA (-3)   /* CUDA runtime error (see rvl_last_error)        */
#define RVL_ESTATE (-4)  /* call order: data/model/priors not yet set      */
#define RVL_ENOMEM (-5)
#define RVL_EPEER (-6)   /* fused all-gather: a peer rank never signalled (bounded wait expired) */

typedef struct rvl_handle rvl_t;

/* A model quantity is either a column of theta (slot >= 0) or a constant
 * (slot == -1, value used).  Mirrors `pardict = free U fixed`
 * (evidence/rvmodel/__init__.py:173-178). */
typedef struct {
    int32_t slot;
    int32_t reserved;
    double value;
} rvl_param;

/* eccentricity parametrisation, branch order of modelk (:425-447) */
#define RVL_ECC_DIRECT 0      /* e1 = ecc,   e2 = omega (no validity check) */
#define RVL_ECC_SECOS_SESIN 1 /* e1 = secos, e2 = sesin; e = c^2+s^2        */
#define RVL_ECC_ECOS_ESIN 2   /* e1 = ecos,  e2 = esin;  e = sqrt(c^2+s^2)  */
/* phase parametrisation (:449-454) */
#define RVL_PHASE_MA0 0 /* phase = ma0                */
#define RVL_PHASE_ML0 1 /* phase = ml0; M0 = ml0 - omega */

typedef struct {
    rvl_param amp;    /* k1, or logk1 when amp_is_log       (:412-415) */
    rvl_param period; /* period, or logperiod when period_is_log (:417-420) */
    rvl_param e1;
    rvl_param e2;
    rvl_param phase;
    rvl_param epoch; /* planet{n}_epoch (:456) */
    int32_t amp_is_log;
    int32_t period_is_log;
    int32_t ecc_mode;
    int32_t phase_mode;
} rvl_planet_desc;

typedef struct {
    int32_t abi_version; /* RVL_ABI_VERSION */
    int32_t ndim;        /* number of free parameters = columns of theta */
    int32_t n_planets;   /* free names containing 'k1'     (:122-124) */
    int32_t n_inst;
    int32_t jitter_in_model; /* some free name contains 'jitter' (:138-139) */
    int32_t drift_in_model;  /* some free name contains 'drift'  (:128-129) */
    int32_t n_linpar;        /* linear-parameter columns         (:210-212) */
    int32_t itmax;           /* Newton cap, reference 10000      (:491)     */
    double tol;              /* Newton |dE| tolerance, reference 1e-4 (:466) */
    double tref;             /* drift reference time: drift_tref or time[0] (:256-260) */
    rvl_planet_desc planet[RVL_MAX_PLANETS];
    rvl_param offset[RVL_MAX_INST]; /* {inst}_offset (:187) */
    rvl_param jitter[RVL_MAX_INST]; /* {inst}_jitter (:190); ignored unless jitter_in_model */
    rvl_param drift[4];             /* lin, quad, cub, quar (:246-253) */
    rvl_param linpar[RVL_MAX_LINPAR];
} rvl_model_desc;

/* prior kinds: ppf(q), evidence/priors.py */
#define RVL_PRIOR_UNIFORM 0     /* p0=xmin p1=xmax : xmin + (xmax-xmin) q          (:41-42)  */
#define RVL_PRIOR_JEFFREYS 1    /* p0=xmin p1=xmax : xmin (xmax/xmin)^q            (:62-63)  */
#define RVL_PRIOR_MODJEFFREYS 2 /* p0=x0   p1=xmax : x0 (1+xmax/x0)^q - x0         (:82-83)  */
#define RVL_PRIOR_UNIFORMFREQ 3 /* p0=xmin p1=xmax : xmin / (1 - q (xmax-xmin)/xmax) (:100-101) */
#define RVL_PRIOR_TRUNCRAYLEIGH 4 /* p0=sigma p1=xmax                              (:249-252) */
#define RVL_PRIOR_NORMAL 5      /* p0=loc p1=scale : loc + scale ndtri(q)  (stats.norm, :436) */
#define RVL_PRIOR_LOGNORMAL 6   /* p0=s p1=loc p2=scale : loc + scale exp(s ndtri(q)) (:437)  */
#define RVL_PRIOR_TABLE 7       /* piecewise-linear inverse CDF through (cdf_k, x_k) knots
                                   (p0 = 1: result is 10**interp, Log10Normal :144;
                                    p1 = 1: a third array of slopes dx/dq follows -> cubic Hermite),
                                   the scheme of the interp1d priors (:118-124,195-202,223-228,
                                   282-287,321-326,349-354); also used for Beta/Gamma/Alpha */

typedef struct {
    int32_t kind;
    int32_t table_len;    /* RVL_PRIOR_TABLE: number of knots */
    int64_t table_offset; /* RVL_PRIOR_TABLE: offset (in doubles) of the knots inside `tables`:
                             cdf[0..len) followed by x[0..len) [and slope[0..len) when p1 = 1] */
    double p[4];
} rvl_prior_desc;

typedef struct {
    uint64_t n_points;       /* lnL evaluations since reset                        */
    uint64_t n_solves;       /* Kepler solves (point x planet x epoch)             */
    uint64_t n_newton_iters; /* total Newton iterations actually taken             */
    uint64_t n_cap_hits;     /* solves that stopped at itmax (reference: :490 ignores -1) */
    uint64_t n_invalid;      /* points returned as -1e30                           */
} rvl_counters_t;

/* ---- lifecycle -------------------------------------------------------- */
int rvl_abi_version(void);
/* device < 0: use the current CUDA device */
int rvl_create(rvl_t **out, int device);
/* One handle over several GPUs of the box, for a single-process caller (a ctypes consumer bound as
 * in INTEGRATION.md gets the whole box through the SAME calls): the staging calls are replicated on
 * every device, and every host-buffer hot call (rvl_transform / rvl_loglike /
 * rvl_transform_loglike) splits its B rows into contiguous blocks -- device i of n owns rows
 * [i*ceil(B/n), min(B, (i+1)*ceil(B/n))), the partition the samplers' MPI ranks use
 * (evidence/ultranest/__init__.py:21-29) -- launches all devices from the calling thread and
 * returns when all have finished.  Page-locked caller buffers are read and written in place by all
 * devices, so the gathered lnL vector is simply the caller's buffer.  devices == NULL /
 * n_devices == 0: every device of the box.  The *_dev entry points need a single-device handle. */
int rvl_create_multi(rvl_t **out, const int32_t *devices, int32_t n_devices);
/* number of devices behind the handle (1 for rvl_create) */
int rvl_device_count(rvl_t *h, int32_t *n);
void rvl_destroy(rvl_t *h);
/* back to the state of a fresh handle after a faulted / aborted launch (work counters, arrival
 * counters and ready stamps only re-arm themselves when a launch runs to its end) */
int rvl_reset(rvl_t *h);
/* h may be NULL: returns the last error of the calling thread (rvl_create failures) */
const char *rvl_last_error(const rvl_t *h);

/* ---- staging (once per run) ------------------------------------------- */
/* Epoch data in the order BaseModel concatenates it (evidence/rvmodel/__init__.py:50-55,
 * 141-146): time (rjd|jdb), vrad, svrad, inst_id in [0, n_inst). */
int rvl_set_data(rvl_t *h, const double *t, const double *rv, const double *err,
                 const int32_t *inst, int32_t n, int32_t n_inst);
/* linpar_dict[name] column (evidence/rvmodel/__init__.py:210-212) */
int rvl_set_linpar(rvl_t *h, int32_t idx, const double *col, int32_t n);
int rvl_set_model(rvl_t *h, const rvl_model_desc *desc);
int rvl_set_priors(rvl_t *h, const rvl_prior_desc *priors, int32_t ndim, const double *tables,
                   int64_t n_table_doubles);
/* knobs, by name; unknown name -> RVL_EINVAL:
 *   "timing"    1: record CUDA events around the likelihood kernel (rvl_last_kernel_ms); default 0
 *   "zero_copy" host-buffer calls: 1 (default) page-locked (pinned) theta / U are read and theta /
 *               lnL written in place over PCIe by the kernels (each theta row is read once,
 *               coalesced, while other warps compute); PAGEABLE buffers up to 32 MiB (numpy arrays)
 *               are bounced through pinned buffers of the handle with one CPU memcpy instead of the
 *               driver's synchronous pageable copy; theta is staged by one DMA copy when the epoch
 *               axis needs several resident ranges; 2: in place even then (through the
 *               once-per-point pass); 0: stage everything with cudaMemcpyAsync
 *   "variant"   0 optimised kernel (default), 1 conservative cross-check (IEEE division, full sin/cos)
 *   "ilp"       epochs per lane in flight, 1..4; 0 (default): 4 for large batches of long points with
 *               four or more planets (N K >= 16384), 2 otherwise
 *   "sched"     1 (default): graded work list -- whole points first, then the points at the end of the
 *               batch cut into 2, 4, .. "max_split" (8) sub-slices with about "phase_items" (200)
 *               percent of one item per warp in each phase, so that all warps run dry together;
 *               0: one uniform slice count ("items_per_warp", "min_chunks")
 *   "setup_items" 1 (default): the constants of the points that are cut into several items are
 *               derived once, by setup items at the head of the kernel's own work list
 *   "prepare"   1: per-point constants from the once-per-point pass even without a transform
 *   "trace"     1: per-warp time stamps of the last launch (rvl_read_trace)
 *   "gather_timeout_ms" bound of the wait for the peers' completion slots in the fused all-gather
 *   "slices", "warps": launch-plan overrides (0 = automatic) */
int rvl_set_option(rvl_t *h, const char *name, int64_t value);

/* ---- hot path: host buffers, synchronous -------------------------------- */
/* replaces the prior(hypercube) closure, one row per point */
int rvl_transform(rvl_t *h, const double *U, int64_t B, double *Theta);
/* replaces the loglike(x) closure / RVModel.log_likelihood, one row per point */
int rvl_loglike(rvl_t *h, const double *Theta, int64_t B, double *lnL);
/* fused u -> theta -> lnL; Theta may be NULL when the sampler does not need it */
int rvl_transform_loglike(rvl_t *h, const double *U, int64_t B, double *Theta, double *lnL);

/* ---- hot path: device buffers, asynchronous on `stream` ------------------
 * The launches of ONE handle share its work counters and scratch buffers: enqueue them in stream
 * order (one stream at a time per handle; use one handle per stream for concurrency). */
int rvl_transform_dev(rvl_t *h, const double *dU, int64_t B, double *dTheta, void *stream);
int rvl_loglike_dev(rvl_t *h, const double *dTheta, int64_t B, double *dlnL, void *stream);
int rvl_transform_loglike_dev(rvl_t *h, const double *dU, int64_t B, double *dTheta,
                              double *dlnL, void *stream);

/* ---- multi-GPU: the all-gather fused into the producing kernel -------------------- */
/* Like rvl_loglike_dev, and additionally every lnL[i] is stored into n_peers peer-mapped device
 * buffers (NVLink peer / symmetric memory of the other ranks, and our own gathered vector) at
 * element `offset + i`, by the same kernel that produces it.  The caller synchronises the ranks
 * afterwards (one signal barrier) instead of running a separate all-gather collective.
 * peer_ptrs: n_peers device addresses as 64-bit integers. */
int rvl_loglike_dev_scatter(rvl_t *h, const double *dTheta, int64_t B, double *dlnL,
                            const uint64_t *peer_ptrs, int32_t n_peers, int64_t offset,
                            void *stream);

/* The whole all-gather inside the likelihood launch.  As rvl_loglike_dev_scatter, and when the
 * launch has finished its last work item it stores `seq` (64-bit, release, system scope) into slot
 * `flag_offset + rank` (in 8-byte elements) of EVERY peer buffer; a one-warp kernel enqueued behind
 * it on `stream` then waits until all n_peers slots of this rank's own buffer (peer_ptrs[rank])
 * hold >= seq.  When that returns -- in stream order -- the gathered vector is complete on this
 * rank: no barrier, no collective.  The caller zeroes the slots once, uses seq = 1, 2, 3, ... per
 * buffer, and alternates two buffers so that a fast rank never overwrites what a slow one still
 * reads (evidence_b200/multigpu.py: FusedGatherLikelihood). */
int rvl_loglike_dev_gather(rvl_t *h, const double *dTheta, int64_t B, double *dlnL,
                           const uint64_t *peer_ptrs, int32_t n_peers, int32_t rank, int64_t offset,
                           int64_t flag_offset, uint64_t seq, void *stream);

/* The same exchange for HOST buffers, one call per rank and step (what a sampler running one
 * process per GPU does where UltraNest's MPI mode gathers the ranks' likelihood values,
 * evidence/ultranest/__init__.py:21-29): this rank's B rows of theta (page-locked: read in place by
 * the kernel) -> lnL of ALL ranks, lnL_all[n_peers * B] in host memory, rank r's block at r*B.
 * peer_ptrs / flag_offset / seq as above; every rank passes the same B.  Synchronous.  A peer that
 * never signals makes the call fail with RVL_EPEER after "gather_timeout_ms" (default 10000)
 * instead of hanging the stream. */
int rvl_loglike_gather(rvl_t *h, const double *Theta, int64_t B, double *lnL_all,
                       const uint64_t *peer_ptrs, int32_t n_peers, int32_t rank,
                       int64_t flag_offset, uint64_t seq);
/* after synchronising the stream of an rvl_loglike_dev_gather: RVL_EPEER if its bounded wait expired */
int rvl_gather_status(rvl_t *h);

/* The gather through a HOST segment shared by the ranks' processes (POSIX shared memory mapped by
 * every rank; evidence_b200/multigpu.py: SharedHostGather) -- for host consumers, the cheapest form:
 * every rank's kernel stores its B lnL values straight into the segment at element `offset`
 * (normally rank * B) over its own PCIe link, overlapped with the arithmetic; no device-side gathered
 * vector, no D2H copy of world * B values per rank.  When the launch has finished, `seq` is stored
 * (release, system scope) into element `flag_offset + rank` of the segment; every process then waits
 * on the host for all ranks' slots (rvl_wait_host_flags: RVL_EPEER after timeout_ms, < 0 = forever;
 * message from rvl_last_error(NULL)).  rvl_host_register page-locks and maps a host range for this
 * device context and returns its device address; each process registers its own mapping. */
int rvl_host_register(void *ptr, int64_t bytes, uint64_t *dev_ptr);
int rvl_host_unregister(void *ptr);
int rvl_loglike_scatter_host(rvl_t *h, const double *Theta, int64_t B, uint64_t shared_dev_ptr,
                             int64_t offset, int64_t flag_offset, int32_t rank, uint64_t seq);
int rvl_wait_host_flags(const uint64_t *flags, int32_t n, uint64_t seq, int32_t timeout_ms);

/* ---- the reference's own native FFI, on the device (trueanomaly.h:4) ----- */
/* Same contract as the reference symbol except: returns -1 when ANY element hit the cap
 * (every nu[i] is still written from the last iterate, the reference leaves the rest 0). */
int rvl_trueanomaly(rvl_t *h, const double *M, int32_t n, double ecc, double *nu,
                    int32_t niterationmax, double tol);

/* ---- model velocity curves: RVModel.kep_rv / modelk (evidence/rvmodel/__init__.py:343-463) ---- */
/* Keplerian part of the model velocity for B theta rows at T caller times:
 *   out[b][j] = sum over the planets p with bit p of planet_mask set, in planet order (kep_rv :383),
 *               of modelk(theta_b, times[j], planet = p + 1)   (:388-463)
 * planet_mask == 0 -> zeros; a bit at or above n_planets -> RVL_EINVAL.  invalid[b] (may be NULL):
 * bit p set when planet p of row b is not a valid Keplerian (e > 1 in the secos/sesin or ecos/esin
 * parametrisation, :425-439); a row with an invalid planet inside planet_mask is NaN.  cap_hits
 * (may be NULL): incremented by the solves that stopped at itmax.  Needs rvl_set_model; Newton
 * tol/itmax are the model's.  Times may be in any order and anywhere (|M| >= 1e5 takes the general
 * Newton loop).  Each element is computed alone: a row's curve does not depend on the batch.  A
 * multi-device handle runs the call on its first device (as rvl_trueanomaly does).  rvl_counters
 * is not touched.  Synchronous. */
int rvl_kepler_rv(rvl_t *h, const double *Theta, int64_t B, const double *times, int32_t T,
                  uint32_t planet_mask, double *out, uint32_t *invalid, uint64_t *cap_hits);
/* the same on device pointers (dCapHits: a device counter, may be NULL), asynchronous on stream;
 * single-device handle; shares the handle's per-point scratch with the likelihood calls (stream
 * order, as for every *_dev call) */
int rvl_kepler_rv_dev(rvl_t *h, const double *dTheta, int64_t B, const double *dTimes, int32_t T,
                      uint32_t planet_mask, double *dOut, uint32_t *dInvalid, uint64_t *dCapHits,
                      void *stream);

/* ---- observability / measurement ---------------------------------------- */
int rvl_counters(rvl_t *h, rvl_counters_t *out);
int rvl_reset_counters(rvl_t *h);
/* duration (ms, CUDA events on the launching stream) of the last likelihood launch of a
 * host-buffer call, kernel only */
int rvl_last_kernel_ms(rvl_t *h, double *ms);
/* option "timing": time (ms) between the end of the likelihood kernel of the last fused all-gather
 * call and the moment every peer's completion slot had arrived (the wait_flags kernel): what the
 * exchange costs this rank beyond its own kernel -- rank skew plus NVLink latency */
int rvl_last_gather_wait_ms(rvl_t *h, double *ms);
/* number of kernel launches issued by this handle so far */
int rvl_launch_count(rvl_t *h, uint64_t *n);
/* register-resident DFMA loop: measured FP64 peak of this device, TFLOP/s (2 flop per DFMA) */
int rvl_fp64_peak(rvl_t *h, double *tflops);
/* option "trace" = 1: every warp of the likelihood kernel records { t_enter, t_ready (epoch data
 * resident), t_done } in ns of the device's global timer and its number of work items; this
 * reads the rows of the last launch (tools/warp_trace.py draws the drain curve from them). */
int rvl_read_trace(rvl_t *h, uint64_t *out, int32_t cap_rows, int32_t *rows);
/* The launch plan as data (no device needed; tests/test_plan.py checks that the work items cover
 * every (point, epoch chunk) exactly once).  in[13] = { ceil(N/32), ncol, wstride, ilp, warps,
 * sm_count, smem_optin, sched, slices, items_per_warp, min_chunks, phase_items, max_split };
 * out[0..8) = { Sm, cpm, grid, n_phases, items per queue, first split point, split points,
 * partial-sum doubles }, then per phase { idx0, S, cps, pt0, part0 }. */
int rvl_plan_describe(const int32_t *in, int64_t B, int64_t *out, int32_t cap);
/* sm count, smem per block opt-in, clock (kHz) */
int rvl_device_info(rvl_t *h, int32_t *sm_count, int32_t *smem_optin, int32_t *clock_khz);

/* ---- next row of the path (SURVEY.md 8f-4): FIP-periodogram accumulation ------------------ */
/* Replaces the per-sample Python loop of evidence/fip_criterion.py:303-338 for ONE (run, k-planet
 * model) block: for each of the n posterior samples (periods[n][k], days; weights[n], any positive
 * normalisation) every grid bin j with nua[j] < f < ... -- precisely the bins
 * range(searchsorted(nub, f, 'right'), searchsorted(nua, f, 'left')) of one of the sample's mean
 * motions f = 2 pi / P (with_alias: also |f +- 2pi/0.99727|, |f +- 2pi/30|, kept when inside
 * [2pi/pmax, 2pi/pmin]) -- receives  fapnu[j] -= pk * weight / sum(weights),  once per sample.
 * nua / nub are the caller's arrays (fip_criterion.py:233-236), searched with the reference's own
 * comparisons.  fapnu[nfreq] is updated in place (host buffer).  Accumulation is 2^-56 fixed point
 * with integer atomics: bit-reproducible.  kernel_ms (optional): CUDA-event time of the two
 * kernels.  No handle: device < 0 = current device.  Errors: rvl_fip_last_error(). */
int rvl_fip_accumulate(int32_t device, const double *nua, const double *nub, int32_t nfreq,
                       const double *periods, int32_t k, const double *weights, int64_t n,
                       double pk, int32_t with_alias, double pmin, double pmax, double *fapnu,
                       double *kernel_ms);
const char *rvl_fip_last_error(void);

/* Replaces the posterior planet-ordering loop of evidence/post_processing.py:104-128: out[n][ndim]
 * = samples[n][ndim] with, in every row whose K planet periods (columns period_cols[K]) are not
 * non-decreasing, the columns of the planets (planet_cols[K][Q]: the Q columns of planet p, in
 * parnames order -- :94-102) gathered through the reference's index list,
 * new[planet_cols[p][q]] = old[planet_cols[rank(p)][q]] with rank = position of p in
 * np.argsort(periods), exactly equal periods in planet order (numpy's default sort leaves ties
 * platform-dependent), NaN last.  (That is the inverse of the sorting permutation; reproduced as is.)
 * Host buffers; out must not alias samples.  Errors: rvl_order_last_error(). */
int rvl_order_planets(int32_t device, const double *samples, int64_t n, int32_t ndim,
                      const int32_t *period_cols, const int32_t *planet_cols, int32_t K, int32_t Q,
                      double *out, double *kernel_ms);
const char *rvl_order_last_error(void);
/* rvl_fip_accumulate and rvl_order_planets keep their device buffers and events per device between
 * calls (no allocation on the second call of a size); this frees them. */
void rvl_post_release(void);

/* ---- next row of the path (SURVEY.md 8f-1): the vectorised proposal step ------------------- */
/* Device-side bookkeeping of a population slice sampler -- the kind of step sampler the reference
 * configures (evidence/ultranest/__init__.py:175), for k walkers at once, with every array on the
 * device and no host read-back inside a move.  One slice move = phase 0 (direction, bracket, all
 * stepping-out positions as candidates) -> likelihood of the k * 2 n_out candidates -> phase 1
 * (bracket from the runs of successes; m shrinkage candidates per walker, each drawn as if the
 * ones before it were rejected) -> likelihood of the k * m candidates -> phase 2 (accept the first
 * candidate above *lmin; m more candidates for the walkers still pending) -> likelihood -> ... ->
 * phase 3 (accept; walkers still pending keep their position).  The likelihood in between is
 * rvl_transform_loglike_dev on `cand_out` (k * 2 n_out rows -> `ll_out`) after phase 0 and on
 * `cand` (k * m rows -> `cand_th`, `cand_ll`) after phases 1 and 2.  Candidates outside the unit cube are clamped for the evaluation and never accepted.
 * All pointers are device addresses (as 64-bit integers); random numbers are Philox4x32-10 keyed by
 * the seed with (move, shrink_round and draw, walker, 0) as the counter: every walker of every seed
 * has its own streams, reproducible for a seed whatever k.
 * evidence_b200/sampler_dev.py drives it. */
typedef struct {
    int32_t k, d, n_out, m;
    uint64_t seed;
    uint32_t move, shrink_round;
    uint64_t lmin;    /* const double*  [1]        constraint: accept iff lnL > *lmin          */
    uint64_t chol;    /* const double*  [d][d]     whitening (lower Cholesky factor, row major)  */
    uint64_t u;       /* double*        [k][d]     walker positions in the unit cube (in/out)    */
    uint64_t theta;   /* double*        [k][d]     their physical parameters (out)               */
    uint64_t lcur;    /* double*        [k]        their lnL (out; untouched until a move lands) */
    uint64_t dirn;    /* double*        [k][d]     scratch                                       */
    uint64_t lo, hi, lo2, hi2; /* double* [k]      scratch                                       */
    uint64_t tval;    /* double*        [k][m]     scratch                                       */
    uint64_t pending; /* int32_t*       [k]        scratch                                       */
    uint64_t cand_out;   /* double*       [k][2 n_out][d] stepping-out candidates (out of phase 0)   */
    uint64_t inside_out; /* uint8_t*      [k][2 n_out]    scratch                                    */
    uint64_t ll_out;     /* const double* [k][2 n_out]    their lnL (in for phase 1)                 */
    uint64_t cand;    /* double*        [k][m][d]  shrinkage candidates (out of phases 1, 2)     */
    uint64_t inside;  /* uint8_t*       [k][m]     scratch                                       */
    uint64_t cand_ll; /* const double*  [k][m]     their lnL (in for phases 2, 3)                */
    uint64_t cand_th; /* const double*  [k][m][d]  their theta                                   */
    uint64_t stats;   /* uint64_t*      [2]        += walkers left unresolved, += accepted moves */
} rvl_slice_args;
int rvl_slice_phase(int32_t phase, const rvl_slice_args *args, void *stream);
/* rvl_slice_phase with circular coordinates: bit j & 31 of wrap_bits[j >> 5] set marks coordinate j
 * as circular (UltraNest's wrapped_params; the reference wraps names containing "omega" or "ml0",
 * evidence/ultranest/__init__.py:159-162).  A candidate's circular coordinate p = u + t dirn is
 * stored as q = p - floor(p), with q = 0 where that rounds to 1 (only for a tiny negative p), and
 * never marks the candidate as outside the cube; an accepted point is that stored value, so u stays
 * in [0, 1).  The other coordinates, directions, brackets, random streams and acceptance are those
 * of rvl_slice_phase.  The walkers then move on the torus, whose uniform measure is the cube's: the
 * moves stay valid for nested sampling whether or not lnL is periodic in that coordinate.
 * wrap_bits NULL or all zero: exactly the launches of rvl_slice_phase.  A bit at or above d:
 * RVL_EINVAL (message in rvl_slice_last_error). */
int rvl_slice_phase_wrapped(int32_t phase, const rvl_slice_args *args, const uint32_t wrap_bits[4],
                            void *stream);

/* An ensemble: R independent runs of one model whose walkers share every launch
 * (evidence_b200/sampler_dev.py: nested_sample_ensemble).  Walker w of a launch is walker
 * walker_of[w] of run run_of[w]; the walkers of a run may sit anywhere in the launch.  It uses that
 * run's constraint lmin[r], whitening chol[r] and counters stats[r], and draws from seeds[r] with
 * walker_of[w] as the walker word of its counters: exactly what walker j of an rvl_slice_phase call
 * with k = k_r and seed = seeds[r] draws.  run_of values must lie in [0, n_runs). */
typedef struct {
    int32_t n_runs, reserved;
    uint64_t run_of;    /* const int32_t*  [k]        run of each walker of the launch             */
    uint64_t walker_of; /* const int32_t*  [k]        its index inside that run                    */
    uint64_t seeds;     /* const uint64_t* [R]                                                     */
    uint64_t lmin;      /* const double*   [R]        each run's constraint                        */
    uint64_t chol;      /* double*         [R][d][d]  each run's whitening (written by _whiten)    */
    uint64_t stats;     /* uint64_t*       [R][2]     each run's counters, as rvl_slice_args.stats */
} rvl_slice_runs;
/* rvl_slice_phase / rvl_slice_phase_wrapped (wrap_bits may be NULL) for the walkers of several runs.
 * args->k is the total number of walkers; args->seed, lmin, chol and stats are ignored (the runs'
 * own are used).  Errors as rvl_slice_phase, and RVL_EINVAL for a NULL runs, n_runs < 1 or a
 * missing address in it. */
int rvl_slice_phase_runs(int32_t phase, const rvl_slice_args *args, const rvl_slice_runs *runs,
                         const uint32_t wrap_bits[4], void *stream);
/* The live points of the R runs of an ensemble, for its set-up calls. */
typedef struct {
    int32_t nlive, d;
    uint32_t round, reserved; /* round: the start draws' counter word (one value per round)    */
    uint64_t u_live;  /* double*        [R][nlive][d] unit-cube live points                      */
    uint64_t th_live; /* const double*  [R][nlive][d] their parameters                           */
    uint64_t l_live;  /* const double*  [R][nlive]    their lnL                                  */
    uint64_t order;   /* const int64_t* [R][nlive]    each run's points by ascending lnL (a stable sort) */
    uint64_t kk;      /* const int64_t* [R]           points retired this round, 1 <= kk[r] <= nlive - 2:
                                                      the survivors of run r are order[r][kk[r]:];
                                                      0: run r takes no part in the round */
    uint64_t start;   /* int64_t*       [k]           out: the slot of each walker's start point  */
    uint64_t lstart;  /* double*        [k]           out: its lnL                                */
} rvl_slice_live;
/* The set-up of an ensemble round, each run's values from its own points and seed alone (whatever R):
 *   _init    u_live[r][p][c] = the uniform of Philox counter (0, 0x494E0000 + c / 2, p, 0) under
 *            seeds[r] (words x, y for even c; z, w for odd c; the u01 of the slice draws).
 *            Reads n_runs, seeds, nlive, d, u_live.
 *   _whiten  one block per run: chol[r] = lower Cholesky factor of 1e-18 I + the covariance of the
 *            survivors of run r (sums over them in order; divided by n - 1), circular coordinates of
 *            wrap_bits (may be NULL) first taken modulo 1 about their circular mean, as
 *            sampler_dev._whitening does; where a pivot is not > 0, diag(sqrt(max(cov_jj, 1e-30))).
 *            The upper triangle is 0.  A run with kk[r] = 0 is skipped (chol[r] is left as it is).
 *   _starts  for each walker w of args (k = args->k, run r = run_of[w], j = walker_of[w]): a start
 *            point, survivor number floor(x n / 2^32) of run r, x the first word of Philox counter
 *            (round, 0x53540000, j, 0) under seeds[r], n = nlive - kk[r]; copied into args->u and
 *            args->theta; args->lcur = NaN; start / lstart = its slot and lnL.  args->d == live->d.
 * Errors: RVL_EINVAL with a message in rvl_slice_last_error for bad sizes or a missing address. */
int rvl_slice_runs_init(const rvl_slice_runs *runs, const rvl_slice_live *live, void *stream);
int rvl_slice_runs_whiten(const rvl_slice_runs *runs, const rvl_slice_live *live,
                          const uint32_t wrap_bits[4], void *stream);
int rvl_slice_runs_starts(const rvl_slice_args *args, const rvl_slice_runs *runs,
                          const rvl_slice_live *live, void *stream);
const char *rvl_slice_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* RVLNL_H */
