/* obe_b200.h -- C ABI of libobe_b200.so: the B200 (sm_100a) particle-filter inference and
 * setting-selection path of usnistgov/optbayesexpt v1.2.0.
 *
 * The reference is pure Python/numpy and has NO FFI of its own: its boundary is the method
 * surface of ParticlePDF / OptBayesExpt / OptBayesExptNoiseParameter.  Each entry point below
 * names the reference method (file:line under /root/reference/optbayesexpt) whose arithmetic
 * it replaces; optbayesexpt_b200/*.py re-creates those classes on top of this ABI via ctypes
 * (INTEGRATION.md shows the binding a reference maintainer would add).
 *
 * Conventions
 *   - plain C: pointers + sizes only.  Pointers named *_dev are DEVICE pointers owned by the
 *     caller (e.g. torch tensors' data_ptr()); everything else is host memory.
 *   - all floating point is IEEE fp64, all indices int64; particles are SoA (d, ld).
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*) unless noted;
 *     the library never allocates device memory behind the caller: scratch comes from the
 *     obe_cloud_t arrays, sized with the obe_*_len() queries.
 *   - return 0 on success, <0 on error; obe_last_error() gives the thread-local message.
 *   - there is no CPU fallback: without a CUDA device every compute entry fails.
 */
#ifndef OBE_B200_H
#define OBE_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OBE_ABI_VERSION 1
#define OBE_TILE_SIZE 2048      /* canonical tile: CDF association, tile_sums granularity   */
#define OBE_STATS_DOUBLES 64    /* length of the device stats block                         */
#define OBE_MAX_PARAMS 8
#define OBE_MAX_CHANNELS 4
#define OBE_MAX_SETTINGS 4
#define OBE_MAX_CONSTANTS 8

/* stats block layout (doubles), written by obe_update / obe_refresh / obe_tile_scan */
enum {
    OBE_STAT_TOTAL = 0,   /* canonical sum of the un-normalised weights (CDF total)          */
    OBE_STAT_INVS = 1,    /* weights_normalised = weights * stats[INVS]                      */
    OBE_STAT_SUMSQ = 2,   /* sum t^2                                                         */
    OBE_STAT_NEFF = 3,    /* 1/sum(w^2) of particlepdf.py:243-244                            */
    OBE_STAT_M1 = 4,      /* [8]  sum t (x_j - pivot_j)                                      */
    OBE_STAT_M2 = 12,     /* [d(d+1)/2] sum t (x_j-p_j)(x_k-p_k), j<=k packed row-major      */
    OBE_STAT_PIVOT = 48,  /* [8]                                                             */
    OBE_STAT_NOISE = 56,  /* [4]  sum t sigma_c^2                                            */
    OBE_STAT_SUMT = 60,   /* sum t from the same pass as the moments                         */
    OBE_STAT_NZERO = 61,  /* particles newly zeroed by the constraint mask                   */
    OBE_STAT_UNIFORM = 62, /* > 0: weights are implicit, every live particle weighs this much */
    OBE_STAT_FIRED = 63   /* 1: the device-side resample test of that update fired (obe_cycle, resample == 2) */
};

/* The particle cloud resident in HBM (ParticlePDF state, particlepdf.py:96-126). */
typedef struct obe_cloud {
    double* particles_dev;    /* (d, ld) row-major: one contiguous row per parameter        */
    double* weights_dev;      /* (n) UN-normalised weights t; normalised = t * stats[INVS]  */
    double* tile_sums_dev;    /* (obe_num_tiles(n))                                         */
    double* tile_prefix_dev;  /* (obe_num_tiles(n) + 1) exclusive prefix; last = CDF total  */
    double* stats_dev;        /* (OBE_STATS_DOUBLES)                                        */
    void* scratch_dev;        /* obe_scratch_bytes(n) bytes, zero-initialised by the caller */
    int64_t n;                /* particles                                                   */
    int64_t ld;               /* row stride in doubles, even (16-byte aligned rows)          */
    int32_t d;                /* parameters per particle (1..OBE_MAX_PARAMS)                 */
    int32_t reserved;
    int64_t* n_dev;           /* NULL, or a device int64 holding the LIVE particle count; `n` is
                                 then only an upper bound (shards of a multi-GPU cloud change
                                 length in a resample without the host being told)            */
} obe_cloud_t;

typedef struct obe_model* obe_model_t; /* opaque device functor for model_function */

/* ---- library ---------------------------------------------------------------------------- */
int obe_abi_version(void);
const char* obe_last_error(void);
int obe_device_count(void);
/* Tuning knobs for tests and A/B runs.  "plan_cluster_min_tiles": tile count (2048 particles each) above
 * which the resample plan runs on a thread-block cluster of 8 CTAs instead of one CTA (default 8192).
 * "utility_lane_fill": the variance utility uses 8/4/2 lanes per setting while n_settings * lanes stays
 * below this percentage of the resident thread count (default 50; 0 = always one thread per setting).
 * Returns 0, or -1 for an unknown name. */
int obe_set_option(const char* name, int64_t value);                 /* 0 without a usable CUDA device                */
int64_t obe_num_tiles(int64_t n);
size_t obe_scratch_bytes(int64_t n);        /* per-cloud scratch (partials, plans, counters) */
size_t obe_select_scratch_bytes(int64_t n_settings);

/* ---- model_function as a device functor (obe_base.py:50-66, 165, 215-222) ---------------- */
/* names: lorentzian_hwhm, lorentzian_fwhm, lorentzian_4p, lorentzian_dip, line, rabi,
 * lockin_coil.  n_params = d of the cloud (>= the model's own parameter count). */
int obe_model_builtin(const char* name, int n_params, obe_model_t* out);
/* User CUDA source compiled by NVRTC for sm_100a.  The source must define
 *   __device__ void <entry>(const double* s, const double* p, const double* c, double* y)
 * `log`/`log_len` receive the compiler log. */
int obe_model_compile(const char* cuda_source, const char* entry, int n_settings, int n_params,
                      int n_model_params, int n_constants, int n_channels, obe_model_t* out,
                      char* log, size_t log_len);
/* A model whose update uses a non-Gaussian measurement likelihood, compiled by NVRTC for sm_100a.
 * The model is the built-in `builtin_name`, or (builtin_name == NULL) `model_source` / `model_entry`
 * with the dimensions of obe_model_compile.  `likelihood`:
 *   "poisson"   record (setting, k_c): y_c is the expected count lambda_c,
 *               log L = sum_c xlogy(k_c, lambda_c) - lambda_c - lgamma(k_c + 1)
 *   "binomial"  record (setting, k_c, n_c): y_c is the success probability p_c,
 *               log L = sum_c lgamma(n+1) - lgamma(k+1) - lgamma(n-k+1) + xlogy(k, p) + xlog1py(n-k, -p)
 *   "user"      `likelihood_source` defines
 *               __device__ double <likelihood_entry>(const double* y_model, const double* y_meas,
 *                                                    const double* aux, int n_channels)
 *               returning log L of the record (y_meas = its second element, aux = its third).
 * The weight factor is exp(choke * log L).  obe_update / obe_cycle / obe_update_from_y_model take such a
 * handle: y_meas carries the counts (the measured values), sigma the third element of the record
 * (trial counts, aux; may be NULL for Poisson), noise_index must be NULL.  The batched and multi-point
 * entries refuse it. */
int obe_model_compile_likelihood(const char* builtin_name, const char* model_source, const char* model_entry,
                                 int n_settings, int n_params, int n_model_params, int n_constants,
                                 int n_channels, const char* likelihood, const char* likelihood_source,
                                 const char* likelihood_entry, obe_model_t* out, char* log, size_t log_len);
int obe_model_info(obe_model_t m, int* n_settings, int* n_model_params, int* n_constants,
                   int* n_channels, int* n_params);
void obe_model_free(obe_model_t m);

/* ---- inference half --------------------------------------------------------------------- */
/* ParticlePDF.__init__/set_pdf (particlepdf.py:121,163-171): weights <- 1/n, stats reset. */
int obe_set_uniform(const obe_cloud_t* c, void* stream);

/* OptBayesExpt.pdf_update without the resample (obe_base.py:381-394):
 *   eval_over_all_parameters (obe_base.py:320) -> likelihood (obe_base.py:451-461 |
 *   obe_noiseparam.py:110-120) -> _normalized_product (particlepdf.py:136-139), plus N_eff
 *   (particlepdf.py:243-244) and the moments of mean/covariance/std (particlepdf.py:173-214),
 *   all in one pass over the cloud.  sigma==NULL with noise_index!=NULL selects the
 *   noise-parameter likelihood.  n_lik_channels = channels that enter the product (zip
 *   truncation).  choke: pass use_choke=0 for choke=None.  pivot[d]: shift for the moment
 *   accumulators (any point near the mean; the previous mean). */
int obe_update(obe_model_t m, const obe_cloud_t* c, const double* setting, const double* constants,
               const double* y_meas, const double* sigma, const int32_t* noise_index,
               int n_lik_channels, int use_choke, double choke, const double* pivot, void* stream);
/* pdf_update(record, y_model_data) (obe_base.py:374-385): model output supplied, (C, ld_y). */
int obe_update_from_y(const obe_cloud_t* c, const double* y_model_dev, int64_t ld_y, int n_channels,
                      const double* y_meas, const double* sigma, const int32_t* noise_index,
                      int n_lik_channels, int use_choke, double choke, const double* pivot,
                      void* stream);
/* obe_update_from_y with the likelihood of the model handle m (obe_update_from_y itself for a
 * Gaussian handle). */
int obe_update_from_y_model(obe_model_t m, const obe_cloud_t* c, const double* y_model_dev, int64_t ld_y,
                            int n_channels, const double* y_meas, const double* sigma,
                            const int32_t* noise_index, int n_lik_channels, int use_choke, double choke,
                            const double* pivot, void* stream);
/* ParticlePDF.bayesian_update(likelihood) (particlepdf.py:216-231): likelihood supplied, (n). */
int obe_update_from_likelihood(const obe_cloud_t* c, const double* likelihood_dev,
                               const double* pivot, void* stream);
/* Recompute tile sums, CDF prefix and moments from the current weights (after the caller wrote
 * weights_dev directly: set_pdf(weights=...), `pdf.particle_weights = ...`), optionally
 * applying enforce_parameter_constraints as data: bit j of mask_le zeroes weights where
 * x_j <= 0 (obe_noiseparam.py:67-71), of mask_lt where x_j < 0 (lockin_of_coil.py:120-128).
 * noise_index (may be NULL) selects the rows whose weighted mean square is accumulated
 * (yvar_noise_model, obe_noiseparam.py:132-136). */
int obe_refresh(const obe_cloud_t* c, uint32_t mask_le, uint32_t mask_lt, const int32_t* noise_index,
                int n_noise, const double* pivot, int renormalise, void* stream);
/* Copy the stats block to host memory (synchronises the stream). */
int obe_fetch_stats(const obe_cloud_t* c, double* stats_host, void* stream);
/* After a systematic resample the weights are IMPLICIT (stats[62] = 1/n_total > 0 and weights_dev is
 * not written: the next update never reads it).  Call this before touching weights_dev directly. */
int obe_materialize_weights(const obe_cloud_t* c, void* stream);
/* Normalised weights (t * INVS, nan_to_num) into out_dev (n). particle_weights getter. */
int obe_normalized_weights(const obe_cloud_t* c, double* out_dev, void* stream);

/* ---- posterior summaries: quantiles and marginal histograms (csrc/obe_summary.cuh) ---------- */
/* Read-only: the cloud, its weights and stats are not written.  Mass is u64 fixed point: a particle of
 * normalised weight w (as obe_normalized_weights) carries wq = rint(w * 2^62); particles with wq == 0 are left
 * out everywhere.  Integer sums make every result independent of the grid and of the run.  Each call ends
 * with one stream synchronisation (the read of its small result into HOST memory).  params: host array of
 * n_params (1..8) parameter rows.  Errors: parameter out of range, bad levels / bins / edges, an empty
 * posterior (sum of wq == 0) and normalised weights that sum to 4 or more (sum of wq >= 2^64).  scratch_dev: device memory of the size the matching query returns. */
size_t obe_quantile_scratch_bytes(int n_params, int n_q);
size_t obe_histogram_scratch_bytes(int n_params, int bins);
size_t obe_histogram2d_scratch_bytes(int bins_x, int bins_y);
/* Streaming passes over the cloud that this thread's last summary call made (range pass included). */
int obe_summary_passes(void);
/* out[r * n_q + i]: the smallest coordinate x* of row params[r] with sum{wq : x <= x*} >= max(1, ceil(q_i W)),
 * W = sum wq (exact).  q: n_q (1..16) levels in [0, 1].  q = 0 gives the minimum and q = 1 the maximum of the
 * positive-weight particles; a zero answer is +0.0. */
int obe_quantile(const obe_cloud_t* c, const int32_t* params, int n_params, const double* q, int n_q,
                 void* scratch_dev, double* out, void* stream);
/* lo_out / hi_out[r]: min / max coordinate of the positive-weight particles of row params[r] (the automatic
 * histogram range).  scratch_dev: obe_histogram_scratch_bytes(n_params, 1) bytes. */
int obe_summary_range(const obe_cloud_t* c, const int32_t* params, int n_params, void* scratch_dev, double* lo_out,
                      double* hi_out, void* stream);
/* Weighted 1-D histograms with np.histogram's uniform-bin rule.  edges: host (n_params, bins + 1), each row
 * non-decreasing, finite, edges[0] < edges[bins]; bins 1..4096.  mass_out / count_out (count_out may be NULL):
 * host (n_params, bins) u64 sums of wq and particle counts. */
int obe_histogram(const obe_cloud_t* c, const int32_t* params, int n_params, const double* edges, int bins,
                  void* scratch_dev, uint64_t* mass_out, uint64_t* count_out, void* stream);
/* Joint histogram of rows param_x, param_y with np.histogram2d's rule; mass_out / count_out: host
 * (bins_x, bins_y), bins_x * bins_y <= 65536. */
int obe_histogram2d(const obe_cloud_t* c, int param_x, int param_y, const double* xedges, int bins_x,
                    const double* yedges, int bins_y, void* scratch_dev, uint64_t* mass_out, uint64_t* count_out,
                    void* stream);

/* ---- weighted draws: Generator.choice(p=w) (particlepdf.py:330-331) ---------------------- */
/* Canonical normalised CDF of the weights into cdf_dev (n). */
int obe_cdf(const obe_cloud_t* c, double* cdf_dev, void* stream);
/* idx[i] = #{k : cdf[k] <= u[i]} clamped to n-1  (searchsorted(cdf, u, 'right')). */
int obe_search(const obe_cloud_t* c, const double* cdf_dev, const double* u_dev, int64_t m,
               int64_t* idx_dev, void* stream);
/* randdraw(K) (particlepdf.py:312-345) without materialising the CDF: K uniforms (host),
 * draws_dev (d, K) row-major, idx_dev (K) optional. */
int obe_draw(const obe_cloud_t* c, const double* u_host, int k, double* draws_dev, int64_t* idx_dev,
             void* stream);

/* ---- resample (particlepdf.py:260-310) --------------------------------------------------- */
/* Gather + Liu-West jitter for given ancestors (reference-parity, multinomial mode):
 *   out[:, i] = in[:, idx[i]] + z[i, :] @ factor ; optional a*out + (1-a)*mean ; w_out = 1/n.
 * factor (d*d row-major) and mean (d) on the host; z_dev (n, d) particle-major standard
 * normals, or NULL to generate them on device (Philox4x32-10, seed, epoch). */
int obe_gather_jitter(const obe_cloud_t* in, const obe_cloud_t* out, const int64_t* idx_dev,
                      const double* factor, const double* mean, const double* z_dev, uint64_t seed,
                      uint32_t epoch, double a_param, int scale, void* stream);
/* Systematic resample (fast path): comb u_i = (i + u0)/n searched in the canonical CDF (plan +
 * ancestors kernels; the uint32 ancestors live in out->scratch_dev), then gather, jitter, implicit
 * weight reset in one elementwise kernel with coalesced writes.  Shards of < 2^32 particles.
 * factor/mean NULL =>
 * Cholesky factor of (1-a^2)*cov and the mean are taken from in->stats_dev on the device.
 * idx_out_dev / z_out_dev (optional) receive the ancestors and the normals used. */
int obe_resample_systematic(const obe_cloud_t* in, const obe_cloud_t* out, double u0,
                            const double* factor, const double* mean, uint64_t seed, uint32_t epoch,
                            double a_param, int scale, int64_t* idx_out_dev, double* z_out_dev,
                            void* stream);

/* ---- sharded clouds (one process per GPU; particles split into contiguous shards) ---------- */
/* The same kernels for one shard of a cloud of n_total particles: this shard's particles own
 * the global comb slots [slot_begin, slot_end) (= out->n of them, which may differ from in->n: shard
 * lengths float, no particle ever crosses NVLink); cdf_offset = summed weight of the lower-ranked
 * shards, cdf_total = global weight; factor/mean are the GLOBAL Liu-West factor and mean (host).
 * RNG counters are global slot numbers, so the jitter does not depend on the number of shards. */
int obe_resample_systematic_sharded(const obe_cloud_t* in, const obe_cloud_t* out, double u0,
                                    int64_t n_total, int64_t slot_begin, int64_t slot_end,
                                    double cdf_offset, double cdf_total, int last_shard,
                                    const double* factor, const double* mean, uint64_t seed,
                                    uint32_t epoch, double a_param, int scale, int64_t* idx_out_dev,
                                    double* z_out_dev, void* stream);
/* Device-resident shard plan (no host round-trip between update, collective and resample):
 * gathered_stats_dev = the all-gathered (world, OBE_STATS_DOUBLES) stats blocks.  Writes plan_dev
 * (OBE_PLAN_DOUBLES doubles: CDF offset/total, slot bounds of every shard, global moments, Cholesky
 * Liu-West factor, pre/post-resample shard totals), the global normaliser into local->stats_dev and
 * the post-resample length of this shard into out->n_dev.  lazy=1: weights are un-normalised. */
#define OBE_PLAN_DOUBLES 512
#define OBE_PLAN_GSTATS 352     /* offset of the combined (global) stats block inside the plan  */
#define OBE_PLAN_COUNTS 416     /* offset of the post-resample shard lengths                    */
#define OBE_PLAN_OVERFLOW 9     /* 1.0 if this shard outgrew its buffer capacity                */
int obe_shard_plan(const double* gathered_stats_dev, int rank, int world, int d, double u0,
                   int64_t n_total, double a_param, int lazy, const obe_cloud_t* local,
                   const obe_cloud_t* out, double* plan_dev, void* stream);
/* ---- peer exchange over NVLink (optional replacement of the small NCCL collectives) -------------
 * Every rank owns one buffer of obe_peer_bytes() (cudaMalloc + CUDA IPC); peer_bufs[g] is rank g's buffer as
 * mapped into THIS process (peer_bufs[rank] = the local one).  Producing kernels write their few doubles
 * straight into every peer's buffer and raise a system-scope flag carrying `epoch`; consumers spin on their
 * own buffer (~20 s timeout -> the plan's overflow word reads 2).  `epoch` is a per-kind counter starting at 1
 * that every rank advances identically; slots are double-buffered by its parity.  1..16 ranks. */
size_t obe_peer_bytes(void);
int obe_peer_alloc(void** dev_ptr, unsigned char* handle64);         /* handle64: cudaIpcMemHandle_t bytes */
int obe_peer_open(const unsigned char* handle64, void** dev_ptr);
int obe_peer_close(void* dev_ptr);
int obe_peer_free(void* dev_ptr);
/* obe_shard_plan with the stats all-gather fused in: publish local->stats_dev to every peer, wait, plan. */
int obe_shard_plan_peer(void* const* peer_bufs, int rank, int world, uint64_t epoch, int d, double u0,
                        int64_t n_total, double a_param, int lazy, const obe_cloud_t* local,
                        const obe_cloud_t* out, double* plan_dev, void* stream);
/* obe_draw_planned with the exchange fused in: owners write their draws into every rank's buffer; a
 * one-CTA kernel then waits for all ranks and copies the (d, k) draws into draws_dev.  k * d <= 1024. */
int obe_draw_planned_peer(const obe_cloud_t* c, const double* u_host, int k, void* const* peer_bufs,
                          int rank, int world, uint64_t epoch, const double* plan_dev, int post,
                          double* draws_dev, void* stream);
/* obe_resample_systematic_sharded with every shard parameter read from plan_dev on the device. */
int obe_resample_systematic_planned(const obe_cloud_t* in, const obe_cloud_t* out, const double* plan_dev,
                                    int64_t n_total, uint64_t seed, uint32_t epoch, double a_param,
                                    int scale, void* stream);
/* Early select (obe_base.py:733-756 opt_setting right after particlepdf.py:260-310 resample): the K draws of the
 * design half are offspring of the resample, so they can be produced from the resample PLAN before the cloud is
 * streamed, and the utility pass can overlap the resample on a second stream.
 *   obe_resample_defer(1)   the calling thread's next obe_resample_systematic[_sharded|_planned] call launches only
 *                           its plan kernel and parks the streaming kernel (0 disarms / drops a parked one);
 *   obe_resample_pick       draw q = the offspring in global slot min(floor(u[q] * n_total), n_total - 1), computed by
 *                           the work unit that owns the slot; (d, k) row-major into draws_dev.  Values are bit-identical
 *                           to what obe_resample_emit stores in that slot.  Sharded: peer_bufs != NULL exchanges the
 *                           draws by peer writes (as obe_draw_planned_peer); peer_bufs == NULL writes zeros for draws
 *                           other shards own (all-reduce(sum) completes them);
 *   obe_resample_emit       launches the parked streaming kernel.
 *   obe_stream_fork/join    side waits for main / main waits for side (cached events, no host synchronisation). */
int obe_resample_defer(int on);
int obe_resample_pick(const double* u_host, int k, double* draws_dev, void* const* peer_bufs, int rank, int world,
                      uint64_t epoch, void* stream);
int obe_resample_emit(void* stream);
int obe_stream_fork(void* main_stream, void* side_stream);
int obe_stream_join(void* main_stream, void* side_stream);
/* One whole cycle in one call: pdf_update (obe_base.py:340-399) -> [forced systematic resample,
 * particlepdf.py:260-310] -> [enforce_parameter_constraints as masks] -> utility + argmax of opt_setting
 * (obe_base.py:628-655,733-756), enqueued with no host work between the launches (a small-cloud cycle is bound by
 * the host, not by the GPU).  It chains the entry points above exactly as the Python classes do:
 *   obe_update
 *   [plan_dev: obe_shard_plan_peer]                                (sharded cloud, peer exchange)
 *   resample != 0: obe_resample_systematic / _planned;  with select != 0 and no constraint mask the emission is
 *                  deferred and the K draws are picked from the plan (obe_resample_pick) so that obe_utility runs
 *                  on side_stream while the cloud streams on `stream`;
 *                  mask_le | mask_lt != 0: obe_refresh(alt, masks) after the resample
 *   select != 0 (not early): obe_draw / obe_draw_planned_peer on the live cloud, then obe_utility.
 * `cloud` is the live buffer, `alt` the output of the resample (the CALLER swaps them after a resampling cycle).
 * The struct is plain data: fill it once, update the per-cycle fields (setting, y_meas, sigma, pivot, u0, epoch,
 * u[], peer epochs) and call. */
typedef struct obe_cycle {
    obe_model_t model;
    const obe_cloud_t* cloud;
    const obe_cloud_t* alt;
    const double* constants;            /* host */
    double setting[OBE_MAX_SETTINGS];
    double y_meas[OBE_MAX_CHANNELS];
    double sigma[OBE_MAX_CHANNELS];     /* used when has_sigma */
    double pivot[OBE_MAX_PARAMS];
    int32_t noise_index[OBE_MAX_CHANNELS];
    int32_t has_sigma, has_noise_index, n_lik_channels, use_choke;
    double choke;
    int32_t resample, scale;            /* resample: 0 = no, 1 = forced systematic, 2 = decided on the device (below) */
    double u0, a_param;
    uint64_t seed;
    uint32_t epoch, mask_le, mask_lt;
    int32_t n_noise;                    /* rows of noise_index the refresh accumulates (noise-parameter engines) */
    /* sharded (plan_dev != NULL): peer exchange only */
    double* plan_dev;
    void* const* peer_bufs;
    int32_t rank, world;
    uint64_t epoch_stats, epoch_draws;
    int64_t n_total;
    /* selection */
    int32_t select, k;
    double u[128];
    double* draws_dev;                  /* (d, k) */
    const double* settings_dev;
    int64_t lds, n_settings;
    double var_noise[OBE_MAX_CHANNELS];
    int32_t noise_from_stats;           /* 1: var_noise is ignored, the noise sums of the live stats block are used */
    int32_t method, log_form, pad0;
    const double* cost_dev;
    const double* kld_noise_dev;
    double* utility_dev;
    void* best_dev;
    void* select_scratch_dev;
    void* stream;
    void* side_stream;                  /* NULL: no overlap, everything on `stream` */
    /* resample == 2: the resample test of particlepdf.py:236-258 is decided ON THE DEVICE by the update kernel
     * (stats[OBE_STAT_FIRED] = N_eff < 0.1 N || N_eff / N < resample_threshold); plan, pick and streaming resample run
     * gated on it, the plain K draws on its complement, the utility pass on whichever draws exist.  Whole clouds only,
     * select != 0, no constraint masks.  The caller reads the outcome from stats_host[OBE_STAT_FIRED] after it has
     * synchronised, and swaps cloud / alt if it fired. */
    double resample_threshold;
    /* optional PINNED host blocks, filled by asynchronous copies behind the cycle's kernels on `stream`:
     * stats_host (64 doubles) <- the stats block the update wrote (stats_src_dev, default cloud->stats_dev);
     * best_host (16 bytes) <- (int64 index, double value) of the argmax, when select != 0.  Valid after
     * obe_stream_sync(stream).  When the blocks are device-visible (cudaHostAlloc / cudaHostRegister memory under
     * UVA) the update and utility kernels store into them directly and no copy is enqueued at all. */
    void* stats_host;
    const double* stats_src_dev;
    void* best_host;
    /* 0: the whole cycle.  1: the update only; 2: everything after it (same struct, completed in between): a
     * small-cloud closed loop gets its first kernel on the device before the host has drawn the uniforms and filled
     * in the selection half. */
    int32_t phase, pad1;
    /* optional completion word (8 bytes of the same kind of pinned host memory as best_host; needs select != 0 and
     * device-visible blocks): the utility kernel stores `seq` there after the argmax pair has landed, so a closed loop
     * can POLL it instead of synchronising the stream (kernels enqueued behind the utility pass -- gated-off launches,
     * the streaming kernel of a resampling cycle -- no longer delay the host).  stats_host is complete when the word
     * appears (the update kernel wrote it, or its copy was enqueued ahead of the selection). */
    uint64_t seq;
    void* seq_host;
} obe_cycle_t;
int obe_cycle(const obe_cycle_t* c);
/* cudaStreamSynchronize(stream): what a closed loop waits on before it reads best_host / stats_host
 * (the reference's opt_setting returns a host value, obe_base.py:733-756). */
int obe_stream_sync(void* stream);
/* randdraw(K) over a sharded cloud: this rank writes the draws it owns (per plan_dev; post=1 uses the
 * post-resample shard totals) and zeros elsewhere; an all-reduce(sum) of draws_dev completes it. */
int obe_draw_planned(const obe_cloud_t* c, const double* u_host, int k, double* draws_dev,
                     const double* plan_dev, int post, void* stream);
/* weights <- 1/n_total for one shard of a cloud of n_total particles. */
int obe_set_uniform_total(const obe_cloud_t* c, int64_t n_total, void* stream);
/* Host twin of the device comb count #{i in [0,n_total) : (i + u0) * (1/n_total) < c}: shard
 * boundaries slot_begin/slot_end are obe_comb_count(cdf_offset / cdf_total ...) evaluated identically
 * on every rank. */
int64_t obe_comb_count(double c, double u0, int64_t n_total);
/* obe_draw writing its m draws into columns of a wider (d, ld_draws) matrix. */
int obe_draw_strided(const obe_cloud_t* c, const double* u_host, int m, double* draws_dev, int ld_draws,
                     int64_t* idx_dev, void* stream);

/* ---- design half ------------------------------------------------------------------------ */
/* utility_variance (obe_base.py:628-655) over the whole grid + argmax of opt_setting
 * (obe_base.py:748).  draws_dev (d, K); settings_dev (s, lds); var_noise[C] host or NULL to use
 * the noise-parameter accumulators of c_stats_dev (obe_noiseparam.py:132-136); cost_dev (S) or
 * NULL (cost_estimate, obe_base.py:566-577); method 0 = variance, 1 = max-min
 * (obe_base.py:602-626), 2 = pseudo (spacing-entropy of the K outputs, obe_base.py:491-518,657-686),
 * 3 = full KLD (obe_base.py:688-720; kld_noise_dev = (K, C) noise samples, single channel);
 * log_form=1 gives log(1 + var/sigma^2).  utility_dev (S) out; best_dev: int64 index then double
 * value (16 bytes). */
int obe_utility(obe_model_t m, const double* draws_dev, int k, const double* settings_dev,
                int64_t lds, int64_t n_settings, const double* constants, const double* var_noise,
                const double* stats_dev, const double* cost_dev, int method, int log_form,
                const double* kld_noise_dev, double* utility_dev, void* best_dev,
                void* select_scratch_dev, void* stream);
/* good_setting (obe_base.py:778-789): index drawn with p ~ nan_to_num(U**pickiness), given its
 * uniform.  idx_dev: int64. */
int obe_pick(const double* utility_dev, int64_t n_settings, double pickiness, double u,
             int64_t* idx_dev, void* select_scratch_dev, void* stream);
/* Multi-point update (the sweeper's pdf_update, demos/sweeper/obe_sweeper.py:87-101: one Bayesian update
 * per point of a sweep, resample test after each): n_points <= 128 records in ONE pass over the cloud.
 * records_dev: (n_points, 12) doubles, row = [0:4) setting, [4:8) y, [8:12) 1/sigma (known-sigma models;
 * ignored when noise_index selects sigma from the particles).  The un-normalised product of the
 * likelihoods goes to weights_out_dev (another row of c->ld doubles, NOT c->weights_dev); lik_scale[c]
 * (may be NULL) multiplies every point's likelihood of channel c -- a particle-independent factor that
 * keeps long sweeps from underflowing.  sums_dev: (n_points, 2) out = sum t_m, sum t_m^2 after every
 * point; result_dev: 2 doubles out = index of the FIRST point after which N_eff / n_total < threshold
 * (the reference's resample test, particlepdf.py:236-258; -1 if none, threshold <= 0 disables) and that
 * ratio.  The caller commits weights_out when result is -1 or n_points-1 (swap the rows, obe_refresh)
 * and otherwise re-runs the first result+1 points, resamples, and continues. */
int obe_update_multi(obe_model_t m, const obe_cloud_t* c, double* weights_out_dev,
                     const double* records_dev, int n_points, const double* constants,
                     const int32_t* noise_index, int n_lik_channels, const double* lik_scale,
                     int use_choke, double choke, double threshold, int64_t n_total,
                     double* sums_dev, double* result_dev, void* stream);
/* Sweeper selection (demos/sweeper/obe_sweeper.py:118-162, sweep_utility + opt_setting): cumsum of the
 * point utility along the swept setting; every (start, stop) pair of setting indices is worth
 * (cum[stop] - cum[start]) / ((stop - start) + cost_of_new_sweep); argmax with np.argmax semantics.
 * pairs_dev: (n_pairs, 2) int32 = start_stop_indices; cumsum_dev: (n_settings) out;
 * pair_utility_dev: (n_pairs) out or NULL; best_dev: int64 pair index then double value (16 bytes).
 * The pair utilities are a plain device vector: obe_pick on them is the sweeper's good_setting. */
int obe_sweep_utility(const double* utility_dev, int64_t n_settings, const int32_t* pairs_dev,
                      int64_t n_pairs, double cost_of_new_sweep, double* cumsum_dev,
                      double* pair_utility_dev, void* best_dev, void* select_scratch_dev, void* stream);
/* eval_over_all_parameters (obe_base.py:298-320) -> y_dev (C, ldy) */
int obe_eval_parameters(obe_model_t m, const obe_cloud_t* c, const double* setting,
                        const double* constants, double* y_dev, int64_t ldy, void* stream);
/* eval_over_all_settings (obe_base.py:322-338) -> y_dev (C, ldy) */
int obe_eval_settings(obe_model_t m, const double* settings_dev, int64_t lds, int64_t n_settings,
                      const double* params, const double* constants, double* y_dev, int64_t ldy,
                      void* stream);

/* ---- batched independent instances (BASELINE config c5: B engines x n particles each) -------- */
/* One SoA cloud: instance b owns particles [b*np, b*np + n) of (d, ld) arrays, np = n rounded up to
 * whole tiles, ld >= n_inst*np.  Two buffers; cur_dev[b] says which one holds instance b (a resample
 * writes the other and flips it).  Per instance: record (setting[4], y_meas[4], sigma[4]), pivot[8],
 * stats block, CDF prefix row (tiles+1), last chosen setting index, resample flag, Philox epoch.
 * Every call below is one or two launches over ALL instances; nothing returns to the host. */
typedef struct obe_batch {
    double* particles_dev[2];
    double* weights_dev[2];
    int32_t* cur_dev;          /* (B)                      */
    double* tile_sums_dev;     /* (B * tiles)              */
    double* tile_prefix_dev;   /* (B * (tiles + 1))        */
    double* stats_dev;         /* (B * OBE_STATS_DOUBLES)  */
    double* pivot_dev;         /* (B * 8)                  */
    double* record_dev;        /* (B * 12)                 */
    int64_t* last_idx_dev;     /* (B)                      */
    double* best_val_dev;      /* (B)                      */
    int32_t* flag_dev;         /* (B) 1 = must resample    */
    int32_t* list_dev;         /* (B) scratch              */
    int32_t* n_list_dev;       /* (1) scratch              */
    uint32_t* epoch_dev;       /* (B) resamples so far     */
    int64_t n_inst, n, np, ld;
    int32_t d, tiles;
} obe_batch_t;
/* weights <- 1/n, buffers/flags reset, tile sums + prefix + moments of every instance. */
int obe_batch_init(const obe_batch_t* b, const int32_t* noise_index, int n_noise, void* stream);
/* pdf_update of every instance (obe_base.py:381-394) with its own record; use_last=1 takes each
 * instance's setting from settings_dev[:, last_idx[b]] (closed loop without a host round-trip).
 * Writes flag_dev[b] = resample decision of particlepdf.py:243-258 (or 1 when force_resample). */
int obe_batch_update(obe_model_t m, const obe_batch_t* b, const double* settings_dev, int64_t lds, int use_last,
                     const double* constants, const int32_t* noise_index, int n_lik_channels, int use_choke,
                     double choke, double resample_threshold, int force_resample, void* stream);
/* systematic resample (particlepdf.py:260-310) of the flagged instances; comb offset = uniform number
 * u0_index of the instance's stream in this cycle; normals from Philox(seed + b, epoch_b); offspring
 * violating the masks get weight 0 (enforce_parameter_constraints); then their stats are rebuilt. */
int obe_batch_resample(const obe_batch_t* b, double a_param, int scale, uint64_t seed, uint64_t uniform_seed,
                       uint32_t cycle, int u0_index, uint32_t mask_le, uint32_t mask_lt, const int32_t* noise_index,
                       int n_noise, void* stream);
int obe_batch_refresh(const obe_batch_t* b, uint32_t mask_le, uint32_t mask_lt, const int32_t* noise_index, int n_noise,
                      void* stream);
/* opt_setting of every instance (obe_base.py:733-756): K draws (uniforms 0..K-1 of the instance's
 * stream in this cycle), variance utility, argmax -> last_idx_dev / best_val_dev.  cost_change > 0
 * applies the sticky cost of demos/lockin/lockin_of_coil.py:135-152. */
int obe_batch_select(obe_model_t m, const obe_batch_t* b, const double* settings_dev, int64_t lds, int64_t n_settings,
                     const double* constants, int k, const double* var_noise, double cost_change, uint64_t uniform_seed,
                     uint32_t cycle, int method, int log_form, double* utility_dev, void* stream);
/* On-device MeasurementSimulator (obe_utils.py:8-53) for the batched engines: instance b measures at the
 * setting it chose last, y_c = model_c(setting, true_params[:, b], constants) + noise_c * z_c, with z the
 * library's Philox/Box-Muller normals (counter b, key seed, epoch cycle), and its record row is filled in
 * on the device (setting, y, and sigma = noise level when write_sigma != 0).  true_params_dev: (np_model,
 * ld_true) SoA; noise_level: host array of n_channels, or noise_level_dev: (B) per instance.  Followed by
 * obe_batch_update(use_last = 1) a closed loop never touches the host. */
int obe_batch_simulate(obe_model_t m, const obe_batch_t* b, const double* settings_dev, int64_t lds,
                       const double* true_params_dev, int64_t ld_true, const double* constants,
                       const double* noise_level, const double* noise_level_dev, uint64_t seed,
                       uint32_t cycle, int write_sigma, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* OBE_B200_H */
