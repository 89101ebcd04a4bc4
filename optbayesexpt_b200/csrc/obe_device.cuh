// obe_device.cuh -- device-side core of the B200 particle-filter path.
//
// Freestanding on purpose (no #include): this file is compiled twice -- by nvcc into
// libobe_b200.so for the built-in model functors, and by NVRTC at run time (sm_100a cubin)
// when a user supplies CUDA source for model_function.  Everything that depends on the
// model functor lives here as a template body; the model-independent kernels live in
// obe_b200.cu.
//
// Data layout in HBM (all fp64, SoA):
//   particles   (d, ld)   one contiguous row per parameter, ld >= n, rows 16 B aligned
//   weights     (n)       UN-normalised weights t_i; the normaliser lives in stats[]
//   tile_sums   (n_tiles) sum of t over each canonical tile of OBE_TILE particles
//   tile_prefix (n_tiles+1) exclusive prefix of tile_sums; [n_tiles] is the CDF total
//   stats       (OBE_STATS_LEN) device-resident scalars, see OBE_ST_* below
//
// Reference semantics implemented by obe_update_body (optbayesexpt v1.2.0):
//   obe_base.py:320      y = model(one_setting, particles, cons)
//   obe_base.py:263-271  L = exp(-((y - y_meas)/sigma)**2 / 2) / sigma      (per channel)
//   obe_base.py:451-461  product over channels (zip truncation), optional L**choke
//   obe_noiseparam.py:110-120  sigma_c = particles[noise_index[c]]
//   particlepdf.py:136-139     w <- nan_to_num(nan_to_num(w*L) / sum)
//   particlepdf.py:243-244     N_eff = 1/sum(w^2)
//   particlepdf.py:173-214     mean / covariance / std   (pivot-shifted moments, same pass)
#ifndef OBE_DEVICE_CUH
#define OBE_DEVICE_CUH

#define OBE_TILE 2048
#define OBE_THREADS 256
#define OBE_EPT 8 /* elements per thread per tile */
#define OBE_MAX_DIMS 8
#define OBE_MAX_CH 4
#define OBE_MAX_SET 4
#define OBE_MAX_CONS 8
#define OBE_MAX_DRAWS 128

// stats block (doubles)
#define OBE_ST_TOTAL 0   /* canonical sum of t = tile_prefix[n_tiles] */
#define OBE_ST_INVS 1    /* multiplier that normalises t (1/total, or exactly 1 after a resample) */
#define OBE_ST_SUMSQ 2   /* sum t^2 */
#define OBE_ST_NEFF 3    /* total^2 / sumsq */
#define OBE_ST_M1 4      /* [8]  sum t (x_j - pivot_j) */
#define OBE_ST_M2 12     /* [36] sum t (x_j - p_j)(x_k - p_k), packed j<=k row-major */
#define OBE_ST_PIVOT 48  /* [8]  pivot used */
#define OBE_ST_NOISE 56  /* [4]  sum t sigma_c^2 (noise-parameter channels) */
#define OBE_ST_SUMT 60   /* plain (non-canonical) sum of t from the same pass */
#define OBE_ST_NZERO 61  /* number of particles zeroed by the constraint mask */
#define OBE_ST_UNIFORM 62 /* > 0: the weights are IMPLICIT, every live particle weighs this much (set by a
                            systematic resample, which then never writes the weight row; cleared by the
                            next update, which never reads it) */
#define OBE_ST_FIRED 63  /* 1.0: the resample test of the update that wrote this block fires (device predicate of
                            obe_cycle's resample == 2; 0 when the update was not asked to decide) */
#define OBE_STATS_LEN 64
#define OBE_NACC_MAX (2 + OBE_MAX_DIMS + 36 + OBE_MAX_CH + 1)

// shard plan block (doubles; integers stored exactly), written by k_shard_plan
#define OBE_PL_OFFSET 0      /* summed weight of the lower-ranked shards */
#define OBE_PL_TOTAL 1       /* global weight total */
#define OBE_PL_U0 2
#define OBE_PL_NTOTAL 3
#define OBE_PL_SLOT0 4       /* first global comb slot owned by this shard */
#define OBE_PL_SLOT1 5
#define OBE_PL_LAST 6        /* 1 on the shard holding the global last particle */
#define OBE_PL_RANK 7
#define OBE_PL_WORLD 8
#define OBE_PL_OVERFLOW 9    /* 1 if a shard outgrew its capacity */
#define OBE_PL_POST_TOTAL 10 /* sum of the post-resample shard totals */
#define OBE_PL_FACTOR 16     /* [64] Liu-West factor, z @ F convention */
#define OBE_PL_MEAN 80       /* [8] */
#define OBE_PL_PRE_OFF 96    /* [64] shard offsets of the CURRENT weights */
#define OBE_PL_PRE_TOT 160   /* [64] shard totals of the current weights */
#define OBE_PL_POST_OFF 224  /* [64] the same after the planned resample (uniform weights) */
#define OBE_PL_POST_TOT 288  /* [64] */
#define OBE_PL_GSTATS 352    /* [64] combined stats block (global TOTAL, INVS, SUMSQ, NEFF, M1, M2, ...) */
#define OBE_PL_COUNTS 416    /* [64] post-resample shard lengths */
#define OBE_PLAN_LEN 512
#define OBE_MAX_SHARDS 64

// likelihood source for obe_update_body
#define OBE_SRC_MODEL 0  /* evaluate the model functor */
#define OBE_SRC_Y 1      /* y_model supplied (pdf_update(..., y_model_data)) */
#define OBE_SRC_LIK 2    /* likelihood supplied (ParticlePDF.bayesian_update) */
#define OBE_SRC_NONE 3   /* no likelihood: moments / tile sums / constraint mask only */
#define OBE_SRC_DRIFT 4  /* no likelihood: the random-walk step of the particles (obe_drift), then their moments */

struct ObeUpdateArgs {
    const double* particles;
    long long ld;
    long long n;
    double* weights;
    double* tile_sums;
    double* partials;        // [gridDim.x][OBE_NACC_MAX]
    unsigned int* counter;   // zero on entry, zero again on exit
    double* stats;
    const double* y_model;   // OBE_SRC_Y: (n_channels, ld_y)
    long long ld_y;
    const double* lik;       // OBE_SRC_LIK: (n)
    const long long* n_dev;  // optional: live particle count on the device (n is then an upper bound)
    double* tile_prefix;     // the last block also scans the tile sums into the CDF prefix ...
    int renormalise;         // ... and sets the normaliser to 1/total (1) or to exactly 1 (0)
    int scale_in;            // 1: w_in = nan_to_num(t * stats[INVS]); 0: raw t
    int write_weights;
    int n_lik_channels;      // min(C, len(y_meas), len(sigma))  -- zip truncation
    int use_choke;
    unsigned int mask_le;    // bit j: weight <- 0 where x_j <= 0   (obe_noiseparam.py:67-71)
    unsigned int mask_lt;    // bit j: weight <- 0 where x_j <  0   (lockin_of_coil.py:120-128)
    double choke;
    double setting[OBE_MAX_SET];
    double cons[OBE_MAX_CONS];
    double y_meas[OBE_MAX_CH];
    double inv_sigma[OBE_MAX_CH]; // 1/sigma_c for a known sigma
    int noise_idx[OBE_MAX_CH];    // >=0: sigma_c is that particle row
    int n_noise;                  // number of noise-parameter channels (0: known sigma)
    double pivot[OBE_MAX_DIMS];
    // device-side resample test (particlepdf.py:236-258), decided by the block that finishes the stats:
    // gate_n > 0: stats[FIRED] = (N_eff < 0.1 gate_n) || (N_eff / gate_n < gate_thr), N_eff = 1 / (sumsq * invs^2)
    double gate_thr;
    double gate_n;
    double* stats_out2;      // optional copy of the finished stats block into device-visible PINNED HOST memory
};

struct ObeUtilityArgs {
    const double* draws;     // (d_model, K) row-major
    int k;
    const double* settings;  // (s, lds)
    long long lds;
    long long n_settings;
    const double* cost;      // (S) or null
    const double* stats;     // noise-parameter mode: var_n[c] = stats[NOISE+c]/stats[SUMT]
    double* utility;         // (S) out
    double* part_val;        // [gridDim.x]
    long long* part_idx;     // [gridDim.x]
    unsigned int* counter;
    long long* best_idx;     // out
    double* best_val;        // out
    int noise_from_stats;
    int log_form;
    int method;              // 0 variance, 1 max-min, 2 pseudo (entropy), 3 full KLD
    int lanes;               // variance utility: lanes per setting (1: one thread walks all K draws)
    int cache;               // lanes == 1: the K x NCH model values of a thread's setting are kept in shared memory
                             // between the two passes of the variance (1) instead of being evaluated twice (0)
    const double* kld_noise; // method 3: (K, C) noise values added to the model outputs
    double var_noise[OBE_MAX_CH];
    double cons[OBE_MAX_CONS];
    long long* best_out2;    // optional second destination of the (index, value) pair: device-visible PINNED HOST
                             // memory, so a closed loop needs no copy after the kernel (obe_cycle, best_host)
    unsigned long long* seq_out2;   // optional: after best_out2 is written (system-scope fence), seq_val is stored here --
    unsigned long long seq_val;     // the host polls this word instead of synchronising the stream (obe_cycle, seq_host)
};

struct ObeEvalArgs {
    const double* a;         // particles (d, ld)  | settings (s, lds)
    long long ld;
    long long n;
    double* y;               // (C, ldy)
    long long ldy;
    double fixed[OBE_MAX_DIMS]; // the one setting | the one parameter set
    double cons[OBE_MAX_CONS];
};

// ---------------------------------------------------------------------------------------------
// small helpers
// ---------------------------------------------------------------------------------------------
#define OBE_DBL_MAX 1.7976931348623157e308

// numpy.nan_to_num defaults: nan -> 0, +inf -> DBL_MAX, -inf -> -DBL_MAX
__device__ __forceinline__ double obe_nan_to_num(double x) {
    if (x != x) return 0.0;
    if (x > OBE_DBL_MAX) return OBE_DBL_MAX;
    if (x < -OBE_DBL_MAX) return -OBE_DBL_MAX;
    return x;
}

// IEEE ops that the compiler may not contract into FMAs: the built-in rational models use
// these so their values are bit-identical to numpy's (which never fuses).
__device__ __forceinline__ double obe_mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double obe_add(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double obe_sub(double a, double b) { return __dadd_rn(a, -b); }
__device__ __forceinline__ double obe_div(double a, double b) { return __ddiv_rn(a, b); }

__device__ __forceinline__ double obe_shfl_xor(double v, int m) {
    return __shfl_xor_sync(0xffffffffu, v, m);
}
__device__ __forceinline__ double obe_warp_sum(double v) {
    v += obe_shfl_xor(v, 16);
    v += obe_shfl_xor(v, 8);
    v += obe_shfl_xor(v, 4);
    v += obe_shfl_xor(v, 2);
    v += obe_shfl_xor(v, 1);
    return v;
}

// streaming 16-byte accesses: every particle byte is touched once per pass
__device__ __forceinline__ double2 obe_ld2(const double* p) {
    double2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(r.x), "=d"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ double2 obe_ld2_rw(const double* p) {
    double2 r;
    asm volatile("ld.global.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(r.x), "=d"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ void obe_st2(double* p, double2 v) {
    asm volatile("st.global.L1::no_allocate.v2.f64 [%0], {%1, %2};" ::"l"(p), "d"(v.x), "d"(v.y) : "memory");
}

// Sum of one double over the block; result valid in every thread. `red` holds >= 8 doubles.
__device__ __forceinline__ double obe_block_sum(double v, double* red) {
    v = obe_warp_sum(v);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    double s = red[0];
#pragma unroll
    for (int w = 1; w < OBE_THREADS / 32; ++w) s += red[w];
    return s;
}

// ---------------------------------------------------------------------------------------------
// mbarrier / bulk-copy (TMA engine, 1-D) primitives
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned obe_smem_addr(const void* p) {
    return (unsigned)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void obe_mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(obe_smem_addr(bar)), "r"(count));
}
__device__ __forceinline__ void obe_mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void obe_mbar_arrive(unsigned long long* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(obe_smem_addr(bar)) : "memory");
}
__device__ __forceinline__ void obe_mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(obe_smem_addr(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void obe_mbar_wait(unsigned long long* bar, unsigned parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "OBE_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra OBE_DONE_%=;\n\t"
        "bra OBE_WAIT_%=;\n\t"
        "OBE_DONE_%=:\n\t"
        "}" ::"r"(obe_smem_addr(bar)), "r"(parity)
        : "memory");
}
// global -> shared bulk copy through the TMA engine; completion is signalled on `bar`
__device__ __forceinline__ void obe_bulk_g2s(void* dst_smem, const void* src_gmem, unsigned bytes,
                                             unsigned long long* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            obe_smem_addr(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(obe_smem_addr(bar))
        : "memory");
}
__device__ __forceinline__ void obe_named_bar(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
// Programmatic dependent launch (sm_90+): a kernel launched with the programmatic-stream-serialization attribute may
// start while its predecessor in the stream is still running; it must call obe_grid_dep_wait() before it touches
// anything the predecessor writes (the call returns once the predecessor grid has completed and its writes are
// visible; a no-op for a normal launch).  obe_grid_dep_launch() in the predecessor lets the dependents be scheduled
// from that point on instead of at its exit.  Used along the cycle's chain of small dependent kernels (update ->
// shard plan -> resample plan -> streaming resample) to take their launch latency and prologues off the critical path.
__device__ __forceinline__ void obe_grid_dep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void obe_grid_dep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------
// The fused Bayesian update: a persistent, warp-specialised kernel, one CTA per SM.
//   producer role (thread 0)   for every stage, 1-D bulk copies (TMA engine, cp.async.bulk +
//                              mbarrier complete_tx) of the weight row and the D particle rows of
//                              the next stage of particles into a ring of shared-memory stages,
//                              NST-1 stages ahead -- HBM stays busy while the FP64 pipe works
//   consumers (all 16 warps)   16-byte conflict-free LDS of their columns, release the stage,
//                              model -> likelihood -> weight product -> moments in registers,
//                              coalesced 16-byte stores of the new weights, tile sums through a
//                              barrier.  (A dedicated 17th producer warp would cap the kernel at
//                              96 registers/thread -- 5 warps on one SM sub-partition -- and spill.)
// Across tiles each consumer keeps sum t^2, the pivot-shifted first/second moments and the noise
// accumulators in registers; they are reduced once per block and combined by the last block to
// finish in a fixed order (run-to-run deterministic).
// ---------------------------------------------------------------------------------------------
#define OBE_CONSUMER_WARPS 16
#define OBE_CONSUMER_THREADS (OBE_CONSUMER_WARPS * 32)
#define OBE_UPDATE_THREADS OBE_CONSUMER_THREADS
#define OBE_SMEM_BUDGET (200 * 1024)

template <int D>
struct ObeAcc {
    double sumsq, sumt, nzero;
    double m1[D];
    double m2[D * (D + 1) / 2];
    double noise[OBE_MAX_CH];
};

// numpy.nan_to_num (nan -> 0, +-inf -> +-DBL_MAX): one integer test on the fast path, the rare
// path out of line so that it is a real branch and not ten predicated instructions per particle.
__device__ __noinline__ double obe_nan_to_num_rare(double x) {
    return (x != x) ? 0.0 : (x > 0.0 ? OBE_DBL_MAX : -OBE_DBL_MAX);
}
__device__ __forceinline__ double obe_nan_to_num_fast(double x) {
    if ((((unsigned)__double2hiint(x)) & 0x7fffffffu) >= 0x7ff00000u) x = obe_nan_to_num_rare(x);
    return x;
}

// 1/x to ~1 ulp for finite, normal, non-zero x: hardware seed + two Newton steps, no slow path.
__device__ __forceinline__ double obe_rcp_fast(double x) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    double e = fma(-x, r, 1.0);
    r = fma(r, e, r);
    e = fma(-x, r, 1.0);
    r = fma(r, e, r);
    return r;
}

// Taylor coefficients 1/13! .. 1/2! of exp, in constant memory so each DFMA takes its
// coefficient as a constant-bank operand (immediates cost two extra moves per FMA).
__constant__ double obe_exp_c[12] = {
    1.6059043836821613e-10, 2.08767569878681e-09, 2.505210838544172e-08, 2.755731922398589e-07,
    2.7557319223985893e-06, 2.48015873015873e-05, 1.984126984126984e-04, 1.3888888888888889e-03,
    8.333333333333333e-03, 4.1666666666666664e-02, 1.6666666666666666e-01, 0.5};

// exp(x) for x <= 0 (the Gaussian log-likelihood): k = rint(x/ln2), r = x - k ln2 in two FMAs,
// degree-13 Taylor polynomial on |r| <= ln2/2 (truncation 4e-18), scaling by 2^k through the
// exponent field.  ~2 ulp; results below 2^-1022 flush to 0 (exact would be a denormal weight).
__device__ __forceinline__ double obe_exp_nonpos(double x) {
    const double t = fma(x, 1.4426950408889634, 6755399441055744.0);   // 1.5 * 2^52: round to int
    int k = __double2loint(t);
    const double kf = t - 6755399441055744.0;
    double r = fma(kf, -6.93147180369123816490e-01, x);
    r = fma(kf, -1.90821492927058770002e-10, r);
    double p = obe_exp_c[0];
#pragma unroll
    for (int i = 1; i < 12; ++i) p = fma(p, r, obe_exp_c[i]);
    p = fma(p, r, 1.0);
    p = fma(p, r, 1.0);
    k = max(k, -1022);
    const double scale = __hiloint2double((k + 1023) << 20, 0);
    return (x < -708.0) ? 0.0 : p * scale;      // also catches -inf; NaN propagates through p
}

// Models may provide a cheaper evaluation for the update pass (reciprocal of a constant hoisted
// out of the particle loop).  Default: the exact functor.
template <class Model>
struct ObeUpdateEval {
    __device__ static __forceinline__ void eval(const double* s, const double* p, const double* c, double* y) {
        Model::eval(s, p, c, y);
    }
};

// record layout of a batched instance (shared memory), see obe_update_batched_body
#define OBE_REC_SET 0      /* [4] setting        */
#define OBE_REC_Y 4        /* [4] y_meas         */
#define OBE_REC_ISIG 8     /* [4] 1/sigma        */
#define OBE_REC_PIVOT 12   /* [8] pivot          */
#define OBE_REC_INVS 20
#define OBE_REC_LEN 24
#define OBE_REC_LCONST 24  /* [4] count likelihoods only: log-factorial constants of the record (ObeBLik) */

// NE elements at once, in one basic block: the per-element chains (reciprocal refinement, the 14-deep exp
// polynomial, ...) are independent, and written this way ptxas interleaves them, which is what hides the
// ~8-cycle FP64 latency at 4 warps per SM sub-partition.  (Element-at-a-time code compiled to one serial
// DFMA chain per particle: ncu showed the FP64 pipe 41 % busy and "wait" the top stall.)
// The underflow cut (x < -708 -> 0, NaN -> 0: nan_to_num zeroes that weight anyway) is applied to the SCALE, on a
// clamped argument: written as `x < -708 ? 0 : p * scale`, ptxas sank each element's polynomial into its own
// branch region and the four 14-deep DFMA chains ran one after the other ("wait" was 30 % of the update kernel's
// stall samples); p * scale with a selected scale has to be evaluated unconditionally, so the chains interleave.
template <int NE>
__device__ __forceinline__ void obe_exp_nonpos_vec(const double (&x)[NE], double (&out)[NE]) {
    double r[NE], p[NE];
    int k[NE];
#pragma unroll
    for (int e = 0; e < NE; ++e) {
        const double xc = fmax(x[e], -708.0);                   // (NaN -> -708: finite polynomial, zero scale below)
        const double t = fma(xc, 1.4426950408889634, 6755399441055744.0);
        k[e] = __double2loint(t);
        const double kf = t - 6755399441055744.0;
        r[e] = fma(kf, -6.93147180369123816490e-01, xc);
        r[e] = fma(kf, -1.90821492927058770002e-10, r[e]);
        p[e] = obe_exp_c[0];
    }
#pragma unroll
    for (int i = 1; i < 12; ++i) {
#pragma unroll
        for (int e = 0; e < NE; ++e) p[e] = fma(p[e], r[e], obe_exp_c[i]);
    }
#pragma unroll
    for (int e = 0; e < NE; ++e) {
        p[e] = fma(p[e], r[e], 1.0);
        p[e] = fma(p[e], r[e], 1.0);
        const int hi = (x[e] >= -708.0) ? ((max(k[e], -1022) + 1023) << 20) : 0;
        out[e] = p[e] * __hiloint2double(hi, 0);
    }
}

// Row `ni` of NE particles held in registers.  `ni` is a kernel argument, uniform over the grid: one branch
// and NE moves instead of a select chain per element.
template <int D, int NE>
__device__ __forceinline__ void obe_pick_rows(const double (&p)[NE][D], int ni, double (&out)[NE], double dflt) {
#define OBE_PICK_CASE(J)                                           \
    case J:                                                        \
        if (J < D) {                                               \
            _Pragma("unroll") for (int e = 0; e < NE; ++e) out[e] = p[e][J < D ? J : 0]; \
            return;                                                \
        }                                                          \
        break;
    switch (ni) {
        OBE_PICK_CASE(0) OBE_PICK_CASE(1) OBE_PICK_CASE(2) OBE_PICK_CASE(3)
        OBE_PICK_CASE(4) OBE_PICK_CASE(5) OBE_PICK_CASE(6) OBE_PICK_CASE(7)
        default: break;
    }
#undef OBE_PICK_CASE
#pragma unroll
    for (int e = 0; e < NE; ++e) out[e] = dflt;
}

// ---- measurement likelihoods of the update pass --------------------------------------------------------------
// A likelihood maps the model outputs y[e][c] of NE particles and the record (r_y[c]: the measured values) to the
// factor lik[e] each weight is multiplied by, choke included.  The zip truncation of obe_base.py:453-455 is
// a.n_lik_channels.

// Gaussian noise with a known sigma, or sigma as a particle row (a.n_noise > 0).  The default.  Its code stays
// inline in obe_update_vec: moved into a functor, ptxas allocated registers differently for one pre-instantiated
// update kernel (k_update_generic<1, OBE_SRC_Y>, 90 -> 88), and the existing kernels are meant to stay as they are.
struct ObeGaussLik {
    static constexpr bool GAUSS = true;
};

// Per-record data of the log-likelihoods, computed on the host: aux[c] is the record's third element (trial counts
// of a binomial, anything a user likelihood wants), lconst[c] the log-factorial terms of a counting pmf.
struct ObeLikParams {
    double aux[OBE_MAX_CH];
    double lconst[OBE_MAX_CH];
};

// xlogy(k, x) = 0 for k == 0 (even at x == 0), k log x otherwise (scipy.special.xlogy)
__device__ __forceinline__ double obe_xlogy(double k, double x) { return k == 0.0 ? 0.0 : k * log(x); }
__device__ __forceinline__ double obe_xlog1py(double k, double x) { return k == 0.0 ? 0.0 : k * log1p(x); }

// Poisson counts: r_y[c] = k_c >= 0, y_c = expected count lambda_c, lconst[c] = lgamma(k_c + 1)
// (scipy.stats.poisson.logpmf).  lambda < 0 / NaN / +inf give NaN (weight 0, like nan_to_num of scipy's nan).
struct ObePoissonPmf {
    static constexpr bool NONPOS = true;
    template <int NY>
    __device__ static __forceinline__ double loglik(const double (&y)[NY], const double* k, const ObeLikParams& q, int n) {
        double ll = 0.0;
#pragma unroll
        for (int c = 0; c < NY; ++c) {
            if (c < n) {
                const double lam = y[c];
                const double lc = (obe_xlogy(k[c], lam) - lam) - q.lconst[c];
                ll += (lam >= 0.0) ? lc : __longlong_as_double(0x7ff8000000000000ll);
            }
        }
        return ll;
    }
};

// Binomial: r_y[c] = k_c successes of aux[c] = n_c trials, y_c = success probability p_c,
// lconst[c] = lgamma(n+1) - lgamma(k+1) - lgamma(n-k+1) (scipy.stats.binom.logpmf).  p outside [0, 1] gives NaN.
struct ObeBinomialPmf {
    static constexpr bool NONPOS = true;
    template <int NY>
    __device__ static __forceinline__ double loglik(const double (&y)[NY], const double* k, const ObeLikParams& q, int n) {
        double ll = 0.0;
#pragma unroll
        for (int c = 0; c < NY; ++c) {
            if (c < n) {
                const double pr = y[c];
                const double lc = (q.lconst[c] + obe_xlogy(k[c], pr)) + obe_xlog1py(q.aux[c] - k[c], -pr);
                ll += (pr >= 0.0 && pr <= 1.0) ? lc : __longlong_as_double(0x7ff8000000000000ll);
            }
        }
        return ll;
    }
};

// A likelihood given as its logarithm per particle: lik = exp(choke * log L), choke = 1 without one.  A pmf has
// log L <= 0 (NONPOS): rounding-level positive sums are clamped to 0 and the lean exp of the Gaussian applies (NaN
// and -inf give 0).  Otherwise (a user likelihood) log L may be positive and goes through the full-range exp.
template <class Pmf>
struct ObeLogLik {
    static constexpr bool GAUSS = false;
    ObeLikParams q;
    template <int D, int NE, int NY>
    __device__ __forceinline__ void operator()(const ObeUpdateArgs& a, const double (&)[NE][D],
                                               const double (&y)[NE][NY], const double* r_y, const double*,
                                               double (&lik)[NE]) const {
        double ll[NE];
#pragma unroll
        for (int e = 0; e < NE; ++e) {
            ll[e] = Pmf::loglik(y[e], r_y, q, a.n_lik_channels);
            if (Pmf::NONPOS) ll[e] = ll[e] > 0.0 ? 0.0 : ll[e];
            if (a.use_choke) ll[e] *= a.choke;
        }
        if (Pmf::NONPOS) {
            obe_exp_nonpos_vec<NE>(ll, lik);
        } else {
#pragma unroll
            for (int e = 0; e < NE; ++e) lik[e] = exp(ll[e]);
        }
    }
};
typedef ObeLogLik<ObePoissonPmf> ObePoissonLik;
typedef ObeLogLik<ObeBinomialPmf> ObeBinomialLik;

// ALLV: every element of the stage is a live particle (all stages but the ragged last one): the valid[] selects vanish.
template <class Model, int D, int SRC, int NE, bool BATCHED, bool ALLV = false, class Lik = ObeGaussLik>
__device__ __forceinline__ void obe_update_vec(const ObeUpdateArgs& a, const double (&p)[NE][D],
                                               const double (&w_in)[NE], const double (&yg)[NE][OBE_MAX_CH],
                                               const double (&lik_given)[NE], const bool (&valid)[NE], double invS,
                                               ObeAcc<D>& acc, const double* rec, double (&t)[NE],
                                               const Lik& likf = Lik()) {
    const double* r_set = BATCHED ? rec + OBE_REC_SET : a.setting;
    const double* r_y = BATCHED ? rec + OBE_REC_Y : a.y_meas;
    const double* r_isig = BATCHED ? rec + OBE_REC_ISIG : a.inv_sigma;
    const double* r_piv = BATCHED ? rec + OBE_REC_PIVOT : a.pivot;
    if (SRC == OBE_SRC_NONE || SRC == OBE_SRC_DRIFT) {
#pragma unroll
        for (int e = 0; e < NE; ++e) t[e] = w_in[e];
    } else {
        double lik[NE];
        if (SRC == OBE_SRC_LIK) {
#pragma unroll
            for (int e = 0; e < NE; ++e) lik[e] = lik_given[e];
        } else {
            constexpr int NY = (SRC == OBE_SRC_MODEL) ? (Model::NCH > 0 ? Model::NCH : 1) : OBE_MAX_CH;
            double y[NE][NY];
#pragma unroll
            for (int e = 0; e < NE; ++e) {
                if (SRC == OBE_SRC_MODEL) {
                    ObeUpdateEval<Model>::eval(r_set, p[e], a.cons, y[e]);
                } else {
#pragma unroll
                    for (int c = 0; c < NY; ++c) y[e][c] = yg[e][c];
                }
                lik[e] = 1.0;
            }
            if constexpr (Lik::GAUSS) {
                // prod_c exp(-((y_c - y_meas_c)/sigma_c)**2 / 2) / sigma_c  (obe_base.py:264-271, 453-455) as ONE
                // exponential of the summed arguments times the product of the reciprocals: the division by sigma
                // is a multiplication by its reciprocal (host's 1/sigma, or one refined rcp per particle for a
                // noise parameter, shared by the channels that name the same row).  For one channel this is the
                // same sequence of operations as exp(arg) * (1/sigma).
                const bool noise = a.n_noise > 0;
                double argsum[NE], isprod[NE], inv_prev[NE];
#pragma unroll
                for (int e = 0; e < NE; ++e) { argsum[e] = 0.0; isprod[e] = 1.0; inv_prev[e] = 1.0; }
                int ni_prev = -2;
#pragma unroll
                for (int c = 0; c < NY; ++c) {
                    if (c < a.n_lik_channels) {
                        const int ni = a.noise_idx[c];
                        double inv_sig[NE];
                        if (!noise) {
#pragma unroll
                            for (int e = 0; e < NE; ++e) inv_sig[e] = r_isig[c];
                        } else if (ni == ni_prev) {
#pragma unroll
                            for (int e = 0; e < NE; ++e) inv_sig[e] = inv_prev[e];
                        } else {
                            double sig[NE];
                            obe_pick_rows<D, NE>(p, ni, sig, 1.0);
#pragma unroll
                            for (int e = 0; e < NE; ++e) inv_sig[e] = obe_rcp_fast(sig[e]);
                        }
#pragma unroll
                        for (int e = 0; e < NE; ++e) {
                            const double q = (y[e][c] - r_y[c]) * inv_sig[e];
                            argsum[e] = fma(-0.5 * q, q, argsum[e]);
                            isprod[e] *= inv_sig[e];
                            inv_prev[e] = inv_sig[e];
                        }
                        ni_prev = ni;
                    }
                }
                {
                    double ex[NE];
                    obe_exp_nonpos_vec<NE>(argsum, ex);
#pragma unroll
                    for (int e = 0; e < NE; ++e) lik[e] = ex[e] * isprod[e];
                }
                if (a.use_choke) {
#pragma unroll
                    for (int e = 0; e < NE; ++e) lik[e] = pow(lik[e], a.choke);
                }
            } else {
                likf(a, p, y, r_y, r_isig, lik);
            }
        }
        // t = nan_to_num(w * lik); w = w_in * invS needs no second nan_to_num (stored weights are finite and
        // <= total; a NaN from 0 * inf propagates into t and is zeroed here like numpy does)
        bool any_bad = false;
#pragma unroll
        for (int e = 0; e < NE; ++e) {
            t[e] = (w_in[e] * invS) * lik[e];
            any_bad |= (((unsigned)__double2hiint(t[e])) & 0x7fffffffu) >= 0x7ff00000u;
        }
        if (any_bad) {
#pragma unroll
            for (int e = 0; e < NE; ++e) t[e] = obe_nan_to_num_fast(t[e]);
        }
    }
    // constraint masks: refresh pass / batched update (the batched drift rejects steps in its move instead)
    if ((SRC == OBE_SRC_NONE || (BATCHED && SRC != OBE_SRC_DRIFT)) && (a.mask_le | a.mask_lt)) {
#pragma unroll
        for (int e = 0; e < NE; ++e) {
            bool bad = false;
#pragma unroll
            for (int j = 0; j < D; ++j) {
                if (((a.mask_le >> j) & 1u) && p[e][j] <= 0.0) bad = true;
                if (((a.mask_lt >> j) & 1u) && p[e][j] < 0.0) bad = true;
            }
            if (bad && (ALLV || valid[e])) {
                if (t[e] != 0.0) acc.nzero += 1.0;
                t[e] = 0.0;
            }
        }
    }
    if (!ALLV) {
#pragma unroll
        for (int e = 0; e < NE; ++e) t[e] = valid[e] ? t[e] : 0.0;
    }
#pragma unroll
    for (int e = 0; e < NE; ++e) {
        acc.sumsq += t[e] * t[e];
        acc.sumt += t[e];
        double dx[D];
#pragma unroll
        for (int j = 0; j < D; ++j) dx[j] = (ALLV || valid[e]) ? p[e][j] - r_piv[j] : 0.0;
        int q = 0;
#pragma unroll
        for (int j = 0; j < D; ++j) {
            const double tj = t[e] * dx[j];
            acc.m1[j] += tj;
#pragma unroll
            for (int k = j; k < D; ++k) acc.m2[q++] += tj * dx[k];
        }
    }
    if (a.n_noise > 0) {
#pragma unroll
        for (int c = 0; c < OBE_MAX_CH; ++c) {
            const int ni = a.noise_idx[c];
            if (ni >= 0) {
                double sig[NE];
                obe_pick_rows<D, NE>(p, ni, sig, 0.0);
#pragma unroll
                for (int e = 0; e < NE; ++e) acc.noise[c] += (ALLV || valid[e]) ? t[e] * (sig[e] * sig[e]) : 0.0;
            }
        }
    }
}

// W chunks of NW*32 consecutive elements scanned at once: ex[e] = exclusive scan of v[e] over the
// block's threads within chunk e (Kogge-Stone over lanes, then over the warp totals), tot[e] = the
// chunk's total.  One set of barriers serves all W chunks, so a single block walks a long array in
// 1/W of the latency-bound rounds.  sm: W * (NW + 1) elements.  Needs NW >= W.
#define OBE_SCANW 8
struct ObeOpSum { template <class T> __device__ __forceinline__ T operator()(T a, T b) const { return a + b; } };
struct ObeOpMax { template <class T> __device__ __forceinline__ T operator()(T a, T b) const { return a > b ? a : b; } };
template <class T, int NW, class Op>
__device__ __forceinline__ void obe_block_excl_scanw(const T (&v)[OBE_SCANW], T (&ex)[OBE_SCANW], T (&tot)[OBE_SCANW],
                                                     T* sm, Op op, T ident, int bar_id) {
    constexpr int W = OBE_SCANW;
    const int lane = threadIdx.x & 31, warp = (threadIdx.x >> 5) % NW;
    T x[W];
#pragma unroll
    for (int e = 0; e < W; ++e) x[e] = v[e];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
#pragma unroll
        for (int e = 0; e < W; ++e) {
            const T y = __shfl_up_sync(0xffffffffu, x[e], o);
            if (lane >= o) x[e] = op(x[e], y);
        }
    }
    obe_named_bar(bar_id, NW * 32);
    if (lane == 31) {
#pragma unroll
        for (int e = 0; e < W; ++e) sm[e * (NW + 1) + warp] = x[e];
    }
    obe_named_bar(bar_id, NW * 32);
    if (warp < W) {
        T* row = sm + warp * (NW + 1);
        T xs = (lane < NW) ? row[lane] : ident;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const T y = __shfl_up_sync(0xffffffffu, xs, o);
            if (lane >= o) xs = op(xs, y);
        }
        T exs = __shfl_up_sync(0xffffffffu, xs, 1);      // exclusive base of each warp
        if (lane == 0) exs = ident;
        if (lane < NW) row[lane] = exs;
        if (lane == 31) row[NW] = xs;
    }
    obe_named_bar(bar_id, NW * 32);
#pragma unroll
    for (int e = 0; e < W; ++e) {
        T exl = __shfl_up_sync(0xffffffffu, x[e], 1);
        if (lane == 0) exl = ident;
        ex[e] = op(sm[e * (NW + 1) + warp], exl);
        tot[e] = sm[e * (NW + 1) + NW];
    }
}

// tile_prefix[k] = sum of tile_sums[0..k) in a fixed association (coalesced chunks of NW*32 with a running
// carry, OBE_SCANW chunks per round); tile_prefix[n_tiles] is THE total every CDF consumer divides by.
// One block.  Also finishes the stats block: canonical total, normaliser, N_eff (and the uniform-weights
// bookkeeping after a resample).  sm: OBE_SCANW * (NW + 1) doubles.
template <int NW>
__device__ __forceinline__ void obe_tile_scan_block(const double* __restrict__ tile_sums, long long n_tiles,
                                                    double* __restrict__ prefix, double* __restrict__ stats,
                                                    int renormalise, long long uniform, long long n, int implicit,
                                                    double* sm, int bar_id, double gate_thr = 0.0,
                                                    double gate_n = 0.0, double* stats_out2 = nullptr) {
    constexpr int T_ = NW * 32;
    const int t = threadIdx.x % T_;
    double carry = 0.0;
    for (long long base = 0; base < n_tiles; base += OBE_SCANW * T_) {
        double v[OBE_SCANW], ex[OBE_SCANW], tot[OBE_SCANW];
#pragma unroll
        for (int e = 0; e < OBE_SCANW; ++e) {
            const long long k = base + e * T_ + t;
            v[e] = (k < n_tiles) ? __ldcg(tile_sums + k) : 0.0;
        }
        obe_block_excl_scanw<double, NW>(v, ex, tot, sm, ObeOpSum(), 0.0, bar_id);
#pragma unroll
        for (int e = 0; e < OBE_SCANW; ++e) {
            const long long k = base + e * T_ + t;
            if (k < n_tiles) prefix[k] = carry + ex[e];
            carry += tot[e];
        }
        obe_named_bar(bar_id, NW * 32);
    }
    const double total = carry;
    if (t == 0) {
        prefix[n_tiles] = total;
        if (stats) {
            stats[OBE_ST_TOTAL] = total;
            if (uniform) {
                // weights are exactly 1/n_total: normaliser is exactly 1 (particlepdf.py:309-310);
                // `uniform` carries n_total (== n for a whole cloud)
                const double wv = 1.0 / (double)uniform;
                stats[OBE_ST_INVS] = 1.0;
                stats[OBE_ST_SUMSQ] = (double)n * wv * wv;
                stats[OBE_ST_SUMT] = (double)n * wv;
                stats[OBE_ST_NEFF] = (double)uniform;
                stats[OBE_ST_UNIFORM] = implicit ? wv : 0.0;
                stats[OBE_ST_FIRED] = 0.0;
            } else {
                const double invs = renormalise ? 1.0 / total : 1.0;
                stats[OBE_ST_INVS] = invs;
                const double ssq = stats[OBE_ST_SUMSQ];
                stats[OBE_ST_NEFF] = (total * total) / ssq;
                double fired = 0.0;
                if (gate_n > 0.0) {
                    // the host's arithmetic (ParticlePDF._n_eff_from / resample_test), operation for operation
                    const double n_eff = 1.0 / obe_mul(ssq, obe_mul(invs, invs));
                    fired = (n_eff < obe_mul(0.1, gate_n) || n_eff / gate_n < gate_thr) ? 1.0 : 0.0;
                }
                stats[OBE_ST_FIRED] = fired;
            }
        }
    }
    if (stats_out2 && stats) {
        // the block is complete (every slot was written by thread 0 of this CTA, before the caller's barriers or just
        // now): 64 threads copy it into the caller's pinned host block -- no D2H copy behind the kernel
        obe_named_bar(bar_id, NW * 32);
        if (t < OBE_STATS_LEN) stats_out2[t] = __ldcg(stats + t);
    }
}

// stage geometry as a function of the number of rows staged per particle
template <int NROWS>
struct ObeStage {
    static constexpr int ELEMS = NROWS <= 4 ? 2048 : (NROWS <= 8 ? 1024 : 512);
    static constexpr int BYTES = NROWS * ELEMS * 8;
    static constexpr int NSTAGES_RAW = OBE_SMEM_BUDGET / BYTES;
    static constexpr int NSTAGES = NSTAGES_RAW > 4 ? 4 : NSTAGES_RAW;
    static constexpr int SUB = OBE_TILE / ELEMS;                 // stages per canonical tile
    static constexpr int EPT = ELEMS / OBE_CONSUMER_THREADS;     // elements per consumer thread per stage
    static constexpr int SMEM = NSTAGES * BYTES + 1024;
};

template <int D, int SRC>
struct ObeUpdateRows {
    static constexpr int NROWS = 1 + D + (SRC == OBE_SRC_Y ? OBE_MAX_CH : 0) + (SRC == OBE_SRC_LIK ? 1 : 0);
};

template <class Model, int D, int SRC, class Lik = ObeGaussLik>
__device__ void obe_update_body(const ObeUpdateArgs& a, const Lik& likf = Lik()) {
    constexpr int NROWS = ObeUpdateRows<D, SRC>::NROWS;
    using ST = ObeStage<NROWS>;
    constexpr int SE = ST::ELEMS, NST = ST::NSTAGES, SUB = ST::SUB, EPT = ST::EPT;
    constexpr int NM2 = D * (D + 1) / 2;
    constexpr int NACC = 3 + D + NM2 + OBE_MAX_CH;
    extern __shared__ __align__(128) unsigned char obe_dyn_smem[];
    double* stage_base = reinterpret_cast<double*>(obe_dyn_smem);
    unsigned long long* full_bar = reinterpret_cast<unsigned long long*>(obe_dyn_smem + NST * ST::BYTES);
    unsigned long long* empty_bar = full_bar + NST;
    __shared__ double red[2][OBE_CONSUMER_WARPS];
    __shared__ double accsm[OBE_CONSUMER_WARPS][OBE_NACC_MAX];
    __shared__ double fin[OBE_NACC_MAX];
    __shared__ unsigned int is_last;

    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    if constexpr (SRC == OBE_SRC_DRIFT) {
        if (!likf.gate_open()) return;           // (uniform over the grid: no block has touched anything yet)
    }
    const long long n = a.n_dev ? *a.n_dev : a.n;
    const long long n_tiles = (n + OBE_TILE - 1) / OBE_TILE;
    // implicit uniform weights (left by a systematic resample): the weight row is neither copied nor read
    const double wuni = a.stats[OBE_ST_UNIFORM];
    const bool implicit = wuni > 0.0;
    // rows actually staged: weights, D particle rows, then the optional extras
    const int n_rows_live = (implicit ? 0 : 1) + D + (SRC == OBE_SRC_Y ? a.n_lik_channels : 0) + (SRC == OBE_SRC_LIK ? 1 : 0);

    if (tid == 0) {
        for (int s = 0; s < NST; ++s) {
            obe_mbar_init(full_bar + s, 1);
            obe_mbar_init(empty_bar + s, OBE_CONSUMER_WARPS);
        }
        obe_mbar_fence_init();
    }
    __syncthreads();

    // ---- producer role: thread 0 issues the bulk copies of iteration p (tile, sub-stage) into
    //      ring slot p % NST, NST-1 iterations ahead of the consumers
    const long long my_tiles = (n_tiles > (long long)blockIdx.x)
                                   ? (n_tiles - 1 - (long long)blockIdx.x) / (long long)gridDim.x + 1 : 0;
    const unsigned total_iters = (unsigned)(my_tiles * SUB);
    auto produce = [&](unsigned p) {
        if (p >= total_iters) return;
        const int s = p % NST;
        const unsigned k = p / NST;
        const long long tile = (long long)blockIdx.x + (long long)(p / SUB) * (long long)gridDim.x;
        const long long base = tile * OBE_TILE + (long long)(p % SUB) * SE;
        long long cnt = a.ld - base;
        if (cnt > SE) cnt = SE;
        obe_mbar_wait(empty_bar + s, (k & 1u) ^ 1u);
        if (cnt <= 0) {                               // sub-stage past the end of a ragged tile
            obe_mbar_arrive(full_bar + s);
            return;
        }
        const unsigned row_bytes = (unsigned)cnt * 8u;
        obe_mbar_expect_tx(full_bar + s, row_bytes * (unsigned)n_rows_live);
        double* dst = stage_base + (size_t)s * (NROWS * SE);
        if (!implicit) obe_bulk_g2s(dst, a.weights + base, row_bytes, full_bar + s);
#pragma unroll
        for (int j = 0; j < D; ++j)
            obe_bulk_g2s(dst + (1 + j) * SE, a.particles + j * a.ld + base, row_bytes, full_bar + s);
        if (SRC == OBE_SRC_Y) {
            for (int c = 0; c < a.n_lik_channels; ++c)
                obe_bulk_g2s(dst + (1 + D + c) * SE, a.y_model + c * a.ld_y + base, row_bytes, full_bar + s);
        }
        if (SRC == OBE_SRC_LIK) obe_bulk_g2s(dst + (1 + D) * SE, a.lik + base, row_bytes, full_bar + s);
    };
    if (tid == 0) {
        for (unsigned p = 0; p + 1 < (unsigned)NST; ++p) produce(p);
    }

    // ---------------------------------------------------------------------- consumers
    const int ct = tid;                   // every thread is a consumer
    const int cwarp = warp;
    const double invS = a.scale_in ? a.stats[OBE_ST_INVS] : 1.0;   // scale_in == 0: raw weights
    const bool write_weights = a.write_weights != 0;
    ObeAcc<D> acc;
    acc.sumsq = 0.0; acc.sumt = 0.0; acc.nzero = 0.0;
#pragma unroll
    for (int j = 0; j < D; ++j) acc.m1[j] = 0.0;
#pragma unroll
    for (int j = 0; j < NM2; ++j) acc.m2[j] = 0.0;
#pragma unroll
    for (int c = 0; c < OBE_MAX_CH; ++c) acc.noise[c] = 0.0;

    unsigned it = 0;
    unsigned tile_par = 0;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, tile_par ^= 1u) {
        double tsum = 0.0;
#pragma unroll 1
        for (int sub = 0; sub < SUB; ++sub, ++it) {
            const int s = it % NST;
            const unsigned k = it / NST;
            const long long base = tile * OBE_TILE + (long long)sub * SE;
            const int n_valid = (base + SE <= n) ? SE : (int)(n - base);   // particles of this stage
            if (tid == 0) produce(it + NST - 1);
            obe_mbar_wait(full_bar + s, k & 1u);
            const double* src = stage_base + (size_t)s * (NROWS * SE);
            // this thread's columns -> registers
            double wv[EPT], pv[D][EPT], yv[SRC == OBE_SRC_Y ? OBE_MAX_CH : 1][EPT], lv[EPT];
            if (EPT >= 2) {
#pragma unroll
                for (int q = 0; q < EPT / 2; ++q) {
                    const int e = 2 * (ct + q * OBE_CONSUMER_THREADS);
                    double2 w2 = make_double2(wuni, wuni);
                    if (!implicit) w2 = *reinterpret_cast<const double2*>(src + e);
                    wv[2 * q] = w2.x; wv[2 * q + 1] = w2.y;
#pragma unroll
                    for (int j = 0; j < D; ++j) {
                        const double2 p2 = *reinterpret_cast<const double2*>(src + (1 + j) * SE + e);
                        pv[j][2 * q] = p2.x; pv[j][2 * q + 1] = p2.y;
                    }
                    if (SRC == OBE_SRC_Y) {
#pragma unroll
                        for (int c = 0; c < OBE_MAX_CH; ++c) {
                            double2 y2 = make_double2(0.0, 0.0);
                            if (c < a.n_lik_channels) y2 = *reinterpret_cast<const double2*>(src + (1 + D + c) * SE + e);
                            yv[SRC == OBE_SRC_Y ? c : 0][2 * q] = y2.x; yv[SRC == OBE_SRC_Y ? c : 0][2 * q + 1] = y2.y;
                        }
                    }
                    if (SRC == OBE_SRC_LIK) {
                        const double2 l2 = *reinterpret_cast<const double2*>(src + (1 + D) * SE + e);
                        lv[2 * q] = l2.x; lv[2 * q + 1] = l2.y;
                    }
                }
            } else {
                wv[0] = implicit ? wuni : src[ct];
#pragma unroll
                for (int j = 0; j < D; ++j) pv[j][0] = src[(1 + j) * SE + ct];
                if (SRC == OBE_SRC_Y) {
#pragma unroll
                    for (int c = 0; c < OBE_MAX_CH; ++c)
                        yv[SRC == OBE_SRC_Y ? c : 0][0] = (c < a.n_lik_channels) ? src[(1 + D + c) * SE + ct] : 0.0;
                }
                if (SRC == OBE_SRC_LIK) lv[0] = src[(1 + D) * SE + ct];
            }
            __syncwarp();
            if (lane == 0) obe_mbar_arrive(empty_bar + s);   // stage can be refilled
            // compute (all EPT elements of this thread together) + store
            {
                double pe[EPT][D], yge[EPT][OBE_MAX_CH], lke[EPT], te[EPT];
                bool valid[EPT];
#pragma unroll
                for (int e = 0; e < EPT; ++e) {
                    const int idx = (EPT >= 2) ? 2 * (ct + (e >> 1) * OBE_CONSUMER_THREADS) + (e & 1) : ct;
                    valid[e] = idx < n_valid;
#pragma unroll
                    for (int j = 0; j < D; ++j) pe[e][j] = pv[j][e];
#pragma unroll
                    for (int c = 0; c < OBE_MAX_CH; ++c) yge[e][c] = (SRC == OBE_SRC_Y) ? yv[SRC == OBE_SRC_Y ? c : 0][e] : 0.0;
                    lke[e] = (SRC == OBE_SRC_LIK) ? lv[e] : 1.0;
                }
                if constexpr (SRC == OBE_SRC_DRIFT) likf.template move<D, EPT>(a, pe, valid, base, ct, n_valid);
                obe_update_vec<Model, D, SRC, EPT, false, false, Lik>(a, pe, wv, yge, lke, valid, invS, acc, nullptr, te, likf);
#pragma unroll
                for (int e = 0; e < EPT; ++e) tsum += te[e];
                if (write_weights) {
#pragma unroll
                    for (int q = 0; q < (EPT >= 2 ? EPT / 2 : 1); ++q) {
                        const int e0 = (EPT >= 2 ? 2 * (ct + q * OBE_CONSUMER_THREADS) : ct);
                        if (EPT >= 2 && e0 + 1 < n_valid) obe_st2(a.weights + base + e0, make_double2(te[2 * q], te[2 * q + 1]));
                        else if (e0 < n_valid) a.weights[base + e0] = te[EPT >= 2 ? 2 * q : 0];
                    }
                }
            }
        }
        // tile sum: warp partials -> one named barrier among the consumers -> fixed-order sum.  (A barrier-free
        // variant -- ring of partial slots, the last warp to arrive sums -- and a select-free path for full stages
        // were measured on top of the interleaved exp and changed nothing: 0.586 vs 0.590 ms at 1e8.)
        if constexpr (SRC != OBE_SRC_DRIFT) {     // (the drift leaves the weights, hence the tile sums, as they are)
            tsum = obe_warp_sum(tsum);
            if (lane == 0) red[tile_par][cwarp] = tsum;
            obe_named_bar(1, OBE_CONSUMER_THREADS);
            if (ct == 0) {
                double s = red[tile_par][0];
#pragma unroll
                for (int w = 1; w < OBE_CONSUMER_WARPS; ++w) s += red[tile_par][w];
                a.tile_sums[tile] = s;
            }
        }
    }

    obe_grid_dep_launch();       // the (tiny) dependents may be scheduled now; they wait for this grid to complete
    // ---- per-block partials, then the last block to arrive combines them in block order
    double vals[NACC];
    vals[0] = acc.sumsq; vals[1] = acc.sumt; vals[2] = acc.nzero;
#pragma unroll
    for (int j = 0; j < D; ++j) vals[3 + j] = acc.m1[j];
#pragma unroll
    for (int j = 0; j < NM2; ++j) vals[3 + D + j] = acc.m2[j];
#pragma unroll
    for (int c = 0; c < OBE_MAX_CH; ++c) vals[3 + D + NM2 + c] = acc.noise[c];
#pragma unroll
    for (int v = 0; v < NACC; ++v) {
        const double sv = obe_warp_sum(vals[v]);
        if (lane == 0) accsm[cwarp][v] = sv;
    }
    obe_named_bar(1, OBE_CONSUMER_THREADS);
    if (ct < NACC) {
        double sv = accsm[0][ct];
#pragma unroll
        for (int w = 1; w < OBE_CONSUMER_WARPS; ++w) sv += accsm[w][ct];
        a.partials[(long long)blockIdx.x * OBE_NACC_MAX + ct] = sv;
    }
    __threadfence();
    obe_named_bar(1, OBE_CONSUMER_THREADS);
    if (ct == 0) is_last = (atomicAdd(a.counter, 1u) == gridDim.x - 1) ? 1u : 0u;
    obe_named_bar(1, OBE_CONSUMER_THREADS);
    if (!is_last) return;
    __threadfence();
    for (int v = cwarp; v < NACC; v += OBE_CONSUMER_WARPS) {
        double sv = 0.0;
        for (unsigned int b = lane; b < gridDim.x; b += 32)
            sv += __ldcg(a.partials + (long long)b * OBE_NACC_MAX + v);
        sv = obe_warp_sum(sv);
        if (lane == 0) fin[v] = sv;
    }
    obe_named_bar(1, OBE_CONSUMER_THREADS);
    if constexpr (SRC == OBE_SRC_DRIFT) {
        // only the moments move: totals, normaliser, N_eff, the implicit-weight word and the tile prefix stay
        if (ct == 0) {
            for (int j = 0; j < D; ++j) { a.stats[OBE_ST_M1 + j] = fin[3 + j]; a.stats[OBE_ST_PIVOT + j] = a.pivot[j]; }
            for (int j = 0; j < NM2; ++j) a.stats[OBE_ST_M2 + j] = fin[3 + D + j];
            for (int c = 0; c < OBE_MAX_CH; ++c)
                if (a.noise_idx[c] >= 0) a.stats[OBE_ST_NOISE + c] = fin[3 + D + NM2 + c];
            *a.counter = 0u;
        }
        if (a.stats_out2) {
            obe_named_bar(1, OBE_CONSUMER_THREADS);
            // the FIRED word of the copy is the update's decision, which this (gated) pass ran under
            if (ct < OBE_STATS_LEN)
                a.stats_out2[ct] = (ct == OBE_ST_FIRED && likf.q.gate) ? *likf.q.gate : __ldcg(a.stats + ct);
        }
        return;
    }
    if (ct == 0) {
        a.stats[OBE_ST_SUMSQ] = fin[0];
        a.stats[OBE_ST_SUMT] = fin[1];
        a.stats[OBE_ST_NZERO] = fin[2];
        for (int j = 0; j < D; ++j) { a.stats[OBE_ST_M1 + j] = fin[3 + j]; a.stats[OBE_ST_PIVOT + j] = a.pivot[j]; }
        for (int j = 0; j < NM2; ++j) a.stats[OBE_ST_M2 + j] = fin[3 + D + j];   // packed j<=k over D dims
        for (int c = 0; c < OBE_MAX_CH; ++c) a.stats[OBE_ST_NOISE + c] = fin[3 + D + NM2 + c];
        if (a.write_weights) a.stats[OBE_ST_UNIFORM] = 0.0;      // the weight row is explicit again
        *a.counter = 0u;
    }
    // the last block also turns the tile sums into the CDF prefix and finishes the stats block (saves a launch)
    obe_named_bar(1, OBE_CONSUMER_THREADS);
    __threadfence();
    obe_tile_scan_block<OBE_CONSUMER_WARPS>(a.tile_sums, n_tiles, a.tile_prefix, a.stats, a.renormalise, 0, n, 0,
                                            &accsm[0][0], 1, a.gate_thr, a.gate_n, a.stats_out2);
}

// ---------------------------------------------------------------------------------------------
// Batched independent instances (BASELINE config c5: 4096 lock-in engines x 1e4 particles).
// One big SoA cloud: instance b owns particles [b*np, b*np + n) of a (d, B*np) array, np = n
// rounded up to whole tiles (padding particles are never read).  Two buffers; cur[b] says which one
// holds instance b (a resample writes the other one and flips it, so instances that do not resample
// are never copied).  Every instance has its own record, pivot, stats block, CDF prefix row,
// resample flag and RNG streams; nothing returns to the host inside a cycle.
// ---------------------------------------------------------------------------------------------
struct ObeBatchArgs {
    ObeUpdateArgs u;              // the fields shared by all instances (cons, noise_idx, masks, choke, ...)
    const double* particles[2];   // (d, ld) each, ld = B * np
    double* weights[2];           // (ld) each
    int* cur;                     // (B) buffer holding instance b
    double* tile_sums;            // (B * T)
    double* prefix;               // (B * (T + 1))
    double* stats;                // (B * OBE_STATS_LEN)
    double* pivot;                // (B * OBE_MAX_DIMS)   updated to the new mean by the kernel
    const double* rec_in;         // (B * 12): setting[4], y_meas[4], sigma[4]
    const double* settings;       // (s, lds) grid, for use_last
    long long lds;
    const long long* last_idx;    // (B) last chosen setting index (use_last)
    int* flag;                    // (B) out: 1 = this instance must resample
    long long n_inst, np;         // instances, padded particles per instance
    int tiles;                    // np / OBE_TILE
    int use_last;                 // 1: the setting of instance b is settings[:, last_idx[b]]
    int n_set;                    // number of setting knobs
    double resample_threshold;
    int force_resample;
    const int* inst_list;         // optional compacted list of instances to process ...
    const int* n_list;            // ... and its length (device)
};

// The move policy of the batched body.  Every kernel but the batched drift (SRC == OBE_SRC_DRIFT, ObeBDrift) runs
// with this one, which is never called.
struct ObeNoMove {};

// Lik: ObeGaussLik (the record's third element is sigma), or ObeBLik of a count / user likelihood (NVRTC modules only:
// the third element is the aux, and the record's log-factorial constants are computed here, per instance, because
// in a closed loop the counts are written on the device).
template <class Model, int D, int SRC, class Mv = ObeNoMove, class Lik = ObeGaussLik>
__device__ void obe_update_batched_body(const ObeBatchArgs& a, const Mv& mv = Mv()) {
    constexpr int NROWS = 1 + D;
    using ST = ObeStage<NROWS>;
    constexpr int SE = ST::ELEMS, NST = ST::NSTAGES, SUB = ST::SUB, EPT = ST::EPT;
    constexpr int NM2 = D * (D + 1) / 2;
    constexpr int NACC = 3 + D + NM2 + OBE_MAX_CH;
    extern __shared__ __align__(128) unsigned char obe_dyn_smem[];
    double* stage_base = reinterpret_cast<double*>(obe_dyn_smem);
    unsigned long long* full_bar = reinterpret_cast<unsigned long long*>(obe_dyn_smem + NST * ST::BYTES);
    unsigned long long* empty_bar = full_bar + NST;
    __shared__ double red[2][OBE_CONSUMER_WARPS];
    __shared__ double accsm[OBE_CONSUMER_WARPS][OBE_NACC_MAX];
    constexpr int RECN = Lik::GAUSS ? OBE_REC_LEN : OBE_REC_LCONST + OBE_MAX_CH;
    __shared__ double rec_s[2][RECN];
    __shared__ double tsum_s[64];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long long n = a.u.n;                     // real particles per instance
    const int T = a.tiles;
    const long long np = a.np;
    if (tid == 0) {
        for (int s = 0; s < NST; ++s) {
            obe_mbar_init(full_bar + s, 1);
            obe_mbar_init(empty_bar + s, OBE_CONSUMER_WARPS);
        }
        obe_mbar_fence_init();
    }
    __syncthreads();
    const long long n_inst = a.inst_list ? (long long)*a.n_list : a.n_inst;
    const long long my_inst = (n_inst > (long long)blockIdx.x)
                                  ? (n_inst - 1 - (long long)blockIdx.x) / (long long)gridDim.x + 1 : 0;
    const unsigned per_inst = (unsigned)(T * SUB);
    const unsigned total_iters = (unsigned)(my_inst * per_inst);
    auto produce = [&](unsigned p) {
        if (p >= total_iters) return;
        const int s = p % NST;
        const unsigned k = p / NST;
        const long long bi = (long long)blockIdx.x + (long long)(p / per_inst) * (long long)gridDim.x;
        const long long b = a.inst_list ? (long long)a.inst_list[bi] : bi;
        const long long off = b * np + (long long)((p % per_inst) / SUB) * OBE_TILE + (long long)(p % SUB) * SE;
        const int cb = a.cur[b];
        obe_mbar_wait(empty_bar + s, (k & 1u) ^ 1u);
        const unsigned row_bytes = (unsigned)SE * 8u;
        obe_mbar_expect_tx(full_bar + s, row_bytes * (unsigned)NROWS);
        double* dst = stage_base + (size_t)s * (NROWS * SE);
        obe_bulk_g2s(dst, a.weights[cb] + off, row_bytes, full_bar + s);
#pragma unroll
        for (int j = 0; j < D; ++j)
            obe_bulk_g2s(dst + (1 + j) * SE, a.particles[cb] + j * a.u.ld + off, row_bytes, full_bar + s);
    };
    if (tid == 0) {
        for (unsigned p = 0; p + 1 < (unsigned)NST; ++p) produce(p);
    }
    const int ct = tid, cwarp = warp;
    const bool write_weights = a.u.write_weights != 0;
    unsigned it = 0, tile_par = 0;
    for (long long ii = 0; ii < my_inst; ++ii) {
        const long long bi = (long long)blockIdx.x + ii * (long long)gridDim.x;
        const long long b = a.inst_list ? (long long)a.inst_list[bi] : bi;
        const int cb = a.cur[b];
        double* rec = rec_s[ii & 1];
        // ---- per-instance record into shared memory
        if (ct < RECN) {
            double v = 0.0;
            if (ct < OBE_REC_Y) {
                if (ct < a.n_set)
                    v = a.use_last ? a.settings[ct * a.lds + a.last_idx[b]] : a.rec_in[b * 12 + ct];
            } else if (ct < OBE_REC_ISIG) {
                v = a.rec_in[b * 12 + ct];
            } else if (ct < OBE_REC_PIVOT) {
                const double sg = a.rec_in[b * 12 + ct];
                if constexpr (Lik::GAUSS) v = (sg != 0.0) ? 1.0 / sg : 1.0;
                else v = sg;                                       // (the aux)
            } else if (ct < OBE_REC_INVS) {
                v = a.pivot[b * OBE_MAX_DIMS + (ct - OBE_REC_PIVOT)];
            } else if (ct == OBE_REC_INVS) {
                v = a.u.scale_in ? a.stats[b * OBE_STATS_LEN + OBE_ST_INVS] : 1.0;
            } else if (ct >= OBE_REC_LCONST) {
                if constexpr (!Lik::GAUSS) {
                    const int c = ct - OBE_REC_LCONST;
                    v = Lik::lconst(a.rec_in[b * 12 + OBE_REC_Y + c], a.rec_in[b * 12 + OBE_REC_ISIG + c]);
                }
            }
            rec[ct] = v;
        }
        if constexpr (SRC == OBE_SRC_DRIFT) mv.template load<D>(b, (int)(ii & 1), ct);
        obe_named_bar(1, OBE_CONSUMER_THREADS);
        const double invS = rec[OBE_REC_INVS];
        ObeAcc<D> acc;
        acc.sumsq = 0.0; acc.sumt = 0.0; acc.nzero = 0.0;
#pragma unroll
        for (int j = 0; j < D; ++j) acc.m1[j] = 0.0;
#pragma unroll
        for (int j = 0; j < NM2; ++j) acc.m2[j] = 0.0;
#pragma unroll
        for (int c = 0; c < OBE_MAX_CH; ++c) acc.noise[c] = 0.0;
        for (int t = 0; t < T; ++t, tile_par ^= 1u) {
            double tsum = 0.0;
#pragma unroll 1
            for (int sub = 0; sub < SUB; ++sub, ++it) {
                const int s = it % NST;
                const unsigned k = it / NST;
                const long long loc = (long long)t * OBE_TILE + (long long)sub * SE;   // offset in the instance
                const long long base = b * np + loc;
                long long nv = n - loc;
                const int n_valid = nv >= SE ? SE : (nv > 0 ? (int)nv : 0);
                if (tid == 0) produce(it + NST - 1);
                obe_mbar_wait(full_bar + s, k & 1u);
                const double* src = stage_base + (size_t)s * (NROWS * SE);
                double wv[EPT], pv[D][EPT];
                // ONE1: a stage of one element per thread (EPT == 1, D = 8).  Only the drift pass handles it; the
                // update and refresh instantiations keep their code (DESIGN §7).
                constexpr bool ONE1 = SRC == OBE_SRC_DRIFT && EPT == 1;
                if constexpr (ONE1) {
                    wv[0] = src[ct];
#pragma unroll
                    for (int j = 0; j < D; ++j) pv[j][0] = src[(1 + j) * SE + ct];
                } else {
#pragma unroll
                    for (int q = 0; q < EPT / 2; ++q) {
                        const int e = 2 * (ct + q * OBE_CONSUMER_THREADS);
                        const double2 w2 = *reinterpret_cast<const double2*>(src + e);
                        wv[2 * q] = w2.x; wv[2 * q + 1] = w2.y;
#pragma unroll
                        for (int j = 0; j < D; ++j) {
                            const double2 p2 = *reinterpret_cast<const double2*>(src + (1 + j) * SE + e);
                            pv[j][2 * q] = p2.x; pv[j][2 * q + 1] = p2.y;
                        }
                    }
                }
                __syncwarp();
                if (lane == 0) obe_mbar_arrive(empty_bar + s);
                {
                    double pe[EPT][D], yge[EPT][OBE_MAX_CH], lke[EPT], te[EPT];
                    bool valid[EPT];
#pragma unroll
                    for (int e = 0; e < EPT; ++e) {
                        valid[e] = (ONE1 ? ct : 2 * (ct + (e >> 1) * OBE_CONSUMER_THREADS) + (e & 1)) < n_valid;
#pragma unroll
                        for (int j = 0; j < D; ++j) pe[e][j] = pv[j][e];
#pragma unroll
                        for (int c = 0; c < OBE_MAX_CH; ++c) yge[e][c] = 0.0;
                        lke[e] = 1.0;
                    }
                    if constexpr (SRC == OBE_SRC_DRIFT)
                        mv.template move<D, EPT>(a.u, pe, valid, b, cb, loc, base, (int)(ii & 1), ct, n_valid);
                    obe_update_vec<Model, D, SRC, EPT, true, false, Lik>(a.u, pe, wv, yge, lke, valid, invS, acc, rec,
                                                                          te);
#pragma unroll
                    for (int e = 0; e < EPT; ++e) tsum += te[e];
                    if (SRC != OBE_SRC_DRIFT && write_weights) {
#pragma unroll
                        for (int q = 0; q < EPT / 2; ++q) {
                            const int e0 = 2 * (ct + q * OBE_CONSUMER_THREADS);
                            if (e0 + 1 < n_valid) obe_st2(a.weights[cb] + base + e0, make_double2(te[2 * q], te[2 * q + 1]));
                            else if (e0 < n_valid) a.weights[cb][base + e0] = te[2 * q];
                        }
                    }
                }
            }
            if constexpr (SRC != OBE_SRC_DRIFT) {     // (the drift leaves the weights, hence the tile sums, as they are)
                tsum = obe_warp_sum(tsum);
                if (lane == 0) red[tile_par][cwarp] = tsum;
                obe_named_bar(1, OBE_CONSUMER_THREADS);
                if (ct == 0) {
                    double s = red[tile_par][0];
#pragma unroll
                    for (int w = 1; w < OBE_CONSUMER_WARPS; ++w) s += red[tile_par][w];
                    a.tile_sums[b * T + t] = s;
                    tsum_s[t] = s;
                }
            }
        }
        // ---- instance epilogue: stats block, CDF prefix row, resample flag, next pivot
        double vals[NACC];
        vals[0] = acc.sumsq; vals[1] = acc.sumt; vals[2] = acc.nzero;
#pragma unroll
        for (int j = 0; j < D; ++j) vals[3 + j] = acc.m1[j];
#pragma unroll
        for (int j = 0; j < NM2; ++j) vals[3 + D + j] = acc.m2[j];
#pragma unroll
        for (int c = 0; c < OBE_MAX_CH; ++c) vals[3 + D + NM2 + c] = acc.noise[c];
#pragma unroll
        for (int v = 0; v < NACC; ++v) {
            const double sv = obe_warp_sum(vals[v]);
            if (lane == 0) accsm[cwarp][v] = sv;
        }
        obe_named_bar(1, OBE_CONSUMER_THREADS);
        double* st = a.stats + b * OBE_STATS_LEN;
        if constexpr (SRC == OBE_SRC_DRIFT) {
            // only the moments move: totals, normaliser, N_eff, SUMT, NZERO, the tile sums, the prefix row and the
            // flag stay; the pivot of the next pass becomes the drifted mean, as after a refresh
            if (ct < NACC) {
                double sv = accsm[0][ct];
#pragma unroll
                for (int w = 1; w < OBE_CONSUMER_WARPS; ++w) sv += accsm[w][ct];
                if (ct >= 3 && ct < 3 + D) st[OBE_ST_M1 + (ct - 3)] = sv;
                else if (ct >= 3 + D && ct < 3 + D + NM2) st[OBE_ST_M2 + (ct - 3 - D)] = sv;
                else if (ct >= 3 + D + NM2 && a.u.noise_idx[ct - 3 - D - NM2] >= 0) st[OBE_ST_NOISE + (ct - 3 - D - NM2)] = sv;
                accsm[0][ct] = sv;
            }
            obe_named_bar(1, OBE_CONSUMER_THREADS);
            if (ct < D) {
                st[OBE_ST_PIVOT + ct] = rec[OBE_REC_PIVOT + ct];
                const double sumt = accsm[0][1];
                if (sumt > 0.0) a.pivot[b * OBE_MAX_DIMS + ct] = rec[OBE_REC_PIVOT + ct] + accsm[0][3 + ct] / sumt;
            }
            obe_named_bar(1, OBE_CONSUMER_THREADS);
            continue;
        }
        if (ct < NACC) {
            double sv = accsm[0][ct];
#pragma unroll
            for (int w = 1; w < OBE_CONSUMER_WARPS; ++w) sv += accsm[w][ct];
            int dst;
            if (ct == 0) dst = OBE_ST_SUMSQ;
            else if (ct == 1) dst = OBE_ST_SUMT;
            else if (ct == 2) dst = OBE_ST_NZERO;
            else if (ct < 3 + D) dst = OBE_ST_M1 + (ct - 3);
            else if (ct < 3 + D + NM2) dst = OBE_ST_M2 + (ct - 3 - D);
            else dst = OBE_ST_NOISE + (ct - 3 - D - NM2);
            st[dst] = sv;
            accsm[0][ct] = sv;        // keep the totals for thread 0 below
        }
        obe_named_bar(1, OBE_CONSUMER_THREADS);
        if (ct == 0) {
            double run = 0.0;
            double* pre = a.prefix + b * (T + 1);
            for (int t = 0; t < T; ++t) { pre[t] = run; run += tsum_s[t]; }
            pre[T] = run;
            const double total = run, ssq = accsm[0][0], sumt = accsm[0][1];
            st[OBE_ST_TOTAL] = total;
            st[OBE_ST_INVS] = 1.0 / total;
            const double neff = (total * total) / ssq;
            st[OBE_ST_NEFF] = neff;
            for (int j = 0; j < D; ++j) {
                st[OBE_ST_PIVOT + j] = rec[OBE_REC_PIVOT + j];
                if (sumt > 0.0) a.pivot[b * OBE_MAX_DIMS + j] = rec[OBE_REC_PIVOT + j] + accsm[0][3 + j] / sumt;
            }
            if (a.flag) {
                const double nn = (double)n;
                a.flag[b] = (a.force_resample || neff < 0.1 * nn || neff / nn < a.resample_threshold) ? 1 : 0;
            }
        }
        obe_named_bar(1, OBE_CONSUMER_THREADS);
    }
}

__device__ __forceinline__ long long obe_min_ll(long long a, long long b) { return a < b ? a : b; }

// ---------------------------------------------------------------------------------------------
// canonical in-tile scan: thread t owns elements [8t, 8t+8) of the tile.
//   incl[e] = (sum of earlier warps' totals, sequential) + (exclusive KS scan over lanes) + running
// The canonical CDF is cdf[j] = (tile_prefix[k] + incl_j) * (1/total), EXCEPT the last valid element
// of each tile, which is tile_prefix[k+1] * (1/total) by definition (so tile_sums may be reduced in
// any order), and the very last particle, which is exactly 1.  (One IEEE multiply by the rounded
// reciprocal instead of a divide per particle: still a fixed, monotone function of the weights that
// numpy reproduces bit for bit as cdf_unnormalised * (1.0 / total).)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tile_load_blocked(const double* __restrict__ w, long long base, long long n,
                                                  double (&v)[OBE_EPT], double wuni = 0.0) {
    const long long i0 = base + (long long)threadIdx.x * OBE_EPT;
    if (wuni > 0.0) {                      // implicit uniform weights: same values an explicit row would hold
#pragma unroll
        for (int e = 0; e < OBE_EPT; ++e) v[e] = (i0 + e < n) ? wuni : 0.0;
        return;
    }
    if (i0 + OBE_EPT <= n) {
#pragma unroll
        for (int e = 0; e < OBE_EPT; e += 2) {
            const double2 x = *reinterpret_cast<const double2*>(w + i0 + e);
            v[e] = x.x; v[e + 1] = x.y;
        }
    } else {
#pragma unroll
        for (int e = 0; e < OBE_EPT; ++e) v[e] = (i0 + e < n) ? w[i0 + e] : 0.0;
    }
}

// PRE_SYNC = false: the caller guarantees that a block barrier separates the previous readers of `sm`
// from this call (saves one barrier per tile in loops that have their own).
template <bool PRE_SYNC = true>
__device__ __forceinline__ void tile_scan_blocked(const double (&v)[OBE_EPT], double (&incl)[OBE_EPT],
                                                  double* sm /*8*/) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double run = 0.0;
#pragma unroll
    for (int e = 0; e < OBE_EPT; ++e) { run += v[e]; incl[e] = run; }
    double x = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    double ex = __shfl_up_sync(0xffffffffu, x, 1);
    if (lane == 0) ex = 0.0;
    if (PRE_SYNC) __syncthreads();
    if (lane == 31) sm[warp] = x;
    __syncthreads();
    double wb = 0.0;
    for (int w2 = 0; w2 < warp; ++w2) wb += sm[w2];
    const double base = wb + ex;
#pragma unroll
    for (int e = 0; e < OBE_EPT; ++e) incl[e] = base + incl[e];
}

// normalised canonical CDF values of this thread's 8 elements of tile k
// Sharded clouds: `offset` is the summed weight of all lower-ranked shards and inv_total the
// reciprocal of the GLOBAL total; last_shard marks the shard that holds the global last particle.
template <bool PRE_SYNC = true>
__device__ __forceinline__ void tile_cdf_blocked(const double* __restrict__ w, const double* __restrict__ prefix,
                                                 long long k, long long n, double inv_total,
                                                 double (&cn)[OBE_EPT], double* sm, double offset = 0.0,
                                                 bool last_shard = true, double wuni = 0.0) {
    double v[OBE_EPT], incl[OBE_EPT];
    const long long base = k * OBE_TILE;
    tile_load_blocked(w, base, n, v, wuni);
    tile_scan_blocked<PRE_SYNC>(v, incl, sm);
    const double p0 = obe_add(offset, prefix[k]);
    const long long last = obe_min_ll(n, base + OBE_TILE) - 1;
    const long long i0 = base + (long long)threadIdx.x * OBE_EPT;
#pragma unroll
    for (int e = 0; e < OBE_EPT; ++e) cn[e] = obe_mul(obe_add(p0, incl[e]), inv_total);
    if (i0 + OBE_EPT > last) {                 // only the thread(s) at the end of the tile
        const double c1 = (last_shard && last == n - 1) ? 1.0 : obe_mul(obe_add(offset, prefix[k + 1]), inv_total);
#pragma unroll
        for (int e = 0; e < OBE_EPT; ++e)
            if (i0 + e >= last) cn[e] = c1;
    }
}

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 + Box-Muller (restated in oracle/obe_oracle.py:device_normals)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void philox4x32_10(unsigned int c0, unsigned int c1, unsigned int c2, unsigned int c3,
                                              unsigned int k0, unsigned int k1, unsigned int (&out)[4]) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const unsigned int hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const unsigned int hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const unsigned int n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// ---------------------------------------------------------------------------------------------
// Box-Muller normals on top of Philox4x32-10 (obe_device.cuh); restated in oracle/obe_oracle.py
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float obe_sqrt_approx(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
// uniform in (0,1): ((x >> 9) + 0.5) * 2^-23, exact in fp32
__device__ __forceinline__ float u24(unsigned int x) {
    // [1,2) from the top 23 bits, minus (1 - 2^-24): 23-bit uniform on the half-integers of 2^-23
    return __uint_as_float(0x3f800000u | (x >> 9)) - 0.99999994039535522461f;
}
// Standard normals for the Liu-West jitter of output slot `slot`: one Philox4x32-10 call yields
// four 24-bit uniforms -> two Box-Muller pairs evaluated in fp32 (the jitter is a random nudge of
// scale sqrt(1-a^2)*sigma; its *value* needs no fp64 accuracy, its arithmetic after this point is
// fp64).  ctr = (slot_lo, slot_hi, call, epoch), key = seed.
template <int D>
__device__ __forceinline__ void device_normals(long long slot, unsigned long long seed, unsigned int epoch,
                                               double (&z)[D]) {
#pragma unroll
    for (int c = 0; c < (D + 3) / 4; ++c) {
        unsigned int r[4];
        philox4x32_10((unsigned int)(slot & 0xffffffffll), (unsigned int)((unsigned long long)slot >> 32),
                      (unsigned int)c, epoch, (unsigned int)(seed & 0xffffffffull), (unsigned int)(seed >> 32), r);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            if (4 * c + 2 * h < D) {
                // MUFU.LG2 / MUFU.RSQ-class approximations: ~1e-6 absolute, ample for a random nudge
                const float rad = obe_sqrt_approx(-2.0f * __logf(u24(r[2 * h])));
                float sn, cs;
                __sincosf(6.2831853071795865f * u24(r[2 * h + 1]), &sn, &cs);
                z[4 * c + 2 * h] = (double)(rad * cs);
                if (4 * c + 2 * h + 1 < D) z[4 * c + 2 * h + 1] = (double)(rad * sn);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Random-walk drift of the parameters between measurements (obe_drift): x <- x + F z, z ~ N(0, I), F F^T = Q
// ---------------------------------------------------------------------------------------------
// Normals of particle slot `slot` in drift step `epoch`: the per-slot layout of device_normals (call c gives four
// 24-bit uniforms -> two float32 Box-Muller pairs for coordinates 4c .. 4c+3) with ctr = (slot_lo, slot_hi,
// 0x40000000 | c, epoch) and key = seed ^ OBE_DRIFT_KEY, so the stream shares neither counters nor key with the
// Liu-West jitter of the same seed.  Restated in oracle/obe_oracle.py:drift_normals.
#define OBE_DRIFT_CTR 0x40000000u
#define OBE_DRIFT_KEY 0x9E3779B97F4A7C15ull
// The random walk of the batched simulator's true parameters (obe_batch_truth_drift) draws the same way with its own
// counter word and key: ctr = (instance_lo, instance_hi, 0x50000000 | c, step), key = seed ^ OBE_TRUTH_KEY.
#define OBE_TRUTH_CTR 0x50000000u
#define OBE_TRUTH_KEY 0xD1B54A32D192ED03ull
template <int D, unsigned int CTR = OBE_DRIFT_CTR, unsigned long long KEY = OBE_DRIFT_KEY>
__device__ __forceinline__ void obe_drift_normals(long long slot, unsigned long long seed, unsigned int epoch,
                                                  double (&z)[D]) {
    const unsigned long long key = seed ^ KEY;
#pragma unroll
    for (int c = 0; c < (D + 3) / 4; ++c) {
        unsigned int r[4];
        philox4x32_10((unsigned int)(slot & 0xffffffffll), (unsigned int)((unsigned long long)slot >> 32),
                      CTR | (unsigned int)c, epoch, (unsigned int)(key & 0xffffffffull),
                      (unsigned int)(key >> 32), r);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            if (4 * c + 2 * h < D) {
                const float rad = obe_sqrt_approx(-2.0f * __logf(u24(r[2 * h])));
                float sn, cs;
                __sincosf(6.2831853071795865f * u24(r[2 * h + 1]), &sn, &cs);
                z[4 * c + 2 * h] = (double)(rad * cs);
                if (4 * c + 2 * h + 1 < D) z[4 * c + 2 * h + 1] = (double)(rad * sn);
            }
        }
    }
}

// The by-value second argument of k_drift<D>.
struct ObeDriftParams {
    double f[OBE_MAX_DIMS * (OBE_MAX_DIMS + 1) / 2];   // F, lower triangle packed row-major: F[j][k] at j(j+1)/2 + k
    double* particles;        // the cloud's rows, moved in place (ObeUpdateArgs::particles is the same memory)
    double* z_out;            // optional (d, ld): the normals of every live slot
    const double* gate;       // optional: the pass runs only when (*gate != 0) == gate_on (obe_cycle, resample == 2)
    double* gate_not;         // optional: block 0 stores (*gate == 0) here before the pass starts or is skipped
    unsigned long long seed;
    unsigned int epoch;
    unsigned int rows;        // bit j: row j of F is not all zero (the other rows are neither moved nor stored)
    int gate_on;
};

// The drift as the "likelihood" of obe_update_body<ObeNoModel, D, OBE_SRC_DRIFT>: the body stages the weights and the
// particle rows, move() steps the particles of a consumer's stage and stores the moved rows, and the body then
// accumulates the moments of the moved cloud with the weights as they are (t = w, like the refresh pass).
// The constraint masks of ObeUpdateArgs reject a step: the particle keeps its previous position exactly.
struct ObeDrift {
    static constexpr bool GAUSS = false;
    ObeDriftParams q;
    __device__ __forceinline__ bool gate_open() const {
        if (!q.gate) return true;
        const bool fired = *q.gate != 0.0;
        if (q.gate_not && blockIdx.x == 0 && threadIdx.x == 0) *q.gate_not = fired ? 0.0 : 1.0;
        return fired == (q.gate_on != 0);
    }
    template <int D, int NE>
    __device__ __forceinline__ void move(const ObeUpdateArgs& a, double (&p)[NE][D], const bool (&valid)[NE],
                                         long long base, int ct, int n_valid) const {
#pragma unroll
        for (int e = 0; e < NE; ++e) {
            if (!valid[e]) continue;
            const long long slot = base + ((NE >= 2) ? 2 * (ct + (e >> 1) * OBE_CONSUMER_THREADS) + (e & 1) : ct);
            double z[D], x[D];
            obe_drift_normals<D>(slot, q.seed, q.epoch, z);
            if (q.z_out) {
#pragma unroll
                for (int j = 0; j < D; ++j) q.z_out[j * a.ld + slot] = z[j];
            }
            bool ok = true;
#pragma unroll
            for (int j = 0; j < D; ++j) {
                x[j] = p[e][j];
                if ((q.rows >> j) & 1u) {
                    double nud = 0.0;
#pragma unroll
                    for (int k = 0; k <= j; ++k) nud = fma(q.f[j * (j + 1) / 2 + k], z[k], nud);
                    x[j] += nud;
                }
                if (((a.mask_le >> j) & 1u) && x[j] <= 0.0) ok = false;
                if (((a.mask_lt >> j) & 1u) && x[j] < 0.0) ok = false;
            }
            if (ok) {
#pragma unroll
                for (int j = 0; j < D; ++j) p[e][j] = x[j];
            }
        }
#pragma unroll
        for (int j = 0; j < D; ++j) {
            if (!((q.rows >> j) & 1u)) continue;
            double* row = q.particles + j * a.ld + base;
#pragma unroll
            for (int u = 0; u < (NE >= 2 ? NE / 2 : 1); ++u) {
                const int e0 = (NE >= 2 ? 2 * (ct + u * OBE_CONSUMER_THREADS) : ct);
                if (NE >= 2 && e0 + 1 < n_valid) obe_st2(row + e0, make_double2(p[2 * u][j], p[2 * u + 1][j]));
                else if (e0 < n_valid) row[e0] = p[NE >= 2 ? 2 * u : 0][j];
            }
        }
    }
    // (never called: obe_update_vec takes the likelihood-free branch for OBE_SRC_DRIFT)
    template <int D, int NE, int NY>
    __device__ __forceinline__ void operator()(const ObeUpdateArgs&, const double (&)[NE][D], const double (&)[NE][NY],
                                               const double*, const double*, double (&lik)[NE]) const {
#pragma unroll
        for (int e = 0; e < NE; ++e) lik[e] = 1.0;
    }
};

// ---- batched drift (obe_batch_drift): the batched refresh body with ObeBDrift as its move policy ----------------
#define OBE_DRIFT_NF (OBE_MAX_DIMS * (OBE_MAX_DIMS + 1) / 2)
// The by-value second argument of k_bdrift<D, PER>.
struct ObeBDriftParams {
    double f[OBE_DRIFT_NF];   // PER == false: the F of every instance, lower triangle packed row-major
    const double* f_dev;      // PER == true: (n_inst, d, d) row-major, one F per instance (the lower triangle is read)
    double* particles[2];     // the two cloud buffers, moved in place (ObeBatchArgs::particles is the same memory)
    unsigned long long seed;
    unsigned int step;
    unsigned int rows;        // PER == false: bit j: row j of F is not all zero
};

// The factor of the instance a CTA is on (PER == true), staged by load() next to the record; two buffers, like rec_s.
struct ObeBDriftSmem {
    double f[2][OBE_DRIFT_NF];
    unsigned int nz[2][OBE_MAX_DIMS];   // row j of F is not all zero
};

// Instance b's slot i steps with obe_drift_normals(slot = (b << 32) | i): ctr = (i, b, 0x40000000 | c, step), the
// single engine's keying with the instance in the high slot word.  A step that would leave the region of the
// constraint masks is not taken; rows of F that are all zero are neither moved nor stored.
template <bool PER>
struct ObeBDrift {
    ObeBDriftParams q;
    __device__ static __forceinline__ ObeBDriftSmem& smem() {
        __shared__ ObeBDriftSmem s;
        return s;
    }
    template <int D>
    __device__ __forceinline__ void load(long long b, int buf, int ct) const {
        if constexpr (PER) {
            if (ct < D) {
                const double* row = q.f_dev + (b * D + ct) * D;
                ObeBDriftSmem& s = smem();
                bool nz = false;
                for (int k = 0; k <= ct; ++k) {
                    const double v = row[k];
                    s.f[buf][ct * (ct + 1) / 2 + k] = v;
                    nz |= v != 0.0;
                }
                s.nz[buf][ct] = nz ? 1u : 0u;
            }
        }
    }
    template <int D, int NE>
    __device__ __forceinline__ void move(const ObeUpdateArgs& a, double (&p)[NE][D], const bool (&valid)[NE],
                                         long long b, int cb, long long loc, long long base, int buf, int ct,
                                         int n_valid) const {
        const double* f = PER ? smem().f[buf] : q.f;
        unsigned int rows = q.rows;
        if constexpr (PER) {
            rows = 0u;
#pragma unroll
            for (int j = 0; j < D; ++j) rows |= smem().nz[buf][j] << j;
        }
#pragma unroll
        for (int e = 0; e < NE; ++e) {
            if (!valid[e]) continue;
            const long long slot = (b << 32) + loc + ((NE >= 2) ? 2 * (ct + (e >> 1) * OBE_CONSUMER_THREADS) + (e & 1) : ct);
            double z[D], x[D];
            obe_drift_normals<D>(slot, q.seed, q.step, z);
            bool ok = true;
#pragma unroll
            for (int j = 0; j < D; ++j) {
                x[j] = p[e][j];
                if ((rows >> j) & 1u) {
                    double nud = 0.0;
#pragma unroll
                    for (int k = 0; k <= j; ++k) nud = fma(f[j * (j + 1) / 2 + k], z[k], nud);
                    x[j] += nud;
                }
                if (((a.mask_le >> j) & 1u) && x[j] <= 0.0) ok = false;
                if (((a.mask_lt >> j) & 1u) && x[j] < 0.0) ok = false;
            }
            if (ok) {
#pragma unroll
                for (int j = 0; j < D; ++j) p[e][j] = x[j];
            }
        }
#pragma unroll
        for (int j = 0; j < D; ++j) {
            if (!((rows >> j) & 1u)) continue;
            double* row = q.particles[cb] + j * a.ld + base;
#pragma unroll
            for (int u = 0; u < (NE >= 2 ? NE / 2 : 1); ++u) {
                const int e0 = (NE >= 2 ? 2 * (ct + u * OBE_CONSUMER_THREADS) : ct);
                if (NE >= 2 && e0 + 1 < n_valid) obe_st2(row + e0, make_double2(p[2 * u][j], p[2 * u + 1][j]));
                else if (e0 < n_valid) row[e0] = p[NE >= 2 ? 2 * u : 0][j];
            }
        }
    }
};

// uniform double in (0,1) from two Philox words
__device__ __forceinline__ double obe_u53(unsigned int lo, unsigned int hi) {
    const unsigned long long x = ((unsigned long long)hi << 32) | lo;
    return ((double)(x >> 11) + 0.5) * 1.1102230246251565e-16;  // 2^-53
}
// the q-th uniform of instance b in cycle `cycle` (batched engines; restated in oracle.batch_uniform)
__device__ __forceinline__ double obe_batch_uniform(unsigned long long seed, unsigned int b, unsigned int cycle,
                                                    unsigned int q) {
    unsigned int r[4];
    philox4x32_10(q, cycle, b, 0x0B5E0001u, (unsigned int)(seed & 0xffffffffull), (unsigned int)(seed >> 32), r);
    return obe_u53(r[0], r[1]);
}

// ---------------------------------------------------------------------------------------------
// Count likelihoods of the batched engines (NVRTC likelihood modules only)
// ---------------------------------------------------------------------------------------------
// The batched simulator's counts.  Draw c of instance b in cycle t takes attempt j's two 53-bit uniforms
// u = u53(x0, x1), v = u53(x2, x3) of Philox4x32-10 with ctr = (b, t, OBE_COUNT_CTR | c, j) and key = the simulator
// seed.  The counter words of the other streams: the Liu-West jitter and the Gaussian simulator (device_normals)
// call word < 2, the packed normals 0x80000000 | D, the drift 0x40000000 | c, the truth walk 0x50000000 | c (both with
// keys of their own), the batch uniforms ctr = (q, cycle, b, 0x0B5E0001); 0x60000000 | c is none of them.
// Below a mean of 10 the count is the inversion of u through the pmf recurrence; at or above it, Hormann's
// transformed rejection (PTRS for Poisson, as numpy; BTRS for binomial, with p > 1/2 by symmetry), at most
// OBE_COUNT_TRIES attempts, NaN if every one is rejected rather than an unbounded loop on a shared GPU.
// Invalid parameters give NaN.  Non-contracted operations throughout: oracle/batched_counts.py restates it bit for bit.
#define OBE_COUNT_CTR 0x60000000u
#define OBE_COUNT_TRIES 64
#define OBE_COUNT_SWITCH 10.0
#define OBE_COUNT_MAX_TRIALS 2147483648.0
__device__ __forceinline__ void obe_count_uniforms(unsigned long long seed, long long b, unsigned int cycle, int c,
                                                   int attempt, double& u, double& v) {
    unsigned int r[4];
    philox4x32_10((unsigned int)b, cycle, OBE_COUNT_CTR | (unsigned int)c, (unsigned int)attempt,
                  (unsigned int)(seed & 0xffffffffull), (unsigned int)(seed >> 32), r);
    u = obe_u53(r[0], r[1]);
    v = obe_u53(r[2], r[3]);
}
__device__ double obe_poisson_draw(double lam, unsigned long long seed, long long b, unsigned int cycle, int c) {
    const double qnan = __longlong_as_double(0x7ff8000000000000ll);
    if (!(lam >= 0.0 && lam <= 1.7976931348623157e308)) return qnan;
    double u, v;
    if (lam < OBE_COUNT_SWITCH) {
        obe_count_uniforms(seed, b, cycle, c, 0, u, v);
        double k = 0.0, p = exp(-lam), F = p;
        while (u > F && p > 0.0) {
            k = obe_add(k, 1.0);
            p = obe_mul(p, obe_div(lam, k));
            F = obe_add(F, p);
        }
        return k;
    }
    const double slam = sqrt(lam), loglam = log(lam);
    const double bb = obe_add(0.931, obe_mul(2.53, slam));
    const double a = obe_add(-0.059, obe_mul(0.02483, bb));
    const double linvalpha = log(obe_add(1.1239, obe_div(1.1328, obe_sub(bb, 3.4))));
    const double vr = obe_sub(0.9277, obe_div(3.6224, obe_sub(bb, 2.0)));
    for (int j = 0; j < OBE_COUNT_TRIES; ++j) {
        obe_count_uniforms(seed, b, cycle, c, j, u, v);
        const double U = obe_sub(u, 0.5), us = obe_sub(0.5, fabs(U));
        const double k = floor(obe_add(obe_add(obe_mul(obe_add(obe_div(obe_mul(2.0, a), us), bb), U), lam), 0.43));
        if (us >= 0.07 && v <= vr) return k;
        if (k < 0.0 || (us < 0.013 && v > us)) continue;
        const double lhs = obe_sub(obe_add(log(v), linvalpha), log(obe_add(obe_div(a, obe_mul(us, us)), bb)));
        const double rhs = obe_sub(obe_add(-lam, obe_mul(k, loglam)), lgamma(obe_add(k, 1.0)));
        if (lhs <= rhs) return k;
    }
    return qnan;
}
__device__ double obe_binomial_draw(double n, double p, unsigned long long seed, long long b, unsigned int cycle,
                                    int c) {
    const double qnan = __longlong_as_double(0x7ff8000000000000ll);
    if (!(p >= 0.0 && p <= 1.0 && n >= 0.0 && n <= OBE_COUNT_MAX_TRIALS && n == floor(n))) return qnan;
    const bool flip = p > 0.5;
    const double q = flip ? obe_sub(1.0, p) : p;
    double u, v, k = qnan;
    if (obe_mul(n, q) < OBE_COUNT_SWITCH) {
        obe_count_uniforms(seed, b, cycle, c, 0, u, v);
        const double r = obe_div(q, obe_sub(1.0, q));
        double pk = exp(obe_mul(n, log1p(-q))), F = pk;
        k = 0.0;
        while (u > F && pk > 0.0 && k < n) {
            k = obe_add(k, 1.0);
            pk = obe_mul(pk, obe_div(obe_mul(r, obe_add(obe_sub(n, k), 1.0)), k));
            F = obe_add(F, pk);
        }
    } else {
        const double qq = obe_sub(1.0, q);
        const double spq = sqrt(obe_mul(obe_mul(n, q), qq));
        const double bb = obe_add(1.15, obe_mul(2.53, spq));
        const double a = obe_add(obe_add(-0.0873, obe_mul(0.0248, bb)), obe_mul(0.01, q));
        const double cc = obe_add(obe_mul(n, q), 0.5);
        const double alpha = obe_mul(obe_add(2.83, obe_div(5.1, bb)), spq);
        const double vr = obe_sub(0.92, obe_div(4.2, bb));
        const double m = floor(obe_mul(obe_add(n, 1.0), q));
        const double lpq = log(obe_div(q, qq));
        const double h = obe_add(lgamma(obe_add(m, 1.0)), lgamma(obe_add(obe_sub(n, m), 1.0)));
        for (int j = 0; j < OBE_COUNT_TRIES; ++j) {
            obe_count_uniforms(seed, b, cycle, c, j, u, v);
            const double U = obe_sub(u, 0.5), us = obe_sub(0.5, fabs(U));
            const double kk = floor(obe_add(obe_mul(obe_add(obe_div(obe_mul(2.0, a), us), bb), U), cc));
            if (kk < 0.0 || kk > n) continue;
            if (us >= 0.07 && v <= vr) { k = kk; break; }
            const double lhs = log(obe_div(obe_mul(v, alpha), obe_add(obe_div(a, obe_mul(us, us)), bb)));
            const double lg = obe_add(lgamma(obe_add(kk, 1.0)), lgamma(obe_add(obe_sub(n, kk), 1.0)));
            const double rhs = obe_add(obe_sub(h, lg), obe_mul(obe_sub(kk, m), lpq));
            if (lhs <= rhs) { k = kk; break; }
        }
    }
    return flip ? obe_sub(n, k) : k;
}

// The per-record side of a likelihood (Pmf of ObeLogLik): the record constant lconst(k, aux) the update subtracts,
// and the simulator's draw (COUNTS).  A user likelihood has neither: lconst 0, no simulator.
template <class Pmf>
struct ObeCounts {
    static constexpr bool COUNTS = false;
    __device__ static __forceinline__ double lconst(double, double) { return 0.0; }
};
template <>
struct ObeCounts<ObePoissonPmf> {
    static constexpr bool COUNTS = true;
    __device__ static __forceinline__ double lconst(double k, double) { return lgamma(obe_add(k, 1.0)); }
    __device__ static __forceinline__ double draw(double lam, double, unsigned long long seed, long long b,
                                                  unsigned int cycle, int c) {
        return obe_poisson_draw(lam, seed, b, cycle, c);
    }
};
template <>
struct ObeCounts<ObeBinomialPmf> {
    static constexpr bool COUNTS = true;
    __device__ static __forceinline__ double lconst(double k, double n) {
        return obe_sub(obe_sub(lgamma(obe_add(n, 1.0)), lgamma(obe_add(k, 1.0))), lgamma(obe_add(obe_sub(n, k), 1.0)));
    }
    __device__ static __forceinline__ double draw(double p, double n, unsigned long long seed, long long b,
                                                  unsigned int cycle, int c) {
        return obe_binomial_draw(n, p, seed, b, cycle, c);
    }
};

// The likelihood of the batched update (Lik of obe_update_batched_body): ObeLogLik<Pmf> with its per-record data
// read from the instance's record in shared memory -- the aux in the third element's slots (r_aux), the constants
// at OBE_REC_LCONST -- instead of from a by-value ObeLikParams.
template <class L>
struct ObeBLik;
template <class Pmf>
struct ObeBLik<ObeLogLik<Pmf>> {
    static constexpr bool GAUSS = false;
    typedef ObeCounts<Pmf> Counts;
    __device__ static __forceinline__ double lconst(double k, double aux) { return Counts::lconst(k, aux); }
    template <int D, int NE, int NY>
    __device__ __forceinline__ void operator()(const ObeUpdateArgs& a, const double (&p)[NE][D],
                                               const double (&y)[NE][NY], const double* r_y, const double* r_aux,
                                               double (&lik)[NE]) const {
        ObeLogLik<Pmf> f;
#pragma unroll
        for (int c = 0; c < OBE_MAX_CH; ++c) {
            f.q.aux[c] = r_aux[c];
            f.q.lconst[c] = r_aux[OBE_REC_LCONST - OBE_REC_ISIG + c];
        }
        f(a, p, y, r_y, r_aux, lik);
    }
};

// ---------------------------------------------------------------------------------------------
// Utility over the setting grid (obe_base.py:463-489, 628-655) fused with the argmax of
// opt_setting (obe_base.py:748).  One thread per setting; the K drawn parameter sets sit in
// shared memory and are re-used by every thread.  The (K,C,S) array of the reference
// (utility_y_space) is never materialised: numpy's two-pass population variance
// (mean = sum/K sequentially over k, var = sum((y-mean)^2)/K) is reproduced by evaluating
// the model twice, with non-contracted IEEE ops so rational models give numpy's bits.
// ---------------------------------------------------------------------------------------------
// Spacing estimators of the differential entropy of n sorted samples, as scipy.stats.differential_entropy
// (method='auto': van Es for n <= 10, Ebrahimi up to 1000) and the reference's copy of it compute them
// (obe_utils.py:116-292); window m = floor(sqrt(n) + 0.5).  Used by utility_pseudo / utility_full_kld
// (obe_base.py:491-518, 657-720).
__device__ __forceinline__ void obe_insertion_sort(double* x, int n) {
    for (int i = 1; i < n; ++i) {
        const double v = x[i];
        int j = i - 1;
        while (j >= 0 && x[j] > v) { x[j + 1] = x[j]; --j; }
        x[j + 1] = v;
    }
}
__device__ __forceinline__ double obe_entropy_sorted(const double* x, int n) {
    const int m = (int)floor(sqrt((double)n) + 0.5);
    const double nd = (double)n, md = (double)m;
    if (n <= 10) {                                      // van Es (obe_utils.py:267-275)
        double sum = 0.0;
        for (int i = 0; i + m < n; ++i) sum += log((nd + 1.0) / md * (x[i + m] - x[i]));
        double harm = 0.0;
        for (int k = m; k <= n; ++k) harm += 1.0 / (double)k;
        return 1.0 / (nd - md) * sum + harm + log(md) - log(nd + 1.0);
    }
    double sum = 0.0;                                   // Ebrahimi (obe_utils.py:278-292)
    for (int i = 0; i < n; ++i) {
        const int hi = (i + m < n) ? i + m : n - 1, lo = (i - m > 0) ? i - m : 0;
        const double i1 = (double)(i + 1);
        double ci = 2.0;
        if (i1 <= md) ci = 1.0 + (i1 - 1.0) / md;
        if (i1 >= nd - md + 1.0) ci = 1.0 + (nd - i1) / md;
        sum += log(nd * (x[hi] - x[lo]) / (ci * md));
    }
    return sum / nd;
}

// np.argmax semantics for combining candidates: the first maximum wins, NaN counts as the maximum
__device__ __forceinline__ void obe_argmax_take(double& best, long long& besti, double ov, long long oi) {
    if (oi < 0) return;
    const bool onan = (ov != ov), bnan = (best != best);
    bool take;
    if (besti < 0) take = true;
    else if (onan && bnan) take = oi < besti;
    else if (onan) take = true;
    else if (bnan) take = false;
    else take = (ov > best) || (ov == best && oi < besti);
    if (take) { best = ov; besti = oi; }
}
// block-wide argmax; the result is valid in thread 0.  bval/bidx: one slot per warp.
__device__ __forceinline__ void obe_block_argmax(double& best, long long& besti, double* bval, long long* bidx) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, best, m);
        const long long oi = __shfl_xor_sync(0xffffffffu, besti, m);
        obe_argmax_take(best, besti, ov, oi);
    }
    if (lane == 0) { bval[warp] = best; bidx[warp] = besti; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w2 = 1; w2 < (int)(blockDim.x >> 5); ++w2) obe_argmax_take(best, besti, bval[w2], bidx[w2]);
    }
}

// ---- noise variance of the design half ---------------------------------------------------------------------------
// The utility divides the spread of the K model curves at a setting by a noise variance.  ObeFixedNoise (the default,
// every pre-instantiated kernel): the constant var_noise[c], or the noise-parameter estimate.  A likelihood policy
// (design_noise='likelihood', NVRTC modules only) uses the likelihood's own variance averaged over the K draws,
// v_c = finish((sum_k nu(y_kc, a_c)) / K, a_c), summed sequentially over k, with a_c = var_noise[c] read as the design
// aux; r_c = 0 where the spread is 0, spread / v_c otherwise (+inf where v_c = 0).  A setting where some draw's output
// is invalid for the likelihood (ok() false) gets utility 0.
struct ObePoissonInfo;   // (the pmf of a likelihood policy, for the information gain: see obe_info_gain_body)
struct ObeBinomialInfo;
struct ObeNoInfo;
struct ObeFixedNoise {
    static constexpr bool LIK = false;
    static constexpr bool NU_IS_Y = false;
};
// Poisson: variance lambda.  nu = y, so v_c is the mean of the variance pass itself.  lambda < 0 / NaN / inf invalid.
struct ObePoissonNoise {
    static constexpr bool LIK = true;
    static constexpr bool NU_IS_Y = true;
    __device__ static __forceinline__ double nu(double y, double) { return y; }
    __device__ static __forceinline__ bool ok(double y, double) { return y >= 0.0 && y <= 1.7976931348623157e308; }
    __device__ static __forceinline__ double finish(double m, double) { return m; }
    typedef ObePoissonInfo Info;                         // (the information gain, obe_info_gain_body)
};
// Binomial in probability units: variance p (1 - p) / n, n = a_c the planned trials.  p outside [0, 1] / NaN invalid.
struct ObeBinomialNoise {
    static constexpr bool LIK = true;
    static constexpr bool NU_IS_Y = false;
    __device__ static __forceinline__ double nu(double y, double) { return obe_mul(y, obe_sub(1.0, y)); }
    __device__ static __forceinline__ bool ok(double y, double) { return y >= 0.0 && y <= 1.0; }
    __device__ static __forceinline__ double finish(double m, double a) { return obe_div(m, a); }
    typedef ObeBinomialInfo Info;
};
// (a user likelihood's policy, nu = its noise_var(y, a), negative or NaN invalid, is generated with its source by
// obe_model_compile_likelihood_design)
__device__ __forceinline__ double obe_design_ratio(double spread, double v) {
    return spread == 0.0 ? 0.0 : obe_div(spread, v);
}

template <class Model, class Noise = ObeFixedNoise>
__device__ void obe_utility_body(const ObeUtilityArgs& a) {
    extern __shared__ double obe_smem[];
    double* sdraw = obe_smem;  // [K][NP]
    __shared__ double bval[OBE_THREADS / 32];
    __shared__ long long bidx[OBE_THREADS / 32];
    __shared__ unsigned int is_last;
    const int tid = threadIdx.x;
    const int K = a.k;
    obe_grid_dep_wait();         // (programmatic dependent launch: the kernel that produces the draws is done)
    for (int q = tid; q < K * Model::NP; q += blockDim.x) {
        const int k = q / Model::NP, j = q % Model::NP;
        sdraw[q] = a.draws[(long long)j * K + k];
    }
    __syncthreads();
    double var_n[Model::NCH];
#pragma unroll
    for (int c = 0; c < Model::NCH; ++c) {
        var_n[c] = a.noise_from_stats ? obe_div(a.stats[OBE_ST_NOISE + c], a.stats[OBE_ST_SUMT]) : a.var_noise[c];
    }
    __shared__ double s_noise_entropy[OBE_MAX_CH];
    if (a.method == 3) {
        if (tid < Model::NCH) {                          // entropy of the noise samples (obe_base.py:718)
            double nz[OBE_MAX_DRAWS];
            for (int k = 0; k < K; ++k) nz[k] = a.kld_noise[k * Model::NCH + tid];
            obe_insertion_sort(nz, K);
            s_noise_entropy[tid] = obe_entropy_sorted(nz, K);
        }
        __syncthreads();
    }
    const double kd = (double)K;
    double best = -1.0;
    long long besti = -1;
    bool have = false;
    if (a.method == 0 && a.lanes > 1) {
        // Variance utility, `lanes` threads per setting.  One thread per setting walks 2K dependent model
        // evaluations (~30 us of pure latency at K = 30, whatever the grid size).  Here the lanes of a group
        // evaluate the K curves of their setting side by side into shared memory, ONCE, and the group's first
        // lane does numpy's two sequential passes over the stored values: same operations in the same order
        // (bit-identical utility), a critical path of K/lanes evaluations plus 2K additions.
        const int G = a.lanes, spb = (int)blockDim.x / G;
        const int sl = tid / G, g = tid % G;
        double* yv = sdraw + K * Model::NP + (long long)sl * Model::NCH * K;       // [NCH][K] of this setting
        for (long long s0 = (long long)blockIdx.x * spb; s0 < a.n_settings; s0 += (long long)gridDim.x * spb) {
            const long long s = s0 + sl;
            const bool valid = s < a.n_settings;
            if (valid) {
                double st[Model::NS > 0 ? Model::NS : 1], y[Model::NCH];
#pragma unroll
                for (int j = 0; j < Model::NS; ++j) st[j] = a.settings[j * a.lds + s];
                for (int k = g; k < K; k += G) {
                    Model::eval(st, sdraw + k * Model::NP, a.cons, y);
#pragma unroll
                    for (int c = 0; c < Model::NCH; ++c) yv[c * K + k] = y[c];
                }
            }
            __syncwarp();
            if (valid && g == 0) {
                double u = 0.0;
                bool ok = true;
#pragma unroll
                for (int c = 0; c < Model::NCH; ++c) {
                    const double* yc = yv + c * K;
                    double mean = 0.0, ss = 0.0, nus = 0.0;
                    for (int k = 0; k < K; ++k) {
                        mean = obe_add(mean, yc[k]);
                        if constexpr (Noise::LIK) {        // the first lane sums nu beside the mean
                            const double nu = Noise::nu(yc[k], var_n[c]);
                            if constexpr (!Noise::NU_IS_Y) nus = obe_add(nus, nu);
                            ok = ok & Noise::ok(yc[k], nu);
                        }
                    }
                    mean = obe_div(mean, kd);
                    for (int k = 0; k < K; ++k) {
                        const double dlt = obe_sub(yc[k], mean);
                        ss = obe_add(ss, obe_mul(dlt, dlt));
                    }
                    double r;
                    if constexpr (Noise::LIK) {
                        const double v = Noise::finish(Noise::NU_IS_Y ? mean : obe_div(nus, kd), var_n[c]);
                        r = obe_design_ratio(obe_div(ss, kd), v);
                    } else {
                        r = obe_div(obe_div(ss, kd), var_n[c]);
                    }
                    u = obe_add(u, a.log_form ? log(obe_add(1.0, r)) : r);
                }
                if (a.cost) u = obe_div(u, a.cost[s]);
                if constexpr (Noise::LIK) u = ok ? u : 0.0;
                a.utility[s] = u;
                const bool unan = (u != u), bnan = (best != best);
                if (!have || (!bnan && (unan || u > best))) { best = u; besti = s; have = true; }
            }
            __syncwarp();
        }
    } else
    for (long long s = (long long)blockIdx.x * blockDim.x + tid; s < a.n_settings;
         s += (long long)gridDim.x * blockDim.x) {
        double st[Model::NS > 0 ? Model::NS : 1];
#pragma unroll
        for (int j = 0; j < Model::NS; ++j) st[j] = a.settings[j * a.lds + s];
        double y[Model::NCH];
        double u = 0.0;
        bool ok = true;                                  // (likelihood noise: every draw's output is valid here)
        double nus[Noise::LIK ? Model::NCH : 1];         // (likelihood noise: sum_k nu(y_kc, a_c))
        if constexpr (Noise::LIK) {
#pragma unroll
            for (int c = 0; c < Model::NCH; ++c) nus[c] = 0.0;
        }
        if (a.method == 0) {
            double mean[Model::NCH], ss[Model::NCH];
#pragma unroll
            for (int c = 0; c < Model::NCH; ++c) { mean[c] = 0.0; ss[c] = 0.0; }
            // numpy's two-pass variance needs every model value twice.  With `cache` the thread parks its K x NCH
            // values in shared memory (column tid of a [K*NCH][blockDim] array: conflict-free) and the second pass
            // reads them back -- the same values in the same order, half the model evaluations (this kernel is
            // FP64-issue-bound on large grids).
            double* ycol = sdraw + K * Model::NP + tid;
            for (int k = 0; k < K; ++k) {
                Model::eval(st, sdraw + k * Model::NP, a.cons, y);
#pragma unroll
                for (int c = 0; c < Model::NCH; ++c) {
                    mean[c] = obe_add(mean[c], y[c]);
                    if (a.cache) ycol[(k * Model::NCH + c) * blockDim.x] = y[c];
                    if constexpr (Noise::LIK) {        // nu is summed in pass 1
                        const double nu = Noise::nu(y[c], var_n[c]);
                        if constexpr (!Noise::NU_IS_Y) nus[c] = obe_add(nus[c], nu);
                        ok = ok & Noise::ok(y[c], nu);
                    }
                }
            }
#pragma unroll
            for (int c = 0; c < Model::NCH; ++c) mean[c] = obe_div(mean[c], kd);
            for (int k = 0; k < K; ++k) {
                if (a.cache) {
#pragma unroll
                    for (int c = 0; c < Model::NCH; ++c) y[c] = ycol[(k * Model::NCH + c) * blockDim.x];
                } else {
                    Model::eval(st, sdraw + k * Model::NP, a.cons, y);
                }
#pragma unroll
                for (int c = 0; c < Model::NCH; ++c) {
                    const double dlt = obe_sub(y[c], mean[c]);
                    ss[c] = obe_add(ss[c], obe_mul(dlt, dlt));
                }
            }
#pragma unroll
            for (int c = 0; c < Model::NCH; ++c) {
                const double var_p = obe_div(ss[c], kd);
                double r;
                if constexpr (Noise::LIK) {
                    const double v = Noise::finish(Noise::NU_IS_Y ? mean[c] : obe_div(nus[c], kd), var_n[c]);
                    r = obe_design_ratio(var_p, v);
                } else {
                    r = obe_div(var_p, var_n[c]);
                }
                u = obe_add(u, a.log_form ? log(obe_add(1.0, r)) : r);
            }
        } else if (a.method >= 2) {
            // entropy-based utilities: the K outputs of one channel are sorted in local memory
            double ys[OBE_MAX_DRAWS];
#pragma unroll 1
            for (int c = 0; c < Model::NCH; ++c) {
                for (int k = 0; k < K; ++k) {
                    Model::eval(st, sdraw + k * Model::NP, a.cons, y);
                    double v = y[0];
#pragma unroll
                    for (int cc = 1; cc < Model::NCH; ++cc)
                        if (cc == c) v = y[cc];
                    if constexpr (Noise::LIK) {
                        const double nu = Noise::nu(v, var_n[c]);
                        nus[c] = obe_add(nus[c], nu);
                        ok = ok & Noise::ok(v, nu);
                    }
                    if (a.method == 3) v = obe_add(v, a.kld_noise[k * Model::NCH + c]);
                    ys[k] = v;
                }
                obe_insertion_sort(ys, K);
                const double h = obe_entropy_sorted(ys, K);
                if (a.method == 2) {
                    // yvar_from_entropy: exp(2H)/(2 pi e)  (obe_base.py:516-517), then var/var_n
                    const double var_p = exp(2.0 * h) / (2.0 * 3.141592653589793 * 2.718281828459045);
                    double r;
                    if constexpr (Noise::LIK) r = obe_design_ratio(var_p, Noise::finish(obe_div(nus[c], kd), var_n[c]));
                    else r = obe_div(var_p, var_n[c]);
                    u = obe_add(u, a.log_form ? log(obe_add(1.0, r)) : r);
                } else {
                    u = exp(h - s_noise_entropy[c]) - 1.0;      // obe_base.py:717-720 (single channel)
                }
            }
        } else {
            // max-min (obe_base.py:520-535, 602-626): span^2 / var_n
            double mx[Model::NCH], mn[Model::NCH];
            for (int k = 0; k < K; ++k) {
                Model::eval(st, sdraw + k * Model::NP, a.cons, y);
#pragma unroll
                for (int c = 0; c < Model::NCH; ++c) {
                    mx[c] = (k == 0 || y[c] > mx[c]) ? y[c] : mx[c];
                    mn[c] = (k == 0 || y[c] < mn[c]) ? y[c] : mn[c];
                    if constexpr (Noise::LIK) {
                        const double nu = Noise::nu(y[c], var_n[c]);
                        nus[c] = obe_add(nus[c], nu);
                        ok = ok & Noise::ok(y[c], nu);
                    }
                }
            }
#pragma unroll
            for (int c = 0; c < Model::NCH; ++c) {
                const double span = obe_sub(mx[c], mn[c]);
                double r;
                if constexpr (Noise::LIK) r = obe_design_ratio(obe_mul(span, span), Noise::finish(obe_div(nus[c], kd), var_n[c]));
                else r = obe_div(obe_mul(span, span), var_n[c]);
                u = obe_add(u, a.log_form ? log(obe_add(1.0, r)) : r);
            }
        }
        if (a.cost) u = obe_div(u, a.cost[s]);
        if constexpr (Noise::LIK) u = ok ? u : 0.0;
        a.utility[s] = u;
        // np.argmax: first maximum, NaN counts as the maximum
        const bool unan = (u != u), bnan = (best != best);
        if (!have || (!bnan && (unan || u > best))) { best = u; besti = s; have = true; }
    }
    // ---- block argmax (lowest index among equals), then the last block combines the per-block results
    const int lane = tid & 31, warp = tid >> 5;
    obe_block_argmax(best, besti, bval, bidx);
    if (tid == 0) {
        a.part_val[blockIdx.x] = best;
        a.part_idx[blockIdx.x] = besti;
        __threadfence();
        is_last = (atomicAdd(a.counter, 1u) == gridDim.x - 1) ? 1u : 0u;
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    best = 0.0; besti = -1;
    for (unsigned int b = tid; b < gridDim.x; b += blockDim.x)      // all threads: no serial tail
        obe_argmax_take(best, besti, __ldcg(a.part_val + b), __ldcg(a.part_idx + b));
    __syncthreads();
    obe_block_argmax(best, besti, bval, bidx);
    if (tid == 0) {
        *a.best_idx = besti;
        *a.best_val = best;
        if (a.best_out2) {
            a.best_out2[0] = besti;
            reinterpret_cast<double*>(a.best_out2)[1] = best;
            if (a.seq_out2) {
                __threadfence_system();                    // the pair (and the stats block of the update kernel before
                *reinterpret_cast<volatile unsigned long long*>(a.seq_out2) = a.seq_val;   // it) land before the flag
            }
        }
        *a.counter = 0u;
    }
    (void)lane; (void)warp;
}

// ---- information gain (utility method 4) ------------------------------------------------------------------------
// The mutual information between the parameters and the next count, for theta uniform over the K draws:
//   I(s) = (1/K) sum_k sum_y p_k(y) log(p_k(y) / pbar(y)),  p_k(y) = P(y | theta_k, s),  pbar = (1/K) sum_j p_j,
// in nats, in [0, log K].  Exact up to the mass outside the windows (< 1e-17 per component):
// - component k contributes the integers of [mu_k - t_k, mu_k + t_k] (clipped to the support), t = sqrt(79 var) + 27
//   (Bernstein: the tail beyond t is below exp(-t^2 / (2 (var + t/3))) < 1e-17), t = 0 for a point mass; y runs over
//   the union of the K windows, so a setting costs K |union| pmf terms;
// - log-pmfs are differences from a reference draw r with an interior output (the one closest to the mean of the K
//   outputs): delta_k(y) = log p_k(y) - log p_r(y), exact 0 for k = r and -inf off a point mass's support;
// - with M = max_k delta_k(y) and L = log1p((1/K) sum_k expm1(delta_k - M)) (log of the mixture over e^M p_r), the
//   term of draw k is pbar(y) phi(d_k), d_k = delta_k - M - L = log(p_k / pbar), phi(d) = d e^d - expm1(d) >= 0:
//   sum_k pbar phi(p_k / pbar) is the KL sum at y because sum_k (pbar - p_k) = 0, and no term cancels another, so
//   an I of 1e-12 keeps its digits;
// - pbar(y) = exp(log p_r(y) + M + L) is the only place lgamma enters.
// An invalid output (ok() false) gives the setting 0; K bitwise-equal outputs give exactly 0.
// Pmf: the likelihood's support, windows, reference log-pmf and the coefficients of delta_k(y).  n: the binomial trials.
struct ObeNoInfo {                    // (a user likelihood without a window: its support is unknown, so no kernel body)
    static constexpr bool EXACT = false;
    enum { USER = 0 };                // (an enum, not a static member: NVRTC would emit one as a global variable)
};
// (a user likelihood with a declared window: ObeUserInfo, generated with its source by compile_likelihood, is the
// policy of obe_info_gain_user_body below: ok(x, a), window(x, a, lo, hi) and logpmf(y, x, a))
// Poisson with mean x: delta_k(y) = y A_k - B_k, A_k = log1p((x_k - x_r) / x_r), B_k = x_k - x_r.
struct ObePoissonInfo {
    static constexpr bool EXACT = true;
    __device__ static __forceinline__ bool ok(double x) { return x >= 0.0 && x <= OBE_DBL_MAX; }
    __device__ static __forceinline__ bool interior(double x) { return x > 0.0; }
    __device__ static __forceinline__ void moments(double x, double, double& mu, double& var) { mu = x; var = x; }
    __device__ static __forceinline__ double top(double) { return OBE_DBL_MAX; }
    __device__ static __forceinline__ void coef(double x, double xr, double, double& A, double& B) {
        B = x - xr;
        A = log1p(B / xr);                               // x = 0: log1p(-1) = -inf
    }
    __device__ static __forceinline__ double delta(double y, double, double A, double B) {
        return y == 0.0 ? -B : fma(y, A, -B);
    }
    __device__ static __forceinline__ double logpmf(double y, double xr, double) {
        return (y == 0.0 ? 0.0 : y * log(xr)) - xr - lgamma(y + 1.0);
    }
};
// Binomial with n trials and success probability x: delta_k(y) = y A_k + (n - y) B_k, A_k = log1p((x_k - x_r) / x_r),
// B_k = log1p((x_r - x_k) / (1 - x_r)); a point mass at 0 (x = 0) or n (x = 1) has A or B = -inf.
struct ObeBinomialInfo {
    static constexpr bool EXACT = true;
    __device__ static __forceinline__ bool ok(double x) { return x >= 0.0 && x <= 1.0; }
    __device__ static __forceinline__ bool interior(double x) { return x > 0.0 && x < 1.0; }
    __device__ static __forceinline__ void moments(double x, double n, double& mu, double& var) {
        mu = n * x;
        var = mu * (1.0 - x);
    }
    __device__ static __forceinline__ double top(double n) { return n; }
    __device__ static __forceinline__ void coef(double x, double xr, double, double& A, double& B) {
        A = log1p((x - xr) / xr);
        B = log1p((xr - x) / (1.0 - xr));
    }
    __device__ static __forceinline__ double delta(double y, double n, double A, double B) {
        const double t = y < n ? (n - y) * B : 0.0;
        return y > 0.0 ? fma(y, A, t) : t;
    }
    __device__ static __forceinline__ double logpmf(double y, double xr, double n) {
        return ((lgamma(n + 1.0) - lgamma(y + 1.0)) - lgamma(n - y + 1.0)) + (y * log(xr) + (n - y) * log1p(-xr));
    }
};

// expm1(x) for x <= 5 (-inf included), from the polynomial of obe_exp_nonpos: on |x| <= ln2/2 the product r p(r)
// (no cancellation), elsewhere 2^k (1 + r p(r)) - 1, whose result is at least 0.29 in magnitude.  ~2 ulp.
__device__ __forceinline__ double obe_expm1_lean(double x) {
    const double xc = fmax(x, -708.0);
    const double t = fma(xc, 1.4426950408889634, 6755399441055744.0);
    const int k = __double2loint(t);
    const double kf = t - 6755399441055744.0;
    double r = fma(kf, -6.93147180369123816490e-01, xc);
    r = fma(kf, -1.90821492927058770002e-10, r);
    double p = obe_exp_c[0];
#pragma unroll
    for (int i = 1; i < 12; ++i) p = fma(p, r, obe_exp_c[i]);
    p = fma(p, r, 1.0);                                  // (e^r - 1) / r
    const double em = p * r;
    if (k == 0) return em;
    const double scale = __hiloint2double((k + 1023) << 20, 0);
    return x < -708.0 ? -1.0 : fma(em, scale, scale - 1.0);
}
// phi(d) = d e^d - expm1(d) = sum_{m >= 2} (m - 1) d^m / m!  (>= 0; phi(-inf) = 1): the series through m = 13 on
// |d| < 1/2 (relative truncation < 1e-13), where the closed form would cancel.
__device__ __forceinline__ double obe_info_phi(double d) {
    if (fabs(d) < 0.5) {
        double p = 1.0 / 518918400.0;
        p = fma(p, d, 1.0 / 43545600.0);
        p = fma(p, d, 1.0 / 3991680.0);
        p = fma(p, d, 1.0 / 403200.0);
        p = fma(p, d, 1.0 / 45360.0);
        p = fma(p, d, 1.0 / 5760.0);
        p = fma(p, d, 1.0 / 840.0);
        p = fma(p, d, 1.0 / 144.0);
        p = fma(p, d, 1.0 / 30.0);
        p = fma(p, d, 0.125);
        p = fma(p, d, 1.0 / 3.0);
        p = fma(p, d, 0.5);
        return p * d * d;
    }
    if (d < -708.0) return 1.0;
    const double em = obe_expm1_lean(d);
    return fma(d, em + 1.0, -em);
}

#define OBE_INFO_ARRAYS 6            // per warp: [6][K] doubles of shared memory
// The union of the K integer windows [ml_k, mh_k] of one warp: the windows ranked by start (ties by k) into sl/sh,
// merged by lane 0 into the disjoint intervals ml/mh with the cumulative counts before each in xb.  Returns the
// number of integers in the union, in every lane.  Call with the K windows visible to the warp (after __syncwarp).
// (obe_info_gain_body keeps its own inline copy of these steps: calling this helper there changes the register
// allocation and the SASS of the Poisson and binomial kernels.)
__device__ __forceinline__ double obe_info_union(int K, int lane, double* ml, double* mh, double* sl, double* sh,
                                                 double* xb) {
    for (int k = lane; k < K; k += 32) {
        const double lo = ml[k];
        int rank = 0;
        for (int j = 0; j < K; ++j) {
            const double lj = ml[j];
            rank += (lj < lo || (lj == lo && j < k)) ? 1 : 0;
        }
        sl[rank] = lo;
        sh[rank] = mh[k];
    }
    __syncwarp();
    double wtot = 0.0;
    if (lane == 0) {                         // merge into ml/mh, cumulative counts into xb
        double clo = sl[0], chi = sh[0], cum = 0.0;
        int nb = 0;
        for (int i = 1; i < K; ++i) {
            const double lo = sl[i], hi = sh[i];
            if (lo <= chi + 1.0) {
                chi = fmax(chi, hi);
            } else {
                ml[nb] = clo; mh[nb] = chi; xb[nb] = cum;
                cum += chi - clo + 1.0;
                ++nb;
                clo = lo; chi = hi;
            }
        }
        ml[nb] = clo; mh[nb] = chi; xb[nb] = cum;
        wtot = cum + (chi - clo + 1.0);
    }
    wtot = __shfl_sync(0xffffffffu, wtot, 0);
    __syncwarp();
    return wtot;
}
// One warp per setting.  The lanes evaluate the K outputs, pick the reference, build the windows (sorted by rank,
// merged by lane 0), then walk the union with a fixed assignment (lane l takes the l-th, (l+32)-th, ... value of y,
// each summing its own terms in order) and reduce in the fixed xor tree of obe_warp_sum: the same bits whatever the
// grid.  The argmax contract is obe_utility_body's.
template <class Model, class Pmf>
__device__ void obe_info_gain_body(const ObeUtilityArgs& a) {
    extern __shared__ double obe_smem[];
    double* sdraw = obe_smem;  // [K][NP]
    __shared__ double bval[OBE_THREADS / 32];
    __shared__ long long bidx[OBE_THREADS / 32];
    __shared__ unsigned int is_last;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int K = a.k;
    obe_grid_dep_wait();
    for (int q = tid; q < K * Model::NP; q += blockDim.x) {
        const int k = q / Model::NP, j = q % Model::NP;
        sdraw[q] = a.draws[(long long)j * K + k];
    }
    __syncthreads();
    const double n = a.var_noise[0];                     // binomial: the planned trials (the design aux)
    const double kd = (double)K;
    double* xa = sdraw + K * Model::NP + (long long)warp * OBE_INFO_ARRAYS * K;  // outputs, then A_k
    double* xb = xa + K;          // cumulative counts of the merged windows
    double* sl = xb + K;          // windows sorted by their start, then B_k
    double* sh = sl + K;
    double* ml = sh + K;          // windows of the K draws, then the merged union
    double* mh = ml + K;
    double best = 0.0;
    long long besti = -1;
    const int wpb = (int)(blockDim.x >> 5);
    for (long long s = (long long)blockIdx.x * wpb + warp; s < a.n_settings; s += (long long)gridDim.x * wpb) {
        double st[Model::NS > 0 ? Model::NS : 1], yv[Model::NCH];
#pragma unroll
        for (int j = 0; j < Model::NS; ++j) st[j] = a.settings[j * a.lds + s];
        for (int k = lane; k < K; k += 32) {
            Model::eval(st, sdraw + k * Model::NP, a.cons, yv);
            xa[k] = yv[0];
        }
        __syncwarp();
        const double x0 = xa[0];
        bool ok = true, same = true;
        double xsum = 0.0;
        for (int k = lane; k < K; k += 32) {
            const double x = xa[k];
            ok = ok & Pmf::ok(x);
            same = same & (x == x0);
            xsum += x;
        }
        ok = __all_sync(0xffffffffu, ok);
        same = __all_sync(0xffffffffu, same);
        double u = 0.0;
        if (ok && !same) {
            // the reference: the interior output closest to the mean, lowest k among equals
            const double mean = obe_warp_sum(xsum) / kd;
            double bd = 0.0;
            int bk = K;                                  // (K: no interior draw seen)
            double m0 = 0.0;                             // (point masses at 0, for a binomial without interior draws)
            for (int k = lane; k < K; k += 32) {
                const double x = xa[k];
                const double dist = fabs(x - mean);
                if (Pmf::interior(x) && (bk == K || dist < bd)) { bd = dist; bk = k; }
                m0 += x == 0.0 ? 1.0 : 0.0;
            }
#pragma unroll
            for (int m = 16; m >= 1; m >>= 1) {
                const double od = __shfl_xor_sync(0xffffffffu, bd, m);
                const int ok2 = __shfl_xor_sync(0xffffffffu, bk, m);
                if (ok2 != K && (bk == K || od < bd || (od == bd && ok2 < bk))) { bd = od; bk = ok2; }
            }
            if (bk == K) {
                // every draw a point mass at 0 or n (binomial), not all at the same one: the entropy of the split
                const double c0 = obe_warp_sum(m0), f0 = c0 / kd, f1 = (kd - c0) / kd;
                u = -(f0 * log(f0) + f1 * log(f1));
            } else {
                const double xr = xa[bk];
                // windows, then their rank by start (ties by k) places them in sl/sh
                for (int k = lane; k < K; k += 32) {
                    double mu, var;
                    Pmf::moments(xa[k], n, mu, var);
                    const double t = var > 0.0 ? sqrt(79.0 * var) + 27.0 : 0.0;
                    ml[k] = fmax(ceil(mu - t), 0.0);
                    mh[k] = fmin(floor(mu + t), Pmf::top(n));
                }
                __syncwarp();
                for (int k = lane; k < K; k += 32) {
                    const double lo = ml[k];
                    int rank = 0;
                    for (int j = 0; j < K; ++j) {
                        const double lj = ml[j];
                        rank += (lj < lo || (lj == lo && j < k)) ? 1 : 0;
                    }
                    sl[rank] = lo;
                    sh[rank] = mh[k];
                }
                __syncwarp();
                double wtot = 0.0;
                if (lane == 0) {                         // merge into ml/mh, cumulative counts into xb
                    double clo = sl[0], chi = sh[0], cum = 0.0;
                    int nb = 0;
                    for (int i = 1; i < K; ++i) {
                        const double lo = sl[i], hi = sh[i];
                        if (lo <= chi + 1.0) {
                            chi = fmax(chi, hi);
                        } else {
                            ml[nb] = clo; mh[nb] = chi; xb[nb] = cum;
                            cum += chi - clo + 1.0;
                            ++nb;
                            clo = lo; chi = hi;
                        }
                    }
                    ml[nb] = clo; mh[nb] = chi; xb[nb] = cum;
                    wtot = cum + (chi - clo + 1.0);
                }
                wtot = __shfl_sync(0xffffffffu, wtot, 0);
                __syncwarp();
                for (int k = lane; k < K; k += 32) {
                    double A, B;
                    Pmf::coef(xa[k], xr, n, A, B);
                    xa[k] = A;
                    sl[k] = B;
                }
                __syncwarp();
                double acc = 0.0;
                int b = 0;
                for (double j = (double)lane; j < wtot; j += 32.0) {
                    while (j >= xb[b] + (mh[b] - ml[b] + 1.0)) ++b;
                    const double y = ml[b] + (j - xb[b]);
                    double M = 0.0;                      // (delta_r = 0)
                    for (int k = 0; k < K; ++k) M = fmax(M, Pmf::delta(y, n, xa[k], sl[k]));
                    double sm = 0.0;
                    for (int k = 0; k < K; ++k) sm += obe_expm1_lean(Pmf::delta(y, n, xa[k], sl[k]) - M);
                    const double L = log1p(sm / kd);
                    double f = 0.0;
                    for (int k = 0; k < K; ++k) f += obe_info_phi((Pmf::delta(y, n, xa[k], sl[k]) - M) - L);
                    const double w = obe_exp_nonpos(fmin((Pmf::logpmf(y, xr, n) + M) + L, 0.0));
                    acc = fma(w, f, acc);
                }
                u = obe_warp_sum(acc) / kd;
            }
        }
        if (a.cost) u = obe_div(u, a.cost[s]);
        u = ok ? u : 0.0;
        if (lane == 0) {
            a.utility[s] = u;
            obe_argmax_take(best, besti, u, s);
        }
        __syncwarp();
    }
    // ---- block argmax (lowest index among equals), then the last block combines the per-block results
    obe_block_argmax(best, besti, bval, bidx);
    if (tid == 0) {
        a.part_val[blockIdx.x] = best;
        a.part_idx[blockIdx.x] = besti;
        __threadfence();
        is_last = (atomicAdd(a.counter, 1u) == gridDim.x - 1) ? 1u : 0u;
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    best = 0.0; besti = -1;
    for (unsigned int b = tid; b < gridDim.x; b += blockDim.x)
        obe_argmax_take(best, besti, __ldcg(a.part_val + b), __ldcg(a.part_idx + b));
    __syncthreads();
    obe_block_argmax(best, besti, bval, bidx);
    if (tid == 0) {
        *a.best_idx = besti;
        *a.best_val = best;
        if (a.best_out2) {
            a.best_out2[0] = besti;
            reinterpret_cast<double*>(a.best_out2)[1] = best;
            if (a.seq_out2) {
                __threadfence_system();
                *reinterpret_cast<volatile unsigned long long*>(a.seq_out2) = a.seq_val;
            }
        }
        *a.counter = 0u;
    }
}
// ---- information gain of a user likelihood with a declared window (cuda_likelihood(..., window=)) -------------
// The same I(s), with the user's log-pmf and count windows in place of the built-in closed forms:
// - draw k contributes the integers of its declared window [lo_k, hi_k]; y runs over the union of the K windows;
// - there is no analytic reference, so at each y: l_k = log p(y | x_k, a), M = max_k l_k,
//   L = log1p((1/K) sum_k expm1(l_k - M)), d_k = l_k - M - L = log(p_k / pbar), pbar = exp(M + L), and the term is
//   pbar sum_k phi(d_k) >= 0 as above.  The per-y maximum (not a reference draw) keeps draws whose supports do not
//   overlap finite; a y where every l_k = -inf contributes 0.  d_k is a difference of two user log-pmfs, so its
//   absolute error is about one ulp of |l|: |dI| <~ 1e-8 I + 1e-14 sqrt(I) (DESIGN.md section 6b);
// - l_k is recomputed, not stored (K doubles per lane per y do not fit beside 8 warps): the first pass over k keeps M
//   and sum_k expm1(l_k - M) online -- when M rises to l the sum becomes sum + expm1(M - l) (sum + k), a sum of
//   non-positive terms, so nothing cancels -- and the second pass sums phi(d_k): 2K log-pmf calls per y.
// A setting gets exactly 0 when some draw is invalid: its noise variance negative or NaN (ok() false), its window
// with NaN or non-integer bounds, lo < 0, lo > hi or hi > 2^53, some l_k NaN or +inf, or a union of more than
// OBE_INFO_USER_MAX_COUNTS integers (a careless window would otherwise hold the GPU for hours); K bitwise-equal outputs
// give exactly 0.  Same fixed lane assignment, xor-tree reduction and argmax contract as obe_info_gain_body.
#define OBE_INFO_USER_MAX_COUNTS 1048576.0
template <class Model, class Info>
__device__ void obe_info_gain_user_body(const ObeUtilityArgs& a) {
    extern __shared__ double obe_smem[];
    double* sdraw = obe_smem;  // [K][NP]
    __shared__ double bval[OBE_THREADS / 32];
    __shared__ long long bidx[OBE_THREADS / 32];
    __shared__ unsigned int is_last;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int K = a.k;
    obe_grid_dep_wait();
    for (int q = tid; q < K * Model::NP; q += blockDim.x) {
        const int k = q / Model::NP, j = q % Model::NP;
        sdraw[q] = a.draws[(long long)j * K + k];
    }
    __syncthreads();
    const double aux = a.var_noise[0];                   // the design aux, passed to the user's functions
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    const double kd = (double)K;
    double* xa = sdraw + K * Model::NP + (long long)warp * OBE_INFO_ARRAYS * K;  // outputs
    double* xb = xa + K;          // cumulative counts of the merged windows
    double* sl = xb + K;          // windows sorted by their start
    double* sh = sl + K;
    double* ml = sh + K;          // windows of the K draws, then the merged union
    double* mh = ml + K;
    double best = 0.0;
    long long besti = -1;
    const int wpb = (int)(blockDim.x >> 5);
    for (long long s = (long long)blockIdx.x * wpb + warp; s < a.n_settings; s += (long long)gridDim.x * wpb) {
        double st[Model::NS > 0 ? Model::NS : 1], yv[Model::NCH];
#pragma unroll
        for (int j = 0; j < Model::NS; ++j) st[j] = a.settings[j * a.lds + s];
        for (int k = lane; k < K; k += 32) {
            Model::eval(st, sdraw + k * Model::NP, a.cons, yv);
            xa[k] = yv[0];
        }
        __syncwarp();
        const double x0 = xa[0];
        bool ok = true, same = true;
        for (int k = lane; k < K; k += 32) {
            const double x = xa[k];
            double lo = 0.0, hi = -1.0;
            Info::window(x, aux, lo, hi);
            ok = ok & Info::ok(x, aux) & (lo >= 0.0) & (lo <= hi) & (hi <= 9007199254740992.0) &
                 (lo == floor(lo)) & (hi == floor(hi));
            same = same & (x == x0);
            ml[k] = lo;
            mh[k] = hi;
        }
        ok = __all_sync(0xffffffffu, ok);
        same = __all_sync(0xffffffffu, same);
        double u = 0.0;
        if (ok && !same) {
            __syncwarp();
            const double wtot = obe_info_union(K, lane, ml, mh, sl, sh, xb);
            if (!(wtot <= OBE_INFO_USER_MAX_COUNTS)) {
                ok = false;
            } else {
                double acc = 0.0;
                bool bad = false;
                int b = 0;
                for (double j = (double)lane; j < wtot; j += 32.0) {
                    while (j >= xb[b] + (mh[b] - ml[b] + 1.0)) ++b;
                    const double y = ml[b] + (j - xb[b]);
                    double M = -inf, sm = 0.0;           // sm = sum_{j < k} expm1(l_j - M); -1 per l_j = -inf
                    for (int k = 0; k < K; ++k) {
                        const double l = Info::logpmf(y, xa[k], aux);
                        bad = bad | !(l < inf);          // NaN or +inf
                        if (l == -inf) sm -= 1.0;
                        else if (l > M) { sm = fma(obe_expm1_lean(M - l), sm + (double)k, sm); M = l; }
                        else sm += obe_expm1_lean(l - M);
                    }
                    if (M == -inf) continue;             // (no draw reaches y)
                    const double L = log1p(sm / kd);
                    double f = 0.0;
                    for (int k = 0; k < K; ++k) f += obe_info_phi((Info::logpmf(y, xa[k], aux) - M) - L);
                    const double w = obe_exp_nonpos(fmin(M + L, 0.0));
                    acc = fma(w, f, acc);
                }
                ok = !__any_sync(0xffffffffu, bad);
                u = obe_warp_sum(acc) / kd;
            }
        }
        if (a.cost) u = obe_div(u, a.cost[s]);
        u = ok ? u : 0.0;
        if (lane == 0) {
            a.utility[s] = u;
            obe_argmax_take(best, besti, u, s);
        }
        __syncwarp();
    }
    // ---- block argmax (lowest index among equals), then the last block combines the per-block results
    obe_block_argmax(best, besti, bval, bidx);
    if (tid == 0) {
        a.part_val[blockIdx.x] = best;
        a.part_idx[blockIdx.x] = besti;
        __threadfence();
        is_last = (atomicAdd(a.counter, 1u) == gridDim.x - 1) ? 1u : 0u;
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    best = 0.0; besti = -1;
    for (unsigned int b = tid; b < gridDim.x; b += blockDim.x)
        obe_argmax_take(best, besti, __ldcg(a.part_val + b), __ldcg(a.part_idx + b));
    __syncthreads();
    obe_block_argmax(best, besti, bval, bidx);
    if (tid == 0) {
        *a.best_idx = besti;
        *a.best_val = best;
        if (a.best_out2) {
            a.best_out2[0] = besti;
            reinterpret_cast<double*>(a.best_out2)[1] = best;
            if (a.seq_out2) {
                __threadfence_system();
                *reinterpret_cast<volatile unsigned long long*>(a.seq_out2) = a.seq_val;
            }
        }
        *a.counter = 0u;
    }
}

// (the kernel of a handle without a pmf is empty: obe_utility refuses method 4 there)
template <class Model, class Pmf>
__device__ __forceinline__ void obe_info_gain_entry(const ObeUtilityArgs& a) {
    if constexpr (Pmf::EXACT) obe_info_gain_body<Model, Pmf>(a);
    else if constexpr (Pmf::USER) obe_info_gain_user_body<Model, Pmf>(a);
}

// ---------------------------------------------------------------------------------------------
// Batched design half: for every instance, K weighted draws through its canonical CDF, the
// variance utility over the setting grid and the argmax -- one CTA per instance, nothing leaves
// the device.  Same arithmetic as k_draw + obe_utility_body, so an instance reproduces what a
// single engine fed the same uniforms would choose.
// ---------------------------------------------------------------------------------------------
struct ObeBSelectArgs {
    const double* particles[2];
    const double* weights[2];
    const int* cur;
    const double* prefix;        // (B * (T + 1))
    const double* stats;         // (B * OBE_STATS_LEN)
    const double* settings;      // (s, lds)
    long long lds, n_settings;
    long long ld, np, n, n_inst;
    int tiles, k;
    long long* last_idx;         // (B) in: previous choice (sticky cost), out: new choice
    double* best_val;            // (B)
    double* utility;             // (B * S) or null
    unsigned long long seed;
    unsigned int cycle;
    int noise_from_stats, log_form, method;
    double cost_change;          // > 0: cost = cost_change except 1 at the previous choice
    double var_noise[OBE_MAX_CH];
    double cons[OBE_MAX_CONS];
};

// Noise: ObeFixedNoise, or a likelihood policy (NVRTC modules: var_noise[c] is then the design aux a_c), with
// obe_utility_body's arithmetic: nu summed beside the mean in the first pass, sequentially over k, and 0 for a setting
// where some draw is invalid for the likelihood.
template <class Model, class Noise = ObeFixedNoise>
__device__ void obe_bselect_body(const ObeBSelectArgs& a) {
    extern __shared__ double obe_smem[];
    double* cn_s = obe_smem;                       // [OBE_TILE]
    double* sdraw = obe_smem + OBE_TILE;           // [K][NP]
    __shared__ double sm[8];
    __shared__ double uq_s[OBE_MAX_DRAWS];
    __shared__ int tq_s[OBE_MAX_DRAWS];
    __shared__ long long iq_s[OBE_MAX_DRAWS];
    __shared__ double bval[OBE_THREADS / 32];
    __shared__ long long bidx[OBE_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int K = a.k, T = a.tiles;
    for (long long b = blockIdx.x; b < a.n_inst; b += gridDim.x) {
        const int cb = a.cur[b];
        const double* w = a.weights[cb] + b * a.np;
        const double* pre = a.prefix + b * (T + 1);
        const double inv_total = 1.0 / pre[T];
        if (tid < K) {
            const double u = obe_batch_uniform(a.seed, (unsigned int)b, a.cycle, (unsigned int)tid);
            int t = 0;
            for (int tt = 0; tt < T; ++tt) {
                const double c = (tt == T - 1) ? 1.0 : obe_mul(pre[tt + 1], inv_total);
                if (c <= u) t = tt + 1;
            }
            uq_s[tid] = u;
            tq_s[tid] = t < T - 1 ? t : T - 1;
        }
        __syncthreads();
        for (int t = 0; t < T; ++t) {
            double cn[OBE_EPT];
            tile_cdf_blocked(w, pre, t, a.n, inv_total, cn, sm);
#pragma unroll
            for (int e = 0; e < OBE_EPT; ++e) cn_s[tid * OBE_EPT + e] = cn[e];
            __syncthreads();
            if (tid < K && tq_s[tid] == t) {
                const long long base = (long long)t * OBE_TILE;
                const int cnt = (int)(obe_min_ll(a.n, base + OBE_TILE) - base);
                const double u = uq_s[tid];
                int lo = 0, hi = cnt;                 // first j with cn_s[j] > u
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (cn_s[mid] <= u) lo = mid + 1; else hi = mid;
                }
                iq_s[tid] = base + (lo < cnt - 1 ? lo : cnt - 1);
            }
            __syncthreads();
        }
        for (int q = tid; q < K * Model::NP; q += blockDim.x) {
            const int kq = q / Model::NP, j = q % Model::NP;
            sdraw[q] = a.particles[cb][j * a.ld + b * a.np + iq_s[kq]];
        }
        __syncthreads();
        double var_n[Model::NCH];
#pragma unroll
        for (int c = 0; c < Model::NCH; ++c) {
            const double* st = a.stats + b * OBE_STATS_LEN;
            var_n[c] = a.noise_from_stats ? obe_div(st[OBE_ST_NOISE + c], st[OBE_ST_SUMT]) : a.var_noise[c];
        }
        const long long prev_choice = a.last_idx[b];
        const double kd = (double)K;
        double best = 0.0;
        long long besti = -1;
        for (long long s = tid; s < a.n_settings; s += blockDim.x) {
            double st[Model::NS > 0 ? Model::NS : 1];
#pragma unroll
            for (int j = 0; j < Model::NS; ++j) st[j] = a.settings[j * a.lds + s];
            double y[Model::NCH], mean[Model::NCH], ss[Model::NCH];
#pragma unroll
            for (int c = 0; c < Model::NCH; ++c) { mean[c] = 0.0; ss[c] = 0.0; }
            bool ok = true;
            double nus[Noise::LIK ? Model::NCH : 1];
            if constexpr (Noise::LIK) {
#pragma unroll
                for (int c = 0; c < Model::NCH; ++c) nus[c] = 0.0;
            }
            for (int k = 0; k < K; ++k) {
                Model::eval(st, sdraw + k * Model::NP, a.cons, y);
#pragma unroll
                for (int c = 0; c < Model::NCH; ++c) {
                    mean[c] = obe_add(mean[c], y[c]);
                    if constexpr (Noise::LIK) {
                        const double nu = Noise::nu(y[c], var_n[c]);
                        if constexpr (!Noise::NU_IS_Y) nus[c] = obe_add(nus[c], nu);
                        ok = ok & Noise::ok(y[c], nu);
                    }
                }
            }
#pragma unroll
            for (int c = 0; c < Model::NCH; ++c) mean[c] = obe_div(mean[c], kd);
            for (int k = 0; k < K; ++k) {
                Model::eval(st, sdraw + k * Model::NP, a.cons, y);
#pragma unroll
                for (int c = 0; c < Model::NCH; ++c) {
                    const double dlt = obe_sub(y[c], mean[c]);
                    ss[c] = obe_add(ss[c], obe_mul(dlt, dlt));
                }
            }
            double u = 0.0;
#pragma unroll
            for (int c = 0; c < Model::NCH; ++c) {
                double r;
                if constexpr (Noise::LIK) {
                    const double v = Noise::finish(Noise::NU_IS_Y ? mean[c] : obe_div(nus[c], kd), var_n[c]);
                    r = obe_design_ratio(obe_div(ss[c], kd), v);
                } else {
                    r = obe_div(obe_div(ss[c], kd), var_n[c]);
                }
                u = obe_add(u, a.log_form ? log(obe_add(1.0, r)) : r);
            }
            if (a.cost_change > 0.0) u = obe_div(u, (s == prev_choice) ? 1.0 : a.cost_change);
            if constexpr (Noise::LIK) u = ok ? u : 0.0;
            if (a.utility) a.utility[b * a.n_settings + s] = u;
            const bool unan = (u != u), bnan = (best != best);
            if (besti < 0 || (!bnan && (unan || u > best))) { best = u; besti = s; }
        }
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, best, m);
            const long long oi = __shfl_xor_sync(0xffffffffu, besti, m);
            const bool onan = (ov != ov), bnan = (best != best);
            bool take = false;
            if (oi >= 0) {
                if (besti < 0) take = true;
                else if (onan && bnan) take = oi < besti;
                else if (onan) take = true;
                else if (bnan) take = false;
                else take = (ov > best) || (ov == best && oi < besti);
            }
            if (take) { best = ov; besti = oi; }
        }
        if (lane == 0) { bval[warp] = best; bidx[warp] = besti; }
        __syncthreads();
        if (tid == 0) {
            for (int w2 = 1; w2 < (int)(blockDim.x >> 5); ++w2) {
                const double ov = bval[w2];
                const long long oi = bidx[w2];
                const bool onan = (ov != ov), bnan = (best != best);
                bool take = false;
                if (oi >= 0) {
                    if (besti < 0) take = true;
                    else if (onan && bnan) take = oi < besti;
                    else if (onan) take = true;
                    else if (bnan) take = false;
                    else take = (ov > best) || (ov == best && oi < besti);
                }
                if (take) { best = ov; besti = oi; }
            }
            a.last_idx[b] = besti;
            a.best_val[b] = best;
        }
        __syncthreads();
    }
}

// eval_over_all_parameters (obe_base.py:298-320): y[c, i] = model(one_setting, particle_i)
template <class Model, int D>
__device__ void obe_eval_params_body(const ObeEvalArgs& a) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < a.n;
         i += (long long)gridDim.x * blockDim.x) {
        double p[D];
#pragma unroll
        for (int j = 0; j < D; ++j) p[j] = a.a[j * a.ld + i];
        double y[Model::NCH];
        Model::eval(a.fixed, p, a.cons, y);
#pragma unroll
        for (int c = 0; c < Model::NCH; ++c) a.y[c * a.ldy + i] = y[c];
    }
}

// eval_over_all_settings (obe_base.py:322-338): y[c, s] = model(setting_s, one_parameter_set)
template <class Model>
__device__ void obe_eval_settings_body(const ObeEvalArgs& a) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < a.n;
         i += (long long)gridDim.x * blockDim.x) {
        double st[Model::NS > 0 ? Model::NS : 1];
#pragma unroll
        for (int j = 0; j < Model::NS; ++j) st[j] = a.a[j * a.ld + i];
        double y[Model::NCH];
        Model::eval(st, a.fixed, a.cons, y);
#pragma unroll
        for (int c = 0; c < Model::NCH; ++c) a.y[c * a.ldy + i] = y[c];
    }
}

// ---------------------------------------------------------------------------------------------
// On-device MeasurementSimulator for the batched engines (obe_utils.py:8-53: model at the "true"
// parameters + Gaussian noise), so that a closed loop of B instances never touches the host:
// instance b measures at the setting it chose last, y_c = model_c + noise_c * z_c with
// z = device_normals(counter b, key seed, epoch cycle), and the record row of b is filled in.
// ---------------------------------------------------------------------------------------------
struct ObeBSimArgs {
    const double* true_pars;     // (NP, ld_true): true parameters of every instance, SoA
    long long ld_true;
    const double* settings;      // (s, lds)
    long long lds;
    const long long* last_idx;   // (B)
    double* record;              // (B * 12): [0:4) setting, [4:8) y, [8:12) sigma
    long long n_inst;
    const double* noise_dev;     // optional (B): per-instance noise level (all channels)
    unsigned long long seed;
    unsigned int cycle;
    int write_sigma;             // 1: also write the noise level into the sigma slots (known-sigma models)
    double noise[OBE_MAX_CH];
    double cons[OBE_MAX_CONS];
};

// Cnt: ObeCounts<void> (Gaussian noise, above), or the ObeCounts of a Poisson / binomial pmf (NVRTC modules): then
// y_c is a count drawn with mean model_c (Poisson, noise ignored) or of noise trials with success probability model_c
// (binomial), and write_sigma writes the noise level -- the trials -- into the record's third element.
template <class Model, class Cnt = ObeCounts<void>>
__device__ void obe_bsimulate_body(const ObeBSimArgs& a) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= a.n_inst) return;
    constexpr int NS = Model::NS > 0 ? Model::NS : 1, NP = Model::NP > 0 ? Model::NP : 1;
    constexpr int NCH = Model::NCH > 0 ? Model::NCH : 1;
    double s[NS], p[NP], y[NCH], z[NCH];
    const long long idx = a.last_idx[b];
#pragma unroll
    for (int j = 0; j < Model::NS; ++j) s[j] = a.settings[j * a.lds + idx];
#pragma unroll
    for (int j = 0; j < Model::NP; ++j) p[j] = a.true_pars[j * a.ld_true + b];
    Model::eval(s, p, a.cons, y);
    if constexpr (Cnt::COUNTS) {
        double* rec = a.record + b * 12;
#pragma unroll
        for (int j = 0; j < Model::NS; ++j) rec[j] = s[j];
        for (int c = 0; c < Model::NCH; ++c) {
            const double nl = a.noise_dev ? a.noise_dev[b] : a.noise[c];
            rec[4 + c] = Cnt::draw(y[c], nl, a.seed, b, a.cycle, c);
            if (a.write_sigma) rec[8 + c] = nl;
        }
        return;
    }
    device_normals<NCH>(b, a.seed, a.cycle, z);
    double* rec = a.record + b * 12;
#pragma unroll
    for (int j = 0; j < Model::NS; ++j) rec[j] = s[j];
#pragma unroll
    for (int c = 0; c < Model::NCH; ++c) {
        const double nl = a.noise_dev ? a.noise_dev[b] : a.noise[c];
        rec[4 + c] = obe_add(y[c], obe_mul(nl, z[c]));
        if (a.write_sigma) rec[8 + c] = nl;
    }
}

// ---------------------------------------------------------------------------------------------
// Multi-point update: the Bayesian updates of M measurement records (a sweep,
// demos/sweeper/obe_sweeper.py:87-101) in ONE pass over the cloud.  Per particle the running product
// t_m = nan_to_num(t_{m-1} * L_m) is carried through the M points in registers; per point the sums
// S1_m = sum t_m and S2_m = sum t_m^2 are reduced (warp shuffle -> per-warp shared rows -> per-CTA
// partials -> last CTA, all in fixed order), which gives N_eff after every point, so the last CTA
// can report the FIRST point at which the reference's resample test (particlepdf.py:236-258) would
// fire.  The caller commits the weights when no point fires (or the last one does) and otherwise
// re-runs the points up to the firing one.  The per-point normalisation of the reference is a
// particle-independent factor and is dropped (lazy normalisation); `lik_scale` removes the
// particle-independent part of 1/sigma so that long sweeps cannot underflow.
// Compute-bound (M model evaluations per particle): plain coalesced loads, no staging.
// ---------------------------------------------------------------------------------------------
#define OBE_MULTI_MAX 128
#define OBE_MULTI_NE 4
struct ObeMultiArgs {
    const double* particles; long long ld; long long n; const long long* n_dev;
    const double* w_in; double* w_out;
    const double* stats;            // of the input weights: normaliser, implicit-uniform value
    const double* records;          // (M, 12): [0:4) setting, [4:8) y, [8:12) 1/sigma (known sigma)
    int m_points, n_lik_channels, n_noise, use_choke;
    int noise_idx[OBE_MAX_CH];
    double choke;
    double lik_scale[OBE_MAX_CH];
    double cons[OBE_MAX_CONS];
    double* partials;               // (grid, 2 * OBE_MULTI_MAX)
    unsigned int* counter;
    double* sums;                   // (M, 2) out: S1_m, S2_m
    double* result;                 // out: [0] first firing point or -1, [1] its N_eff / n_total
    double threshold;               // fire when N_eff / n_total < threshold (<= 0: never)
    long long n_total;
};

template <class Model, int D>
__device__ void obe_update_multi_body(const ObeMultiArgs& a) {
    __shared__ double rec_s[OBE_MULTI_MAX * 12];
    __shared__ double acc_s[OBE_THREADS / 32][2 * OBE_MULTI_MAX];
    __shared__ unsigned int is_last;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int M = a.m_points;
    for (int q = tid; q < M * 12; q += OBE_THREADS) rec_s[q] = a.records[q];
    for (int q = lane; q < 2 * M; q += 32) acc_s[warp][q] = 0.0;
    __syncthreads();
    const long long n = a.n_dev ? *a.n_dev : a.n;
    const double invS = a.stats[OBE_ST_INVS], wuni = a.stats[OBE_ST_UNIFORM];
    constexpr int NE = OBE_MULTI_NE;   // particles per thread and round: amortises the two warp reductions per point
    constexpr int NY = Model::NCH > 0 ? Model::NCH : 1;
    for (long long base = (long long)blockIdx.x * (NE * OBE_THREADS); base < n;
         base += (long long)gridDim.x * (NE * OBE_THREADS)) {
        double p[NE][D], t[NE];
        bool valid[NE];
#pragma unroll
        for (int e = 0; e < NE; ++e) {
            const long long i = base + e * OBE_THREADS + tid;
            valid[e] = i < n;
            const long long ii = valid[e] ? i : 0;
#pragma unroll
            for (int j = 0; j < D; ++j) p[e][j] = a.particles[j * a.ld + ii];
            const double w = (wuni > 0.0) ? wuni : a.w_in[ii];
            t[e] = valid[e] ? w * invS : 0.0;
        }
        // a noise parameter is a particle coordinate: its reciprocal does not depend on the point
        double isg_p[NE][NY];
        if (a.n_noise > 0) {
#pragma unroll
            for (int e = 0; e < NE; ++e) {
#pragma unroll
                for (int c = 0; c < NY; ++c) {
                    const int ni = a.noise_idx[c];
                    double sig = 1.0;
#pragma unroll
                    for (int j = 0; j < D; ++j)
                        if (j == ni) sig = p[e][j];
                    isg_p[e][c] = obe_rcp_fast(sig);
                }
            }
        }
        for (int m = 0; m < M; ++m) {
            const double* r = rec_s + m * 12;
#pragma unroll
            for (int e = 0; e < NE; ++e) {
                double y[NY];
                ObeUpdateEval<Model>::eval(r, p[e], a.cons, y);
                double lik = 1.0;
#pragma unroll
                for (int c = 0; c < NY; ++c) {
                    if (c < a.n_lik_channels) {
                        const double isg = (a.n_noise > 0) ? isg_p[e][c] : r[8 + c];
                        const double q = (y[c] - r[4 + c]) * isg;
                        lik *= obe_exp_nonpos(-0.5 * (q * q)) * (isg * a.lik_scale[c]);
                    }
                }
                if (a.use_choke) lik = pow(lik, a.choke);
                t[e] = obe_nan_to_num_fast(t[e] * lik);
            }
            double s1 = 0.0, s2 = 0.0;
#pragma unroll
            for (int e = 0; e < NE; ++e) { s1 += t[e]; s2 += t[e] * t[e]; }
            s1 = obe_warp_sum(s1);
            s2 = obe_warp_sum(s2);
            if (lane == 0) { acc_s[warp][2 * m] += s1; acc_s[warp][2 * m + 1] += s2; }
        }
#pragma unroll
        for (int e = 0; e < NE; ++e) {
            const long long i = base + e * OBE_THREADS + tid;
            if (valid[e]) a.w_out[i] = t[e];
        }
    }
    __syncthreads();
    for (int q = tid; q < 2 * M; q += OBE_THREADS) {
        double v = 0.0;
#pragma unroll
        for (int w2 = 0; w2 < OBE_THREADS / 32; ++w2) v += acc_s[w2][q];
        a.partials[(long long)blockIdx.x * (2 * OBE_MULTI_MAX) + q] = v;
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) is_last = (atomicAdd(a.counter, 1u) == gridDim.x - 1) ? 1u : 0u;
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    for (int q = tid; q < 2 * M; q += OBE_THREADS) {
        double v = 0.0;
        for (unsigned int b = 0; b < gridDim.x; ++b) v += __ldcg(a.partials + (long long)b * (2 * OBE_MULTI_MAX) + q);
        a.sums[q] = v;
        rec_s[q] = v;
    }
    __syncthreads();
    if (tid == 0) {
        double first = -1.0, ratio = 0.0;
        if (a.threshold > 0.0) {
            for (int m = 0; m < M; ++m) {
                const double s1 = rec_s[2 * m], s2 = rec_s[2 * m + 1];
                const double frac = (s1 * s1) / s2 / (double)a.n_total;      // N_eff / n  (particlepdf.py:243-244)
                if (frac < a.threshold) { first = (double)m; ratio = frac; break; }
            }
        }
        a.result[0] = first;
        a.result[1] = ratio;
        *a.counter = 0u;
    }
}

// A model that is never evaluated: instantiates the update body for the OBE_SRC_Y /
// OBE_SRC_LIK / OBE_SRC_NONE sources (moments, tile sums, constraint mask).
struct ObeNoModel {
    enum { NS = 0, NP = 0, NCONS = 0, NCH = 0 };
    __device__ static __forceinline__ void eval(const double*, const double*, const double*, double*) {}
};

#define OBE_DEFINE_MODEL_KERNELS(MODEL, D, SUFFIX)                                                        \
    extern "C" __global__ void __launch_bounds__(OBE_UPDATE_THREADS, 1) obe_k_update_##SUFFIX(const ObeUpdateArgs a) { \
        obe_update_body<MODEL, D, OBE_SRC_MODEL>(a);                                                                   \
    }                                                                                                     \
    extern "C" __global__ void __launch_bounds__(OBE_THREADS) obe_k_evalp_##SUFFIX(const ObeEvalArgs a) {  \
        obe_eval_params_body<MODEL, D>(a);                                                                \
    }                                                                                                     \
    extern "C" __global__ void __launch_bounds__(OBE_THREADS) obe_k_multi_##SUFFIX(const ObeMultiArgs a) { \
        obe_update_multi_body<MODEL, D>(a);                                                               \
    }

#define OBE_DEFINE_BATCH_KERNELS(MODEL, D, SUFFIX)                                                              \
    extern "C" __global__ void __launch_bounds__(OBE_UPDATE_THREADS, 1) obe_k_bupdate_##SUFFIX(const ObeBatchArgs a) { \
        obe_update_batched_body<MODEL, D, OBE_SRC_MODEL>(a);                                                    \
    }                                                                                                          \
    extern "C" __global__ void __launch_bounds__(OBE_THREADS) obe_k_bselect_##SUFFIX(const ObeBSelectArgs a) {   \
        obe_bselect_body<MODEL>(a);                                                                            \
    }                                                                                                          \
    extern "C" __global__ void __launch_bounds__(OBE_THREADS) obe_k_bsim_##SUFFIX(const ObeBSimArgs a) {         \
        obe_bsimulate_body<MODEL>(a);                                                                          \
    }

// A model with a non-Gaussian likelihood LIK (compiled by NVRTC per handle): the model-evaluating update, the update
// from a supplied y_model, and the model evaluation over the cloud.  No multi-point kernel; the batched ones are
// OBE_DEFINE_LIK_BATCH_KERNELS.
#define OBE_DEFINE_LIK_KERNELS(MODEL, LIK, D)                                                                  \
    extern "C" __global__ void __launch_bounds__(OBE_UPDATE_THREADS, 1) obe_k_update_lik(const ObeUpdateArgs a, \
                                                                                         const ObeLikParams q) { \
        obe_update_body<MODEL, D, OBE_SRC_MODEL, LIK>(a, LIK{q});                                               \
    }                                                                                                          \
    extern "C" __global__ void __launch_bounds__(OBE_UPDATE_THREADS, 1) obe_k_updatey_lik(const ObeUpdateArgs a, \
                                                                                          const ObeLikParams q) { \
        obe_update_body<ObeNoModel, D, OBE_SRC_Y, LIK>(a, LIK{q});                                              \
    }                                                                                                          \
    extern "C" __global__ void __launch_bounds__(OBE_THREADS) obe_k_evalp_lik(const ObeEvalArgs a) {           \
        obe_eval_params_body<MODEL, D>(a);                                                                     \
    }

// The batched engine of a non-Gaussian likelihood LIK (compiled by NVRTC per handle, beside OBE_DEFINE_LIK_KERNELS):
// the update reads the record's third element as the aux, the selection runs NOISE (ObeFixedNoise for a plain handle,
// the likelihood's policy for a design handle), the simulator draws counts (empty for a user likelihood).
template <class Model, class L>
__device__ __forceinline__ void obe_bsim_lik_entry(const ObeBSimArgs& a) {
    if constexpr (ObeBLik<L>::Counts::COUNTS) obe_bsimulate_body<Model, typename ObeBLik<L>::Counts>(a);
}
#define OBE_DEFINE_LIK_BATCH_KERNELS(MODEL, LIK, NOISE, D)                                                      \
    extern "C" __global__ void __launch_bounds__(OBE_UPDATE_THREADS, 1) obe_k_bupdate_lik(const ObeBatchArgs a) { \
        obe_update_batched_body<MODEL, D, OBE_SRC_MODEL, ObeNoMove, ObeBLik<LIK>>(a);                           \
    }                                                                                                          \
    extern "C" __global__ void __launch_bounds__(OBE_THREADS) obe_k_bselect_lik(const ObeBSelectArgs a) {       \
        obe_bselect_body<MODEL, NOISE>(a);                                                                     \
    }                                                                                                          \
    extern "C" __global__ void __launch_bounds__(OBE_THREADS) obe_k_bsim_lik(const ObeBSimArgs a) {             \
        obe_bsim_lik_entry<MODEL, LIK>(a);                                                                     \
    }

// The utility of a likelihood-aware design (design_noise='likelihood'): var_noise[c] is the design aux a_c and NOISE
// the likelihood's noise-variance policy, NOISE::Info its pmf for the information gain (obe_k_utility_info, method 4).
// Compiled by NVRTC per handle, beside OBE_DEFINE_LIK_KERNELS.
#define OBE_DEFINE_DESIGN_KERNELS(MODEL, NOISE)                                                               \
    extern "C" __global__ void __launch_bounds__(OBE_THREADS) obe_k_utility_design(const ObeUtilityArgs a) {  \
        obe_utility_body<MODEL, NOISE>(a);                                                                    \
    }                                                                                                         \
    extern "C" __global__ void __launch_bounds__(OBE_THREADS) obe_k_evals_design(const ObeEvalArgs a) {       \
        obe_eval_settings_body<MODEL>(a);                                                                     \
    }                                                                                                         \
    extern "C" __global__ void __launch_bounds__(OBE_THREADS) obe_k_utility_info(const ObeUtilityArgs a) {    \
        obe_info_gain_entry<MODEL, NOISE::Info>(a);                                                              \
    }

#define OBE_DEFINE_GRID_KERNELS(MODEL, SUFFIX)                                                             \
    extern "C" __global__ void __launch_bounds__(OBE_THREADS) obe_k_utility_##SUFFIX(const ObeUtilityArgs a) { \
        obe_utility_body<MODEL>(a);                                                                       \
    }                                                                                                     \
    extern "C" __global__ void __launch_bounds__(OBE_THREADS) obe_k_evals_##SUFFIX(const ObeEvalArgs a) {  \
        obe_eval_settings_body<MODEL>(a);                                                                 \
    }

#endif  // OBE_DEVICE_CUH
