// obe_summary.cuh -- posterior summaries on the device: weighted quantiles and 1-D / 2-D marginal histograms.
//
// Included at the end of obe_b200.cu (it uses that file's error helpers, check_cloud and obe_sms).  None of these
// kernels writes the cloud: they read the particle rows and the weights and leave results in caller scratch.
//
// Mass is summed in unsigned 64-bit fixed point: a particle of normalised weight w (exactly as
// obe_normalized_weights computes it) carries wq = rint(w * 2^62).  Integer sums do not depend on the order of the
// additions, so every result below is the same bits at any grid size and from run to run, and a sharded cloud can
// reduce its bins with an integer all-reduce.  Particles with wq == 0 are outside the posterior everywhere.
//
//   quantile:  T = max(1, ceil(q W)) with W = sum wq (exact 128-bit product); the answer is the smallest
//              coordinate x* with sum{wq : x <= x*} >= T -- always one particle's coordinate, bit for bit
//              (a zero answer is +0.0).
//   histogram: numpy's uniform-bin rule against caller-supplied edges (np.histogram's computed index with its
//              decrement / increment correction; np.histogram2d's searchsorted rule), last bin closed, values
//              outside dropped.
//
// Quantile search.  Coordinates are mapped to order-preserving 64-bit keys.  Every requested (parameter, q) pair
// keeps an interval [lo, hi] of keys that holds its answer and the exact mass below lo.  A pass histograms, for each
// distinct interval, the particles inside it into 2^k sub-bins of 2^shift keys each (membership is an integer shift,
// exact), and a one-CTA decision kernel walks the integer bins to the sub-bin where the cumulative mass crosses T.
// Each pass takes log2(sub-bins) bits off the key span, so a pair ends after at most ceil(64 / k) passes: when its
// interval is one key (every particle in it shares one value), or earlier when it holds at most OBE_SUM_CAP
// particles -- those are then gathered in the next pass, sorted and walked exactly.  The host launches the bounded
// number of passes; the ones with nothing left to do exit on the device.
#ifndef OBE_SUMMARY_CUH
#define OBE_SUMMARY_CUH

#define OBE_SUM_THREADS 512
#define OBE_SUM_MAX_Q 16
#define OBE_SUM_MAX_PAIRS (OBE_MAX_DIMS * OBE_SUM_MAX_Q)
#define OBE_SUM_SLOTS 16384        /* shared-memory bins of one CTA: 3 u32 words = 12 B each (192 KB) */
#define OBE_SUM_LOG_KMAX 11        /* at most 2048 sub-bins per interval and pass */
#define OBE_SUM_CAP 4096           /* an interval with at most this many particles is gathered and sorted */
#define OBE_SUM_MAX_BINS 4096      /* 1-D bins per parameter */
#define OBE_SUM_MAX_BINS2D 65536   /* bins_x * bins_y */
#define OBE_SUM_WSCALE 4611686018427387904.0   /* 2^62 */

enum { OBE_SUM_DONE = 0, OBE_SUM_REFINE = 1, OBE_SUM_GATHER = 2 };

typedef unsigned long long obe_u64;

// ---------------------------------------------------------------------------------------------
// shared pieces
// ---------------------------------------------------------------------------------------------
struct ObeSumSrc {
    const double* particles;
    long long ld;
    long long n;
    const long long* n_dev;   // optional live count (n is then a bound)
    const double* weights;
    const double* stats;
};

__device__ __forceinline__ obe_u64 obe_sum_wq(double t, double inv) {
    return __double2ull_rn(__dmul_rn(obe_nan_to_num(__dmul_rn(t, inv)), OBE_SUM_WSCALE));
}
// order-preserving key of a coordinate (-0.0 and +0.0 share the key of +0.0)
__device__ __forceinline__ obe_u64 obe_sum_key(double x) {
    if (x == 0.0) x = 0.0;
    const obe_u64 u = (obe_u64)__double_as_longlong(x);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double obe_sum_value(obe_u64 k) {
    return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffull) : ~k));
}

// Calls f(row_slot, x, wq) for every live particle with wq > 0 and every row r < nr (rows[r] = parameter index),
// two particles per thread and step with 16-byte loads.  uniform weights (stats[UNIFORM] > 0) skip the weight row.
template <class F>
__device__ __forceinline__ void obe_sum_stream(const ObeSumSrc& s, const int* rows, int nr, F&& f) {
    long long n = s.n;
    if (s.n_dev) n = *s.n_dev;
    const double inv = s.stats[OBE_ST_INVS], wuni = s.stats[OBE_ST_UNIFORM];
    const bool uni = wuni > 0.0;
    const obe_u64 wq_uni = uni ? obe_sum_wq(wuni, inv) : 0ull;   // as obe_sum_uniform_wq
    const long long n_pairs = (n + 1) >> 1;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < n_pairs; p += stride) {
        const long long i = 2 * p;
        const bool two = i + 1 < n;
        obe_u64 w0, w1;
        if (uni) {
            w0 = wq_uni;
            w1 = two ? wq_uni : 0ull;
        } else if (two) {
            const double2 w = __ldcs(reinterpret_cast<const double2*>(s.weights + i));
            w0 = obe_sum_wq(w.x, inv);
            w1 = obe_sum_wq(w.y, inv);
        } else {
            w0 = obe_sum_wq(__ldcs(s.weights + i), inv);
            w1 = 0ull;
        }
        if (!(w0 | w1)) continue;
        double x0[OBE_MAX_DIMS], x1[OBE_MAX_DIMS];
#pragma unroll
        for (int r = 0; r < OBE_MAX_DIMS; ++r) {
            x0[r] = 0.0; x1[r] = 0.0;
            if (r < nr) {
                const double* row = s.particles + (long long)rows[r] * s.ld;
                if (two) {
                    const double2 x = __ldcs(reinterpret_cast<const double2*>(row + i));
                    x0[r] = x.x; x1[r] = x.y;
                } else {
                    x0[r] = __ldcs(row + i);
                }
            }
        }
        // particle by particle, its rows in order (the 2-D histogram pairs row 0 with row 1)
        if (w0) {
#pragma unroll
            for (int r = 0; r < OBE_MAX_DIMS; ++r)
                if (r < nr) f(r, x0[r], w0);
        }
        if (w1) {
#pragma unroll
            for (int r = 0; r < OBE_MAX_DIMS; ++r)
                if (r < nr) f(r, x1[r], w1);
        }
    }
}

// W = sum wq is accumulated as the sums of the 32-bit halves of every wq, which cannot wrap.  Normalised weights
// give W ~ 2^62; a weight row that sums to 4 or more (weights assigned un-normalised) would wrap the 64-bit W and is
// refused instead.  Returns 1 in that case.
__host__ __device__ __forceinline__ int obe_sum_total(obe_u64 lo, obe_u64 hi, obe_u64* W) {
    *W = (hi << 32) + lo;
    return ((hi + (lo >> 32)) >> 32) != 0ull;
}

__device__ __forceinline__ obe_u64 obe_sum_warp_add(obe_u64 v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ obe_u64 obe_sum_warp_max(obe_u64 v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const obe_u64 w = __shfl_xor_sync(0xffffffffu, v, o);
        v = w > v ? w : v;
    }
    return v;
}

// Shared-memory bins of one CTA: three u32 words per bin.  A 64-bit shared atomicAdd is a compare-and-swap loop on
// this part; the mass goes in as two native 32-bit adds instead (the low word's old value gives the carry).  With
// implicit uniform weights every particle carries the same wq, so only the count is accumulated and the mass is
// count * wq when the bins are flushed.
struct ObeSumBins {
    unsigned int* lo;
    unsigned int* hi;
    unsigned int* cnt;
    obe_u64 wq_uni;           // > 0: uniform weights
    __device__ __forceinline__ void init(unsigned char* smem, int nb, obe_u64 uni) {
        lo = reinterpret_cast<unsigned int*>(smem);
        hi = lo + nb;
        cnt = hi + nb;
        wq_uni = uni;
        for (int b = threadIdx.x; b < 3 * nb; b += blockDim.x) lo[b] = 0u;
    }
    __device__ __forceinline__ void add(int b, obe_u64 m, unsigned int c) {
        atomicAdd(cnt + b, c);
        if (!wq_uni) {
            const unsigned int l = (unsigned int)m;
            const unsigned int old = atomicAdd(lo + b, l);
            atomicAdd(hi + b, (unsigned int)(m >> 32) + (old + l < old ? 1u : 0u));
        }
    }
    // shared bins [0, nb) -> global, non-zero bins only
    __device__ __forceinline__ void flush(int nb, obe_u64* g_mass, obe_u64* g_cnt) const {
        for (int b = threadIdx.x; b < nb; b += blockDim.x) {
            const unsigned int c = cnt[b];
            if (c) {
                atomicAdd(g_mass + b, wq_uni ? wq_uni * c : ((obe_u64)hi[b] << 32) + lo[b]);
                atomicAdd(g_cnt + b, (obe_u64)c);
            }
        }
    }
};
__device__ __forceinline__ obe_u64 obe_sum_uniform_wq(const ObeSumSrc& s) {
    const double wuni = s.stats[OBE_ST_UNIFORM];
    return wuni > 0.0 ? obe_sum_wq(wuni, s.stats[OBE_ST_INVS]) : 0ull;
}

// Per-thread run cache of one histogram row: consecutive hits on one bin are summed in registers and reach the
// shared bins as one update.  A narrow cloud that piles most particles into a few bins would otherwise serialise
// on those bins' shared atomics; a broad one pays one compare per particle.
struct ObeSumRun {
    int bin;
    unsigned int cnt;
    obe_u64 mass;
    __device__ __forceinline__ void flush(ObeSumBins& sb) {
        if (cnt) sb.add(bin, mass, cnt);
    }
    __device__ __forceinline__ void add(int b, obe_u64 wq, ObeSumBins& sb) {
        if (b != bin) {
            flush(sb);
            bin = b; mass = 0ull; cnt = 0u;
        }
        mass += wq;
        ++cnt;
    }
};

// ---------------------------------------------------------------------------------------------
// range pass: W, the number of positive-weight particles, and min / max key of each requested row
// out[0] / out[OBE_SUM_RANGE_WHI] = sums of the low / high 32-bit halves of wq (see obe_sum_total), out[1] = count,
// out[2 + 2r] = ~min key, out[3 + 2r] = max key  (all zero on entry, atomicMax only)
// ---------------------------------------------------------------------------------------------
#define OBE_SUM_RANGE_WHI (2 + 2 * OBE_MAX_DIMS)
#define OBE_SUM_RANGE_LEN (3 + 2 * OBE_MAX_DIMS)
struct ObeSumRangeArgs {
    ObeSumSrc s;
    int rows[OBE_MAX_DIMS];
    int nr;
    obe_u64* out;
};

__global__ void __launch_bounds__(256) k_sum_range(const ObeSumRangeArgs a) {
    obe_u64 wlo = 0ull, whi = 0ull, cnt = 0ull;
    obe_u64 nmin[OBE_MAX_DIMS], vmax[OBE_MAX_DIMS];
#pragma unroll
    for (int r = 0; r < OBE_MAX_DIMS; ++r) { nmin[r] = 0ull; vmax[r] = 0ull; }
    obe_sum_stream(a.s, a.rows, a.nr, [&](int r, double x, obe_u64 wq) {
        const obe_u64 k = obe_sum_key(x);
#pragma unroll
        for (int rr = 0; rr < OBE_MAX_DIMS; ++rr)
            if (rr == r) {
                nmin[rr] = max(nmin[rr], ~k);
                vmax[rr] = max(vmax[rr], k);
            }
        if (r == 0) { wlo += wq & 0xffffffffull; whi += wq >> 32; ++cnt; }
    });
    wlo = obe_sum_warp_add(wlo);
    whi = obe_sum_warp_add(whi);
    cnt = obe_sum_warp_add(cnt);
    const bool lead = (threadIdx.x & 31) == 0;
    if (lead && cnt) { atomicAdd(a.out, wlo); atomicAdd(a.out + OBE_SUM_RANGE_WHI, whi); atomicAdd(a.out + 1, cnt); }
#pragma unroll
    for (int r = 0; r < OBE_MAX_DIMS; ++r) {
        if (r >= a.nr) break;
        const obe_u64 m0 = obe_sum_warp_max(nmin[r]), m1 = obe_sum_warp_max(vmax[r]);
        if (lead && cnt) { atomicMax(a.out + 2 + 2 * r, m0); atomicMax(a.out + 3 + 2 * r, m1); }
    }
}

// ---------------------------------------------------------------------------------------------
// histogram pass
// ---------------------------------------------------------------------------------------------
struct ObeSumHistArgs {
    ObeSumSrc s;
    int rows[OBE_MAX_DIMS];   // 1-D: the parameters of this launch; 2-D: rows[0] = x, rows[1] = y
    int nr;
    int bins, bins_y;         // 1-D: bins per row; 2-D: bins along x and along y
    int win0, nwin;           // 2-D: this launch counts the flat bins [win0, win0 + nwin)
    const double* edges;      // 1-D: (nr, bins + 1); 2-D: x edges (bins + 1) then y edges (bins_y + 1)
    obe_u64* mass;            // global bins of this launch (1-D: nr * bins; 2-D: nwin)
    obe_u64* count;
    obe_u64* wsum;            // optional: [0] += low and [1] += high 32-bit halves of every wq (obe_sum_total)
};

// np.histogram's bin of x for uniform edges e[0..nb] (-1: outside).  searchsorted: correct the computed index
// until it is exact, as np.histogram2d's searchsorted(edges, x, 'right') with the last edge closed.
template <bool SEARCHSORTED>
__device__ __forceinline__ int obe_sum_bin(double x, const double* __restrict__ e, int nb) {
    const double first = e[0], last = e[nb];
    if (!(x >= first && x <= last)) return -1;
    const double f = __dmul_rn(__ddiv_rn(__dsub_rn(x, first), __dsub_rn(last, first)), (double)nb);
    int k = (int)f;
    if (k >= nb) k = nb - 1;
    if (SEARCHSORTED) {
        while (k > 0 && x < e[k]) --k;
        while (k < nb - 1 && x >= e[k + 1]) ++k;
    } else {
        if (x < e[k]) --k;
        if (k != nb - 1 && x >= e[k + 1]) ++k;
    }
    return k;
}

template <bool TWO_D>
__global__ void __launch_bounds__(OBE_SUM_THREADS) k_sum_hist(const ObeSumHistArgs a) {
    extern __shared__ __align__(16) unsigned char obe_sum_smem[];
    const int nb = TWO_D ? a.nwin : a.nr * a.bins;
    ObeSumBins sb;
    sb.init(obe_sum_smem, nb, obe_sum_uniform_wq(a.s));
    __syncthreads();
    ObeSumRun run[TWO_D ? 1 : OBE_MAX_DIMS];
#pragma unroll
    for (int r = 0; r < (TWO_D ? 1 : OBE_MAX_DIMS); ++r) { run[r].bin = -1; run[r].cnt = 0u; run[r].mass = 0ull; }
    obe_u64 wlo = 0ull, whi = 0ull;
    int bx = -1;
    obe_sum_stream(a.s, a.rows, TWO_D ? 2 : a.nr, [&](int r, double x, obe_u64 wq) {
        if (TWO_D) {
            if (r == 0) {
                wlo += wq & 0xffffffffull; whi += wq >> 32;
                bx = obe_sum_bin<true>(x, a.edges, a.bins);
                return;
            }
            if (bx < 0) return;
            const int by = obe_sum_bin<true>(x, a.edges + a.bins + 1, a.bins_y);
            if (by < 0) return;
            const int b = bx * a.bins_y + by - a.win0;
            if (b >= 0 && b < a.nwin) run[0].add(b, wq, sb);
        } else {
            if (r == 0) { wlo += wq & 0xffffffffull; whi += wq >> 32; }
            const int b = obe_sum_bin<false>(x, a.edges + (long long)r * (a.bins + 1), a.bins);
            if (b < 0) return;
#pragma unroll
            for (int rr = 0; rr < OBE_MAX_DIMS; ++rr)
                if (rr == r) run[rr].add(r * a.bins + b, wq, sb);
        }
    });
#pragma unroll
    for (int r = 0; r < (TWO_D ? 1 : OBE_MAX_DIMS); ++r) run[r].flush(sb);
    if (a.wsum) {
        wlo = obe_sum_warp_add(wlo);
        whi = obe_sum_warp_add(whi);
        if ((threadIdx.x & 31) == 0) { atomicAdd(a.wsum, wlo); atomicAdd(a.wsum + 1, whi); }
    }
    __syncthreads();
    sb.flush(nb, a.mass, a.count);
}

// ---------------------------------------------------------------------------------------------
// quantile search
// ---------------------------------------------------------------------------------------------
struct ObeSumPair {
    int row, state, slot, pad;
    obe_u64 target, below, lo, hi;   // T, exact mass below lo, key interval holding the answer
};
struct ObeSumSlot {
    int row, kind, shift, pad;
    obe_u64 lo, hi;
};
struct ObeSumCtl {
    int n_slots, log_k, status, passes;  // status: 1 empty posterior, 2 W overflows; passes: passes that ran
    int row_first[OBE_MAX_DIMS], row_count[OBE_MAX_DIMS];
};
struct ObeSumQArgs {
    ObeSumSrc s;
    int rows[OBE_MAX_DIMS];
    int nr, nq, n_pairs, first;
    double q[OBE_SUM_MAX_Q];
    ObeSumCtl* ctl;
    ObeSumPair* pairs;
    ObeSumSlot* slots;
    const obe_u64* range;      // k_sum_range output
    obe_u64* g_mass;           // OBE_SUM_SLOTS
    obe_u64* g_cnt;            // OBE_SUM_SLOTS
    unsigned int* g_fill;      // OBE_SUM_MAX_PAIRS gather fill counters
    obe_u64* g_keys;           // OBE_SUM_MAX_PAIRS * OBE_SUM_CAP (key, wq) pairs
    double* result;            // n_pairs
};

// T = max(1, ceil(q W)), exact: q = m 2^-s with m < 2^53, the product m W in 128 bits
__device__ __forceinline__ obe_u64 obe_sum_target(double q, obe_u64 W) {
    if (!(q > 0.0)) return 1ull;
    int ex;
    const double f = frexp(q, &ex);
    const obe_u64 m = (obe_u64)ldexp(f, 53);
    const int s = 53 - ex;
    const obe_u64 lo = m * W, hi = __umul64hi(m, W);
    obe_u64 fl, rem;
    if (s >= 128) {
        fl = 0ull; rem = lo | hi;
    } else if (s >= 64) {
        const int t = s - 64;
        fl = hi >> t;
        rem = lo | (t ? (hi & ((1ull << t) - 1ull)) : 0ull);
    } else {
        fl = (lo >> s) | (hi << (64 - s));
        rem = lo & ((1ull << s) - 1ull);
    }
    const obe_u64 T = fl + (rem ? 1ull : 0ull);
    return T ? T : 1ull;
}

// One pass: sub-bin histograms of the REFINE intervals, (key, wq) of the GATHER intervals.
__global__ void __launch_bounds__(OBE_SUM_THREADS) k_sum_refine(const ObeSumQArgs a) {
    extern __shared__ __align__(16) unsigned char obe_sum_smem[];
    __shared__ ObeSumSlot sl[OBE_SUM_MAX_PAIRS];
    __shared__ int rfirst[OBE_MAX_DIMS], rcount[OBE_MAX_DIMS], rows[OBE_MAX_DIMS], n_act;
    const int n_slots = a.ctl->n_slots;
    if (n_slots == 0) return;                           // nothing left to refine: gated off
    const int log_k = a.ctl->log_k;
    const int nb = n_slots << log_k;
    ObeSumBins sb;
    sb.init(obe_sum_smem, nb, obe_sum_uniform_wq(a.s));
    for (int t = threadIdx.x; t < n_slots; t += blockDim.x) sl[t] = a.slots[t];
    if (threadIdx.x < OBE_MAX_DIMS) {
        rfirst[threadIdx.x] = a.ctl->row_first[threadIdx.x];
        rcount[threadIdx.x] = a.ctl->row_count[threadIdx.x];
    }
    __syncthreads();
    // rows with no open interval are not read at all
    if (threadIdx.x == 0) {
        int m = 0;
        for (int r = 0; r < a.nr; ++r)
            if (rcount[r]) rows[m++] = r;
        n_act = m;
    }
    __syncthreads();
    const int nr = n_act;
    int prow[OBE_MAX_DIMS];
#pragma unroll
    for (int r = 0; r < OBE_MAX_DIMS; ++r) prow[r] = r < nr ? a.rows[rows[r]] : 0;
    ObeSumRun run[OBE_MAX_DIMS];
#pragma unroll
    for (int r = 0; r < OBE_MAX_DIMS; ++r) { run[r].bin = -1; run[r].cnt = 0u; run[r].mass = 0ull; }
    obe_sum_stream(a.s, prow, nr, [&](int r, double x, obe_u64 wq) {
        const obe_u64 k = obe_sum_key(x);
        const int row = rows[r];
        const int s0 = rfirst[row], s1 = s0 + rcount[row];
        for (int s = s0; s < s1; ++s) {
            if (k < sl[s].lo || k > sl[s].hi) continue;
            if (sl[s].kind == OBE_SUM_REFINE) {
                const int b = (s << log_k) + (int)((k - sl[s].lo) >> sl[s].shift);
#pragma unroll
                for (int rr = 0; rr < OBE_MAX_DIMS; ++rr)
                    if (rr == r) run[rr].add(b, wq, sb);
            } else {
                const unsigned int at = atomicAdd(a.g_fill + s, 1u);
                if (at < OBE_SUM_CAP) {
                    obe_u64* dst = a.g_keys + 2 * ((long long)s * OBE_SUM_CAP + at);
                    dst[0] = k;
                    dst[1] = wq;
                }
            }
            break;                                      // the open intervals of one row are disjoint
        }
    });
#pragma unroll
    for (int r = 0; r < OBE_MAX_DIMS; ++r) run[r].flush(sb);
    __syncthreads();
    sb.flush(nb, a.g_mass, a.g_cnt);
}

__device__ __forceinline__ obe_u64 obe_sum_warp_incl_scan(obe_u64 v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const obe_u64 t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += t;
    }
    return v;
}

// Decision: one CTA.  Resolves the gathered intervals (sort + exact walk), moves every refining pair to the
// sub-bin where its cumulative mass crosses T, clears the global bins, and lays out the intervals of the next pass.
__global__ void __launch_bounds__(OBE_SUM_THREADS) k_sum_decide(const ObeSumQArgs a) {
    extern __shared__ __align__(16) unsigned char obe_sum_smem[];
    obe_u64* keys = reinterpret_cast<obe_u64*>(obe_sum_smem);      // OBE_SUM_CAP
    obe_u64* wqs = keys + OBE_SUM_CAP;                              // OBE_SUM_CAP
    __shared__ int leader[OBE_SUM_MAX_PAIRS];
    __shared__ int old_slots, old_log_k;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    ObeSumCtl* ctl = a.ctl;
    if (tid == 0) { old_slots = a.first ? 0 : ctl->n_slots; old_log_k = ctl->log_k; }
    __syncthreads();
    if (!a.first && old_slots == 0) return;            // everything was decided in an earlier pass
    if (!a.first && tid == 0) ++ctl->passes;
    if (a.first) {
        obe_u64 W;
        const int over = obe_sum_total(a.range[0], a.range[OBE_SUM_RANGE_WHI], &W);
        const obe_u64 npos = a.range[1];
        if (tid < a.n_pairs) {
            ObeSumPair p;
            p.row = tid / a.nq; p.slot = -1; p.pad = 0;
            p.target = obe_sum_target(a.q[tid % a.nq], W);
            p.below = 0ull;
            p.lo = ~a.range[2 + 2 * p.row];
            p.hi = a.range[3 + 2 * p.row];
            if (W == 0ull || over) {
                p.state = OBE_SUM_DONE;
                a.result[tid] = __longlong_as_double(0x7ff8000000000000ll);
            } else if (p.lo == p.hi) {
                p.state = OBE_SUM_DONE;
                a.result[tid] = obe_sum_value(p.lo);
            } else {
                p.state = npos <= OBE_SUM_CAP ? OBE_SUM_GATHER : OBE_SUM_REFINE;
            }
            a.pairs[tid] = p;
        }
        if (tid == 0) ctl->status = over ? 2 : (W == 0ull ? 1 : 0);
    } else {
        // gathered intervals: sort their (key, wq) by key, prefix-sum wq, and walk from the mass below
        for (int s = 0; s < old_slots; ++s) {
            if (a.slots[s].kind != OBE_SUM_GATHER) continue;
            const unsigned int fill = a.g_fill[s];
            const int c = (int)(fill < OBE_SUM_CAP ? fill : OBE_SUM_CAP);
            int np2 = 1;
            while (np2 < c) np2 <<= 1;
            for (int t = tid; t < np2; t += blockDim.x) {
                if (t < c) {
                    keys[t] = a.g_keys[2 * ((long long)s * OBE_SUM_CAP + t)];
                    wqs[t] = a.g_keys[2 * ((long long)s * OBE_SUM_CAP + t) + 1];
                } else {
                    keys[t] = ~0ull; wqs[t] = 0ull;
                }
            }
            __syncthreads();
            for (int k = 2; k <= np2; k <<= 1)                          // bitonic sort by key
                for (int j = k >> 1; j > 0; j >>= 1) {
                    for (int t = tid; t < np2; t += blockDim.x) {
                        const int u = t ^ j;
                        if (u > t) {
                            const bool up = (t & k) == 0;
                            const obe_u64 kt = keys[t], ku = keys[u];
                            if ((kt > ku) == up) {
                                keys[t] = ku; keys[u] = kt;
                                const obe_u64 w = wqs[t]; wqs[t] = wqs[u]; wqs[u] = w;
                            }
                        }
                    }
                    __syncthreads();
                }
            if (warp == 0) {                                           // inclusive prefix of wq (one warp)
                obe_u64 carry = 0ull;
                for (int b = 0; b < c; b += 32) {
                    const obe_u64 v = b + lane < c ? wqs[b + lane] : 0ull;
                    const obe_u64 incl = obe_sum_warp_incl_scan(v, lane) + carry;
                    if (b + lane < c) wqs[b + lane] = incl;
                    carry = __shfl_sync(0xffffffffu, incl, 31);
                }
            }
            __syncthreads();
            if (tid < a.n_pairs) {
                ObeSumPair& p = a.pairs[tid];
                if (p.state == OBE_SUM_GATHER && p.slot == s) {
                    const obe_u64 need = p.target - p.below;            // > 0: below < T
                    int lo = 0, hi = c;                                 // first index with prefix >= need
                    while (lo < hi) {
                        const int mid = (lo + hi) >> 1;
                        if (wqs[mid] >= need) hi = mid; else lo = mid + 1;
                    }
                    a.result[tid] = lo < c ? obe_sum_value(keys[lo]) : __longlong_as_double(0x7ff8000000000000ll);
                    p.state = OBE_SUM_DONE;
                }
            }
            __syncthreads();
        }
        // refining pairs: one warp each walks its interval's sub-bins to the crossing
        for (int t = warp; t < a.n_pairs; t += blockDim.x >> 5) {
            ObeSumPair p = a.pairs[t];
            if (p.state != OBE_SUM_REFINE) continue;
            const ObeSumSlot sl = a.slots[p.slot];
            const int nbin = (int)((sl.hi - sl.lo) >> sl.shift) + 1;
            const obe_u64* gm = a.g_mass + ((long long)p.slot << old_log_k);
            const obe_u64* gc = a.g_cnt + ((long long)p.slot << old_log_k);
            const obe_u64 need = p.target - p.below;
            obe_u64 carry = 0ull;
            int k = -1;
            obe_u64 below_k = 0ull;
            for (int b = 0; b < nbin; b += 32) {
                const obe_u64 v = b + lane < nbin ? gm[b + lane] : 0ull;
                const obe_u64 incl = obe_sum_warp_incl_scan(v, lane) + carry;
                const unsigned int hit = __ballot_sync(0xffffffffu, b + lane < nbin && incl >= need);
                if (hit) {
                    const int f = __ffs(hit) - 1;
                    k = b + f;
                    below_k = __shfl_sync(0xffffffffu, incl - v, f);
                    break;
                }
                carry = __shfl_sync(0xffffffffu, incl, 31);
            }
            if (lane == 0) {
                if (k < 0) {                                             // cannot happen: mass below + inside >= T
                    p.state = OBE_SUM_DONE;
                    a.result[t] = __longlong_as_double(0x7ff8000000000000ll);
                } else {
                    const obe_u64 lo = sl.lo + ((obe_u64)k << sl.shift);
                    const obe_u64 wm1 = (1ull << sl.shift) - 1ull;
                    const obe_u64 hi = (sl.hi - lo <= wm1) ? sl.hi : lo + wm1;
                    p.lo = lo; p.hi = hi;
                    p.below += below_k;
                    if (lo == hi) {
                        p.state = OBE_SUM_DONE;
                        a.result[t] = obe_sum_value(lo);
                    } else {
                        p.state = gc[k] <= OBE_SUM_CAP ? OBE_SUM_GATHER : OBE_SUM_REFINE;
                    }
                }
                a.pairs[t] = p;
            }
        }
        __syncthreads();
        // clear what this pass used
        for (int b = tid; b < (old_slots << old_log_k); b += blockDim.x) { a.g_mass[b] = 0ull; a.g_cnt[b] = 0ull; }
        for (int s = tid; s < old_slots; s += blockDim.x) a.g_fill[s] = 0u;
    }
    __syncthreads();
    // next pass: one slot per distinct open interval (pairs of one row are contiguous, so are their slots)
    if (tid < a.n_pairs) {
        const ObeSumPair p = a.pairs[tid];
        int l = -1;
        if (p.state != OBE_SUM_DONE) {
            for (int u = p.row * a.nq; u <= tid; ++u) {
                const ObeSumPair o = a.pairs[u];
                if (o.state != OBE_SUM_DONE && o.lo == p.lo && o.hi == p.hi) { l = u; break; }
            }
        }
        leader[tid] = l;
    }
    __syncthreads();
    if (tid == 0) {
        int ns = 0;
        for (int r = 0; r < OBE_MAX_DIMS; ++r) { ctl->row_first[r] = 0; ctl->row_count[r] = 0; }
        for (int t = 0; t < a.n_pairs; ++t) {
            if (leader[t] != t) continue;
            const ObeSumPair p = a.pairs[t];
            if (ctl->row_count[p.row] == 0) ctl->row_first[p.row] = ns;
            ++ctl->row_count[p.row];
            leader[t] = -2 - ns;                                       // slot id, told apart from pair ids
            ObeSumSlot sl;
            sl.row = p.row; sl.kind = p.state; sl.lo = p.lo; sl.hi = p.hi; sl.pad = 0; sl.shift = 0;
            a.slots[ns++] = sl;
        }
        int log_k = OBE_SUM_LOG_KMAX;
        while (log_k > 0 && (ns << log_k) > OBE_SUM_SLOTS) --log_k;
        for (int s = 0; s < ns; ++s) {
            const obe_u64 span = a.slots[s].hi - a.slots[s].lo;
            const int bits = 64 - __clzll((long long)span);
            a.slots[s].shift = bits > log_k ? bits - log_k : 0;
        }
        ctl->n_slots = ns;
        ctl->log_k = log_k;
    }
    __syncthreads();
    if (tid < a.n_pairs) {
        const int l = leader[tid];
        if (l != -1) a.pairs[tid].slot = l <= -2 ? -2 - l : -2 - leader[l];
    }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static thread_local int g_sum_passes = 0;   // streaming passes over the cloud of this thread's last summary call

struct ObeSumQScratch {
    obe_u64* range;           // OBE_SUM_RANGE_LEN
    ObeSumCtl* ctl;
    ObeSumPair* pairs;
    ObeSumSlot* slots;
    double* result;
    obe_u64* g_mass;
    obe_u64* g_cnt;
    unsigned int* g_fill;
    obe_u64* g_keys;
    size_t zero_bytes;        // [range, g_keys) is cleared at the start of a call
};
static size_t sum_q_layout(void* base, ObeSumQScratch* o) {
    size_t b = 0;
    unsigned char* p = (unsigned char*)base;
    auto take = [&](size_t bytes) { unsigned char* r = p ? p + b : nullptr; b += align_up(bytes, 256); return r; };
    ObeSumQScratch s;
    s.range = (obe_u64*)take(OBE_SUM_RANGE_LEN * sizeof(obe_u64));
    s.ctl = (ObeSumCtl*)take(sizeof(ObeSumCtl));
    s.pairs = (ObeSumPair*)take(OBE_SUM_MAX_PAIRS * sizeof(ObeSumPair));
    s.slots = (ObeSumSlot*)take(OBE_SUM_MAX_PAIRS * sizeof(ObeSumSlot));
    s.result = (double*)take(OBE_SUM_MAX_PAIRS * sizeof(double));
    s.g_mass = (obe_u64*)take(OBE_SUM_SLOTS * sizeof(obe_u64));
    s.g_cnt = (obe_u64*)take(OBE_SUM_SLOTS * sizeof(obe_u64));
    s.g_fill = (unsigned int*)take(OBE_SUM_MAX_PAIRS * sizeof(unsigned int));
    s.zero_bytes = b;
    s.g_keys = (obe_u64*)take((size_t)OBE_SUM_MAX_PAIRS * OBE_SUM_CAP * 2 * sizeof(obe_u64));
    if (o) *o = s;
    return b;
}

static ObeSumSrc sum_src(const obe_cloud_t* c) {
    ObeSumSrc s;
    s.particles = c->particles_dev; s.ld = c->ld; s.n = c->n; s.n_dev = (const long long*)c->n_dev;
    s.weights = c->weights_dev; s.stats = c->stats_dev;
    return s;
}
static int sum_check_params(const obe_cloud_t* c, const int32_t* params, int n_params) {
    if (!c || !params) return obe_fail("null argument%s%s");
    if (n_params < 1 || n_params > OBE_MAX_DIMS) return obe_fail("n_params must be 1..8%s%s");
    for (int r = 0; r < n_params; ++r)
        if (params[r] < 0 || params[r] >= c->d) return obe_fail("parameter index out of range%s%s");
    return 0;
}
// a streaming grid: as many CTAs per SM as the shared memory allows
template <class K>
static int sum_grid(K kernel, int threads, size_t smem, int* grid) {
    if (smem > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return obe_fail("cudaFuncSetAttribute(max dynamic smem): %s%s", cudaGetErrorString(e));
    }
    int per_sm = 0;
    OBE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
    *grid = obe_sms() * (per_sm > 0 ? per_sm : 1);
    return 0;
}
static int sum_range(const obe_cloud_t* c, const int32_t* params, int n_params, obe_u64* out, cudaStream_t st) {
    ObeSumRangeArgs a;
    memset(&a, 0, sizeof(a));
    a.s = sum_src(c);
    for (int r = 0; r < n_params; ++r) a.rows[r] = params[r];
    a.nr = n_params;
    a.out = out;
    int grid;
    if (sum_grid(k_sum_range, 256, 0, &grid)) return -1;
    k_sum_range<<<grid, 256, 0, st>>>(a);
    OBE_LAUNCH_CHECK("k_sum_range");
    g_sum_passes = 1;
    return 0;
}

static int sum_check_total(obe_u64 lo, obe_u64 hi, obe_u64* W) {
    if (obe_sum_total(lo, hi, W))
        return obe_fail("the normalised weights sum to 4 or more: summaries need weights that sum to 1%s%s");
    if (*W == 0) return obe_fail("the posterior is empty: every particle has zero weight%s%s");
    return 0;
}
static size_t sum_hist_bytes(int64_t rows_bins, int64_t edges) {
    return 256 + align_up((size_t)edges * sizeof(double), 256) + 2 * align_up((size_t)rows_bins * sizeof(obe_u64), 256);
}

// launches + the one synchronising read shared by the two histogram entries
static int sum_hist_run(const obe_cloud_t* c, bool two_d, const int32_t* rows, int n_rows, int bins, int bins_y,
                        const double* edges_host, int64_t n_edges, void* scratch_dev, uint64_t* mass_out,
                        uint64_t* count_out, cudaStream_t st) {
    const int64_t total = two_d ? (int64_t)bins * bins_y : (int64_t)n_rows * bins;
    unsigned char* base = (unsigned char*)scratch_dev;
    obe_u64* wsum = (obe_u64*)base;
    double* edges = (double*)(base + 256);
    obe_u64* mass = (obe_u64*)(base + 256 + align_up((size_t)n_edges * sizeof(double), 256));
    obe_u64* count = mass + align_up((size_t)total * sizeof(obe_u64), 256) / sizeof(obe_u64);
    OBE_CUDA(cudaMemsetAsync(wsum, 0, 2 * sizeof(obe_u64), st));
    OBE_CUDA(cudaMemsetAsync(mass, 0, (char*)(count + total) - (char*)mass, st));
    OBE_CUDA(cudaMemcpyAsync(edges, edges_host, n_edges * sizeof(double), cudaMemcpyHostToDevice, st));
    ObeSumHistArgs a;
    memset(&a, 0, sizeof(a));
    a.s = sum_src(c);
    a.bins = bins; a.bins_y = bins_y;
    int passes = 0;
    if (two_d) {
        a.rows[0] = rows[0]; a.rows[1] = rows[1]; a.nr = 2;
        a.edges = edges;
        for (int64_t w0 = 0; w0 < total; w0 += OBE_SUM_SLOTS) {
            a.win0 = (int)w0;
            a.nwin = (int)(total - w0 < OBE_SUM_SLOTS ? total - w0 : OBE_SUM_SLOTS);
            a.mass = mass + w0; a.count = count + w0;
            a.wsum = w0 == 0 ? wsum : nullptr;
            const size_t smem = (size_t)a.nwin * 12;
            int grid;
            if (sum_grid(k_sum_hist<true>, OBE_SUM_THREADS, smem, &grid)) return -1;
            k_sum_hist<true><<<grid, OBE_SUM_THREADS, smem, st>>>(a);
            OBE_LAUNCH_CHECK("k_sum_hist<2d>");
            ++passes;
        }
    } else {
        const int per = OBE_SUM_SLOTS / bins < OBE_MAX_DIMS ? OBE_SUM_SLOTS / bins : OBE_MAX_DIMS;
        for (int r0 = 0; r0 < n_rows; r0 += per) {
            a.nr = n_rows - r0 < per ? n_rows - r0 : per;
            for (int r = 0; r < a.nr; ++r) a.rows[r] = rows[r0 + r];
            a.edges = edges + (int64_t)r0 * (bins + 1);
            a.mass = mass + (int64_t)r0 * bins; a.count = count + (int64_t)r0 * bins;
            a.wsum = r0 == 0 ? wsum : nullptr;
            const size_t smem = (size_t)a.nr * bins * 12;
            int grid;
            if (sum_grid(k_sum_hist<false>, OBE_SUM_THREADS, smem, &grid)) return -1;
            k_sum_hist<false><<<grid, OBE_SUM_THREADS, smem, st>>>(a);
            OBE_LAUNCH_CHECK("k_sum_hist<1d>");
            ++passes;
        }
    }
    obe_u64 wh[2] = {0, 0}, W;
    OBE_CUDA(cudaMemcpyAsync(mass_out, mass, total * sizeof(obe_u64), cudaMemcpyDeviceToHost, st));
    if (count_out) OBE_CUDA(cudaMemcpyAsync(count_out, count, total * sizeof(obe_u64), cudaMemcpyDeviceToHost, st));
    OBE_CUDA(cudaMemcpyAsync(wh, wsum, sizeof(wh), cudaMemcpyDeviceToHost, st));
    OBE_CUDA(cudaStreamSynchronize(st));
    g_sum_passes = passes;
    return sum_check_total(wh[0], wh[1], &W);
}
static int sum_check_edges(const double* e, int bins) {
    if (!e) return obe_fail("null argument%s%s");
    if (!(e[0] < e[bins])) return obe_fail("bin edges must increase (edges[0] < edges[bins])%s%s");
    for (int k = 0; k <= bins; ++k) {
        if (!std::isfinite(e[k])) return obe_fail("bin edges must be finite%s%s");
        if (k && e[k] < e[k - 1]) return obe_fail("bin edges must not decrease%s%s");
    }
    return 0;
}

extern "C" {

int obe_summary_passes(void) { return g_sum_passes; }
size_t obe_quantile_scratch_bytes(int n_params, int n_q) {
    (void)n_params; (void)n_q;
    return sum_q_layout(nullptr, nullptr);
}
size_t obe_histogram_scratch_bytes(int n_params, int bins) {
    return sum_hist_bytes((int64_t)n_params * bins, (int64_t)n_params * (bins + 1));
}
size_t obe_histogram2d_scratch_bytes(int bins_x, int bins_y) {
    return sum_hist_bytes((int64_t)bins_x * bins_y, (int64_t)bins_x + bins_y + 2);
}

int obe_summary_range(const obe_cloud_t* c, const int32_t* params, int n_params, void* scratch_dev, double* lo_out,
                      double* hi_out, void* stream) {
    if (sum_check_params(c, params, n_params)) return -1;
    if (!scratch_dev || !lo_out || !hi_out) return obe_fail("null argument%s%s");
    if (check_cloud(c)) return -1;
    cudaStream_t st = (cudaStream_t)stream;
    obe_u64* out = (obe_u64*)scratch_dev;
    const size_t nb = OBE_SUM_RANGE_LEN * sizeof(obe_u64);
    OBE_CUDA(cudaMemsetAsync(out, 0, nb, st));
    if (sum_range(c, params, n_params, out, st)) return -1;
    obe_u64 host[OBE_SUM_RANGE_LEN], W;
    OBE_CUDA(cudaMemcpyAsync(host, out, nb, cudaMemcpyDeviceToHost, st));
    OBE_CUDA(cudaStreamSynchronize(st));
    if (sum_check_total(host[0], host[OBE_SUM_RANGE_WHI], &W)) return -1;
    for (int r = 0; r < n_params; ++r) {
        const obe_u64 kmin = ~host[2 + 2 * r], kmax = host[3 + 2 * r];
        obe_u64 b = (kmin >> 63) ? (kmin & 0x7fffffffffffffffull) : ~kmin;
        memcpy(&lo_out[r], &b, 8);
        b = (kmax >> 63) ? (kmax & 0x7fffffffffffffffull) : ~kmax;
        memcpy(&hi_out[r], &b, 8);
    }
    return 0;
}

int obe_quantile(const obe_cloud_t* c, const int32_t* params, int n_params, const double* q, int n_q,
                 void* scratch_dev, double* out, void* stream) {
    if (sum_check_params(c, params, n_params)) return -1;
    if (!q || !scratch_dev || !out) return obe_fail("null argument%s%s");
    if (n_q < 1 || n_q > OBE_SUM_MAX_Q) return obe_fail("n_q must be 1..16%s%s");
    for (int i = 0; i < n_q; ++i)
        if (!(q[i] >= 0.0 && q[i] <= 1.0)) return obe_fail("quantile levels must lie in [0, 1]%s%s");
    if (check_cloud(c)) return -1;
    cudaStream_t st = (cudaStream_t)stream;
    ObeSumQScratch s;
    sum_q_layout(scratch_dev, &s);
    OBE_CUDA(cudaMemsetAsync(scratch_dev, 0, s.zero_bytes, st));
    if (sum_range(c, params, n_params, s.range, st)) return -1;
    ObeSumQArgs a;
    memset(&a, 0, sizeof(a));
    a.s = sum_src(c);
    for (int r = 0; r < n_params; ++r) a.rows[r] = params[r];
    a.nr = n_params; a.nq = n_q; a.n_pairs = n_params * n_q;
    for (int i = 0; i < n_q; ++i) a.q[i] = q[i];
    a.ctl = s.ctl; a.pairs = s.pairs; a.slots = s.slots; a.range = s.range;
    a.g_mass = s.g_mass; a.g_cnt = s.g_cnt; a.g_fill = s.g_fill; a.g_keys = s.g_keys; a.result = s.result;
    const size_t dsmem = (size_t)OBE_SUM_CAP * 2 * sizeof(obe_u64);
    OBE_CUDA(cudaFuncSetAttribute(k_sum_decide, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dsmem));
    a.first = 1;
    k_sum_decide<<<1, OBE_SUM_THREADS, dsmem, st>>>(a);
    OBE_LAUNCH_CHECK("k_sum_decide");
    a.first = 0;
    // every pass takes at least log_k bits off each open key span: after ceil(64 / log_k) passes all are decided
    int log_k = OBE_SUM_LOG_KMAX;
    while (log_k > 0 && (a.n_pairs << log_k) > OBE_SUM_SLOTS) --log_k;
    const int passes = (64 + log_k - 1) / log_k;
    const size_t rsmem = (size_t)OBE_SUM_SLOTS * 12;
    int grid;
    if (sum_grid(k_sum_refine, OBE_SUM_THREADS, rsmem, &grid)) return -1;
    for (int p = 0; p < passes; ++p) {
        k_sum_refine<<<grid, OBE_SUM_THREADS, rsmem, st>>>(a);
        OBE_LAUNCH_CHECK("k_sum_refine");
        k_sum_decide<<<1, OBE_SUM_THREADS, dsmem, st>>>(a);
        OBE_LAUNCH_CHECK("k_sum_decide");
    }
    ObeSumCtl ctl;
    OBE_CUDA(cudaMemcpyAsync(out, s.result, a.n_pairs * sizeof(double), cudaMemcpyDeviceToHost, st));
    OBE_CUDA(cudaMemcpyAsync(&ctl, s.ctl, sizeof(ctl), cudaMemcpyDeviceToHost, st));
    OBE_CUDA(cudaStreamSynchronize(st));
    g_sum_passes = 1 + ctl.passes;
    if (ctl.status == 1) return obe_fail("the posterior is empty: every particle has zero weight%s%s");
    if (ctl.status == 2)
        return obe_fail("the normalised weights sum to 4 or more: summaries need weights that sum to 1%s%s");
    return 0;
}

int obe_histogram(const obe_cloud_t* c, const int32_t* params, int n_params, const double* edges, int bins,
                  void* scratch_dev, uint64_t* mass_out, uint64_t* count_out, void* stream) {
    if (sum_check_params(c, params, n_params)) return -1;
    if (!edges || !scratch_dev || !mass_out) return obe_fail("null argument%s%s");
    if (bins < 1 || bins > OBE_SUM_MAX_BINS) return obe_fail("bins must be 1..4096%s%s");
    for (int r = 0; r < n_params; ++r)
        if (sum_check_edges(edges + (int64_t)r * (bins + 1), bins)) return -1;
    if (check_cloud(c)) return -1;
    return sum_hist_run(c, false, params, n_params, bins, 0, edges, (int64_t)n_params * (bins + 1), scratch_dev,
                        mass_out, count_out, (cudaStream_t)stream);
}

int obe_histogram2d(const obe_cloud_t* c, int param_x, int param_y, const double* xedges, int bins_x,
                    const double* yedges, int bins_y, void* scratch_dev, uint64_t* mass_out, uint64_t* count_out,
                    void* stream) {
    const int32_t rows[2] = {param_x, param_y};
    if (sum_check_params(c, rows, 2)) return -1;
    if (!xedges || !yedges || !scratch_dev || !mass_out) return obe_fail("null argument%s%s");
    if (bins_x < 1 || bins_y < 1 || (int64_t)bins_x * bins_y > OBE_SUM_MAX_BINS2D)
        return obe_fail("bins must be >= 1 along each axis with bins_x * bins_y <= 65536%s%s");
    if (sum_check_edges(xedges, bins_x) || sum_check_edges(yedges, bins_y)) return -1;
    if (check_cloud(c)) return -1;
    std::vector<double> e((size_t)bins_x + bins_y + 2);
    memcpy(e.data(), xedges, (bins_x + 1) * sizeof(double));
    memcpy(e.data() + bins_x + 1, yedges, (bins_y + 1) * sizeof(double));
    return sum_hist_run(c, true, rows, 2, bins_x, bins_y, e.data(), (int64_t)e.size(), scratch_dev, mass_out,
                        count_out, (cudaStream_t)stream);
}

}  // extern "C"

#endif  // OBE_SUMMARY_CUH
