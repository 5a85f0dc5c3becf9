// Exact ranking metrics on the device: ROC AUC, average precision and the Youden threshold over fp32 scores
// (sklearn roc_auc_score / average_precision_score / roc_curve as called at src/plot.py:103-107,131 of the
// reference; torchmetrics BinaryAUROC / BinaryAveragePrecision at pangnn.py:27-30,220-222,262-268).
//
// Pipeline (pangnn_metric_runs, then pangnn_metric_reduce):
//   key pass     (score, label) -> 32-bit key that sorts ascending in DECREASING score order (-0 folded onto +0),
//                0/1 label; device flags for NaN scores and labels outside {0, 1}
//   sort         pangnn_sort_pairs_u64 with key_bits = 32 (four 8-bit passes), the label as the value
//   compaction   one row (key, pos, neg) per distinct key, in sorted order: tile statistics -> one-block scan
//                over the tiles -> emit.  A run's counts are (inclusive prefix at its last element) - (exclusive
//                prefix at its first element); the first element's prefix comes through shared memory when the run
//                starts inside the tile, else from the "carry" of the tile scan (the exclusive prefix at the last
//                head before the tile: a prefix MAX, since both cumulative counts grow with the position).  Runs
//                of any length, across any number of tiles, need nothing else.
//                The same kernels take already-compacted runs (multi-GPU merge): their counts are gathered
//                through the sort's permutation and equal keys are summed.
//   reduce       over runs with offsets (TP_0, FP_0) and the global (P, N): scan, then per-tile partials of the
//                128-bit AUROC numerator  sum_k neg_k (TP_{k-1} + TP_k),  the 128-bit AP numerator
//                sum_k pos_k floor(TP_k 2^s / (TP_k + FP_k)) with s = 127 - bitlen(P), and the Youden arg-max
//                (fp64 TP_k/P - FP_k/N, earliest run = smallest key on ties); one fixed final reduction.
//   curve        (pangnn_metric_curve) over runs with the same params: per-tile (kept, pos, neg) sums -> the tile
//                scan -> emit, which recomputes the cumulative counts and writes each kept run's (score, TP, FP) at
//                its compacted position.  A run's keep decision (sklearn roc_curve / precision_recall_curve
//                drop_intermediate) needs only the next run: read from `runs`, or from `bound` after the last run.
// Integer sums are exact, so the result does not depend on tiles, input order or the rank split.
#include "common.cuh"

namespace pangnn {

namespace {

typedef unsigned long long u64;
typedef unsigned __int128 u128;

constexpr int kMThreads = 256;
constexpr int kMItems = 8;                                   // consecutive items per thread
constexpr int kMTile = kMThreads * kMItems;                  // 2048
constexpr int kScanThreads1 = 1024;                          // the one-block tile scan
constexpr int kHistBins = 65536;

struct Tri {
    u64 a, b, c;
};
__device__ __forceinline__ Tri tri_add(Tri x, Tri y) { return {x.a + y.a, x.b + y.b, x.c + y.c}; }
__device__ __forceinline__ Tri tri_sub(Tri x, Tri y) { return {x.a - y.a, x.b - y.b, x.c - y.c}; }

// Exclusive block scan of Tri (THREADS threads); `total` = block sum.  Re-entrant within a kernel.
template <int THREADS>
__device__ __forceinline__ Tri block_exscan3(Tri v, Tri &total) {
    __shared__ Tri wsum[THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    Tri inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const u64 a = __shfl_up_sync(0xffffffffu, inc.a, o);
        const u64 b = __shfl_up_sync(0xffffffffu, inc.b, o);
        const u64 c = __shfl_up_sync(0xffffffffu, inc.c, o);
        if (lane >= o) inc = tri_add(inc, {a, b, c});
    }
    if (lane == 31) wsum[warp] = inc;
    __syncthreads();
    Tri off = {0, 0, 0}, tot = {0, 0, 0};
    for (int w = 0; w < THREADS / 32; ++w) {
        const Tri s = wsum[w];
        if (w < warp) off = tri_add(off, s);
        tot = tri_add(tot, s);
    }
    total = tot;
    __syncthreads();
    return tri_sub(tri_add(off, inc), v);
}

// Exclusive block prefix max of u64 (THREADS threads), 0 for thread 0.
template <int THREADS>
__device__ __forceinline__ u64 block_exmax(u64 v) {
    __shared__ u64 wmax[THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    u64 inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const u64 t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc = t > inc ? t : inc;
    }
    if (lane == 31) wmax[warp] = inc;
    u64 ex = __shfl_up_sync(0xffffffffu, inc, 1);
    if (lane == 0) ex = 0;
    __syncthreads();
    for (int w = 0; w < warp; ++w) ex = wmax[w] > ex ? wmax[w] : ex;
    __syncthreads();
    return ex;
}

// ---- key pass ------------------------------------------------------------------------------------------------
// Ascending order of the key = decreasing order of the score; -0.0 and +0.0 share a key; +-inf are ordinary.
__device__ __forceinline__ uint32_t score_key(float s) {
    uint32_t u = __float_as_uint(s);
    if (u == 0x80000000u) u = 0u;
    const uint32_t asc = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
    return ~asc;
}

__device__ __forceinline__ bool label_at(const void *labels, int kind, int64_t i, uint32_t &lab) {
    switch (kind) {
        case PANGNN_LABEL_F32: {
            const float v = static_cast<const float *>(labels)[i];
            lab = v == 1.f ? 1u : 0u;
            return v == 0.f || v == 1.f;
        }
        case PANGNN_LABEL_I32: {
            const int32_t v = static_cast<const int32_t *>(labels)[i];
            lab = (uint32_t)(v == 1);
            return v == 0 || v == 1;
        }
        case PANGNN_LABEL_I64: {
            const int64_t v = static_cast<const int64_t *>(labels)[i];
            lab = (uint32_t)(v == 1);
            return v == 0 || v == 1;
        }
        default: {
            const uint8_t v = static_cast<const uint8_t *>(labels)[i];
            lab = (uint32_t)(v == 1);
            return v <= 1;
        }
    }
}

__global__ void __launch_bounds__(256)
metric_keys_kernel(const float *__restrict__ scores, const void *__restrict__ labels, int kind, int64_t n,
                   uint64_t *__restrict__ keys, uint32_t *__restrict__ vals, int64_t *__restrict__ info) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float s = scores[i];
    uint32_t lab;
    const bool ok = label_at(labels, kind, i, lab);
    keys[i] = score_key(s);
    vals[i] = lab;
    const int f = (isnan(s) ? PANGNN_METRIC_NAN : 0) | (ok ? 0 : PANGNN_METRIC_BAD_LABEL);
    if (f) atomicOr(reinterpret_cast<unsigned long long *>(info + 5), (u64)f);
}

// runs given as input (multi-GPU merge): the sort key of row i
__global__ void __launch_bounds__(256)
metric_run_keys_kernel(const int64_t *__restrict__ runs_in, int64_t n, uint64_t *__restrict__ keys) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) keys[i] = (uint64_t)runs_in[3 * i];
}

// ---- compaction ----------------------------------------------------------------------------------------------
// Sorted element i: key (low 32 bits of the sorted key), counts = (label, 1 - label), or the counts of input
// run vals[i] when runs_in is given.
struct Sorted {
    const uint64_t *keys;
    const uint32_t *vals;
    const int64_t *runs_in;
    int64_t n;
    __device__ __forceinline__ void get(int64_t i, uint32_t &key, u64 &pos, u64 &neg) const {
        key = (uint32_t)keys[i];
        const uint32_t v = vals[i];
        if (runs_in) {
            pos = (u64)runs_in[3 * (int64_t)v + 1];
            neg = (u64)runs_in[3 * (int64_t)v + 2];
        } else {
            pos = v;
            neg = 1u - v;
        }
    }
};

// Per tile: [0] heads (first elements of runs), [1] positives, [2] negatives, [3..4] (pos, neg) exclusive prefix,
// local to the tile, at the tile's last head (0 when the tile has none).  Layout tstat[5][nb].
__global__ void __launch_bounds__(kMThreads)
runs_tile_stats_kernel(Sorted s, u64 *__restrict__ tstat, uint32_t nb) {
    __shared__ int last_thread;
    if (threadIdx.x == 0) last_thread = -1;
    const int64_t i0 = (int64_t)blockIdx.x * kMTile + (int64_t)threadIdx.x * kMItems;
    uint32_t prev = (i0 > 0 && i0 < s.n) ? (uint32_t)s.keys[i0 - 1] : 0u;
    Tri sum = {0, 0, 0}, last_ex = {0, 0, 0};
    bool has_head = false;
#pragma unroll
    for (int r = 0; r < kMItems; ++r) {
        const int64_t i = i0 + r;
        if (i < s.n) {
            uint32_t key;
            u64 pos, neg;
            s.get(i, key, pos, neg);
            const bool head = i == 0 || key != prev;
            if (head) {
                has_head = true;
                last_ex = sum;
            }
            sum = tri_add(sum, {head ? 1ull : 0ull, pos, neg});
            prev = key;
        }
    }
    Tri total;
    const Tri ex = block_exscan3<kMThreads>(sum, total);        // (syncs: last_thread is initialised)
    if (has_head) atomicMax(&last_thread, (int)threadIdx.x);
    __syncthreads();
    const uint32_t b = blockIdx.x;
    if (threadIdx.x == 0) {
        tstat[0 * (size_t)nb + b] = total.a;
        tstat[1 * (size_t)nb + b] = total.b;
        tstat[2 * (size_t)nb + b] = total.c;
        if (last_thread < 0) {
            tstat[3 * (size_t)nb + b] = 0;
            tstat[4 * (size_t)nb + b] = 0;
        }
    }
    if ((int)threadIdx.x == last_thread) {
        tstat[3 * (size_t)nb + b] = ex.b + last_ex.b;
        tstat[4 * (size_t)nb + b] = ex.c + last_ex.c;
    }
}

// One block over the tiles: toff[5][nb] = exclusive scans of (heads, pos, neg) and, with carry, the (pos, neg)
// exclusive prefix at the last head before each tile.  totals (optional) = (runs, P, N).
__global__ void __launch_bounds__(kScanThreads1)
tile_scan_kernel(const u64 *__restrict__ tstat, uint32_t nb, int carry, u64 *__restrict__ toff,
                 int64_t *__restrict__ totals) {
    const uint32_t per = (nb + kScanThreads1 - 1) / kScanThreads1;
    const uint32_t j0 = min(nb, threadIdx.x * per), j1 = min(nb, j0 + per);
    Tri run = {0, 0, 0};
    u64 cand_p = 0, cand_n = 0;
    bool has = false;
    for (uint32_t j = j0; j < j1; ++j) {
        const Tri st = {tstat[j], tstat[(size_t)nb + j], tstat[2 * (size_t)nb + j]};
        if (carry && st.a) {
            has = true;
            cand_p = run.b + tstat[3 * (size_t)nb + j];
            cand_n = run.c + tstat[4 * (size_t)nb + j];
        }
        run = tri_add(run, st);
    }
    Tri total;
    const Tri ex = block_exscan3<kScanThreads1>(run, total);
    u64 cp = 0, cn = 0;
    if (carry) {
        cp = block_exmax<kScanThreads1>(has ? ex.b + cand_p : 0);
        cn = block_exmax<kScanThreads1>(has ? ex.c + cand_n : 0);
    }
    Tri cur = ex;
    for (uint32_t j = j0; j < j1; ++j) {
        const Tri st = {tstat[j], tstat[(size_t)nb + j], tstat[2 * (size_t)nb + j]};
        toff[j] = cur.a;
        toff[(size_t)nb + j] = cur.b;
        toff[2 * (size_t)nb + j] = cur.c;
        if (carry) {
            toff[3 * (size_t)nb + j] = cp;
            toff[4 * (size_t)nb + j] = cn;
            if (st.a) {
                cp = cur.b + tstat[3 * (size_t)nb + j];
                cn = cur.c + tstat[4 * (size_t)nb + j];
            }
        }
        cur = tri_add(cur, st);
    }
    if (totals && threadIdx.x == 0) {
        totals[0] = (int64_t)total.a;
        totals[1] = (int64_t)total.b;
        totals[2] = (int64_t)total.c;
    }
}

// Every last element of a run writes runs_out[r] = (key, pos, neg) and counts the run in hist[key >> 16].
__global__ void __launch_bounds__(kMThreads)
runs_emit_kernel(Sorted s, const u64 *__restrict__ toff, uint32_t nb, int64_t *__restrict__ runs_out,
                 unsigned long long *__restrict__ hist) {
    __shared__ u64 start_p[kMTile + 1], start_n[kMTile + 1];  // exclusive prefix at the head of local run h
    const uint32_t b = blockIdx.x;
    const int64_t i0 = (int64_t)b * kMTile + (int64_t)threadIdx.x * kMItems;
    uint32_t key[kMItems];
    u64 pos[kMItems], neg[kMItems];
    uint32_t head = 0, end = 0;                                // bit r: item r starts / ends a run
    uint32_t prev = (i0 > 0 && i0 < s.n) ? (uint32_t)s.keys[i0 - 1] : 0u;
    Tri sum = {0, 0, 0};
#pragma unroll
    for (int r = 0; r < kMItems; ++r) {
        const int64_t i = i0 + r;
        key[r] = 0; pos[r] = 0; neg[r] = 0;
        if (i < s.n) {
            s.get(i, key[r], pos[r], neg[r]);
            const bool h = i == 0 || key[r] != prev;
            head |= (uint32_t)h << r;
            if (r > 0 && h) end |= 1u << (r - 1);
            sum = tri_add(sum, {h ? 1ull : 0ull, pos[r], neg[r]});
            prev = key[r];
        }
    }
    {
        const int64_t il = i0 + kMItems - 1;                  // the thread's last item ends a run?
        if (il < s.n) {
            if (il == s.n - 1 || (uint32_t)s.keys[il + 1] != key[kMItems - 1]) end |= 1u << (kMItems - 1);
        } else if (i0 < s.n) {
            end |= 1u << (int)(s.n - 1 - i0);                 // the global last element
        }
    }
    Tri total;
    const Tri ex = block_exscan3<kMThreads>(sum, total);
    const u64 base = toff[b], op = toff[(size_t)nb + b], on = toff[2 * (size_t)nb + b];
    if (threadIdx.x == 0) {
        start_p[0] = toff[3 * (size_t)nb + b];
        start_n[0] = toff[4 * (size_t)nb + b];
    }
    Tri cur = ex;
#pragma unroll
    for (int r = 0; r < kMItems; ++r) {
        if ((head >> r) & 1u) {
            const u64 h = cur.a + 1;
            start_p[h] = op + cur.b;
            start_n[h] = on + cur.c;
        }
        cur = tri_add(cur, {(u64)((head >> r) & 1u), pos[r], neg[r]});
    }
    __syncthreads();
    cur = ex;
#pragma unroll
    for (int r = 0; r < kMItems; ++r) {
        cur = tri_add(cur, {(u64)((head >> r) & 1u), pos[r], neg[r]});
        if ((end >> r) & 1u) {
            const u64 h = cur.a;                               // local run index (0 = run carried in)
            const u64 run = base + h - 1;
            runs_out[3 * run] = (int64_t)key[r];
            runs_out[3 * run + 1] = (int64_t)(op + cur.b - start_p[h]);
            runs_out[3 * run + 2] = (int64_t)(on + cur.c - start_n[h]);
            if (hist) atomicAdd(hist + (key[r] >> 16), 1ull);
        }
    }
}

// ---- reduction over runs -------------------------------------------------------------------------------------
// params: [0] runs, [1] P, [2] N, [3] TP_0, [4] FP_0
__global__ void __launch_bounds__(kMThreads)
reduce_tile_stats_kernel(const int64_t *__restrict__ runs, const int64_t *__restrict__ params,
                         u64 *__restrict__ tstat, uint32_t nb) {
    const int64_t R = params[0];
    const int64_t i0 = (int64_t)blockIdx.x * kMTile + (int64_t)threadIdx.x * kMItems;
    Tri sum = {0, 0, 0};
#pragma unroll
    for (int r = 0; r < kMItems; ++r) {
        const int64_t i = i0 + r;
        if (i < R) sum = tri_add(sum, {0ull, (u64)runs[3 * i + 1], (u64)runs[3 * i + 2]});
    }
    Tri total;
    block_exscan3<kMThreads>(sum, total);
    if (threadIdx.x == 0) {
        tstat[blockIdx.x] = 0;
        tstat[(size_t)nb + blockIdx.x] = total.b;
        tstat[2 * (size_t)nb + blockIdx.x] = total.c;
    }
}

struct Partial {
    u64 auc_lo, auc_hi, ap_lo, ap_hi;
    double j;
    u64 key;
};

__device__ __forceinline__ u128 shfl_xor_u128(u128 v, int o) {
    const u64 lo = __shfl_xor_sync(0xffffffffu, (u64)v, o);
    const u64 hi = __shfl_xor_sync(0xffffffffu, (u64)(v >> 64), o);
    return ((u128)hi << 64) | lo;
}

// (j, key) is better than (bj, bkey): larger j, or equal j and the earlier run (smaller key)
__device__ __forceinline__ bool better(double j, u64 key, double bj, u64 bkey) {
    return j > bj || (j == bj && key < bkey);
}

// Block reduction of (auc, ap, j, key) to thread 0 (fixed shuffle tree: deterministic).
__device__ __forceinline__ void block_reduce_partial(u128 &auc, u128 &ap, double &j, u64 &key) {
    __shared__ u128 s_auc[kMThreads / 32], s_ap[kMThreads / 32];
    __shared__ double s_j[kMThreads / 32];
    __shared__ u64 s_key[kMThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        auc += shfl_xor_u128(auc, o);
        ap += shfl_xor_u128(ap, o);
        const double oj = __shfl_xor_sync(0xffffffffu, j, o);
        const u64 ok = __shfl_xor_sync(0xffffffffu, key, o);
        if (better(oj, ok, j, key)) { j = oj; key = ok; }
    }
    if (lane == 0) { s_auc[warp] = auc; s_ap[warp] = ap; s_j[warp] = j; s_key[warp] = key; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < kMThreads / 32; ++w) {
            auc += s_auc[w];
            ap += s_ap[w];
            if (better(s_j[w], s_key[w], j, key)) { j = s_j[w]; key = s_key[w]; }
        }
    }
}

__device__ __forceinline__ int ap_shift(u64 P) { return 127 - (P ? 64 - __clzll((long long)P) : 0); }

__global__ void __launch_bounds__(kMThreads)
reduce_tile_kernel(const int64_t *__restrict__ runs, const int64_t *__restrict__ params, const u64 *__restrict__ toff,
                   uint32_t nb, Partial *__restrict__ part) {
    const int64_t R = params[0];
    const u64 P = (u64)params[1], N = (u64)params[2];
    const int shift = ap_shift(P);
    const int64_t i0 = (int64_t)blockIdx.x * kMTile + (int64_t)threadIdx.x * kMItems;
    Tri sum = {0, 0, 0};
#pragma unroll
    for (int r = 0; r < kMItems; ++r) {
        const int64_t i = i0 + r;
        if (i < R) sum = tri_add(sum, {0ull, (u64)runs[3 * i + 1], (u64)runs[3 * i + 2]});
    }
    Tri total;
    const Tri ex = block_exscan3<kMThreads>(sum, total);
    u64 tp = (u64)params[3] + toff[(size_t)nb + blockIdx.x] + ex.b;
    u64 fp = (u64)params[4] + toff[2 * (size_t)nb + blockIdx.x] + ex.c;
    u128 auc = 0, ap = 0;
    double bj = -INFINITY;
    u64 bkey = ~0ull;
    const bool both = P > 0 && N > 0;
    for (int r = 0; r < kMItems; ++r) {
        const int64_t i = i0 + r;
        if (i >= R) break;
        const u64 key = (u64)runs[3 * i], pos = (u64)runs[3 * i + 1], neg = (u64)runs[3 * i + 2];
        const u64 tp1 = tp + pos, fp1 = fp + neg;
        auc += (u128)neg * (u128)(tp + tp1);
        if (pos) ap += (u128)pos * (((u128)tp1 << shift) / (u128)(tp1 + fp1));
        if (both) {
            const double j = (double)tp1 / (double)P - (double)fp1 / (double)N;
            if (better(j, key, bj, bkey)) { bj = j; bkey = key; }
        }
        tp = tp1;
        fp = fp1;
    }
    block_reduce_partial(auc, ap, bj, bkey);
    if (threadIdx.x == 0)
        part[blockIdx.x] = {(u64)auc, (u64)(auc >> 64), (u64)ap, (u64)(ap >> 64), bj, bkey};
}

// out: [0..1] AUROC numerator (lo, hi), [2..3] AP numerator (lo, hi), [4] Youden j (fp64 bits, -inf: none),
// [5] key of that run (all ones: none), [6] runs, [7] AP fixed-point shift
__global__ void __launch_bounds__(kMThreads)
reduce_final_kernel(const Partial *__restrict__ part, uint32_t nb, const int64_t *__restrict__ params,
                    int64_t *__restrict__ out) {
    u128 auc = 0, ap = 0;
    double bj = -INFINITY;
    u64 bkey = ~0ull;
    for (uint32_t b = threadIdx.x; b < nb; b += kMThreads) {
        const Partial p = part[b];
        auc += ((u128)p.auc_hi << 64) | p.auc_lo;
        ap += ((u128)p.ap_hi << 64) | p.ap_lo;
        if (better(p.j, p.key, bj, bkey)) { bj = p.j; bkey = p.key; }
    }
    block_reduce_partial(auc, ap, bj, bkey);
    if (threadIdx.x == 0) {
        out[0] = (int64_t)(u64)auc;
        out[1] = (int64_t)(u64)(auc >> 64);
        out[2] = (int64_t)(u64)ap;
        out[3] = (int64_t)(u64)(ap >> 64);
        out[4] = __double_as_longlong(bj);
        out[5] = (int64_t)bkey;
        out[6] = params[0];
        out[7] = ap_shift((u64)params[1]);
    }
}

// ---- curve points over runs ----------------------------------------------------------------------------------
// bound: [0] pos, [1] neg of the run that follows the last of these runs, [2] PANGNN_CURVE_* flags.
// The thread's kMItems runs and which of them are kept: run i is kept if it is the first run of the curve, the last
// one, or passes the mode's rule against run i+1 (read across the thread's and the tile's edge from `runs`, and from
// `bound` after the last run).
struct CurveItems {
    u64 key[kMItems], pos[kMItems], neg[kMItems];
    uint32_t keep;                                             // bit r: item r is kept
};

__device__ __forceinline__ bool curve_rule(int mode, u64 pos, u64 neg, u64 npos, u64 nneg) {
    if (mode == PANGNN_CURVE_ROC) return pos != npos || neg != nneg;
    if (mode == PANGNN_CURVE_PR) return pos != 0 || npos != 0;
    return true;
}

__device__ __forceinline__ void curve_items(const int64_t *__restrict__ runs, int64_t R, int64_t i0,
                                            const int64_t *__restrict__ bound, int mode, CurveItems &it) {
    const int64_t flags = bound[2];
    it.keep = 0;
#pragma unroll
    for (int r = 0; r < kMItems; ++r) {
        const int64_t i = i0 + r;
        it.key[r] = 0; it.pos[r] = 0; it.neg[r] = 0;
        if (i < R) {
            it.key[r] = (u64)runs[3 * i];
            it.pos[r] = (u64)runs[3 * i + 1];
            it.neg[r] = (u64)runs[3 * i + 2];
        }
    }
    u64 npos, nneg;                                            // run i0 + kMItems
    bool has_next;
    {
        const int64_t i = i0 + kMItems;
        has_next = i < R || (flags & PANGNN_CURVE_FOLLOWED);
        npos = i < R ? (u64)runs[3 * i + 1] : (u64)bound[0];
        nneg = i < R ? (u64)runs[3 * i + 2] : (u64)bound[1];
    }
#pragma unroll
    for (int r = kMItems - 1; r >= 0; --r) {
        const int64_t i = i0 + r;
        if (i < R) {
            const bool first = i == 0 && (flags & PANGNN_CURVE_FIRST);
            if (i + 1 == R) {                                  // the next run is the bound's, if any
                has_next = (flags & PANGNN_CURVE_FOLLOWED) != 0;
                npos = (u64)bound[0];
                nneg = (u64)bound[1];
            }
            if (first || !has_next || curve_rule(mode, it.pos[r], it.neg[r], npos, nneg)) it.keep |= 1u << r;
        }
        npos = it.pos[r];
        nneg = it.neg[r];
        has_next = true;
    }
}

// Per tile: [0] kept runs, [1] positives, [2] negatives.  Layout tstat[3][nb].
__global__ void __launch_bounds__(kMThreads)
curve_tile_stats_kernel(const int64_t *__restrict__ runs, const int64_t *__restrict__ params,
                        const int64_t *__restrict__ bound, int mode, u64 *__restrict__ tstat, uint32_t nb) {
    const int64_t R = params[0];
    const int64_t i0 = (int64_t)blockIdx.x * kMTile + (int64_t)threadIdx.x * kMItems;
    CurveItems it;
    curve_items(runs, R, i0, bound, mode, it);
    Tri sum = {(u64)__popc(it.keep), 0, 0};
#pragma unroll
    for (int r = 0; r < kMItems; ++r) sum = tri_add(sum, {0ull, it.pos[r], it.neg[r]});
    Tri total;
    block_exscan3<kMThreads>(sum, total);
    if (threadIdx.x == 0) {
        tstat[blockIdx.x] = total.a;
        tstat[(size_t)nb + blockIdx.x] = total.b;
        tstat[2 * (size_t)nb + blockIdx.x] = total.c;
    }
}

// Inverse of score_key: the fp32 score of a key (+0.0 for the folded zeros).
__device__ __forceinline__ float key_score(u64 key) {
    const uint32_t asc = ~(uint32_t)key;
    return __uint_as_float((asc & 0x80000000u) ? (asc & 0x7fffffffu) : ~asc);
}

// Kept run i -> thr[c] (its score), tp[c] = TP_0 + TP_i, fp[c] = FP_0 + FP_i, c = kept runs before it.
__global__ void __launch_bounds__(kMThreads)
curve_emit_kernel(const int64_t *__restrict__ runs, const int64_t *__restrict__ params,
                  const int64_t *__restrict__ bound, int mode, const u64 *__restrict__ toff, uint32_t nb,
                  float *__restrict__ thr, int64_t *__restrict__ tp_out, int64_t *__restrict__ fp_out) {
    const int64_t R = params[0];
    const int64_t i0 = (int64_t)blockIdx.x * kMTile + (int64_t)threadIdx.x * kMItems;
    CurveItems it;
    curve_items(runs, R, i0, bound, mode, it);
    Tri sum = {(u64)__popc(it.keep), 0, 0};
#pragma unroll
    for (int r = 0; r < kMItems; ++r) sum = tri_add(sum, {0ull, it.pos[r], it.neg[r]});
    Tri total;
    const Tri ex = block_exscan3<kMThreads>(sum, total);
    u64 c = toff[blockIdx.x] + ex.a;
    u64 tp = (u64)params[3] + toff[(size_t)nb + blockIdx.x] + ex.b;
    u64 fp = (u64)params[4] + toff[2 * (size_t)nb + blockIdx.x] + ex.c;
#pragma unroll
    for (int r = 0; r < kMItems; ++r) {
        tp += it.pos[r];
        fp += it.neg[r];
        if ((it.keep >> r) & 1u) {
            thr[c] = key_score(it.key[r]);
            tp_out[c] = (int64_t)tp;
            fp_out[c] = (int64_t)fp;
            ++c;
        }
    }
}

uint32_t tiles(int64_t n) { return (uint32_t)((n + kMTile - 1) / kMTile); }

size_t runs_ws_bytes(int64_t n) {
    const size_t nb = tiles(n);
    size_t b = 0;
    b += 2 * align_up((size_t)n * sizeof(uint64_t), 256);     // keys, sorted keys
    b += 2 * align_up((size_t)n * sizeof(uint32_t), 256);     // labels / permutation, sorted
    b += 2 * align_up(5 * nb * sizeof(u64), 256);             // tile statistics, tile offsets
    b += align_up(pangnn_sort_pairs_workspace_bytes(n), 256);
    return b + 1024;
}

size_t reduce_ws_bytes(int64_t max_runs) {
    const size_t nb = tiles(max_runs);
    return 2 * align_up(3 * nb * sizeof(u64), 256) + align_up(nb * sizeof(Partial), 256) + 1024;
}

size_t curve_ws_bytes(int64_t max_runs) { return 2 * align_up(3 * (size_t)tiles(max_runs) * sizeof(u64), 256) + 1024; }

}  // namespace
}  // namespace pangnn

using namespace pangnn;

extern "C" {

size_t pangnn_metric_runs_workspace_bytes(int64_t n) { return runs_ws_bytes(n < 0 ? 0 : n); }

int pangnn_metric_runs(const float *scores, const void *labels, int label_kind, const int64_t *runs_in, int64_t n,
                       int64_t *runs_out, int64_t *info, int64_t *hist, void *ws, size_t ws_bytes, void *stream) {
    PANGNN_REQUIRE(info && n >= 0, "bad arguments");
    PANGNN_REQUIRE(n < ((int64_t)1 << 32), "more than 2^32 - 1 scores on one device (the sort's limit)");
    PANGNN_REQUIRE(n == 0 || (runs_out && ws && (runs_in || (scores && labels))), "null pointer");
    PANGNN_REQUIRE(runs_in || (label_kind >= PANGNN_LABEL_F32 && label_kind <= PANGNN_LABEL_U8), "bad label kind");
    cudaStream_t st = (cudaStream_t)stream;
    int rc = check_cuda(cudaMemsetAsync(info, 0, 6 * sizeof(int64_t), st), "memset(info)");
    if (!rc && hist) rc = check_cuda(cudaMemsetAsync(hist, 0, kHistBins * sizeof(int64_t), st), "memset(hist)");
    if (rc || n == 0) return rc;
    if (ws_bytes < runs_ws_bytes(n)) {
        set_error("metric_runs: workspace too small (%zu < %zu)", ws_bytes, runs_ws_bytes(n));
        return PANGNN_EWORKSPACE;
    }
    const uint32_t nb = tiles(n);
    Workspace w(ws, ws_bytes);
    uint64_t *keys = w.take<uint64_t>(n), *skeys = w.take<uint64_t>(n);
    uint32_t *vals = w.take<uint32_t>(n), *svals = w.take<uint32_t>(n);
    u64 *tstat = w.take<u64>(5 * (size_t)nb), *toff = w.take<u64>(5 * (size_t)nb);
    w.off = align_up(w.off, 256);
    void *sort_ws = w.base + w.off;
    const size_t sort_bytes = ws_bytes - w.off;
    const unsigned blocks = (unsigned)((n + 255) / 256);
    if (runs_in) {
        metric_run_keys_kernel<<<blocks, 256, 0, st>>>(runs_in, n, keys);
        PANGNN_CHECK_LAUNCH("metric_run_keys");
    } else {
        metric_keys_kernel<<<blocks, 256, 0, st>>>(scores, labels, label_kind, n, keys, vals, info);
        PANGNN_CHECK_LAUNCH("metric_keys");
    }
    rc = pangnn_sort_pairs_u64(keys, runs_in ? nullptr : vals, skeys, svals, n, 32, sort_ws, sort_bytes, st);
    if (rc) return rc;
    const Sorted s = {skeys, svals, runs_in, n};
    runs_tile_stats_kernel<<<nb, kMThreads, 0, st>>>(s, tstat, nb);
    PANGNN_CHECK_LAUNCH("runs_tile_stats");
    tile_scan_kernel<<<1, kScanThreads1, 0, st>>>(tstat, nb, 1, toff, info);
    PANGNN_CHECK_LAUNCH("runs_tile_scan");
    runs_emit_kernel<<<nb, kMThreads, 0, st>>>(s, toff, nb, runs_out, reinterpret_cast<unsigned long long *>(hist));
    PANGNN_CHECK_LAUNCH("runs_emit");
    return PANGNN_OK;
}

size_t pangnn_metric_reduce_workspace_bytes(int64_t max_runs) { return reduce_ws_bytes(max_runs < 0 ? 0 : max_runs); }

int pangnn_metric_reduce(const int64_t *runs, int64_t max_runs, const int64_t *params, int64_t *out, void *ws,
                         size_t ws_bytes, void *stream) {
    PANGNN_REQUIRE(params && out && max_runs >= 0, "bad arguments");
    PANGNN_REQUIRE(max_runs == 0 || (runs && ws), "null pointer");
    if (ws_bytes < reduce_ws_bytes(max_runs)) {
        set_error("metric_reduce: workspace too small (%zu < %zu)", ws_bytes, reduce_ws_bytes(max_runs));
        return PANGNN_EWORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const uint32_t nb = tiles(max_runs);
    Workspace w(ws, ws_bytes);
    u64 *tstat = w.take<u64>(3 * (size_t)nb), *toff = w.take<u64>(3 * (size_t)nb);
    Partial *part = w.take<Partial>(nb);
    if (nb) {
        reduce_tile_stats_kernel<<<nb, kMThreads, 0, st>>>(runs, params, tstat, nb);
        PANGNN_CHECK_LAUNCH("reduce_tile_stats");
        tile_scan_kernel<<<1, kScanThreads1, 0, st>>>(tstat, nb, 0, toff, nullptr);
        PANGNN_CHECK_LAUNCH("reduce_tile_scan");
        reduce_tile_kernel<<<nb, kMThreads, 0, st>>>(runs, params, toff, nb, part);
        PANGNN_CHECK_LAUNCH("reduce_tile");
    }
    reduce_final_kernel<<<1, kMThreads, 0, st>>>(part, nb, params, out);
    PANGNN_CHECK_LAUNCH("reduce_final");
    return PANGNN_OK;
}

size_t pangnn_metric_curve_workspace_bytes(int64_t max_runs) { return curve_ws_bytes(max_runs < 0 ? 0 : max_runs); }

int pangnn_metric_curve(const int64_t *runs, int64_t max_runs, const int64_t *params, const int64_t *bound, int mode,
                        float *thresholds, int64_t *tp, int64_t *fp, int64_t *count, void *ws, size_t ws_bytes,
                        void *stream) {
    PANGNN_REQUIRE(params && bound && count && max_runs >= 0, "bad arguments");
    PANGNN_REQUIRE(mode >= PANGNN_CURVE_ALL && mode <= PANGNN_CURVE_PR, "bad curve mode");
    PANGNN_REQUIRE(max_runs == 0 || (runs && thresholds && tp && fp && ws), "null pointer");
    if (ws_bytes < curve_ws_bytes(max_runs)) {
        set_error("metric_curve: workspace too small (%zu < %zu)", ws_bytes, curve_ws_bytes(max_runs));
        return PANGNN_EWORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const uint32_t nb = tiles(max_runs);
    if (nb == 0) return check_cuda(cudaMemsetAsync(count, 0, 3 * sizeof(int64_t), st), "memset(count)");
    Workspace w(ws, ws_bytes);
    u64 *tstat = w.take<u64>(3 * (size_t)nb), *toff = w.take<u64>(3 * (size_t)nb);
    curve_tile_stats_kernel<<<nb, kMThreads, 0, st>>>(runs, params, bound, mode, tstat, nb);
    PANGNN_CHECK_LAUNCH("curve_tile_stats");
    tile_scan_kernel<<<1, kScanThreads1, 0, st>>>(tstat, nb, 0, toff, count);
    PANGNN_CHECK_LAUNCH("curve_tile_scan");
    curve_emit_kernel<<<nb, kMThreads, 0, st>>>(runs, params, bound, mode, toff, nb, thresholds, tp, fp);
    PANGNN_CHECK_LAUNCH("curve_emit");
    return PANGNN_OK;
}

}  // extern "C"
