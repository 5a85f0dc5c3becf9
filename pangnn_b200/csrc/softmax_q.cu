// Candidate normalisation on the device: hit table -> unique sorted hits -> per (query, target
// genome) segment temperature softmax + Q-score -> compacted (src, dst, w, y) edge list.
//
// Replaces (reference, all pure-Python dict loops):
//   src/preprocessing.py:413-416  groupby / dict(zip)   (duplicate (query,target): last row wins)
//   src/preprocessing.py:370-385  remove_trivial_cases
//   src/preprocessing.py:430-443  softmax_with_temperature (scipy logsumexp, fp64)
//   src/preprocessing.py:454-548  normalize_sim_scores
//   src/preprocessing.py:73-118   build_edge_index, :264-325 map_edge_weights,
//   src/preprocessing.py:122-156  map_labels_to_edge_index
//
// Roofline: HBM; algorithmic bytes of the softmax kernel = n*(4 q + 4 t + 8 bits + 4 w + 4 y + 1 keep)
// + 8 per segment.  Eight lanes per segment, persistent grid; fp64 shuffle reductions.
#include <cmath>

#include "common.cuh"

namespace pangnn {

int exclusive_scan_u32(const uint32_t *in, uint32_t *out, int64_t n, uint32_t *total, void *ws,
                       size_t ws_bytes, cudaStream_t st);
int sort_pairs_u64(const uint64_t *keys_in, const uint32_t *vals_in, uint64_t *keys_out,
                   uint32_t *vals_out, int64_t n, int key_bits, void *ws, size_t ws_bytes,
                   cudaStream_t st, int first_bit = 0);

static int bits_for_nodes(int64_t n) {
    int b = 1;
    while (((int64_t)1 << b) < n) ++b;
    return b;
}

__global__ void hits_pack_kernel(const int32_t *__restrict__ q, const int32_t *__restrict__ t,
                                 int64_t n, int nbits, uint64_t *__restrict__ keys) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) keys[i] = ((uint64_t)(uint32_t)q[i] << nbits) | (uint64_t)(uint32_t)t[i];
}

// flag = 1 on the LAST element of every run of equal keys (stable sort => last original row)
__global__ void hits_last_flag_kernel(const uint64_t *__restrict__ keys, int64_t n,
                                      uint32_t *__restrict__ flag) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flag[i] = (i == n - 1 || keys[i] != keys[i + 1]) ? 1u : 0u;
}

__global__ void hits_unpack_kernel(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ vals,
                                   const uint32_t *__restrict__ pos, const double *__restrict__ bits,
                                   int64_t n, int nbits, int32_t *__restrict__ q,
                                   int32_t *__restrict__ t, double *__restrict__ bits_out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (i != n - 1 && keys[i] == keys[i + 1]) return;
    const uint32_t p = pos[i];
    const uint64_t k = keys[i];
    q[p] = (int32_t)(k >> nbits);
    t[p] = (int32_t)(k & ((1ull << nbits) - 1ull));
    bits_out[p] = bits[vals[i]];
}

// head[i] = 1 where a (query, genome_of[target]) segment starts
__global__ void seg_head_kernel(const int32_t *__restrict__ q, const int32_t *__restrict__ t,
                                const int32_t *__restrict__ genome_of, int64_t n,
                                uint32_t *__restrict__ head) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t h = 1u;
    if (i > 0) h = (q[i] != q[i - 1] || genome_of[t[i]] != genome_of[t[i - 1]]) ? 1u : 0u;
    head[i] = h;
}

// seg_start[seg_id] = i for heads; seg_start[num_seg] = n
__global__ void seg_start_kernel(const uint32_t *__restrict__ head_pos, const int32_t *__restrict__ q,
                                 const int32_t *__restrict__ t, const int32_t *__restrict__ genome_of,
                                 int64_t n, const uint32_t *__restrict__ num_seg,
                                 int64_t *__restrict__ seg_start) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const bool h = (i == 0) || q[i] != q[i - 1] || genome_of[t[i]] != genome_of[t[i - 1]];
    if (h) seg_start[head_pos[i]] = i;
    if (i == n - 1) seg_start[*num_seg] = n;
}

// One group of kGL = 8 lanes per (query, genome) segment, persistent grid-stride over segments
// (simulated and real candidate sets hold a handful of members: p50 4, p90 9; the NegBin tail
// reaches thousands and is walked by the same 8 lanes).  Segments of <= 8 entries — the bulk — are
// handled in ONE pass: each lane loads its entry once and keeps exp() in a register; larger ones
// take the three-pass route (max, sum, emit).  fp64 throughout as in the reference (numpy / scipy
// logsumexp); reductions are xor-shuffles inside the group with the group's own mask.
constexpr int kGL = 8;

__device__ __forceinline__ double group_max(double v, unsigned m) {
#pragma unroll
    for (int o = kGL / 2; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(m, v, o));
    return v;
}
__device__ __forceinline__ double group_sum(double v, unsigned m) {
#pragma unroll
    for (int o = kGL / 2; o > 0; o >>= 1) v += __shfl_xor_sync(m, v, o);
    return v;
}
__device__ __forceinline__ int group_sum(int v, unsigned m) {
#pragma unroll
    for (int o = kGL / 2; o > 0; o >>= 1) v += __shfl_xor_sync(m, v, o);
    return v;
}

// w = -10 log10(clip(1 - p, eps, 1 - eps)) + pseudo.  The clip saturates almost every entry (simulated
// data: 10 % at the upper constant 81, 89 % at the lower one), so log10 is evaluated only for the few
// unsaturated values; w_lo / w_hi are the two constants, computed once per thread with the same formula.
__device__ __forceinline__ void emit_entry(int64_t i, int32_t qi, int32_t ti, bool self, bool trivial, int members,
                                           double e, double sum, double eps, double pseudo, float w_lo, float w_hi,
                                           const int32_t *__restrict__ group_of, float *__restrict__ w,
                                           float *__restrict__ y, uint32_t *__restrict__ keep) {
    float wi = 0.f;
    if (!self) {
        // 1 - p = (S - e_i) / S: the subtraction in fp64 (S was accumulated in fp64 from the very e_i it removes,
        // so it is exact), the quotient of the two positive numbers and the logarithm in fp32 (1e-7 relative on
        // 1 - p = 4e-7 absolute on w); an fp64 division + log10 per entry was a fifth of the kernel's instructions
        // 1 - p is not representable in fp32 near 1 (ulp 6e-8 > eps = 1e-8), so that end is taken from p itself:
        // -10 log10(1 - p) = -10 / ln(10) log1p(-p), which rounds to the same float as the fp64 formula
        float om = 0.f, pf = 1.f;
        if (members > 1) {
            om = (float)(sum - e) / (float)sum;
            pf = (float)e / (float)sum;
        }
        if (om <= (float)eps) wi = w_hi;                       // np.clip(1-p, eps, 1-eps)
        else if (pf <= (float)eps) wi = w_lo;
        else if (pf < 0.5f) wi = fmaf(-4.342944819032518f, log1pf(-pf), (float)pseudo);
        else wi = fmaf(-10.f, log10f(om), (float)pseudo);
    }
    w[i] = wi;
    float yi = 0.f;
    if (group_of && !self) {
        const int32_t gq = group_of[qi];
        yi = (gq >= 0 && gq == group_of[ti]) ? 1.f : 0.f;
    }
    y[i] = yi;
    keep[i] = (!self && !trivial) ? 1u : 0u;
}

constexpr int kElemMaxSeg = 32;     // segments up to this size take the thread-per-entry kernel

// exp(x - mx) for the softmax: the DIFFERENCE is formed in fp64 (exact to 1e-16), the exponential is
// evaluated in fp32 (1e-7 relative) and accumulated in fp64.  An fp64 exp() per candidate made this
// path fp64-pipe-bound (0.8 ms for 1.8e7 entries); the Q-score needs 1 - p to ~1e-6 relative for the
// 1e-5 bar on w, which this keeps (the subtraction sum - e stays exact because e is the very value
// that was added into sum).
__device__ __forceinline__ double exp_diff(double x, double mx) { return (double)expf((float)(x - mx)); }

// Thread per ENTRY for the bulk of the table (segments of <= kElemMaxSeg entries: p50 4, p90 9, 78 % singletons
// on C3), in two phases so that exp() is evaluated ONCE per candidate (ncu on the one-phase version: 76 % issue
// utilisation, 36 % of it in the per-neighbour exp — every entry recomputed its whole segment):
//   phase A: the entry finds its segment through the head scan, walks its few neighbours (L1-resident) for the
//            maximum score (plain compares) and the member count, stores e_i = exp((x_i - max) / T);
//            heads of longer segments append their segment id to `long_list` for the cooperative kernel;
//   phase B: sums the e_j of its segment (fp64 adds of the stored fp32 values), forms 1 - p, emits w / y / keep.
struct SegOf {
    int64_t s0, s1;
};
__device__ __forceinline__ SegOf segment_of(int64_t i, const uint32_t *__restrict__ head_excl,
                                            const int64_t *__restrict__ seg_start) {
    int64_t seg = head_excl[i];                                // #heads before i
    int64_t s0 = seg_start[seg];
    if (s0 != i) {                                             // i is not a head: it belongs to the previous segment
        --seg;
        s0 = seg_start[seg];
    }
    return SegOf{s0, seg_start[seg + 1]};
}

// Windows overlap by 32 - kSoftmaxStride entries, so that every segment of up to 32 - kSoftmaxStride + 1 entries
// (p90 of the candidate sets is 9) lies completely inside at least one window; the first such window owns it.
constexpr int kSoftmaxStride = 24;
constexpr int kLongListDiv = 32 - kSoftmaxStride + 2;          // a listed segment has at least this many entries

// Bulk kernel: one thread per ENTRY, one pass.  A warp looks at 32 consecutive entries of the sorted table; the
// heads among them (from the head scan, read coalesced) give every lane the first and last lane of its segment,
// and a segment that lies completely inside the warp's window (the bulk: p50 4 entries, p90 9) is reduced with
// segmented suffix scans over shuffles — max of the non-self scores, then e_i = expf((x_i - max) / T) ONCE per
// candidate, then the fp64 sum of the e_j — with no per-entry index chain (head scan -> segment bounds ->
// neighbours), no divergence and no round trip of e through HBM.  Segments that cross the window are left to
// the boundary kernel below.
__global__ void __launch_bounds__(256)
segment_softmax_q_warp_kernel(const int32_t *__restrict__ q, const int32_t *__restrict__ t,
                              const double *__restrict__ bits, const uint32_t *__restrict__ head_excl,
                              const uint32_t *__restrict__ num_seg, int64_t n,
                              const int32_t *__restrict__ group_of, double inv_temp, double eps, double pseudo,
                              float w_lo, float w_hi, int drop_trivial, float *__restrict__ w, float *__restrict__ y,
                              uint32_t *__restrict__ keep) {
    const int lane = threadIdx.x & 31;
    const int64_t window = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t i = window * kSoftmaxStride + lane;          // windows of 32 entries every kSoftmaxStride entries
    const unsigned full = 0xffffffffu;
    const bool active = i < n;
    const uint32_t nseg = *num_seg;
    // #heads before entry k, continued past the table so that every k >= n counts as a head
    auto heads_before = [&](int64_t k) -> uint32_t { return k < n ? head_excl[k] : nseg + (uint32_t)(k - n); };
    const uint32_t he = heads_before(i);
    uint32_t he_next = __shfl_down_sync(full, he, 1);
    uint32_t he_next2 = 0;
    if (lane == 31) {
        he_next = heads_before(i + 1);
        he_next2 = heads_before(i + 2);
    }
    const bool is_head = (he_next - he) == 1;
    const unsigned hb = __ballot_sync(full, is_head);
    const bool after_is_head = __shfl_sync(full, (int)((he_next2 - he_next) == 1), 31) != 0;
    const unsigned upto = (lane == 31) ? full : ((2u << lane) - 1u);         // lanes 0 .. lane
    const unsigned le = hb & upto, gt = hb & ~upto;
    const int sl = le ? 31 - __clz(le) : 0;
    const int el = gt ? __ffs(gt) - 2 : 31;
    const bool interior = active && le != 0 && (gt != 0 || after_is_head);
    const int my_el = interior ? el : lane;                                   // others never absorb a neighbour

    int32_t qi = 0, ti = 0;
    double x = 0.0;
    if (active) {
        qi = q[i];
        ti = t[i];
        x = bits[i];
    }
    const bool self = qi == ti;
    const unsigned segmask = (el == 31 ? full : ((2u << el) - 1u)) & ~((1u << sl) - 1u);
    const int members = __popc(__ballot_sync(full, active && !self) & segmask);
    // segmented suffix max of the non-self scores, broadcast from the segment's first lane.  A softmax is
    // shift-invariant, so the shift only has to be NEAR the maximum: it is taken over the scores rounded to fp32
    // (one shuffle per step instead of two, fp32 max instead of fp64 compare + select); the difference
    // x - shift below is still formed in fp64
    float v = (active && !self) ? (float)x : -INFINITY;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const float o = __shfl_down_sync(full, v, d);
        if (lane + d <= my_el) v = fmaxf(v, o);
    }
    const double bmax = (double)__shfl_sync(full, v, sl);
    float e = 0.f;
    if (interior && !self && members > 1) e = expf((float)((x - bmax) * inv_temp));
    double sum = (double)e;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const double o = __shfl_down_sync(full, sum, d);
        if (lane + d <= my_el) sum += o;
    }
    sum = __shfl_sync(full, sum, sl);
    // a segment that also lies completely inside the PREVIOUS window (it ends within the overlap) is emitted there
    if (!interior || (window > 0 && el < 32 - kSoftmaxStride)) return;
    emit_entry(i, qi, ti, self, drop_trivial && el == sl, members, (double)e, sum > 0.0 ? sum : 1.0, eps, pseudo,
               w_lo, w_hi, group_of, w, y, keep);
}

// Segments that fit in NO window (longer than the overlap allows at their position; the warp kernel above skips
// them): a segment starting in [S k, S k + S) (S = kSoftmaxStride) fits window k iff it ends by S k + 32, so an
// unfit one contains entry p = S k + 32.  One thread per window k looks at the segment holding p and handles it
// when it starts at or after S k: its id goes to `long_list` for the cooperative kernel.  Each unfit segment is
// seen by exactly one thread.
__global__ void __launch_bounds__(256)
segment_softmax_q_boundary_kernel(const int32_t *__restrict__ q, const int32_t *__restrict__ t,
                                  const double *__restrict__ bits, const uint32_t *__restrict__ head_excl,
                                  const int64_t *__restrict__ seg_start, const uint32_t *__restrict__ num_seg,
                                  int64_t n, const int32_t *__restrict__ group_of, double inv_temp, double eps,
                                  double pseudo, float w_lo, float w_hi, int drop_trivial, float *__restrict__ w,
                                  float *__restrict__ y, uint32_t *__restrict__ keep,
                                  uint32_t *__restrict__ long_count, uint32_t *__restrict__ long_list) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t p = k * kSoftmaxStride + 32;
    if (p >= n) return;
    // most p are heads (78 % of the C3 segments are singletons): decided from two neighbouring counters, before
    // the dependent seg_start lookups
    const uint32_t hp = head_excl[p], hn = p + 1 < n ? head_excl[p + 1] : *num_seg;
    if (hn - hp == 1u) return;
    const int64_t seg = (int64_t)hp - 1;                       // segment of the entry BEFORE p ...
    const int64_t s0 = seg_start[seg], s1 = seg_start[seg + 1];
    if (s1 <= p) return;                                       // ... ends at p: entry p is a head
    if (s0 < k * kSoftmaxStride) return;                       // starts in an earlier window's range: handled there
    if (s0 >= (k + 1) * kSoftmaxStride) return;                // starts in the NEXT window's range: fits there, or is
                                                               // found by that window's thread
    // every unfit segment (10 or more entries) goes to the cooperative kernel, 8 lanes per segment with coalesced
    // loads.  (Until round 2 segments of up to 32 entries were handled right here, serially by this one thread:
    // three dependent walks over the segment in one lane made this filter pass latency-bound at 0.10 ms.)
    long_list[atomicAdd(long_count, 1u)] = (uint32_t)seg;      // disjoint outputs: any order
}

__global__ void __launch_bounds__(256)
segment_softmax_q_kernel(const int32_t *__restrict__ q, const int32_t *__restrict__ t,
                         const double *__restrict__ bits, const int64_t *__restrict__ seg_start,
                         const uint32_t *__restrict__ num_seg, const uint32_t *__restrict__ seg_list,
                         const int32_t *__restrict__ group_of,
                         double inv_temp, double eps, double pseudo, float w_lo, float w_hi, int drop_trivial,
                         float *__restrict__ w, float *__restrict__ y, uint32_t *__restrict__ keep) {
    const int lane = threadIdx.x & 31, gl = lane & (kGL - 1);
    const unsigned gmask = ((1u << kGL) - 1u) << (lane & ~(kGL - 1));
    const int64_t ngroups = (int64_t)gridDim.x * blockDim.x / kGL;
    const int64_t nseg = (int64_t)*num_seg;                    // number of entries of seg_list (or of segments)
    for (int64_t k = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / kGL; k < nseg; k += ngroups) {
        const int64_t seg = seg_list ? (int64_t)seg_list[k] : k;
        const int64_t s0 = seg_start[seg], s1 = seg_start[seg + 1];
        const bool trivial = drop_trivial && (s1 - s0) == 1;    // the self hit counts (a1)
        if (s1 - s0 == 1) {
            // ---- singleton (with the default filter: trivial, dropped later): p = 1, w saturates
            if (gl == 0) {
                const int32_t qi = q[s0], ti = t[s0];
                emit_entry(s0, qi, ti, qi == ti, trivial, 1, 0.0, 1.0, eps, pseudo, w_lo, w_hi, group_of, w, y, keep);
            }
        } else if (s1 - s0 <= kGL) {
            // ---- single pass: one entry per lane
            const int64_t i = s0 + gl;
            const bool have = i < s1;
            int32_t qi = 0, ti = 0;
            double x = -INFINITY;
            bool self = true;
            if (have) {
                qi = q[i]; ti = t[i];
                self = qi == ti;
                if (!self) x = bits[i] * inv_temp;
            }
            const int members = group_sum((have && !self) ? 1 : 0, gmask);
            const double mx = group_max(x, gmask);
            const double e = (have && !self && members > 1) ? exp_diff(x, mx) : 0.0;
            const double sum = group_sum(e, gmask);
            if (have) emit_entry(i, qi, ti, self, trivial, members, e, sum, eps, pseudo, w_lo, w_hi, group_of, w, y, keep);
        } else {
            // ---- long segment: max, sum, emit
            double mx = -INFINITY;
            int members = 0;
            for (int64_t i = s0 + gl; i < s1; i += kGL)
                if (q[i] != t[i]) {
                    mx = fmax(mx, bits[i] * inv_temp);
                    ++members;
                }
            mx = group_max(mx, gmask);
            members = group_sum(members, gmask);
            double sum = 0.0;
            if (members > 1)
                for (int64_t i = s0 + gl; i < s1; i += kGL)
                    if (q[i] != t[i]) sum += exp_diff(bits[i] * inv_temp, mx);
            sum = group_sum(sum, gmask);
            for (int64_t i = s0 + gl; i < s1; i += kGL) {
                const int32_t qi = q[i], ti = t[i];
                const bool self = qi == ti;
                const double e = (!self && members > 1) ? exp_diff(bits[i] * inv_temp, mx) : 0.0;
                emit_entry(i, qi, ti, self, false, members, e, sum, eps, pseudo, w_lo, w_hi, group_of, w, y, keep);
            }
        }
    }
}

// ---- max-candidate baseline (src/helper.py:437-485, 494-576): label = 1 iff no candidate of the same
// (query, target genome) segment scores strictly higher.  Same segmentation as the softmax: thread per
// entry for segments <= kElemMaxSeg, 8 lanes per listed long segment.
template <typename T>
__global__ void __launch_bounds__(256)
segment_max_label_entry_kernel(const T *__restrict__ score, const uint32_t *__restrict__ head_excl,
                               const int64_t *__restrict__ seg_start, int64_t n, int32_t *__restrict__ label,
                               uint32_t *__restrict__ long_count, uint32_t *__restrict__ long_list) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int64_t seg = head_excl[i];
    int64_t s0 = seg_start[seg];
    if (s0 != i) {
        --seg;
        s0 = seg_start[seg];
    }
    const int64_t s1 = seg_start[seg + 1];
    if (s1 - s0 > kElemMaxSeg) {
        if (s0 == i) long_list[atomicAdd(long_count, 1u)] = (uint32_t)seg;
        return;
    }
    const T mine = score[i];
    bool top = true;
    for (int64_t j = s0; j < s1; ++j) top = top && !(score[j] > mine);
    label[i] = top ? 1 : 0;
}

template <typename T>
__global__ void __launch_bounds__(256)
segment_max_label_long_kernel(const T *__restrict__ score, const int64_t *__restrict__ seg_start,
                              const uint32_t *__restrict__ long_count, const uint32_t *__restrict__ long_list,
                              int32_t *__restrict__ label) {
    const int lane = threadIdx.x & 31, gl = lane & (kGL - 1);
    const unsigned gmask = ((1u << kGL) - 1u) << (lane & ~(kGL - 1));
    const int64_t ngroups = (int64_t)gridDim.x * blockDim.x / kGL;
    const int64_t nlong = (int64_t)*long_count;
    for (int64_t k = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / kGL; k < nlong; k += ngroups) {
        const int64_t seg = long_list[k];
        const int64_t s0 = seg_start[seg], s1 = seg_start[seg + 1];
        double mx = -INFINITY;
        for (int64_t i = s0 + gl; i < s1; i += kGL) mx = fmax(mx, (double)score[i]);
        mx = group_max(mx, gmask);
        for (int64_t i = s0 + gl; i < s1; i += kGL) label[i] = ((double)score[i] >= mx) ? 1 : 0;
    }
}

__global__ void compact_edges_kernel(const int32_t *__restrict__ q, const int32_t *__restrict__ t,
                                     const float *__restrict__ w, const float *__restrict__ y,
                                     const uint32_t *__restrict__ keep, const uint32_t *__restrict__ pos,
                                     int64_t n, int32_t *__restrict__ src, int32_t *__restrict__ dst,
                                     float *__restrict__ w_out, float *__restrict__ y_out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !keep[i]) return;
    const uint32_t p = pos[i];
    src[p] = q[i];
    dst[p] = t[i];
    w_out[p] = w[i];
    y_out[p] = y[i];
}

}  // namespace pangnn

using namespace pangnn;

extern "C" {

size_t pangnn_scan_workspace_bytes(int64_t n);
size_t pangnn_sort_pairs_workspace_bytes(int64_t n);

size_t pangnn_hits_sort_unique_workspace_bytes(int64_t n) {
    return 2 * align_up((size_t)n * 8, 256) + 3 * align_up((size_t)n * 4, 256) +
           pangnn_sort_pairs_workspace_bytes(n) + pangnn_scan_workspace_bytes(n) + 2048;
}

int pangnn_hits_sort_unique(const int32_t *q, const int32_t *t, const double *bits, int64_t n,
                            int32_t num_nodes, int32_t *q_out, int32_t *t_out, double *bits_out,
                            uint32_t *count, void *ws, size_t ws_bytes, void *stream) {
    PANGNN_REQUIRE(count, "null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    if (n == 0) return check_cuda(cudaMemsetAsync(count, 0, 4, st), "memset");
    PANGNN_REQUIRE(q && t && bits && q_out && t_out && bits_out && ws, "null pointer");
    if (ws_bytes < pangnn_hits_sort_unique_workspace_bytes(n)) {
        set_error("hits_sort_unique: workspace too small");
        return PANGNN_EWORKSPACE;
    }
    Workspace w(ws, ws_bytes);
    uint64_t *ka = w.take<uint64_t>(n);
    uint64_t *kb = w.take<uint64_t>(n);
    uint32_t *vals = w.take<uint32_t>(n);
    uint32_t *flag = w.take<uint32_t>(n);
    const size_t scan_bytes = pangnn_scan_workspace_bytes(n);
    void *scan_ws = w.take<char>(scan_bytes);
    const size_t sort_bytes = pangnn_sort_pairs_workspace_bytes(n);
    void *sort_ws = w.take<char>(sort_bytes);
    const int nbits = bits_for_nodes(num_nodes > 1 ? num_nodes : 2);
    const unsigned blocks = (unsigned)((n + 255) / 256);
    hits_pack_kernel<<<blocks, 256, 0, st>>>(q, t, n, nbits, ka);
    PANGNN_CHECK_LAUNCH("hits_pack");
    int rc = sort_pairs_u64(ka, nullptr, kb, vals, n, 2 * nbits, sort_ws, sort_bytes, st);
    if (rc) return rc;
    hits_last_flag_kernel<<<blocks, 256, 0, st>>>(kb, n, flag);
    PANGNN_CHECK_LAUNCH("hits_last_flag");
    rc = exclusive_scan_u32(flag, flag, n, count, scan_ws, scan_bytes, st);
    if (rc) return rc;
    hits_unpack_kernel<<<blocks, 256, 0, st>>>(kb, vals, flag, bits, n, nbits, q_out, t_out, bits_out);
    PANGNN_CHECK_LAUNCH("hits_unpack");
    return PANGNN_OK;
}

size_t pangnn_hits_normalize_workspace_bytes(int64_t n) {
    return align_up((size_t)(n + 1) * 8, 256) + 6 * align_up((size_t)n * 4, 256) +
           pangnn_scan_workspace_bytes(n) + 4096;
}

int pangnn_hits_normalize(const int32_t *q, const int32_t *t, const double *bits, int64_t n,
                          const int32_t *genome_of, const int32_t *group_of, double temp, double eps,
                          double pseudo, int drop_trivial, int32_t *src, int32_t *dst, float *w_out,
                          float *y_out, uint32_t *count, void *ws, size_t ws_bytes, void *stream) {
    PANGNN_REQUIRE(count, "null pointer");
    PANGNN_REQUIRE(temp > 0.0, "temperature must be > 0");
    cudaStream_t st = (cudaStream_t)stream;
    if (n == 0) return check_cuda(cudaMemsetAsync(count, 0, 4, st), "memset");
    PANGNN_REQUIRE(q && t && bits && genome_of && src && dst && w_out && y_out && ws, "null pointer");
    if (ws_bytes < pangnn_hits_normalize_workspace_bytes(n)) {
        set_error("hits_normalize: workspace too small");
        return PANGNN_EWORKSPACE;
    }
    Workspace wk(ws, ws_bytes);
    int64_t *seg_start = wk.take<int64_t>(n + 1);
    uint32_t *flag = wk.take<uint32_t>(n);           // heads, then keep flags / positions
    float *w = wk.take<float>(n);
    float *y = wk.take<float>(n);
    uint32_t *num_seg = wk.take<uint32_t>(64);
    const size_t scan_bytes = pangnn_scan_workspace_bytes(n);
    void *scan_ws = wk.take<char>(scan_bytes);
    uint32_t *keep = wk.take<uint32_t>(n);
    uint32_t *long_list = wk.take<uint32_t>(n / kLongListDiv + 1);
    const unsigned blocks = (unsigned)((n + 255) / 256);

    seg_head_kernel<<<blocks, 256, 0, st>>>(q, t, genome_of, n, flag);
    PANGNN_CHECK_LAUNCH("seg_head");
    int rc = exclusive_scan_u32(flag, flag, n, num_seg, scan_ws, scan_bytes, st);
    if (rc) return rc;
    seg_start_kernel<<<blocks, 256, 0, st>>>(flag, q, t, genome_of, n, num_seg, seg_start);
    PANGNN_CHECK_LAUNCH("seg_start");
    // bulk: thread per entry in overlapping 32-entry windows; tail (segments that fit no window, listed by the boundary
    // kernel): 8 lanes per
    // segment, persistent grid.
    uint32_t *long_count = num_seg + 1;
    rc = check_cuda(cudaMemsetAsync(long_count, 0, sizeof(uint32_t), st), "memset");
    if (rc) return rc;
    // the two values the clip saturates to, computed once with the kernel's formula
    const float w_hi = (float)(-10.0 * log10(eps) + pseudo), w_lo = (float)(-10.0 * log10(1.0 - eps) + pseudo);
    const int64_t windows = (n + kSoftmaxStride - 1) / kSoftmaxStride;
    segment_softmax_q_warp_kernel<<<(unsigned)((windows * 32 + 255) / 256), 256, 0, st>>>(
        q, t, bits, flag, num_seg, n, group_of, 1.0 / temp, eps, pseudo, w_lo, w_hi, drop_trivial, w, y, keep);
    PANGNN_CHECK_LAUNCH("segment_softmax_q_warp");
    if (n > 32) {
        segment_softmax_q_boundary_kernel<<<(unsigned)((windows + 255) / 256), 256, 0, st>>>(
            q, t, bits, flag, seg_start, num_seg, n, group_of, 1.0 / temp, eps, pseudo, w_lo, w_hi, drop_trivial, w, y,
            keep, long_count, long_list);
        PANGNN_CHECK_LAUNCH("segment_softmax_q_boundary");
    }
    const int64_t want = (n / kLongListDiv * kGL + 255) / 256;
    const unsigned wblocks = (unsigned)(want < (int64_t)kNumSMs * 8 ? (want > 0 ? want : 1) : (int64_t)kNumSMs * 8);
    segment_softmax_q_kernel<<<wblocks, 256, 0, st>>>(q, t, bits, seg_start, long_count, long_list, group_of, 1.0 / temp,
                                                      eps, pseudo, w_lo, w_hi, drop_trivial, w, y, keep);
    PANGNN_CHECK_LAUNCH("segment_softmax_q");
    rc = exclusive_scan_u32(keep, flag, n, count, scan_ws, scan_bytes, st);
    if (rc) return rc;
    compact_edges_kernel<<<blocks, 256, 0, st>>>(q, t, w, y, keep, flag, n, src, dst, w_out, y_out);
    PANGNN_CHECK_LAUNCH("compact_edges");
    return PANGNN_OK;
}

size_t pangnn_segment_max_labels_workspace_bytes(int64_t n) {
    return align_up((size_t)(n + 1) * 8, 256) + 2 * align_up((size_t)n * 4, 256) + pangnn_scan_workspace_bytes(n) + 4096;
}

int pangnn_segment_max_labels(const int32_t *q, const int32_t *t, const void *score, int score_is_f64, int64_t n,
                              const int32_t *genome_of, int32_t *label, void *ws, size_t ws_bytes, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (n == 0) return PANGNN_OK;
    PANGNN_REQUIRE(q && t && score && genome_of && label && ws, "null pointer");
    if (ws_bytes < pangnn_segment_max_labels_workspace_bytes(n)) {
        set_error("segment_max_labels: workspace too small");
        return PANGNN_EWORKSPACE;
    }
    Workspace wk(ws, ws_bytes);
    int64_t *seg_start = wk.take<int64_t>(n + 1);
    uint32_t *flag = wk.take<uint32_t>(n);
    uint32_t *long_list = wk.take<uint32_t>(n / kLongListDiv + 1);
    uint32_t *num_seg = wk.take<uint32_t>(64);
    const size_t scan_bytes = pangnn_scan_workspace_bytes(n);
    void *scan_ws = wk.take<char>(scan_bytes);
    const unsigned blocks = (unsigned)((n + 255) / 256);
    seg_head_kernel<<<blocks, 256, 0, st>>>(q, t, genome_of, n, flag);
    PANGNN_CHECK_LAUNCH("seg_head");
    int rc = exclusive_scan_u32(flag, flag, n, num_seg, scan_ws, scan_bytes, st);
    if (rc) return rc;
    seg_start_kernel<<<blocks, 256, 0, st>>>(flag, q, t, genome_of, n, num_seg, seg_start);
    PANGNN_CHECK_LAUNCH("seg_start");
    uint32_t *long_count = num_seg + 1;
    rc = check_cuda(cudaMemsetAsync(long_count, 0, sizeof(uint32_t), st), "memset");
    if (rc) return rc;
    const int64_t want = (n / kLongListDiv * kGL + 255) / 256;
    const unsigned wblocks = (unsigned)(want < (int64_t)kNumSMs * 8 ? (want > 0 ? want : 1) : (int64_t)kNumSMs * 8);
    if (score_is_f64) {
        const double *sc = static_cast<const double *>(score);
        segment_max_label_entry_kernel<double><<<blocks, 256, 0, st>>>(sc, flag, seg_start, n, label, long_count, long_list);
        PANGNN_CHECK_LAUNCH("segment_max_label_entry");
        segment_max_label_long_kernel<double><<<wblocks, 256, 0, st>>>(sc, seg_start, long_count, long_list, label);
    } else {
        const float *sc = static_cast<const float *>(score);
        segment_max_label_entry_kernel<float><<<blocks, 256, 0, st>>>(sc, flag, seg_start, n, label, long_count, long_list);
        PANGNN_CHECK_LAUNCH("segment_max_label_entry");
        segment_max_label_long_kernel<float><<<wblocks, 256, 0, st>>>(sc, seg_start, long_count, long_list, label);
    }
    PANGNN_CHECK_LAUNCH("segment_max_label_long");
    return PANGNN_OK;
}

}  // extern "C"
