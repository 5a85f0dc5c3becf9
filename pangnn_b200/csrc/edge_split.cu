// Held-out validation and test edges of whole-graph training (--edge_split VAL TEST, pangnn_b200/edge_split.py).
// A scored edge (s, d) is assigned by its unordered pair a = min(s, d), b = max(s, d): x = the first word of the
// Philox4x32-10 stream keyed by (seed, purpose 5) at counter (0, a, b, 0); validation if x < t_val, test if
// x < t_val + t_test, else train.  Both directions of a pair fall in the same split, and the split depends on
// (seed, a, b) alone: every rank of a genome partition splits its own edges with no communication, at any world size.
// Roofline: HBM, 8 B read and 1 B written per edge; runs once per graph.
#include "common.cuh"
#include "philox.cuh"

namespace pangnn {
namespace {

constexpr uint32_t kSplitPurpose = 5;     // purposes 1-4 are simulate.cu's

__global__ void __launch_bounds__(256)
edge_split_kernel(const int32_t *__restrict__ src, const int32_t *__restrict__ dst, int64_t num_edges, uint64_t seed,
                  uint32_t t_val, uint64_t t_vt, int8_t *__restrict__ split) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= num_edges) return;
    const uint32_t s = (uint32_t)src[e], d = (uint32_t)dst[e];
    Philox g(seed, kSplitPurpose, s < d ? s : d, s < d ? d : s);
    const uint32_t x = g.next();
    split[e] = x < t_val ? (int8_t)PANGNN_SPLIT_VAL : ((uint64_t)x < t_vt ? (int8_t)PANGNN_SPLIT_TEST
                                                                           : (int8_t)PANGNN_SPLIT_TRAIN);
}

}  // namespace
}  // namespace pangnn

using namespace pangnn;

extern "C" int pangnn_edge_split(const int32_t *src, const int32_t *dst, int64_t num_edges, uint64_t seed,
                                 uint32_t t_val, uint32_t t_test, int8_t *split, void *stream) {
    PANGNN_REQUIRE(num_edges >= 0, "negative edge count");
    if (num_edges == 0) return PANGNN_OK;
    PANGNN_REQUIRE(src && dst && split, "null pointer");
    const uint64_t t_vt = (uint64_t)t_val + t_test;
    PANGNN_REQUIRE(t_vt <= (1ull << 32), "t_val + t_test exceeds 2^32");
    edge_split_kernel<<<(unsigned)((num_edges + 255) / 256), 256, 0, (cudaStream_t)stream>>>(src, dst, num_edges, seed,
                                                                                             t_val, t_vt, split);
    PANGNN_CHECK_LAUNCH("edge_split");
    return PANGNN_OK;
}
