// Data-parallel gradient average over NVLink peer memory (new; the reference gets it from DDP's NCCL all-reduce
// behind accelerator.backward, pangnn.py:207).  Two stream-ordered launches per step, both legal in a CUDA-graph
// capture and correct on every replay:
//   push:    gradients -> this rank's bucket half (e & 1); the last CTA signals e + 1 to every peer
//   reduce:  wait for all peers' e + 1, grad = (b_0 + ... + b_{W-1}) * fp32(1/W) in rank order; last CTA: e += 1
// Nothing host-side is baked into a captured launch except the pointers themselves (gradients by value in the
// kernel parameters, symmetric-memory mappings that live as long as the group): the epoch, and so the bucket
// half and the signal value, are read from device memory at run time.
//
// Bucket layout: tensor t occupies floats [off_t, off_t + numel_t) of a half, off_t a multiple of 4 (so the
// bucket side is read and written as float4; the gradient side is element-wise, no alignment assumed).
#include "common.cuh"

namespace pangnn {

constexpr int kGradThreads = 256;

struct GradList {
    float *ptr[PANGNN_GRAD_REDUCE_MAX_TENSORS];
    int64_t numel[PANGNN_GRAD_REDUCE_MAX_TENSORS];
    int64_t off4[PANGNN_GRAD_REDUCE_MAX_TENSORS + 1];     // bucket offsets in float4 units; off4[count] = total
    int32_t count;
};

struct PeerPtrs {
    const float *bucket[PANGNN_GRAD_REDUCE_MAX_RANKS];
    int32_t *signal[PANGNN_GRAD_REDUCE_MAX_RANKS];
};

enum { kEpoch = 0, kPushTicket = 1, kReduceTicket = 2, kStatus = 3 };

__device__ __forceinline__ int find_tensor(const GradList &g, int64_t i4) {
    int t = 0;
    while (t + 1 < g.count && g.off4[t + 1] <= i4) ++t;
    return t;
}

__device__ __forceinline__ void st_release_sys(int32_t *p, int32_t v) {
    asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

__device__ __forceinline__ int32_t ld_acquire_sys(const int32_t *p) {
    int32_t v;
    asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ uint64_t globaltimer() {
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// Ticket of a one-shot grid: true in the last CTA to arrive (after every other CTA's fence), which also resets
// the counter for the next launch.
__device__ __forceinline__ bool last_cta(int32_t *ticket) {
    __shared__ bool last;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence_system();                               // this CTA's stores before its ticket
        last = atomicAdd(ticket, 1) == (int32_t)gridDim.x - 1;
        if (last) {
            *ticket = 0;
            __threadfence_system();                           // every CTA's stores before what the last one does
        }
    }
    __syncthreads();
    return last;
}

__global__ void __launch_bounds__(kGradThreads)
grad_push_kernel(const __grid_constant__ GradList g, float *__restrict__ bucket, int64_t half_floats,
                 const __grid_constant__ PeerPtrs peers, int32_t world, int32_t rank, int32_t *ctrl) {
    const int32_t e = *(volatile int32_t *)(ctrl + kEpoch);
    float4 *dst = reinterpret_cast<float4 *>(bucket + (int64_t)(e & 1) * half_floats);
    const int64_t total4 = g.off4[g.count];
    for (int64_t i4 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i4 < total4;
         i4 += (int64_t)gridDim.x * blockDim.x) {
        const int t = find_tensor(g, i4);
        const int64_t j = (i4 - g.off4[t]) * 4;
        const float *src = g.ptr[t];
        const int64_t n = g.numel[t];
        float v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k] = (src != nullptr && j + k < n) ? src[j + k] : 0.f;
        dst[i4] = make_float4(v[0], v[1], v[2], v[3]);
    }
    if (last_cta(ctrl + kPushTicket) && threadIdx.x == 0)
        for (int p = 0; p < world; ++p) st_release_sys(peers.signal[p] + rank, e + 1);
}

__global__ void __launch_bounds__(kGradThreads)
grad_reduce_kernel(const __grid_constant__ GradList g, int64_t half_floats, const __grid_constant__ PeerPtrs peers,
                   const int32_t *signal, int32_t world, float scale, int32_t *ctrl, int64_t timeout_ns) {
    __shared__ int32_t missing;
    const int32_t e = *(volatile int32_t *)(ctrl + kEpoch);
    if (threadIdx.x == 0) {
        missing = -1;
        const uint64_t t0 = globaltimer();
        unsigned ns = 32;
        for (int p = 0; p < world && missing < 0; ++p) {
            while ((int32_t)(ld_acquire_sys(signal + p) - (e + 1)) < 0) {     // signals only grow (wrap-safe)
                if ((int64_t)(globaltimer() - t0) > timeout_ns) {
                    missing = p;
                    break;
                }
                __nanosleep(ns);
                ns = ns < 4096 ? ns * 2 : ns;
            }
        }
        if (missing >= 0) atomicCAS(ctrl + kStatus, 0, 1 + missing);
    }
    __syncthreads();
    if (missing < 0) {
        const int64_t total4 = g.off4[g.count];
        const int64_t h = (int64_t)(e & 1) * half_floats;
        for (int64_t i4 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i4 < total4;
             i4 += (int64_t)gridDim.x * blockDim.x) {
            const int t = find_tensor(g, i4);
            float *out = g.ptr[t];
            if (out == nullptr) continue;
            // peer memory written by another kernel: L2-coherent loads, never the non-coherent path
            float4 acc = __ldcg(reinterpret_cast<const float4 *>(peers.bucket[0] + h) + i4);
            for (int p = 1; p < world; ++p) {
                const float4 b = __ldcg(reinterpret_cast<const float4 *>(peers.bucket[p] + h) + i4);
                acc.x += b.x; acc.y += b.y; acc.z += b.z; acc.w += b.w;
            }
            const float r[4] = {acc.x * scale, acc.y * scale, acc.z * scale, acc.w * scale};
            const int64_t j = (i4 - g.off4[t]) * 4, n = g.numel[t];
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (j + k < n) out[j + k] = r[k];
        }
    }
    if (last_cta(ctrl + kReduceTicket) && threadIdx.x == 0) *(volatile int32_t *)(ctrl + kEpoch) = e + 1;
}

int64_t bucket_floats(const int64_t *numels, int32_t count, int64_t *off4) {
    int64_t o = 0;
    for (int32_t t = 0; t < count; ++t) {
        if (numels[t] < 0) return -1;
        if (off4) off4[t] = o;
        o += (numels[t] + 3) / 4;
    }
    if (off4) off4[count] = o;
    return o * 4;
}

int make_list(float *const *grads, const int64_t *numels, int32_t count, int64_t half_floats, GradList &g) {
    PANGNN_REQUIRE(count >= 1 && count <= PANGNN_GRAD_REDUCE_MAX_TENSORS, "1 <= count <= 32 gradient tensors");
    PANGNN_REQUIRE(grads && numels, "null gradient table");
    const int64_t need = bucket_floats(numels, count, g.off4);
    PANGNN_REQUIRE(need >= 0, "negative tensor size");
    PANGNN_REQUIRE(half_floats >= need && half_floats % 4 == 0, "bucket half too small or not a multiple of 4 floats");
    g.count = count;
    for (int32_t t = 0; t < count; ++t) {
        g.ptr[t] = grads[t];
        g.numel[t] = numels[t];
    }
    return PANGNN_OK;
}

unsigned grad_grid(const GradList &g) {
    const int64_t blocks = (g.off4[g.count] + kGradThreads - 1) / kGradThreads;
    return (unsigned)(blocks < 1 ? 1 : (blocks > kNumSMs ? kNumSMs : blocks));
}

}  // namespace pangnn

using namespace pangnn;

extern "C" {

int64_t pangnn_grad_bucket_floats(const int64_t *numels, int32_t count) {
    if (!numels || count < 0) return -1;
    return bucket_floats(numels, count, nullptr);
}

int pangnn_grad_push(float *const *grads, const int64_t *numels, int32_t count, float *bucket, int64_t half_floats,
                     int32_t *const *peer_signals, int32_t world, int32_t rank, int32_t *ctrl, void *stream) {
    PANGNN_REQUIRE(world >= 1 && world <= PANGNN_GRAD_REDUCE_MAX_RANKS, "1 <= world <= 8");
    PANGNN_REQUIRE(rank >= 0 && rank < world, "0 <= rank < world");
    PANGNN_REQUIRE(bucket && ctrl && peer_signals && (uintptr_t)bucket % 16 == 0, "null or misaligned buffer");
    GradList g;
    int rc = make_list(grads, numels, count, half_floats, g);
    if (rc != PANGNN_OK) return rc;
    PeerPtrs peers = {};
    for (int32_t p = 0; p < world; ++p) {
        PANGNN_REQUIRE(peer_signals[p], "null peer signal array");
        peers.signal[p] = peer_signals[p];
    }
    grad_push_kernel<<<grad_grid(g), kGradThreads, 0, (cudaStream_t)stream>>>(g, bucket, half_floats, peers, world,
                                                                              rank, ctrl);
    PANGNN_CHECK_LAUNCH("grad_push");
    return PANGNN_OK;
}

int pangnn_grad_reduce(float *const *grads, const int64_t *numels, int32_t count, const float *const *peer_buckets,
                       int64_t half_floats, const int32_t *signal, int32_t world, int32_t rank, int32_t *ctrl,
                       int64_t timeout_ns, void *stream) {
    PANGNN_REQUIRE(world >= 1 && world <= PANGNN_GRAD_REDUCE_MAX_RANKS, "1 <= world <= 8");
    PANGNN_REQUIRE(rank >= 0 && rank < world, "0 <= rank < world");
    PANGNN_REQUIRE(signal && ctrl && peer_buckets && timeout_ns > 0, "null buffer or non-positive timeout");
    GradList g;
    int rc = make_list(grads, numels, count, half_floats, g);
    if (rc != PANGNN_OK) return rc;
    PeerPtrs peers = {};
    for (int32_t p = 0; p < world; ++p) {
        PANGNN_REQUIRE(peer_buckets[p] && (uintptr_t)peer_buckets[p] % 16 == 0, "null or misaligned peer bucket");
        peers.bucket[p] = peer_buckets[p];
    }
    const float scale = 1.0f / (float)world;
    grad_reduce_kernel<<<grad_grid(g), kGradThreads, 0, (cudaStream_t)stream>>>(g, half_floats, peers, signal, world,
                                                                                scale, ctrl, timeout_ns);
    PANGNN_CHECK_LAUNCH("grad_reduce");
    return PANGNN_OK;
}

}  // extern "C"
