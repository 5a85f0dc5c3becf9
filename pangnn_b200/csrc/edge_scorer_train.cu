// Training form of the fused edge scorer on the tcgen05 tensor cores (3xTF32, fp32-grade): endpoint gather +
// 3-layer MLP + BCE-with-logits loss + the whole backward in ONE pass over the scored edges.  Replaces
// src/gnn.py:171-177, pangnn.py:98,203 and their autograd backward (pangnn.py:207).  The inference form lives in
// edge_scorer_tc.cu.
//
// Per 128-edge tile (layer 1 is hoisted to the nodes, pq[n] = [h W1a^T | h W1b^T]):
//   gather   r1 = relu(pq[src,0:64] + pq[dst,64:128] + w1c*skip + b1)  -> smem X (K-major hi / lo, operand A of G1)
//            and smem R (row-major hi / lo, operand B of G3); its relu mask -> 4-bit nibbles for epilogue 2
//   G1       a2 = r1 W2^T                                  D1 [128 x 64]
//   epi-1a   r2 = relu(a2 + b2); the relu MASK m2 as 1.0 / 0.0 -> TENSOR MEMORY (tcgen05.st, this thread's lane)
//   G2       g = m2 W2'   with W2'[j][k] = w3[j] W2[j][k]    D2 [128 x 64], A operand read from tensor memory.
//            dr1 = da2 W2 = dz (.) (m2 W2') row by row, so G2 needs neither dz nor a hi / lo split of its A operand
//            (a 0 / 1 matrix is exact in TF32: 2 products per k-step instead of 3) and is issued BEFORE the logit
//            reduction, the loss and the sigmoid — it runs underneath them.
//   epi-1b   z = r2 . w3 + b3 (one CTA barrier: partial sums of the 4 column slices); logit, loss, dz (an edge
//            without a label, y < 0, gets no loss term and dz = 0, so every gradient contribution vanishes);
//            dz m2 (hi / lo of the ROW scalar dz, selected by the mask) row-major -> smem over X (operand A of G3)
//   G3       [P_hi ; P_lo] += [dz m2 hi | dz m2 lo]^T (r1_hi + r1_lo)   D3 [128 x 64], both operands MN-major (the
//            row-major tiles themselves in the 128B / 32-byte-atom swizzle, umma.cuh); accumulates across the CTA's
//            tiles, drained into registers every 4 tiles (truncating accumulation); dW2[j][k] = w3[j] (P_hi + P_lo)
//   epi-2    da1 = dz (.) g (.) [r1 > 0] -> HBM [E, 64] (quad-transposed: 64 contiguous bytes per lane quad and
//            edge row); db1, dw1c column sums
//
// Hand-offs: a dedicated warp group only issues MMAs (one elected lane); compute warps arrive on `bar_ops` when
// their part of an operand set is written, the issuer commits each contraction to its own mbarrier (bar1/2/3).
// One CTA-wide barrier per tile; index staging and mask nibbles are double-buffered by tile parity.
//
// Roofline: HBM.  Bytes / edge: 8 idx + 512 gathered rows + 4 logit + 4 skip + 4 y + 256 da1 = 784.
#include "edge_scorer.cuh"
#include "umma.cuh"

namespace pangnn {

#ifdef PANGNN_SCORER_PROF
// development build only (python -m pangnn_b200.build --prof): per-phase cycle totals of thread 0 of every CTA
__device__ unsigned long long g_scorer_prof[16];
#define PROF_T(i) do { if (tid == 0) { const long long _c = clock64(); prof[i] += _c - prof_t; prof_t = _c; } } while (0)
#else
#define PROF_T(i) do { } while (0)
#endif

namespace {

constexpr int D = kScD;
constexpr int BM = 128;
constexpr int NT = 512;                          // compute threads: warp w serves TMEM lane group w % 4 (edge slots
constexpr int CPT = 16;                          // 32 (w%4) .. +31) and the column slice w / 4 of width 16
constexpr uint32_t CH = BM * 16 + 16;            // chunk stride of a [128 rows] K-major operand
constexpr uint32_t CHW = D * 16 + 16;            // chunk stride of a [64 rows] operand (W2, W2'^T)
constexpr uint32_t kOpBytes = (D / 4) * CH;      // 33024: one [128 x 64] K-major operand (hi or lo)
constexpr uint32_t kWBytes = (D / 4) * CHW;      // 16640: one [64 x 64] operand
constexpr uint32_t kPanel = BM * 128;            // 16 KB: 128 edge rows x 32 floats of an MN-major operand

// shared-memory map (bytes, relative to a 1024-byte aligned base)
constexpr uint32_t oXh = 0, oXl = oXh + kOpBytes;                       // r1 K-major; later P = dz m2 row-major (4 panels)
constexpr uint32_t oRh = (oXl + kOpBytes + 1023) / 1024 * 1024, oRl = oRh + 2 * kPanel;     // r1 row-major, hi / lo
constexpr uint32_t oWh = oRl + 2 * kPanel, oWl = oWh + kWBytes;         // W2 [j][k] (G1)
constexpr uint32_t oWTh = oWl + kWBytes, oWTl = oWTh + kWBytes;         // W2' [k][j] = w3[j] W2[j][k] (G2)
constexpr uint32_t oVec = oWTl + kWBytes;                               // b1, w1c, b2, w3: 4 x 64 floats
constexpr uint32_t oZp = oVec + 4 * D * 4;                              // [4][128] partial logits
constexpr uint32_t oSkip = oZp + 4 * BM * 4;                            // [2][128]
constexpr uint32_t oSrc = oSkip + 2 * BM * 4, oDst = oSrc + 2 * BM * 4;
constexpr uint32_t oM1 = oDst + 2 * BM * 4;                             // [2][128][16] relu-mask nibbles of r1
constexpr uint32_t oEnd = oM1 + 2 * BM * 16;
static_assert(4 * kPanel <= 2 * kOpBytes, "X must also hold the row-major [P_hi | P_lo] operand");
static_assert(oEnd + 1024 + 2048 <= 227 * 1024, "shared memory budget");

__device__ __forceinline__ float4 shfl_xor4(float4 v, int m) {
    v.x = __shfl_xor_sync(0xffffffffu, v.x, m); v.y = __shfl_xor_sync(0xffffffffu, v.y, m);
    v.z = __shfl_xor_sync(0xffffffffu, v.z, m); v.w = __shfl_xor_sync(0xffffffffu, v.w, m);
    return v;
}
// 4 x 4 transpose of float4 elements inside every quad of lanes: in, lane r of the quad holds S[c] = M[r][c];
// out, lane i holds S[j] = M[j][i].  Two exchange rounds (lane ^ 2, lane ^ 1), half of the data each.
__device__ __forceinline__ void quad_transpose(float4 (&S)[4], int lane) {
    const bool up = lane & 2, odd = lane & 1;
    float4 s0 = up ? S[0] : S[2], s1 = up ? S[1] : S[3];
    s0 = shfl_xor4(s0, 2); s1 = shfl_xor4(s1, 2);
    if (up) { S[0] = s0; S[1] = s1; } else { S[2] = s0; S[3] = s1; }
    s0 = odd ? S[0] : S[1]; s1 = odd ? S[2] : S[3];
    s0 = shfl_xor4(s0, 1); s1 = shfl_xor4(s1, 1);
    if (odd) { S[0] = s0; S[2] = s1; } else { S[1] = s0; S[3] = s1; }
}

// 512 compute threads + one warp GROUP (4 warps, one working lane) that only issues tcgen05.mma and hands registers
// to the compute warps (setmaxnreg 24 / 112: the CTA's pool is what it was launched with, 640 x 96 registers, so
// 512 x 120 + 128 x 24 does not fit — asking for 120 deadlocks; a single extra warp would put 5 warps on one
// scheduler = 96 registers each).
__global__ void __launch_bounds__(NT + 128, 1)
edge_score_train_kernel(const ScorerArgs p) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    // the swizzled MN-major operands want a 1024-byte aligned base (dynamic shared memory starts after the statics)
    uint8_t *smem = smem_raw + ((1024u - (umma::smem_u32(smem_raw) & 1023u)) & 1023u);
    __shared__ __align__(8) uint64_t bar_ops, bar1, bar2, bar3;      // operands ready; G1 / G2 / G3 complete
    __shared__ uint32_t tmem_base_s;
    __shared__ double lred[BM];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int q = warp & 3, h = warp >> 2;                   // TMEM lane group, column slice (compute warps)
    const int row = q * 32 + lane;                           // this thread's edge slot in the epilogues
    const uint32_t sb = umma::smem_u32(smem);
    float *sVec = reinterpret_cast<float *>(smem + oVec);
    float *sZp = reinterpret_cast<float *>(smem + oZp);
    float *sSkip = reinterpret_cast<float *>(smem + oSkip);
    int32_t *sSrc = reinterpret_cast<int32_t *>(smem + oSrc);
    int32_t *sDst = reinterpret_cast<int32_t *>(smem + oDst);
    uint8_t *sM1 = smem + oM1;
    constexpr uint32_t kTmemCols = 256;                      // D1 | D2 | D3 | m2 (64 columns each)

    // ---- one-time setup
    if (warp == 0) umma::tmem_alloc(&tmem_base_s, kTmemCols);
    if (tid == 32) {
        umma::mbar_init(&bar_ops, NT / 32);
        umma::mbar_init(&bar1, 1);
        umma::mbar_init(&bar2, 1);
        umma::mbar_init(&bar3, 1);
        umma::fence_mbar_init();
    }
    const bool issuer = warp >= NT / 32;
    auto sync_compute = [&]() { asm volatile("bar.sync 1, %0;" :: "n"(NT) : "memory"); };
    // this warp's part of an operand set is written (shared memory: visible to the async proxy; tensor memory:
    // stores complete): tell the issuer
    auto ops_ready = [&]() {
        umma::fence_async_smem();
        umma::fence_before_sync();
        __syncwarp();
        if (lane == 0) umma::mbar_arrive(&bar_ops);
    };
    for (int i = tid; i < D * D && !issuer; i += NT) {       // W2[j][k]: rows j over k; W2'[k][j]: rows k over j
        const int j = i / D, k = i % D;
        const float v = p.w2[i];
        const float hi = umma::tf32_hi(v), lo = umma::tf32_lo(v, hi);
        const uint32_t off = (uint32_t)(k >> 2) * CHW + (uint32_t)j * 16 + (uint32_t)(k & 3) * 4;
        *reinterpret_cast<float *>(smem + oWh + off) = hi;
        *reinterpret_cast<float *>(smem + oWl + off) = lo;
        const float vt = p.w3[j] * v;
        const float hit = umma::tf32_hi(vt), lot = umma::tf32_lo(vt, hit);
        const uint32_t offT = (uint32_t)(j >> 2) * CHW + (uint32_t)k * 16 + (uint32_t)(j & 3) * 4;
        *reinterpret_cast<float *>(smem + oWTh + offT) = hit;
        *reinterpret_cast<float *>(smem + oWTl + offT) = lot;
    }
    if (tid < D) {
        sVec[tid] = p.b1[tid];
        sVec[D + tid] = (p.skip && p.w1c) ? p.w1c[tid] : 0.f;
        sVec[2 * D + tid] = p.b2[tid];
        sVec[3 * D + tid] = p.w3[tid];
    }
    const float b3 = p.b3[0];
    umma::fence_async_smem();
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tD1 = tmem_base_s, tD2 = tmem_base_s + 64, tD3 = tmem_base_s + 128, tA = tmem_base_s + 192;
    const uint32_t lane_off = (uint32_t)(q * 32) << 16;
    constexpr uint32_t idesc = umma::idesc_tf32(BM, D, false, false);     // M = 128, N = 64, K-major x K-major
    constexpr int kG3Flush = 4;     // D3 is drained into registers every 4 tiles (the tensor core's fp32 accumulation
                                    // truncates, ~2e-8 relative per tcgen05.mma in the chain)
    const int64_t num_tiles = (p.E + BM - 1) / BM;

    if (issuer) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 24;");
        if (warp == NT / 32 && lane == 0) {
            // small code on purpose (24 registers per thread): rolled loops, descriptors advanced incrementally.
            // Measured and rejected: full unrolling (4.78 ms: the issuer spills on 24 registers); G3 as one N = 128
            // instruction per k-step over [r1_hi | r1_lo] (3.26 vs 3.04 ms); r1 handed to G1 through tensor memory
            // as well (quad-mapped gather + register transpose, R stores after G1: 3.33 ms — twice the load
            // wavefronts and 64 more shuffles per thread cost more than the G3 wait they remove); the next tile's
            // endpoint rows prefetched into registers across epilogue 2 (3.81 vs 3.53 ms on the previous kernel).
            uint32_t ready = 0;         // completed phases of bar_ops
            int64_t it = 0;
            const uint64_t dXh = umma::smem_desc(sb + oXh, CH, 128), dXl = umma::smem_desc(sb + oXl, CH, 128);
            const uint64_t dWh = umma::smem_desc(sb + oWh, CHW, 128), dWl = umma::smem_desc(sb + oWl, CHW, 128);
            const uint64_t dWTh = umma::smem_desc(sb + oWTh, CHW, 128), dWTl = umma::smem_desc(sb + oWTl, CHW, 128);
            const uint64_t dRh = umma::smem_desc_mn(sb + oRh, kPanel), dRl = umma::smem_desc_mn(sb + oRl, kPanel);
            const uint64_t dPmn = umma::smem_desc_mn(sb + oXh, kPanel);                     // 4 panels: hi j 0-63, lo j 0-63
            constexpr uint32_t idesc_mn = umma::idesc_tf32(BM, D, true, true);
            constexpr uint64_t stepX = (2 * CH) >> 4, stepW = (2 * CHW) >> 4;
            for (int64_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
                // G1: D1 = r1 W2^T
                umma::mbar_wait(&bar_ops, ready++ & 1);
                umma::fence_after_sync();
                {
                    uint64_t ah = dXh, al = dXl, bh = dWh, bl = dWl;
#pragma unroll 1
                    for (int s = 0; s < D / 8; ++s, ah += stepX, al += stepX, bh += stepW, bl += stepW) {
                        umma::mma_tf32(tD1, al, bh, idesc, s > 0 ? 1u : 0u);      // small terms first
                        umma::mma_tf32(tD1, ah, bl, idesc, 1u);
                        umma::mma_tf32(tD1, ah, bh, idesc, 1u);
                    }
                }
                umma::mma_commit(&bar1);
                // G2: D2 = m2 W2'  (A = the 0 / 1 mask in tensor memory, 8 columns per k-step; exact in TF32)
                umma::mbar_wait(&bar_ops, ready++ & 1);
                umma::fence_after_sync();
                {
                    uint64_t bh = dWTh, bl = dWTl;
                    uint32_t a = tA;
#pragma unroll 1
                    for (int s = 0; s < D / 8; ++s, a += 8, bh += stepW, bl += stepW) {
                        umma::mma_tf32_ts(tD2, a, bl, idesc, s > 0 ? 1u : 0u);
                        umma::mma_tf32_ts(tD2, a, bh, idesc, 1u);
                    }
                }
                umma::mma_commit(&bar2);
                // G3: D3 += [P_hi | P_lo]^T (r1_hi + r1_lo), both operands MN-major
                umma::mbar_wait(&bar_ops, ready++ & 1);
                umma::fence_after_sync();
                {
                    uint32_t acc = (it % kG3Flush) == 0 ? 0u : 1u;
                    uint64_t a = dPmn, bh = dRh, bl = dRl;
#pragma unroll 1
                    for (int s = 0; s < BM / 8; ++s, a += 64, bh += 64, bl += 64) {    // 8 edge rows = 1024 B per k-step
                        umma::mma_tf32(tD3, a, bl, idesc_mn, acc);
                        umma::mma_tf32(tD3, a, bh, idesc_mn, 1u);
                        acc = 1u;
                    }
                }
                umma::mma_commit(&bar3);
            }
        }
        __syncwarp();
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 112;");
        // per-thread column sums, live across tiles
        float gw3[CPT], gq2[CPT], g3acc[CPT];        // dw3; sum_e dz m2 (db2 = w3 (.) that); drained D3
        float4 gb1q = make_float4(0.f, 0.f, 0.f, 0.f), gw1cq = make_float4(0.f, 0.f, 0.f, 0.f);   // 4 columns x this quad's rows
        float gb3 = 0.f, loss_acc = 0.f;
#pragma unroll
        for (int c = 0; c < CPT; ++c) gw3[c] = gq2[c] = g3acc[c] = 0.f;
        int g3_tiles = 0;               // tiles accumulated in D3 since the last drain

        // indices of the tile after the staged one travel in registers (threads 0..127)
        int32_t nsrc = 0, ndst = 0;
        float nskip = 0.f;
        auto load_indices = [&](int64_t t) {
            nsrc = ndst = 0;
            nskip = 0.f;
            if (tid < BM && t < num_tiles) {
                const int64_t e = t * BM + tid;
                if (e < p.E) {
                    nsrc = p.src[e];
                    ndst = p.dst[e];
                    if (p.skip) nskip = p.skip[e];
                }
            }
        };
        auto stage_indices = [&](int b) {
            if (tid < BM) {
                sSrc[b * BM + tid] = nsrc;
                sDst[b * BM + tid] = ndst;
                sSkip[b * BM + tid] = nskip;
            }
        };
        load_indices(blockIdx.x);
        stage_indices(0);
        sync_compute();
        load_indices((int64_t)blockIdx.x + gridDim.x);
        // gather mapping: 16 lanes x float4 per endpoint row, 32 edges per pass, 4 passes
        const int fl = tid & 15, sub = tid >> 4;
        const float4 b1v = *reinterpret_cast<const float4 *>(sVec + fl * 4);
        const float4 w1cv = *reinterpret_cast<const float4 *>(sVec + D + fl * 4);
#ifdef PANGNN_SCORER_PROF
        long long prof[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}, prof_t = clock64();
#endif
        uint32_t it = 0;                // local tile counter: buffer / barrier parity
        for (int64_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
            const int b = it & 1;       // staging buffer of this tile (written during the previous tile)
            const uint32_t par = it & 1;
            const int64_t e0 = tile * BM;
            // ---- gather + layer-1 epilogue
            {
                float4 pv[4], qv[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int e = u * 32 + sub;
                    pv[u] = __ldg(reinterpret_cast<const float4 *>(p.pq + (int64_t)sSrc[b * BM + e] * (2 * D)) + fl);
                    qv[u] = __ldg(reinterpret_cast<const float4 *>(p.pq + (int64_t)sDst[b * BM + e] * (2 * D) + D) + fl);
                }
                if (it > 0) {                                // X / R are still being read by the previous tile's G3
                    umma::mbar_wait(&bar3, (it - 1) & 1);
                    if (g3_tiles == kG3Flush) {              // drain D3 (uniform branch)
                        umma::fence_after_sync();
                        float t[CPT];
                        umma::tmem_ld<CPT>(tD3 + lane_off + (uint32_t)(h * CPT), t);
#pragma unroll
                        for (int c = 0; c < CPT; ++c) g3acc[c] += t[c];
                        g3_tiles = 0;
                    }
                }
                PROF_T(0);
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int e = u * 32 + sub;
                    const float sk = sSkip[b * BM + e];
                    float4 a;
                    a.x = fmaxf(pv[u].x + qv[u].x + fmaf(w1cv.x, sk, b1v.x), 0.f);
                    a.y = fmaxf(pv[u].y + qv[u].y + fmaf(w1cv.y, sk, b1v.y), 0.f);
                    a.z = fmaxf(pv[u].z + qv[u].z + fmaf(w1cv.z, sk, b1v.z), 0.f);
                    a.w = fmaxf(pv[u].w + qv[u].w + fmaf(w1cv.w, sk, b1v.w), 0.f);
                    float4 ahi, alo;
                    umma::split4(a, ahi, alo);
                    const uint32_t offK = (uint32_t)fl * CH + (uint32_t)e * 16;
                    *reinterpret_cast<float4 *>(smem + oXh + offK) = ahi;
                    *reinterpret_cast<float4 *>(smem + oXl + offK) = alo;
                    const uint32_t offM = umma::mn_off((uint32_t)e, (uint32_t)fl * 4, kPanel);
                    *reinterpret_cast<float4 *>(smem + oRh + offM) = ahi;
                    *reinterpret_cast<float4 *>(smem + oRl + offM) = alo;
                    // relu mask of these 4 columns for epilogue 2 (r1 >= 0: positive <=> non-zero)
                    sM1[(b * BM + e) * 16 + fl] = (uint8_t)((a.x > 0.f ? 1u : 0u) | (a.y > 0.f ? 2u : 0u) |
                                                            (a.z > 0.f ? 4u : 0u) | (a.w > 0.f ? 8u : 0u));
                }
            }
            PROF_T(1);
            ops_ready();                                     // G1
            // while G1 runs: pull the next tile's endpoint rows into L2 (their indices are still in registers)
            if (tid < BM && tile + gridDim.x < num_tiles) {
                const char *ps = reinterpret_cast<const char *>(p.pq + (int64_t)nsrc * (2 * D));
                const char *pd = reinterpret_cast<const char *>(p.pq + (int64_t)ndst * (2 * D) + D);
                asm volatile("prefetch.global.L2 [%0];" :: "l"(ps));
                asm volatile("prefetch.global.L2 [%0];" :: "l"(ps + 128));
                asm volatile("prefetch.global.L2 [%0];" :: "l"(pd));
                asm volatile("prefetch.global.L2 [%0];" :: "l"(pd + 128));
            }
            PROF_T(2);
            // this edge slot's label, loaded before the G1 wait so that its latency hides under the contraction
            const int64_t e = e0 + row;
            const bool ok = e < p.E;
            const float yy = (ok && p.y) ? __ldg(p.y + e) : 0.f;
            umma::mbar_wait(&bar1, par);
            umma::fence_after_sync();
            PROF_T(3);
            // ---- epilogue 1a: thread = edge slot `row`, columns h*16 .. h*16+15: r2 and its mask
            float v[CPT];
            umma::tmem_ld<CPT>(tD1 + lane_off + (uint32_t)(h * CPT), v);
            uint32_t m2 = 0;                                 // bit c: a2[row][h*16 + c] + b2 > 0
            float zp = 0.f;
#pragma unroll
            for (int c0 = 0; c0 < CPT; c0 += 8) {
                float mk[8];
#pragma unroll
                for (int c = c0; c < c0 + 8; c += 4) {
                    const float4 b2v = *reinterpret_cast<const float4 *>(sVec + 2 * D + h * CPT + c);
                    const float4 w3v = *reinterpret_cast<const float4 *>(sVec + 3 * D + h * CPT + c);
                    v[c + 0] = fmaxf(v[c + 0] + b2v.x, 0.f);                          // r2
                    v[c + 1] = fmaxf(v[c + 1] + b2v.y, 0.f);
                    v[c + 2] = fmaxf(v[c + 2] + b2v.z, 0.f);
                    v[c + 3] = fmaxf(v[c + 3] + b2v.w, 0.f);
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const bool on = v[c + i] > 0.f;
                        m2 |= (on ? 1u : 0u) << (c + i);
                        mk[c - c0 + i] = on ? 1.f : 0.f;
                    }
                    zp = fmaf(v[c + 0], w3v.x, zp); zp = fmaf(v[c + 1], w3v.y, zp);
                    zp = fmaf(v[c + 2], w3v.z, zp); zp = fmaf(v[c + 3], w3v.w, zp);
                }
                umma::tmem_st8(tA + lane_off + (uint32_t)(h * CPT + c0), mk);
            }
            umma::tmem_st_wait();
            ops_ready();                                     // G2 (its A operand is complete: the mask)
            PROF_T(4);
            sZp[h * BM + row] = zp;
            stage_indices(b ^ 1);                            // the next tile's indices, published by the barrier below
            sync_compute();
            load_indices(tile + 2 * (int64_t)gridDim.x);
            PROF_T(5);
            // ---- epilogue 1b: logit, loss, dz
            const float zz = sZp[row] + sZp[BM + row] + sZp[2 * BM + row] + sZp[3 * BM + row] + b3;
            // y < 0: no label (held out): no loss term, dz = 0.  Selects, not branches: the loss branch stays uniform
            const bool labelled = yy >= 0.f;
            if (h == 0 && ok) {
                if (p.logits) p.logits[e] = zz;
                if (p.prob || p.pred) {
                    const float pr = 1.f / (1.f + expf(-zz));
                    if (p.prob) p.prob[e] = pr;
                    if (p.pred) p.pred[e] = pr >= p.threshold ? 1 : 0;
                }
                if (p.y && p.loss_partial) {
                    // torch BCEWithLogits(pos_weight): (1-y) z + (1+(pw-1)y) (log1p(exp(-|z|)) + max(-z,0))
                    const float lw = fmaf(p.pos_weight - 1.f, yy, 1.f);
                    const float term = (1.f - yy) * zz + lw * (log1pf(expf(-fabsf(zz))) + fmaxf(-zz, 0.f));
                    loss_acc += labelled ? term : 0.f;
                }
            }
            float dz = 0.f;
            if (ok) {
                if (p.dlogits) {
                    dz = p.dlogits[e] * p.scale;
                } else {
                    // torch's backward: ((pw*y + 1 - y) * sigmoid(z) - pw*y) * grad
                    const float sg = 1.f / (1.f + expf(-zz));
                    const float t = p.pos_weight * yy;
                    const float g = ((t + 1.f - yy) * sg - t) * p.scale;
                    dz = labelled ? g : 0.f;
                }
            }
            if (h == 0) gb3 += dz;
            const float4 sk4 = *reinterpret_cast<const float4 *>(sSkip + b * BM + (row & ~3));     // this quad's 4 edge slots
            uint32_t m1;                                     // bit c: r1[row][h*16 + c] > 0
            {
                const uint32_t nb = *reinterpret_cast<const uint32_t *>(sM1 + (b * BM + row) * 16 + h * 4);
                m1 = (nb & 0xfu) | ((nb >> 4) & 0xf0u) | ((nb >> 8) & 0xf00u) | ((nb >> 12) & 0xf000u);
            }
            // P = dz m2 row-major -> X (MN-major A operand of G3: panels hi j 0-31, 32-63, lo j 0-31, 32-63).  X's K-major
            // r1 is dead: G1 has completed.  The hi / lo split is the row scalar's.
            {
                const float dzh = umma::tf32_hi(dz), dzl = umma::tf32_lo(dz, dzh);
#pragma unroll
                for (int c = 0; c < CPT; c += 4) {
                    const int j = h * CPT + c;
                    float4 ph, pl;
                    ph.x = (m2 >> (c + 0)) & 1u ? dzh : 0.f; pl.x = (m2 >> (c + 0)) & 1u ? dzl : 0.f;
                    ph.y = (m2 >> (c + 1)) & 1u ? dzh : 0.f; pl.y = (m2 >> (c + 1)) & 1u ? dzl : 0.f;
                    ph.z = (m2 >> (c + 2)) & 1u ? dzh : 0.f; pl.z = (m2 >> (c + 2)) & 1u ? dzl : 0.f;
                    ph.w = (m2 >> (c + 3)) & 1u ? dzh : 0.f; pl.w = (m2 >> (c + 3)) & 1u ? dzl : 0.f;
                    const uint32_t off = umma::mn_off((uint32_t)row, (uint32_t)j, kPanel);
                    *reinterpret_cast<float4 *>(smem + oXh + off) = ph;
                    *reinterpret_cast<float4 *>(smem + oXh + 2 * kPanel + off) = pl;
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        gw3[c + i] = fmaf(dz, v[c + i], gw3[c + i]);
                        gq2[c + i] += (m2 >> (c + i)) & 1u ? dz : 0.f;
                    }
                }
            }
            ops_ready();                                     // G3
            PROF_T(6);
            umma::mbar_wait(&bar2, par);
            umma::fence_after_sync();
            PROF_T(7);
            // ---- epilogue 2: da1 = dz g [r1 > 0] -> HBM; db1, dw1c.  The 4 lanes of a quad exchange their float4
            // pieces so that every store instruction writes 64 contiguous bytes per edge row (8 rows per warp
            // instruction instead of 32 rows x 16 bytes).
            umma::tmem_ld<CPT>(tD2 + lane_off + (uint32_t)(h * CPT), v);
            {
                float4 T[4];
#pragma unroll
                for (int c = 0; c < 16; c += 4) {
                    T[c / 4].x = (m1 >> (c + 0)) & 1u ? dz * v[c + 0] : 0.f;
                    T[c / 4].y = (m1 >> (c + 1)) & 1u ? dz * v[c + 1] : 0.f;
                    T[c / 4].z = (m1 >> (c + 2)) & 1u ? dz * v[c + 2] : 0.f;
                    T[c / 4].w = (m1 >> (c + 3)) & 1u ? dz * v[c + 3] : 0.f;
                }
                quad_transpose(T, lane);        // T[j] = da1[edge slot (row & ~3) + j][h*16 + 4 (lane & 3) .. + 3]
                const int64_t eq = e0 + (row & ~3);
                float *dst = p.da1 + eq * D + h * 16 + 4 * (lane & 3);
                const float skj[4] = {sk4.x, sk4.y, sk4.z, sk4.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    gb1q.x += T[j].x; gb1q.y += T[j].y; gb1q.z += T[j].z; gb1q.w += T[j].w;
                    gw1cq.x = fmaf(T[j].x, skj[j], gw1cq.x); gw1cq.y = fmaf(T[j].y, skj[j], gw1cq.y);
                    gw1cq.z = fmaf(T[j].z, skj[j], gw1cq.z); gw1cq.w = fmaf(T[j].w, skj[j], gw1cq.w);
                    if (eq + j < p.E) *reinterpret_cast<float4 *>(dst + j * D) = T[j];
                }
            }
            ++g3_tiles;
            PROF_T(8);
        }
        if (it > 0) {
            umma::mbar_wait(&bar3, (it - 1) & 1);
            umma::fence_after_sync();
        }
#ifdef PANGNN_SCORER_PROF
        if (tid == 0)
            for (int i = 0; i < 12; ++i) atomicAdd(&g_scorer_prof[i], (unsigned long long)prof[i]);
#endif

        // ---- CTA epilogue
        if (p.loss_partial) {
            if (tid < BM) lred[tid] = (double)loss_acc;          // tid < 128 <=> h == 0, row == tid
            sync_compute();
            if (tid == 0) {
                double s = 0.0;
                for (int i = 0; i < BM; ++i) s += lred[i];
                p.loss_partial[blockIdx.x] = s;
            }
        }
        float *out = p.partial + (int64_t)blockIdx.x * kScNGP;
        float *red = reinterpret_cast<float *>(smem);        // [128][64] floats = 32 KB (reuses X)
        // dW2[j][k] = w3[j] (D3[j][k] + D3[64 + j][k])
        float v[CPT];
#pragma unroll
        for (int c = 0; c < CPT; ++c) v[c] = 0.f;
        if (g3_tiles > 0) umma::tmem_ld<CPT>(tD3 + lane_off + (uint32_t)(h * CPT), v);
#pragma unroll
        for (int c = 0; c < CPT; ++c) v[c] += g3acc[c];
        sync_compute();
#pragma unroll
        for (int c = 0; c < CPT; ++c) red[row * D + h * CPT + c] = v[c];
        sync_compute();
        for (int i = tid; i < D * D; i += NT) out[kG_W2 + i] = sVec[3 * D + i / D] * (red[i] + red[D * D + i]);
        // column sums over the 128 edge slots, fixed order
        auto reduce_cols = [&](const float (&acc)[CPT], int off, bool times_w3) {
            sync_compute();
#pragma unroll
            for (int c = 0; c < CPT; ++c) red[row * D + h * CPT + c] = acc[c];
            sync_compute();
            if (tid < D) {
                float s = 0.f;
                for (int r = 0; r < BM; ++r) s += red[r * D + tid];
                out[off + tid] = times_w3 ? sVec[3 * D + tid] * s : s;
            }
        };
        reduce_cols(gq2, kG_B2, true);
        reduce_cols(gw3, kG_W3, false);
        // db1 / dw1c: 32 partial rows (4 lane groups x 8 quads), 4 columns per thread
        auto reduce_cols_q = [&](const float4 acc, int off) {
            sync_compute();
            *reinterpret_cast<float4 *>(red + (q * 8 + (lane >> 2)) * D + h * 16 + 4 * (lane & 3)) = acc;
            sync_compute();
            if (tid < D) {
                float s = 0.f;
                for (int r = 0; r < 32; ++r) s += red[r * D + tid];
                out[off + tid] = s;
            }
        };
        reduce_cols_q(gb1q, kG_B1);
        reduce_cols_q(gw1cq, kG_W1C);
        sync_compute();
        if (h == 0) red[row] = gb3;
        sync_compute();
        if (tid == 0) {
            float s = 0.f;
            for (int r = 0; r < BM; ++r) s += red[r];
            out[kG_B3] = s;
        }
    }   // compute warps
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_dealloc(tmem_base_s, kTmemCols);
}

}  // namespace

int launch_edge_score_train(const ScorerArgs &a, int *grid_out, cudaStream_t st) {
    const size_t smem_train = oEnd + 1024 + 128;             // + alignment slack
    static bool attr_set = false;
    if (!attr_set) {
        int rc = check_cuda(cudaFuncSetAttribute(edge_score_train_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 (int)smem_train), "cudaFuncSetAttribute(edge_score train)");
        if (rc) return rc;
        attr_set = true;
    }
    const int64_t tiles = (a.E + BM - 1) / BM;
    const int grid = (int)(tiles < kNumSMs ? (tiles > 0 ? tiles : 1) : kNumSMs);
    *grid_out = grid;
    edge_score_train_kernel<<<grid, NT + 128, smem_train, st>>>(a);
    PANGNN_CHECK_LAUNCH("edge_score_train");
    return PANGNN_OK;
}

}  // namespace pangnn

#ifdef PANGNN_SCORER_PROF
// development build only: read (and optionally reset) the per-phase cycle totals
extern "C" int pangnn_debug_scorer_prof(unsigned long long *out, int reset) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out, pangnn::g_scorer_prof, sizeof(unsigned long long) * 16);
    if (reset) {
        unsigned long long z[16] = {0};
        cudaMemcpyToSymbol(pangnn::g_scorer_prof, z, sizeof(z));
    }
    return 0;
}
#endif
