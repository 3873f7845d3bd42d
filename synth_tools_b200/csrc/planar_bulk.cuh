// planar_bulk.cuh -- generic staged render of PLANAR 32-bit streams ([inst][F], what the
// reference hosts hand over), shared by square_grain, pdm raw, pwm, the one-pole and the word
// clock.  Lane r of a warp owns instance r of the warp's 32.  The stream is a 2-D tensor
// [inst][F] (box = 32 words x 32 instances, SWIZZLE_128B): per tile of 64 frames one elected
// lane moves the warp's two boxes into a shared-memory stage with two tensor-TMA copies, every
// lane walks its row with LDS.128 / STS.128 in place -- lane r finds 16-byte chunk c of its row
// at r*128 + ((c ^ (r & 7)) << 4) -- and the elected lane sends the tile back with two tensor-TMA
// stores.  Loads run one tile ahead, stores drain one tile behind.
//
// Op (by value, trivially copyable):
//   static constexpr int NIN      0: no per-instance input stream (output only), 1: one
//   void     load(uint64_t i)     state / params of instance i from the SoA rows
//   void     store(uint64_t i)
//   uint32_t tick(uint32_t x, uint64_t t)   one frame; x = the input word (NIN == 1)
// Requirements (checked by launch, which declines otherwise): F % 4 == 0, in/out 16-byte
// aligned; in may alias out exactly.
#pragma once
#include "common.cuh"
#include <cuda.h>

namespace pbulk {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile("{\n\t.reg .pred p;\n\t"
                 "W: mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
                 "@p bra D;\n\tbra W;\n\tD:\n\t}" ::"r"(bar), "r"(parity) : "memory");
}

constexpr int WARPS = 2;

typedef CUresult (*encode_tiled_t)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                   const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline encode_tiled_t encode_fn() {
    static encode_tiled_t fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void *q = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &q, cudaEnableDefault, &qr) == cudaSuccess && qr == cudaDriverEntryPointSuccess) fn = (encode_tiled_t)q;
        else cudaGetLastError();
    }
    return fn;
}
// [rows][words] stream of 32-bit words, row pitch = words * 4 bytes (a multiple of 16)
inline bool encode_rows_u32(CUtensorMap *tm, const void *base, uint64_t words, uint64_t rows) {
    encode_tiled_t enc = encode_fn();
    if (!enc || words >= (1ull << 31) || rows >= (1ull << 31) || (words & 3) || ((uintptr_t)base & 15)) return false;
    const cuuint64_t dims[2] = {words, rows}, strides[1] = {words * 4};
    const cuuint32_t box[2] = {32, 32}, estr[2] = {1, 1};
    return enc(tm, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, (void *)base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
               CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// [rows][bytes] stream of bytes (PDM v2 duty rows): box = 128 bytes x 32 rows
inline bool encode_rows_u8(CUtensorMap *tm, const void *base, uint64_t bytes, uint64_t rows) {
    encode_tiled_t enc = encode_fn();
    if (!enc || bytes >= (1ull << 31) || rows >= (1ull << 31) || (bytes & 15) || ((uintptr_t)base & 15)) return false;
    const cuuint64_t dims[2] = {bytes, rows}, strides[1] = {bytes};
    const cuuint32_t box[2] = {128, 32}, estr[2] = {1, 1};
    return enc(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, (void *)base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
               CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// [rows][mid][words]: box = 32 words x 1 x 32 rows (the generated graph kernels: [inst][stream][F])
inline bool encode_rows3_u32(CUtensorMap *tm, const void *base, uint64_t words, uint64_t mid, uint64_t rows) {
    encode_tiled_t enc = encode_fn();
    if (!enc || words >= (1ull << 31) || rows >= (1ull << 31) || mid == 0 || mid >= (1ull << 31) || (words & 3) || ((uintptr_t)base & 15)) return false;
    const cuuint64_t dims[3] = {words, mid, rows}, strides[2] = {words * 4, mid * words * 4};
    const cuuint32_t box[3] = {32, 1, 32}, estr[3] = {1, 1, 1};
    return enc(tm, CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, (void *)base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
               CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

constexpr int T_STAGES = 3;
constexpr uint32_t T_BOXB = 4096, T_STAGEB = 2 * T_BOXB;           // 64 words per tile
constexpr size_t t_smem_bytes() { return (size_t)WARPS * T_STAGES * T_STAGEB + WARPS * T_STAGES * 8 + 1024; }

template <class Op>
__global__ void __launch_bounds__(WARPS * 32) k_planar_tma(Op op, const __grid_constant__ CUtensorMap tm_in, const __grid_constant__ CUtensorMap tm_out, uint64_t n, uint64_t F) {
    extern __shared__ __align__(1024) uint8_t pt_smem[];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t g0 = ((uint64_t)blockIdx.x * WARPS + warp) * 32;
    if (g0 >= n) return;
    const uint32_t rows = n - g0 < 32 ? (uint32_t)(n - g0) : 32u;
    const bool mine = lane < rows;
    const uint32_t sm0 = (smem_u32(pt_smem) + 1023u) & ~1023u;
    const uint32_t base = sm0 + warp * (T_STAGES * T_STAGEB);
    const uint32_t bar0 = sm0 + WARPS * T_STAGES * T_STAGEB + warp * (T_STAGES * 8);
    if (Op::NIN && lane == 0) {
#pragma unroll
        for (int s = 0; s < T_STAGES; ++s) asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar0 + 8 * s), "r"(1));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    if (mine) op.load(g0 + lane);
    const uint32_t n_tiles = (uint32_t)((F + 63) / 64);
    const uint64_t tmi = reinterpret_cast<uint64_t>(&tm_in), tmo = reinterpret_cast<uint64_t>(&tm_out);
    auto cols_of = [&](uint32_t k) { const uint64_t left = F - (uint64_t)k * 64; return left < 64 ? (uint32_t)left : 64u; };
    auto issue = [&](uint32_t k) {                                   // lane 0 only
        const uint32_t s = k % T_STAGES, nbox = cols_of(k) > 32 ? 2u : 1u;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar0 + 8 * s), "r"(nbox * T_BOXB) : "memory");
        for (uint32_t h = 0; h < nbox; ++h)
            asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                         ::"r"(base + s * T_STAGEB + h * T_BOXB), "l"(tmi), "r"((int32_t)(k * 64 + h * 32)), "r"((int32_t)g0), "r"(bar0 + 8 * s) : "memory");
    };
    if (Op::NIN && lane == 0) for (uint32_t k = 0; k < T_STAGES - 2 && k < n_tiles; ++k) issue(k);
#pragma unroll 1
    for (uint32_t k = 0; k < n_tiles; ++k) {
        const uint32_t s = k % T_STAGES, cols = cols_of(k);
        if (Op::NIN) {
            if (k + T_STAGES - 2 < n_tiles && lane == 0) {           // that stage last held tile k-2: its stores must have read it out
                asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
                issue(k + T_STAGES - 2);
            }
            mbar_wait(bar0 + 8 * s, (k / T_STAGES) & 1);
        } else {
            if (lane == 0) asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(T_STAGES - 1) : "memory");   // the stores of tile k-STAGES have left this stage
            __syncwarp();
        }
        if (mine) {
            const uint64_t t0 = (uint64_t)k * 64;
#pragma unroll 4
            for (uint32_t c = 0; c < cols / 4; ++c) {
                const uint32_t a = base + s * T_STAGEB + (c >> 3) * T_BOXB + lane * 128 + (((c & 7) ^ (lane & 7)) << 4);
                uint32_t x0 = 0, x1 = 0, x2 = 0, x3 = 0;
                if (Op::NIN) asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(x0), "=r"(x1), "=r"(x2), "=r"(x3) : "r"(a));
                const uint64_t t = t0 + 4 * c;
                x0 = op.tick(x0, t); x1 = op.tick(x1, t + 1); x2 = op.tick(x2, t + 2); x3 = op.tick(x3, t + 3);
                asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(x0), "r"(x1), "r"(x2), "r"(x3) : "memory");
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) {
            const uint32_t nbox = cols > 32 ? 2u : 1u;
            for (uint32_t h = 0; h < nbox; ++h)
                asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%1, %2}], [%3];"
                             ::"l"(tmo), "r"((int32_t)(k * 64 + h * 32)), "r"((int32_t)g0), "r"(base + s * T_STAGEB + h * T_BOXB) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncwarp();
    if (mine) op.store(g0 + lane);
}

// Renders the streams with k_planar_tma and returns true, or returns false when they cannot be staged (F % 4 != 0, a
// stream off 16-byte alignment, or no tensor map encodes them): the caller then runs its scalar kernel.  A CUDA error is
// left for the caller's launch check (CK_LAUNCH).
template <class Op>
bool launch(cproc_cuda_ctx *ctx, const Op &op, const uint32_t *in, uint32_t *out, uint64_t n, uint64_t F) {
    CUtensorMap tin, tout;
    if (!encode_rows_u32(&tout, out, F, n) || !encode_rows_u32(&tin, Op::NIN ? (const void *)in : (const void *)out, F, n)) return false;
    static bool attr_set[64] = {};
    if (!attr_set[ctx->device & 63]) {
        if (cudaFuncSetAttribute(k_planar_tma<Op>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)t_smem_bytes()) != cudaSuccess) return true;
        attr_set[ctx->device & 63] = true;
    }
    k_planar_tma<Op><<<(unsigned)ceil_div_u64(n, WARPS * 32), WARPS * 32, t_smem_bytes(), ctx->stream>>>(op, tin, tout, n, F);
    return true;
}

// ---- INTERLEAVED streams [F][inst]: four adjacent instances per thread ---------------------------------------------------
// Rows are coalesced as they are; what a thread-per-instance kernel lacks is bytes in flight (one 4-byte load per thread and tick).
// Here a thread owns instances i..i+3 (128-bit accesses: a block covers 2 KiB of every row) and loads a batch of four frames
// before it ticks them.  n % 4 == 0, 16-byte aligned streams; `in` may alias `out`.
template <class Op>
__global__ void __launch_bounds__(128) k_interleaved4(Op op0, const uint32_t *in, uint32_t *out, uint64_t n, uint64_t F) {
    const uint64_t i = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i >= n) return;
    Op a = op0, b = op0, c = op0, d = op0;
    a.load(i); b.load(i + 1); c.load(i + 2); d.load(i + 3);
    const uint4 *src = reinterpret_cast<const uint4 *>(in + i);
    uint4 *dst = reinterpret_cast<uint4 *>(out + i);
    const uint64_t row = n >> 2;                                     // row pitch in uint4
    uint64_t t = 0;
    for (; t + 4 <= F; t += 4) {
        uint4 x[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) x[k] = Op::NIN ? __ldcs(src + (t + k) * row) : make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
        for (int k = 0; k < 4; ++k)
            __stcs(dst + (t + k) * row, make_uint4(a.tick(x[k].x, t + k), b.tick(x[k].y, t + k), c.tick(x[k].z, t + k), d.tick(x[k].w, t + k)));
    }
    for (; t < F; ++t) {
        const uint4 x = Op::NIN ? __ldcs(src + t * row) : make_uint4(0u, 0u, 0u, 0u);
        __stcs(dst + t * row, make_uint4(a.tick(x.x, t), b.tick(x.y, t), c.tick(x.z, t), d.tick(x.w, t)));
    }
    a.store(i); b.store(i + 1); c.store(i + 2); d.store(i + 3);
}

inline bool usable_interleaved4(uint64_t n, const void *in, const void *out) {
    return n % 4 == 0 && ((uintptr_t)in & 15) == 0 && ((uintptr_t)out & 15) == 0;
}

template <class Op>
void launch_interleaved4(cproc_cuda_ctx *ctx, const Op &op, const uint32_t *in, uint32_t *out, uint64_t n, uint64_t F) {
    k_interleaved4<Op><<<(unsigned)ceil_div_u64(n / 4, 128), 128, 0, ctx->stream>>>(op, in, out, n, F);
}

}  // namespace pbulk
