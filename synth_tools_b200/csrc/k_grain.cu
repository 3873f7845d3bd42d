// k_grain.cu -- square_grain~ (linux/synth_tools.c:85-100): a Schmitt-trigger
// squarer with a one-sample output delay.
//
//   out[i] = state;
//   if (state >= 0 && in[i] < -thresh) state = -0.5f;
//   else if (state < 0 && in[i] > thresh) state = +0.5f;
//
// Outputs are exactly {0, +0.5, -0.5}, so the result is bit-exact.  The
// hysteresis makes the recurrence a 3-state machine that is serial in time;
// the grain axis carries the parallelism (one thread per grain).
//
// GrainOp: PLANAR [grain][F] streams go through the staging templates of
//   planar_bulk.cuh (k_planar_tma), INTERLEAVED [F][grain] streams
//   through k_interleaved4 (four grains per thread), as the other stream processors.
// k_grain_planar: the PLANAR fallback (planar_bulk = 0, F % 4 != 0 or rows off
//   16-byte alignment).  A warp owns 32 grains and walks the frame axis in 32-frame
//   tiles: the tile is loaded with 32 coalesced 128-byte row reads into padded
//   shared memory, each lane then runs its own grain along its row IN PLACE (in may
//   alias out, as in Pd), and the tile is written back with 32 coalesced row stores.
// k_grain_interleaved: the INTERLEAVED fallback, one grain per thread.
// k_grain_mix: config C3b -- input from a per-grain phasor, integer stereo mix.
//   k_grain_mix2 / k_grain_mix3 are its faster generations; all three take <BUS>: with
//   a mix bus attached (cproc_cuda_bus_attach) the launch exchanges its mix itself.
#include "common.cuh"
#include "planar_bulk.cuh"
#include "bus_fused.cuh"

struct GrainParams {
    float *state;            // SoA [1][npad]
    const float *thresh;     // SoA [1][npad]
    uint64_t n, F;
    const float *in;
    float *out;
};

__device__ __forceinline__ float grain_step(float &state, float val, float thresh) {
    const float o = state;                                   // :91
    if (state >= 0.0f && val < -thresh) state = -0.5f;       // :92-94
    else if (state < 0.0f && val > thresh) state = 0.5f;     // :95-97
    return o;
}

// one grain as an Op of the PLANAR / INTERLEAVED stream templates (planar_bulk.cuh)
struct GrainOp {
    static constexpr int NIN = 1;
    float *state; const float *thresh;
    float st, th;
    __device__ __forceinline__ void load(uint64_t i) { st = state[i]; th = thresh[i]; }
    __device__ __forceinline__ void store(uint64_t i) { state[i] = st; }
    __device__ __forceinline__ uint32_t tick(uint32_t x, uint64_t) { return __float_as_uint(grain_step(st, __uint_as_float(x), th)); }
};

#define GRAIN_WARPS 4
__global__ void __launch_bounds__(GRAIN_WARPS * 32) k_grain_planar(const GrainParams p) {
    __shared__ float tile[GRAIN_WARPS][32][33];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t g0 = ((uint64_t)blockIdx.x * GRAIN_WARPS + warp) * 32;
    if (g0 >= p.n) return;
    const uint32_t rows = p.n - g0 < 32 ? (uint32_t)(p.n - g0) : 32u;
    float (*tl)[33] = tile[warp];
    const bool mine = lane < rows;
    float state = mine ? p.state[g0 + lane] : 0.0f;
    const float th = mine ? p.thresh[g0 + lane] : 0.0f;
    for (uint64_t t0 = 0; t0 < p.F; t0 += 32) {
        const uint32_t cols = p.F - t0 < 32 ? (uint32_t)(p.F - t0) : 32u;
        if (lane < cols)
            for (uint32_t r = 0; r < rows; ++r) tl[r][lane] = __ldcs(p.in + (g0 + r) * p.F + t0 + lane);
        __syncwarp();
        if (mine)
            for (uint32_t i = 0; i < cols; ++i) tl[lane][i] = grain_step(state, tl[lane][i], th);
        __syncwarp();
        if (lane < cols)
            for (uint32_t r = 0; r < rows; ++r) __stcs(p.out + (g0 + r) * p.F + t0 + lane, tl[r][lane]);
        __syncwarp();
    }
    if (mine) p.state[g0 + lane] = state;
}

// [F][grain] streams: a warp's 32 grains are 128 contiguous bytes of every frame row.
// in and out may be the same buffer, so the compiler cannot move loads across stores:
// the 16-frame batches make the independent loads explicit (all in flight, then the
// serial trigger steps, then the stores).
#define GI_BLOCK 128
#define GI_BATCH 16
__global__ void __launch_bounds__(GI_BLOCK) k_grain_interleaved(const GrainParams p) {
    const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= p.n) return;
    float state = p.state[g];
    const float th = p.thresh[g];
    const float *src = p.in + g;
    float *dst = p.out + g;
    uint64_t t = 0;
    for (; t + GI_BATCH <= p.F; t += GI_BATCH) {
        float v[GI_BATCH];
#pragma unroll
        for (int i = 0; i < GI_BATCH; ++i) v[i] = __ldcs(src + (t + i) * p.n);
#pragma unroll
        for (int i = 0; i < GI_BATCH; ++i) v[i] = grain_step(state, v[i], th);
#pragma unroll
        for (int i = 0; i < GI_BATCH; ++i) __stcs(dst + (t + i) * p.n, v[i]);
    }
    for (; t < p.F; ++t) {
        const float v = __ldcs(src + t * p.n);
        __stcs(dst + t * p.n, grain_step(state, v, th));
    }
    p.state[g] = state;
}

int launch_square_grain(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io) {
    cproc_cuda_ctx *ctx = b->ctx;
    if (!io->in || !io->out) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "square_grain: in/out is NULL");
    if (io->layout == CPROC_CUDA_TILED) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "square_grain: TILED layout not supported");
    if (F == 0) return 0;
    GrainOp op; op.state = (float *)b->d_state; op.thresh = (const float *)b->d_param; op.st = 0.f; op.th = 0.f;
    if (ctx->planar_bulk && io->layout == CPROC_CUDA_PLANAR && pbulk::launch(ctx, op, (const uint32_t *)io->in, (uint32_t *)io->out, b->n, F)) {
        CK_LAUNCH(ctx, "k_grain (bulk)");
        return 0;
    }
    if (ctx->planar_bulk && io->layout == CPROC_CUDA_INTERLEAVED && pbulk::usable_interleaved4(b->n, io->in, io->out)) {
        pbulk::launch_interleaved4(ctx, op, (const uint32_t *)io->in, (uint32_t *)io->out, b->n, F);
        CK_LAUNCH(ctx, "k_grain (interleaved4)");
        return 0;
    }
    GrainParams p;
    p.state = (float *)b->d_state; p.thresh = (const float *)b->d_param; p.n = b->n; p.F = F;
    p.in = (const float *)io->in; p.out = (float *)io->out;
    if (io->layout == CPROC_CUDA_INTERLEAVED)
        k_grain_interleaved<<<(unsigned)ceil_div_u64(p.n, GI_BLOCK), GI_BLOCK, 0, ctx->stream>>>(p);
    else
        k_grain_planar<<<(unsigned)ceil_div_u64(p.n, GRAIN_WARPS * 32), GRAIN_WARPS * 32, 0, ctx->stream>>>(p);
    CK_LAUNCH(ctx, "k_grain");
    return 0;
}

// ---------------------------------------------------------------------------
// C3b: per-grain phasor input, dyadic pan, integer stereo mix (units of 2^-7).
struct GrainMixParams {
    uint32_t *st;            // SoA [2][npad]: state (float bits), phase
    const uint32_t *prm;     // SoA [4][npad]: threshold (float bits), inc, gl, gr
    uint64_t npad, n, F;
    int32_t *imix;           // [2][F], zeroed by the launcher; with a bus: [2][F] + ticket, zero between launches
};

// With a mix bus attached (BUS) and pipelined (mode 2), block 0 runs the previous frame block's exchange and the
// render blocks are 1..gridDim.x-1.  Block 0, not the last block: k_grain_mix is one thread per grain, many waves,
// and a last block would start only after the last wave.  Returns false for the exchange block.
template <bool BUS>
__device__ __forceinline__ bool grain_render_block(const BusFused &bf, uint32_t &blk, uint32_t &nblk) {
    blk = blockIdx.x; nblk = gridDim.x;
    if (BUS && bf.mode == 2) {
        if (blk == 0) { bus_exchange_block(bf); return false; }
        --blk; --nblk;
    }
    return true;
}

// With a bus attached the render blocks accumulate into the batch's [2][F] accumulator (zero between launches), then
// take a ticket; the last render block of the launch reads every word back with atomicExch(.., 0), which leaves the
// accumulator zero for the next launch, emits it to the bus and completes the exchange (mode 1) or stages it (mode 2).
// The kernels call it under `if constexpr (BUS)`: a plain `if` changes the register allocation of the BUS = false
// instantiation, which is meant to stay the kernel without a bus, instruction for instruction.
__device__ __forceinline__ void grain_bus_tail(int32_t *acc, uint64_t F, const BusFused &bf, uint32_t nblk) {
    __shared__ uint32_t last_s;
    uint32_t *ticket = (uint32_t *)(acc + 2 * F);
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last_s = atomicAdd(ticket, 1u) == nblk - 1u;
    __syncthreads();
    if (!last_s) return;                      // (uniform over the block)
    __threadfence();
    for (uint64_t i = threadIdx.x; i < 2 * F; i += blockDim.x) bus_emit_word(bf, i, (uint32_t)atomicExch(acc + i, 0));
    if (threadIdx.x == 0) *ticket = 0;
    bus_participant_done(bf);
}

#define GMIX_BLOCK 256
#define GMIX_CHUNK 32
template <bool BUS>
__global__ void __launch_bounds__(GMIX_BLOCK) k_grain_mix(const GrainMixParams p, const BusFused bf) {
    // Each lane keeps one grain in registers.  Left and right gains (0..64) are
    // packed into one word so one REDUX.SUM per frame reduces both channels
    // over the warp; warp sums are accumulated per block in shared memory and
    // flushed to the global integer mix once per chunk of frames.
    __shared__ int32_t acc[2][GMIX_CHUNK];
    uint32_t blk, nblk;
    if (!grain_render_block<BUS>(bf, blk, nblk)) return;
    const uint64_t g = (uint64_t)blk * blockDim.x + threadIdx.x;
    const bool mine = g < p.n;
    const uint32_t lane = threadIdx.x & 31;
    float state = 0.0f, th = 0.0f;
    uint32_t ph = 0, inc = 0;
    int32_t pk = 0;
    if (mine) {
        state = __uint_as_float(p.st[g]); ph = p.st[p.npad + g];
        th = __uint_as_float(p.prm[g]); inc = p.prm[p.npad + g];
        pk = (int32_t)((p.prm[3 * p.npad + g] << 16) + p.prm[2 * p.npad + g]);
    }
    for (uint64_t t0 = 0; t0 < p.F; t0 += GMIX_CHUNK) {
        if (threadIdx.x < 2 * GMIX_CHUNK) (&acc[0][0])[threadIdx.x] = 0;
        __syncthreads();
        const uint32_t cols = p.F - t0 < GMIX_CHUNK ? (uint32_t)(p.F - t0) : GMIX_CHUNK;
        int32_t keep = 0;
        for (uint32_t i = 0; i < cols; ++i) {
            const float val = __int2float_rn((int32_t)ph) * 0x1p-31f;   // acc -> signed saw
            ph += inc;                                                  // cproc.h:141
            const float o = grain_step(state, val, th);
            const int32_t c = o > 0.0f ? pk : (o < 0.0f ? -pk : 0);
            const int32_t s = __reduce_add_sync(0xFFFFFFFFu, c);
            if (lane == (i & 31)) keep = s;
        }
        if (lane < cols) {
            const int32_t l = (int32_t)(int16_t)(keep & 0xFFFF);        // |sum L| <= 32*64
            const int32_t r = (keep - l) >> 16;
            atomicAdd(&acc[0][lane], l);
            atomicAdd(&acc[1][lane], r);
        }
        __syncthreads();
        if (threadIdx.x < cols) {
            atomicAdd(p.imix + t0 + threadIdx.x, acc[0][threadIdx.x]);
            atomicAdd(p.imix + p.F + t0 + threadIdx.x, acc[1][threadIdx.x]);
        }
        __syncthreads();
    }
    if (mine) { p.st[g] = __float_as_uint(state); p.st[p.npad + g] = ph; }
    if constexpr (BUS) grain_bus_tail(p.imix, p.F, bf, nblk);
}

// ---------------------------------------------------------------------------
// C3b, second generation.  Two changes against k_grain_mix:
//  * the comparisons run on the integer phase.  val = (float)(int)ph * 2^-31 is a
//    monotone function of the signed phase, so `val < -thresh` is `x < lo` and
//    `val > thresh` is `x > hi` for two per-grain integers found once per parameter
//    upload by bisection with the very same I2F / FMUL / FSETP (k_grain_thresholds):
//    no conversion, no multiply in the loop, and still bit-exact.
//  * the mix leaves the inner loop: a thread keeps 32 packed (right << 16) + left
//    accumulators for a 64-frame chunk in registers and walks ITS grains through the
//    chunk one after the other; the state machine output m in {-1, 0, +1} enters the
//    bus as one IMAD (acc += m * pk).  One warp reduction per frame per chunk instead
//    of one per grain-sample.
// This generation and the third write back only the reference's states (+-0, +-0.5): a
// batch with any other state uploaded (grain_odd_state, abi.cu) runs k_grain_mix.
__global__ void k_grain_thresholds(const uint32_t *prm, uint64_t n, uint64_t npad, int32_t *lo, int32_t *hi, int32_t *pk, uint32_t *weird) {
    const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n) return;
    const float th = __uint_as_float(prm[g]);
    pk[g] = (int32_t)((prm[3 * npad + g] << 16) + prm[2 * npad + g]);
    // a negative threshold lets both flip conditions hold at once; only the literal
    // two-branch form (k_grain_mix / k_grain_mix2) orders them like the reference
    if (th < 0.0f) atomicOr(weird, 2u);
    auto val = [](int64_t x) { return __int2float_rn((int32_t)x) * 0x1p-31f; };
    // lo: smallest x with !(val(x) < -th); the predicate is true below, false from lo on
    int64_t a = INT32_MIN, b = INT32_MAX;
    if (!(val(a) < -th)) lo[g] = INT32_MIN;
    else if (val(b) < -th) { lo[g] = INT32_MAX; atomicOr(weird, 1u); }       // true for every phase: not representable
    else {
        while (b - a > 1) { const int64_t m = a + (b - a) / 2; if (val(m) < -th) a = m; else b = m; }
        lo[g] = (int32_t)b;
    }
    // hi: largest x with !(val(x) > th); the predicate is false up to hi, true above
    a = INT32_MIN; b = INT32_MAX;
    if (!(val(b) > th)) hi[g] = INT32_MAX;
    else if (val(a) > th) { hi[g] = INT32_MIN; atomicOr(weird, 1u); }
    else {
        while (b - a > 1) { const int64_t m = a + (b - a) / 2; if (val(m) > th) b = m; else a = m; }
        hi[g] = (int32_t)a;
    }
}

#define GM2_BLOCK 128
#define GM2_CHUNK 64
struct GrainMix2Params {
    GrainMixParams g;
    const int32_t *lo, *hi;
};

__device__ __forceinline__ void gm2_tick(int32_t &m, uint32_t &ph, uint32_t inc, int32_t pk, int32_t lo, int32_t hi, int32_t &acc) {
    const int32_t x = (int32_t)ph;
    ph += inc;                                              // cproc.h:141
    acc = m * pk + acc;                                     // out = state (synth_tools.c:91), panned into the bus
    // if (state >= 0 && in < -thresh) state = -0.5; else if (state < 0 && in > thresh) state = +0.5;   (:92-97)
    // three compares with the sign predicate folded in, two selects (ptxas makes 8+ of the C form)
    asm("{ .reg .pred pn, pd, pu;\n\t"
        "setp.lt.s32 pn, %0, 0;\n\t"
        "setp.lt.and.s32 pd, %1, %2, !pn;\n\t"
        "setp.gt.and.s32 pu, %1, %3, pn;\n\t"
        "selp.s32 %0, -1, %0, pd;\n\t"
        "selp.s32 %0, 1, %0, pu; }" : "+r"(m) : "r"(x), "r"(lo), "r"(hi));
}

struct GM2Grain { float st; uint32_t ph, inc; int32_t pk, lo, hi; };
__device__ __forceinline__ void gm2_load(GM2Grain &v, const GrainMix2Params &p, uint64_t g) {
    const uint64_t npad = p.g.npad;
    v.st = __uint_as_float(__ldcg(p.g.st + g));
    v.ph = __ldcg(p.g.st + npad + g);
    v.inc = __ldg(p.g.prm + npad + g);
    v.pk = (int32_t)((__ldg(p.g.prm + 3 * npad + g) << 16) + __ldg(p.g.prm + 2 * npad + g));
    v.lo = __ldg(p.lo + g); v.hi = __ldg(p.hi + g);
}

template <bool BUS>
__global__ void __launch_bounds__(GM2_BLOCK) k_grain_mix2(const GrainMix2Params p, const BusFused bf) {
    __shared__ int32_t sacc[2][GM2_CHUNK];
    uint32_t blk, nblk;
    if (!grain_render_block<BUS>(bf, blk, nblk)) return;
    const uint64_t T = (uint64_t)nblk * GM2_BLOCK;
    const uint64_t tid = (uint64_t)blk * GM2_BLOCK + threadIdx.x;
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t n = p.g.n, npad = p.g.npad;
    for (uint64_t t0 = 0; t0 < p.g.F; t0 += GM2_CHUNK) {
        const uint32_t cols = p.g.F - t0 < GM2_CHUNK ? (uint32_t)(p.g.F - t0) : GM2_CHUNK;
        if (threadIdx.x < 2 * GM2_CHUNK) (&sacc[0][0])[threadIdx.x] = 0;
        __syncthreads();
        int32_t acc[GM2_CHUNK];
#pragma unroll
        for (int k = 0; k < GM2_CHUNK; ++k) acc[k] = 0;
        // software pipeline: the next grain's seven words are in flight while this one runs its 32 frames
        GM2Grain nx = {};
        if (tid < n) gm2_load(nx, p, tid);
        for (uint64_t g = tid; g < n; g += T) {
            const GM2Grain cur = nx;
            if (g + T < n) gm2_load(nx, p, g + T);
            int32_t m = cur.st > 0.0f ? 1 : (cur.st < 0.0f ? -1 : 0);
            uint32_t ph = cur.ph;
            const uint32_t inc = cur.inc;
            const int32_t pk = cur.pk, lo = cur.lo, hi = cur.hi;
            if (cols == GM2_CHUNK) {
#pragma unroll
                for (int k = 0; k < GM2_CHUNK; ++k) gm2_tick(m, ph, inc, pk, lo, hi, acc[k]);
            } else {
#pragma unroll
                for (int k = 0; k < GM2_CHUNK; ++k) if (k < (int)cols) gm2_tick(m, ph, inc, pk, lo, hi, acc[k]);
            }
            if (m != 0) p.g.st[g] = __float_as_uint(0.5f * (float)m);    // never flipped from 0.0: unchanged
            p.g.st[npad + g] = ph;
        }
#pragma unroll
        for (int h = 0; h < GM2_CHUNK / 32; ++h) {
            int32_t keepl = 0, keepr = 0;
#pragma unroll
            for (int k = 0; k < 32; ++k) {
                const int32_t a = acc[h * 32 + k];
                const int32_t l = (int32_t)(int16_t)(a & 0xFFFF);        // |sum L| <= grains_per_thread * 64 < 2^15
                const int32_t r = (a - l) >> 16;
                const int32_t sl = __reduce_add_sync(0xFFFFFFFFu, l), sr = __reduce_add_sync(0xFFFFFFFFu, r);
                if (lane == k) { keepl = sl; keepr = sr; }
            }
            if (h * 32 + lane < cols) { atomicAdd(&sacc[0][h * 32 + lane], keepl); atomicAdd(&sacc[1][h * 32 + lane], keepr); }
        }
        __syncthreads();
        if (threadIdx.x < cols) {
            atomicAdd(p.g.imix + t0 + threadIdx.x, sacc[0][threadIdx.x]);
            atomicAdd(p.g.imix + p.g.F + t0 + threadIdx.x, sacc[1][threadIdx.x]);
        }
        __syncthreads();
    }
    if constexpr (BUS) grain_bus_tail(p.g.imix, p.g.F, bf, nblk);
}

// ---------------------------------------------------------------------------
// C3b, third generation: the trigger state lives in a predicate.  For thresh >= 0
// (lo <= hi) the two-branch update of synth_tools.c:92-97 is the Schmitt trigger
//     neg' = (x < lo) | (neg & (x <= hi))
// which is two ISETP with a predicate operand (ISETP.LE.AND, ISETP.LT.OR); the bus
// term is `neg ? -pk : pk` (one SEL) added by an IMAD.IADD, the phasor a second
// IMAD.IADD: 5 instructions per grain-sample, 3 on the ALU pipe, 2 on the FMA pipe
// (k_grain_mix2: 7 and 5).  A grain whose state is still the initial 0.0 outputs 0
// until its first flip (synth_tools.c:91: out = state), so it walks its chunk with
// the literal form; once flipped it never returns to 0.
#define GM3_BLOCK 128
#define GM3_CHUNK 64
struct GrainMix3Params {
    GrainMixParams g;
    const int32_t *lo, *hi, *pk;
};
struct GM3Grain { float st; uint32_t ph, inc; int32_t pk, lo, hi; };
__device__ __forceinline__ void gm3_load(GM3Grain &v, const GrainMix3Params &p, uint64_t g) {
    v.st = __uint_as_float(__ldcg(p.g.st + g));
    v.ph = __ldcg(p.g.st + p.g.npad + g);
    v.inc = __ldg(p.g.prm + p.g.npad + g);
    v.pk = __ldg(p.pk + g); v.lo = __ldg(p.lo + g); v.hi = __ldg(p.hi + g);
}

__device__ __forceinline__ void gm3_chunk(const GM3Grain &cur, uint32_t cols, int32_t (&acc)[GM3_CHUNK], float &st_out, uint32_t &ph_out) {
    uint32_t ph = cur.ph;
    const uint32_t inc = cur.inc;
    const int32_t pk = cur.pk, npk = -cur.pk, lo = cur.lo, hi = cur.hi;
    if (cols == GM3_CHUNK && cur.st != 0.0f) {
        bool neg = cur.st < 0.0f;
#pragma unroll
        for (int k = 0; k < GM3_CHUNK; ++k) {
            const int32_t x = (int32_t)ph;
            ph += inc;                                       // cproc.h:141
            acc[k] += neg ? npk : pk;                        // out = state (:91), panned into the bus
            neg = (x < lo) | (neg & (x <= hi));              // :92-97
        }
        st_out = neg ? -0.5f : 0.5f;
    } else {
        // initial 0.0 state or a ragged last chunk: the literal form, tick by tick
        int32_t m = cur.st > 0.0f ? 1 : (cur.st < 0.0f ? -1 : 0);
#pragma unroll
        for (int k = 0; k < GM3_CHUNK; ++k)
            if (k < (int)cols) gm2_tick(m, ph, inc, pk, lo, hi, acc[k]);
        st_out = m != 0 ? 0.5f * (float)m : cur.st;
    }
    ph_out = ph;
}

template <bool BUS>
__global__ void __launch_bounds__(GM3_BLOCK) k_grain_mix3(const GrainMix3Params p, const BusFused bf) {
    __shared__ int32_t sacc[2][GM3_CHUNK];
    uint32_t blk, nblk;
    if (!grain_render_block<BUS>(bf, blk, nblk)) return;
    const uint64_t T = (uint64_t)nblk * GM3_BLOCK;
    const uint64_t tid = (uint64_t)blk * GM3_BLOCK + threadIdx.x;
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t n = p.g.n, npad = p.g.npad;
    for (uint64_t t0 = 0; t0 < p.g.F; t0 += GM3_CHUNK) {
        const uint32_t cols = p.g.F - t0 < GM3_CHUNK ? (uint32_t)(p.g.F - t0) : GM3_CHUNK;
        if (threadIdx.x < 2 * GM3_CHUNK) (&sacc[0][0])[threadIdx.x] = 0;
        __syncthreads();
        int32_t acc[GM3_CHUNK];
#pragma unroll
        for (int k = 0; k < GM3_CHUNK; ++k) acc[k] = 0;
        GM3Grain nx = {};
        if (tid < n) gm3_load(nx, p, tid);
        for (uint64_t g = tid; g < n; g += T) {
            const GM3Grain cur = nx;
            if (g + T < n) gm3_load(nx, p, g + T);               // in flight while this grain runs its chunk
            float st; uint32_t ph;
            gm3_chunk(cur, cols, acc, st, ph);
            p.g.st[g] = __float_as_uint(st);
            p.g.st[npad + g] = ph;
        }
#pragma unroll
        for (int h = 0; h < GM3_CHUNK / 32; ++h) {
            int32_t keepl = 0, keepr = 0;
#pragma unroll
            for (int k = 0; k < 32; ++k) {
                const int32_t a = acc[h * 32 + k];
                const int32_t l = (int32_t)(int16_t)(a & 0xFFFF);        // |sum L| <= grains_per_thread * 64 < 2^15
                const int32_t r = (a - l) >> 16;
                const int32_t sl = __reduce_add_sync(0xFFFFFFFFu, l), sr = __reduce_add_sync(0xFFFFFFFFu, r);
                if (lane == k) { keepl = sl; keepr = sr; }
            }
            if (h * 32 + lane < cols) { atomicAdd(&sacc[0][h * 32 + lane], keepl); atomicAdd(&sacc[1][h * 32 + lane], keepr); }
        }
        __syncthreads();
        if (threadIdx.x < cols) {
            atomicAdd(p.g.imix + t0 + threadIdx.x, sacc[0][threadIdx.x]);
            atomicAdd(p.g.imix + p.g.F + t0 + threadIdx.x, sacc[1][threadIdx.x]);
        }
        __syncthreads();
    }
    if constexpr (BUS) grain_bus_tail(p.g.imix, p.g.F, bf, nblk);
}

__global__ void k_imix_to_float(const int32_t *imix, float *mix, uint64_t count, float scale) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) mix[i] = __int2float_rn(imix[i]) * scale;
}

int launch_square_grain_mix(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io) {
    cproc_cuda_ctx *ctx = b->ctx;
    if (!io->out && !io->mix) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "square_grain_mix: out and mix are both NULL");
    if (F == 0) return 0;
    int32_t *imix = (int32_t *)io->mix;
    if (b->bus) {
        // the launch exchanges its mix itself: a [2][F] accumulator + ticket that every launch leaves zero, no memset
        const size_t need = sizeof(int32_t) * (2 * F + 1);
        if (b->cap_acc < need) {
            if (b->d_acc) cudaFree(b->d_acc);
            b->d_acc = nullptr; b->cap_acc = 0;
            CK(ctx, cudaMalloc(&b->d_acc, need));
            CK(ctx, cudaMemsetAsync(b->d_acc, 0, need, ctx->stream));   // once
            b->cap_acc = need;
        }
        imix = (int32_t *)b->d_acc;
    } else {
        if (!imix) {
            size_t need = sizeof(int32_t) * 2 * F;
            if (b->cap_mix < need) {
                if (b->d_mix) cudaFree(b->d_mix);
                b->d_mix = nullptr; b->cap_mix = 0;
                CK(ctx, cudaMalloc(&b->d_mix, need));
                b->cap_mix = need;
            }
            imix = (int32_t *)b->d_mix;
        }
        CK(ctx, cudaMemsetAsync(imix, 0, sizeof(int32_t) * 2 * F, ctx->stream));
    }
    GrainMixParams p;
    p.st = b->d_state; p.prm = b->d_param; p.npad = b->npad; p.n = b->n; p.F = F; p.imix = imix;
    if (b->aux_dirty) {                                   // integer thresholds, once per parameter upload
        if (!b->d_aux) CK(ctx, cudaMalloc(&b->d_aux, sizeof(uint32_t) * (3 * b->npad + 4)));
        uint32_t *weird = b->d_aux + 3 * b->npad;
        CK(ctx, cudaMemsetAsync(weird, 0, sizeof(uint32_t), ctx->stream));
        k_grain_thresholds<<<(unsigned)ceil_div_u64(b->n, 128), 128, 0, ctx->stream>>>(b->d_param, b->n, b->npad, (int32_t *)b->d_aux, (int32_t *)b->d_aux + b->npad, (int32_t *)b->d_aux + 2 * b->npad, weird);
        CK_LAUNCH(ctx, "k_grain_thresholds");
        uint32_t h = 0;
        CK(ctx, cudaMemcpyAsync(&h, weird, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
        CK(ctx, cudaStreamSynchronize(ctx->stream));
        b->aux_weird = h;
        b->aux_dirty = false;
    }
    // one pusher: the last render block of the launch; the bus writes io->mix (int32) and io->out ((float)x * 2^-7)
    BusFused bf;
    int rc = cproc_bus_fused_begin(b, &bf, 2 * F, 0u, 3u, 1u, (int32_t *)io->mix, (float *)io->out);
    if (rc) return rc;
    // a pipelined bus adds block 0, which completes the previous frame block's exchange; the capped grids below keep
    // it a free slot from the start
    const uint32_t xb = bf.world && bf.mode == 2 ? 1u : 0u;
#define GRAIN_MIX_LAUNCH(K, blocks, BLK, q) do { \
        if (bf.world) K<true><<<(unsigned)(blocks) + xb, BLK, 0, ctx->stream>>>(q, bf); \
        else K<false><<<(unsigned)(blocks), BLK, 0, ctx->stream>>>(q, bf); } while (0)
    if (ctx->grain_mix2 >= 2 && !b->aux_weird && !b->grain_odd_state) {
        GrainMix3Params q;
        q.g = p; q.lo = (const int32_t *)b->d_aux; q.hi = q.lo + b->npad; q.pk = q.lo + 2 * b->npad;
        uint64_t blocks = ceil_div_u64(p.n, GM3_BLOCK);
        const uint64_t cap = (uint64_t)ctx->n_sm * (uint64_t)ctx->grain_blocks_per_sm - xb;
        if (blocks > cap) blocks = cap;
        const uint64_t min_blocks = ceil_div_u64(p.n, (uint64_t)GM3_BLOCK * 500);   // packed 16-bit bus fields: <= 500 grains per thread
        if (blocks < min_blocks) blocks = min_blocks;
        GRAIN_MIX_LAUNCH(k_grain_mix3, blocks, GM3_BLOCK, q);
        CK_LAUNCH(ctx, "k_grain_mix3");
    } else if (ctx->grain_mix2 && !(b->aux_weird & 1u) && !b->grain_odd_state) {
        GrainMix2Params q;
        q.g = p; q.lo = (const int32_t *)b->d_aux; q.hi = (const int32_t *)b->d_aux + b->npad;
        uint64_t blocks = ceil_div_u64(p.n, GM2_BLOCK);
        const uint64_t cap = (uint64_t)ctx->n_sm * (uint64_t)ctx->grain_blocks_per_sm - xb;
        if (blocks > cap) blocks = cap;
        const uint64_t min_blocks = ceil_div_u64(p.n, (uint64_t)GM2_BLOCK * 500);   // packed 16-bit bus fields: <= 500 grains per thread
        if (blocks < min_blocks) blocks = min_blocks;
        GRAIN_MIX_LAUNCH(k_grain_mix2, blocks, GM2_BLOCK, q);
        CK_LAUNCH(ctx, "k_grain_mix2");
    } else {
        GRAIN_MIX_LAUNCH(k_grain_mix, ceil_div_u64(p.n, GMIX_BLOCK), GMIX_BLOCK, p);
        CK_LAUNCH(ctx, "k_grain_mix");
    }
#undef GRAIN_MIX_LAUNCH
    if (io->out && !bf.world) {
        k_imix_to_float<<<(unsigned)ceil_div_u64(2 * F, 256), 256, 0, ctx->stream>>>(imix, (float *)io->out, 2 * F, 0x1p-7f);
        CK_LAUNCH(ctx, "k_imix_to_float");
    }
    return 0;
}
