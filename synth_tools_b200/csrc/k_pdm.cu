// k_pdm.cu -- sigma-delta / PDM kernels other than the v2 modulator (k_pdm_v2.cu); integer, serial in time, bit-exact.
//
//   k_pdm_v1_*    stm32f103/mod_pdm.c:230-264 (carry-bit PDM, shared dither)
//   k_pdm_raw     stm32f103/pdm.h:13-77 (pdmK_update on an input stream)
//   k_pwm         stm32f103/mod_pdm.c:167-175
//
// Scheduling of the persistent v1 kernel.  A warp of 32 banks is a "chain" of G time groups that must run
// in order.  The kernel runs W <= C worker warps and cuts the C*G work units into W equal contiguous pieces
// (McNaughton's wrap-around rule for preemptive scheduling): a worker runs the HEAD of its last chain first,
// then its whole chains, then the TAIL of its first chain, whose head was run first thing by the previous
// worker.  The hand-over goes through the state arrays in L2 plus a release/acquire progress word; by
// construction the producer is always ahead, so the wait is a safety net.
#include "common.cuh"
#include "pdm_common.cuh"
#include "planar_bulk.cuh"

// McNaughton wrap-around schedule over C chains x G groups for W workers.
struct Sched {
    uint64_t C, G, W, Lg;            // Lg = ceil(C*G / W) >= G
    unsigned long long *flags;       // [C] progress words: (epoch << 32) | groups done
    unsigned long long epoch;
};

struct Segment { uint64_t chain, g0, g1; bool wait, signal; };

// Segment k of worker w in execution order (k < sched_count(s, w)).
__device__ __forceinline__ uint32_t sched_count(const Sched &s, uint64_t w, uint64_t *ca, uint64_t *ga, uint64_t *cb, uint64_t *gb) {
    const uint64_t total = s.C * s.G;
    const uint64_t u0 = w * s.Lg;
    if (u0 >= total) return 0;
    const uint64_t u1 = u0 + s.Lg < total ? u0 + s.Lg : total;
    *ca = u0 / s.G; *ga = u0 % s.G;
    *cb = (u1 - 1) / s.G; *gb = (u1 - 1) % s.G + 1;
    return (uint32_t)(*cb - *ca + 1);
}
__device__ __forceinline__ Segment sched_segment(const Sched &s, uint32_t k, uint32_t nseg, uint64_t ca, uint64_t ga, uint64_t cb, uint64_t gb) {
    if (nseg == 1) return Segment{ca, ga, gb, ga > 0, gb < s.G};
    if (k == 0) return Segment{cb, 0, gb, false, gb < s.G};          // head of the last chain: no dependency
    if (k == nseg - 1) return Segment{ca, ga, s.G, ga > 0, false};   // tail of the first chain
    return Segment{ca + k, 0, s.G, false, false};                    // whole chains in between
}

__device__ __forceinline__ void sched_wait(const Sched &s, const Segment &sg, uint32_t lane) {
    if (!sg.wait) return;
    if (lane == 0) {
        const unsigned long long want = (s.epoch << 32) | sg.g0;
        while (ld_acquire_u64(s.flags + sg.chain) != want) __nanosleep(100);
    }
    __syncwarp();
}
__device__ __forceinline__ void sched_signal(const Sched &s, const Segment &sg, uint32_t lane) {
    if (!sg.signal) return;
    __threadfence();
    __syncwarp();
    if (lane == 0) st_release_u64(s.flags + sg.chain, (s.epoch << 32) | sg.g1);
}

// Workers for C chains: as many warps as there are chains, up to `per_sm` warps
// on each of the SMs; always W <= C so that Lg >= G.
static int sched_setup(cproc_cuda_batch *b, Sched *s, uint64_t C, uint64_t G, int per_sm) {
    cproc_cuda_ctx *ctx = b->ctx;
    if (b->n_flags < C) {
        if (b->d_flags) cudaFree(b->d_flags);
        b->d_flags = nullptr; b->n_flags = 0;
        CK(ctx, cudaMalloc(&b->d_flags, sizeof(unsigned long long) * C));
        CK(ctx, cudaMemsetAsync(b->d_flags, 0, sizeof(unsigned long long) * C, ctx->stream));
        b->n_flags = C;
    }
    uint64_t W = (uint64_t)ctx->n_sm * per_sm;
    if (W > C) W = C;
    s->C = C; s->G = G; s->W = W; s->Lg = ceil_div_u64(C * G, W);
    s->flags = b->d_flags;
    s->epoch = ++b->epoch;
    return 0;
}

// pdm_persist: 0 never, 2 always, 1 auto -- only where a plain grid would leave
// the warp schedulers badly unbalanced (between 1 and 1.6 chains per scheduler;
// measured on B200: 683 chains -> +20 %, 1024 chains -> -9 %).
static bool persist_wanted(const cproc_cuda_ctx *ctx, uint64_t C) {
    if (ctx->pdm_persist == 0) return false;
    if (ctx->pdm_persist >= 2) return true;
    const uint64_t smsp = 4ull * ctx->n_sm;
    return C > smsp && C * 10 < smsp * 16;
}

// ---------------------------------------------------------------------------
// v1: carry-bit PDM.  32 ticks -> one packed word (sample t at bit t & 31).
struct PdmV1Params {
    uint32_t *st;              // SoA [2][npad]: setpoint, accu
    uint64_t npad, n, n_banks;
    uint32_t bank_size;
    const uint32_t *prng;      // generator state at the start of the run
    uint32_t *prng_out;        // ... at its end: another buffer (a bank replayed by several blocks must not see a write-back); the host swaps
    const uint32_t *dither_ext;
    uint32_t *out;
    uint64_t F;
    uint32_t dmask, layout;
    const uint32_t *jump16;    // M^16 of xorshift32 as 4 byte-indexed LUTs (two-chain PRNG) or null
    uint32_t *prng_live;       // persistent kernel (thread == bank, segments of one bank run in order): state updated in place
    Sched sched;
};

// accu += x with the carry out shifted into the LSB of bits (ARM: adds + adc;
// mod_pdm.c:236-240 uses rrx, i.e. the MSB: the final __brev gives the same
// time order LSB-first).
__device__ __forceinline__ void add_carry_shift(uint32_t &accu, uint32_t &bits, uint32_t x) {
    asm("add.cc.u32 %0, %0, %2;\n\taddc.u32 %1, %1, %1;" : "+r"(accu), "+r"(bits) : "r"(x));
}

// 32 ticks of B channels -> one packed word per channel
template <int B, bool DEXT>
__device__ __forceinline__ void v1_word(const uint32_t (&sp)[B], uint32_t (&acc)[B], uint32_t &rng, const uint32_t *dext32,
                                        uint32_t dmask, uint32_t (&wv)[B]) {
    uint32_t bits[B];
#pragma unroll
    for (int j = 0; j < B; ++j) bits[j] = 0;
#pragma unroll
    for (int i = 0; i < 32; ++i) {
        uint32_t d;
        if (DEXT) d = dext32[i] & dmask;
        else { rng = xorshift32_step(rng); d = rng & dmask; }       // mod_pdm.c:261
#pragma unroll
        for (int j = 0; j < B; ++j) add_carry_shift(acc[j], bits[j], sp[j] + d);   // :235-240
    }
#pragma unroll
    for (int j = 0; j < B; ++j) wv[j] = __brev(bits[j]);
}

// The same word with the bank's generator run as TWO interleaved chains (xorshift32 is a 6-deep
// dependent chain per tick and there are fewer than two warps per scheduler at the C2 shape, so
// one chain leaves the issue slots idle), software pipelined: while the accumulators consume the
// 32 dither values of word w (registers `cur`), the generator produces the 32 values of word w+1
// (`nxt`) -- chain A ticks 0..15, chain B (started 16 steps ahead with the GF(2) jump table M^16)
// ticks 16..31.  The accumulate chain (one dependent add per tick) is then never paced by the
// 6-deep xorshift chain.
// GEN = false for the last word of a group: nothing is generated beyond it.
template <int B, bool GEN>
__device__ __forceinline__ void v1_word_pipe(const uint32_t (&sp)[B], uint32_t (&acc)[B], const uint32_t (&cur)[32], uint32_t (&nxt)[32],
                                             uint32_t &rng, const uint32_t (*jt)[256], uint32_t dmask, uint32_t (&wv)[B]) {
    uint32_t bits[B];
#pragma unroll
    for (int j = 0; j < B; ++j) bits[j] = 0;
    uint32_t xa = rng, xb = GEN ? jump_apply(jt, rng) : 0u;          // rng = generator state at the start of word w+1
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        if (GEN) {
            xa = xorshift32_step(xa); nxt[i] = xa & dmask;            // mod_pdm.c:261
            xb = xorshift32_step(xb); nxt[16 + i] = xb & dmask;
        }
#pragma unroll
        for (int j = 0; j < B; ++j) add_carry_shift(acc[j], bits[j], sp[j] + cur[2 * i]);       // :235-240
#pragma unroll
        for (int j = 0; j < B; ++j) add_carry_shift(acc[j], bits[j], sp[j] + cur[2 * i + 1]);
    }
    if (GEN) rng = xb;                                               // state at the start of word w+2
#pragma unroll
    for (int j = 0; j < B; ++j) wv[j] = __brev(bits[j]);
}

// One group of four words with the two-chain generator, software pipelined: the first word's dither is generated up front, the last
// word of the group generates nothing (the next group starts over: one un-overlapped word in four keeps the generator state exact
// at every group boundary).
template <int B>
__device__ __forceinline__ void v1_group_pipe(const PdmV1Params &p, const uint32_t (&sp)[B], uint32_t (&acc)[B], uint32_t &rng, const uint32_t (*jt)[256],
                                              uint32_t (&q)[4][B]) {
    uint32_t da[32], db[32];
    {
        uint32_t xa = rng, xb = jump_apply(jt, rng);
#pragma unroll
        for (int i = 0; i < 16; ++i) { xa = xorshift32_step(xa); da[i] = xa & p.dmask; xb = xorshift32_step(xb); da[16 + i] = xb & p.dmask; }
        rng = xb;
    }
    v1_word_pipe<B, true>(sp, acc, da, db, rng, jt, p.dmask, q[0]);
    v1_word_pipe<B, true>(sp, acc, db, da, rng, jt, p.dmask, q[1]);
    v1_word_pipe<B, true>(sp, acc, da, db, rng, jt, p.dmask, q[2]);
    v1_word_pipe<B, false>(sp, acc, db, da, rng, jt, p.dmask, q[3]);
}

// words [w0, w1) of one thread's B channels
template <int B, bool DEXT>
__device__ __forceinline__ void v1_run_segment(const PdmV1Params &p, const uint32_t (&sp)[B], uint32_t (&acc)[B], uint32_t &rng,
                                               uint64_t c0, uint64_t bank, uint64_t w0, uint64_t w1, const uint32_t (*jt)[256] = nullptr) {
    const uint64_t words = p.F >> 5;
    const uint32_t *dext = DEXT ? p.dither_ext + bank * p.F : nullptr;
    // Groups of four words (128 ticks): the TILED layout's unit, and -- with the two-chain generator -- the unit of the software
    // pipeline for the other layouts too when the run is whole groups (PLANAR: one 128-bit store per channel and group when the
    // rows allow it; INTERLEAVED: four coalesced word stores).  The TILED loop is kept on its own: it is the measured one
    // (sharing it with the other layouts' store selection cost it 3.5 %).
    if (p.layout == CPROC_CUDA_TILED) {
        for (uint64_t g = w0; g < w1; g += 4) {
            uint32_t q[4][B];
            if (!DEXT && jt) v1_group_pipe<B>(p, sp, acc, rng, jt, q);
            else
#pragma unroll
            for (int k = 0; k < 4; ++k) v1_word<B, DEXT>(sp, acc, rng, DEXT ? dext + ((g + k) << 5) : nullptr, p.dmask, q[k]);
#pragma unroll
            for (int j = 0; j < B; ++j)
                if (c0 + j < p.n) st_v4_stream(p.out + (((g >> 2) * p.n + c0 + j) << 2), make_uint4(q[0][j], q[1][j], q[2][j], q[3][j]));
        }
        return;
    }
    const bool il = p.layout == CPROC_CUDA_INTERLEAVED;
    if (!DEXT && jt && ((w0 | w1 | words) & 3) == 0) {
        const bool row16 = !il && (((uintptr_t)p.out) & 15) == 0;        // PLANAR rows of whole groups from an aligned base
        for (uint64_t g = w0; g < w1; g += 4) {
            uint32_t q[4][B];
            v1_group_pipe<B>(p, sp, acc, rng, jt, q);
#pragma unroll
            for (int j = 0; j < B; ++j) {
                if (c0 + j >= p.n) continue;
                if (il) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) __stcs(p.out + (g + k) * p.n + c0 + j, q[k][j]);
                } else if (row16) st_v4_stream(p.out + (c0 + j) * words + g, make_uint4(q[0][j], q[1][j], q[2][j], q[3][j]));
                else {
#pragma unroll
                    for (int k = 0; k < 4; ++k) __stcs(p.out + (c0 + j) * words + g + k, q[k][j]);
                }
            }
        }
        return;
    }
    for (uint64_t g = w0; g < w1; ++g) {
        uint32_t wv[B];
        v1_word<B, DEXT>(sp, acc, rng, DEXT ? dext + (g << 5) : nullptr, p.dmask, wv);
#pragma unroll
        for (int j = 0; j < B; ++j)
            if (c0 + j < p.n) __stcs(p.out + (il ? g * p.n + c0 + j : (c0 + j) * words + g), wv[j]);
    }
}

template <int B>
__global__ void __launch_bounds__(128, 4) k_pdm_v1_persist(const PdmV1Params p, uint32_t unit_words) {
    __shared__ uint32_t jt[4][256];
    if (p.jump16) {
        for (uint32_t k = threadIdx.x; k < 1024; k += blockDim.x) (&jt[0][0])[k] = __ldg(p.jump16 + k);
        __syncthreads();
    }
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t worker = (uint64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (worker >= p.sched.W) return;
    uint64_t ca, ga, cb, gb;
    const uint32_t nseg = sched_count(p.sched, worker, &ca, &ga, &cb, &gb);
    for (uint32_t k = 0; k < nseg; ++k) {
        const Segment sg = sched_segment(p.sched, k, nseg, ca, ga, cb, gb);
        const uint64_t bank = sg.chain * 32 + lane;
        sched_wait(p.sched, sg, lane);
        if (bank < p.n_banks) {
            const uint64_t c0 = bank * B;
            uint32_t sp[B], acc[B];
#pragma unroll
            for (int j = 0; j < B; ++j) { sp[j] = __ldcg(p.st + c0 + j); acc[j] = __ldcg(p.st + p.npad + c0 + j); }
            uint32_t rng = __ldcg(p.prng_live + bank);
            v1_run_segment<B, false>(p, sp, acc, rng, c0, bank, sg.g0 * unit_words, sg.g1 * unit_words, p.jump16 ? jt : nullptr);
#pragma unroll
            for (int j = 0; j < B; ++j) __stcg(p.st + p.npad + c0 + j, acc[j]);
            __stcg(p.prng_live + bank, rng);
        }
        sched_signal(p.sched, sg, lane);
    }
}

template <int B, bool TPB, bool DEXT>
__global__ void __launch_bounds__(128) k_pdm_v1_simple(const PdmV1Params p) {
    __shared__ uint32_t jt[(TPB && !DEXT) ? 4 : 1][256];
    const bool two = TPB && !DEXT && p.jump16 != nullptr;
    if (two) {
        for (uint32_t k = threadIdx.x; k < 1024; k += blockDim.x) (&jt[0][0])[k] = __ldg(p.jump16 + k);
        __syncthreads();
    }
    const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= (TPB ? p.n_banks : p.n_banks * p.bank_size)) return;
    const uint64_t c0 = tid * B;
    const uint64_t bank = TPB ? tid : tid / p.bank_size;
    const bool rng_owner = TPB ? true : (tid % p.bank_size == 0);
    uint32_t sp[B], acc[B];
#pragma unroll
    for (int j = 0; j < B; ++j) { sp[j] = p.st[c0 + j]; acc[j] = p.st[p.npad + c0 + j]; }
    uint32_t rng = __ldg(p.prng + bank);
    v1_run_segment<B, DEXT>(p, sp, acc, rng, c0, bank, 0, p.F >> 5, two ? jt : nullptr);
#pragma unroll
    for (int j = 0; j < B; ++j) p.st[p.npad + c0 + j] = acc[j];
    if (rng_owner && !DEXT) p.prng_out[bank] = rng;
}

int launch_pdm_v1(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io) {
    cproc_cuda_ctx *ctx = b->ctx;
    const cproc_cuda_config &c = b->cfg;
    if (!io->out) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "pdm_v1: out is NULL");
    if (F & 31) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "pdm_v1: F must be a multiple of 32 (packed bit output)");
    if (io->layout == CPROC_CUDA_TILED && (F & 127)) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "pdm_v1: TILED needs F %% 128 == 0");
    if (io->layout == CPROC_CUDA_TILED && ((uintptr_t)io->out & 15)) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "pdm_v1: TILED needs a 16-byte aligned out");
    if (F == 0) return 0;
    PdmV1Params p;
    p.st = b->d_state; p.npad = b->npad; p.n = b->n; p.n_banks = b->n_banks; p.bank_size = c.bank_size;
    if (!b->d_prng2) CK(ctx, cudaMalloc(&b->d_prng2, sizeof(uint32_t) * b->n_banks));
    p.prng = b->d_prng; p.prng_out = b->d_prng2; p.prng_live = b->d_prng;
    p.dither_ext = (const uint32_t *)io->in2; p.out = (uint32_t *)io->out; p.F = F;
    p.dmask = c.dither_mask; p.layout = io->layout;
    p.sched = Sched{};
    p.jump16 = nullptr;
    const int blk = ctx->pdm_block;
    const bool dext = io->in2 != nullptr;
    // Thread per bank (3 instructions per channel-tick + 7 for the generator, once per bank) or thread per channel (every thread replays
    // the generator: 10 per channel-tick, but bank_size times the warps).  Auto: per bank unless the banks are fewer warps than the chip
    // has schedulers while the channels are not -- 65,536 channels in banks of 4 are 512 bank-warps on 592 schedulers: 1.89e12 per bank,
    // 2.21e12 per channel (tools/layout_matrix.py).
    bool tpb = ctx->pdm_tpb && c.bank_size <= 4;
    if (ctx->pdm_tpb == 2 && tpb && c.bank_size >= 2 && ceil_div_u64(p.n_banks, 32) < 4ull * ctx->n_sm) tpb = false;
    const uint64_t C = ceil_div_u64(p.n_banks, 32);
    bool swap_prng = false;
    if (ctx->pdm_v1_chains == 2 && tpb && !dext && (F & 127) == 0) {            // whole 128-tick groups: the two-chain, software-pipelined words in every layout
        if (!ctx->d_jump16) {                                 // M^16 of xorshift32 as 4 byte-indexed LUTs
            std::vector<uint32_t> h(1024);
            jump_table_fill(h.data(), 16);
            CK(ctx, cudaMalloc(&ctx->d_jump16, h.size() * 4));
            CK(ctx, cudaMemcpyAsync(ctx->d_jump16, h.data(), h.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
            CK(ctx, cudaStreamSynchronize(ctx->stream));
        }
        p.jump16 = ctx->d_jump16;
    }
    if (tpb && !dext && (F & 127) == 0 && persist_wanted(ctx, C)) {
        int rc = sched_setup(b, &p.sched, C, F >> 7, 4 * ctx->pdm_warps_per_smsp);   // unit = 128 ticks = 4 words
        if (rc) return rc;
        const unsigned grid = (unsigned)ceil_div_u64(p.sched.W, 4);
        switch (c.bank_size) {
        case 1: k_pdm_v1_persist<1><<<grid, 128, 0, ctx->stream>>>(p, 4); break;
        case 2: k_pdm_v1_persist<2><<<grid, 128, 0, ctx->stream>>>(p, 4); break;
        case 3: k_pdm_v1_persist<3><<<grid, 128, 0, ctx->stream>>>(p, 4); break;
        default: k_pdm_v1_persist<4><<<grid, 128, 0, ctx->stream>>>(p, 4); break;
        }
    } else {
        swap_prng = !dext;
#define V1_SIMPLE(BB, TT) do { \
        const unsigned grid = (unsigned)ceil_div_u64((TT) ? p.n_banks : p.n_banks * p.bank_size, blk); \
        if (dext) k_pdm_v1_simple<BB, TT, true><<<grid, blk, 0, ctx->stream>>>(p); \
        else k_pdm_v1_simple<BB, TT, false><<<grid, blk, 0, ctx->stream>>>(p); } while (0)
        if (tpb) {
            switch (c.bank_size) {
            case 1: V1_SIMPLE(1, true); break;
            case 2: V1_SIMPLE(2, true); break;
            case 3: V1_SIMPLE(3, true); break;
            default: V1_SIMPLE(4, true); break;
            }
        } else V1_SIMPLE(1, false);
#undef V1_SIMPLE
    }
    CK_LAUNCH(ctx, "k_pdm_v1");
    if (swap_prng) { uint32_t *t = b->d_prng; b->d_prng = b->d_prng2; b->d_prng2 = t; }
    return 0;
}

// ---------------------------------------------------------------------------
// raw pdmK_update over an input stream (pdm.h), uint32 quantiser output.
struct PdmRawParams {
    uint32_t *st;               // SoA [K][npad]
    const uint32_t *param;      // SoA [1][npad] constant input
    uint64_t npad, n;
    const uint32_t *in;         // [inst][F] / [F][inst] or null
    const uint32_t *dither;     // [F] or null
    uint32_t *out;
    uint64_t F;
    uint32_t sh, layout;
};

template <int K>
__global__ void k_pdm_raw(const PdmRawParams p) {
    const uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= p.n) return;
    uint32_t s[K];
#pragma unroll
    for (int k = 0; k < K; ++k) s[k] = p.st[k * p.npad + c];
    const uint32_t cst = p.param[c];
    const bool il = p.layout == CPROC_CUDA_INTERLEAVED;
    for (uint64_t t = 0; t < p.F; ++t) {
        uint64_t idx = il ? t * p.n + c : c * p.F + t;
        uint32_t x = p.in ? p.in[idx] : cst;
        uint32_t d = p.dither ? p.dither[t] : 0u;
        p.out[idx] = pdm_step<K>(s, x, p.sh, d);
    }
#pragma unroll
    for (int k = 0; k < K; ++k) p.st[k * p.npad + c] = s[k];
}

// PLANAR streams through the staging template (planar_bulk.cuh): the per-thread row walk of
// k_pdm_raw touches 32 different lines per warp instruction.
template <int K, int HAS_IN>
struct PdmRawOp {
    static constexpr int NIN = HAS_IN;
    uint32_t *st; const uint32_t *param; const uint32_t *dither;
    uint64_t npad; uint32_t sh;
    uint32_t s[K], cst;
    __device__ __forceinline__ void load(uint64_t i) {
#pragma unroll
        for (int k = 0; k < K; ++k) s[k] = st[k * npad + i];
        cst = param[i];
    }
    __device__ __forceinline__ void store(uint64_t i) {
#pragma unroll
        for (int k = 0; k < K; ++k) st[k * npad + i] = s[k];
    }
    __device__ __forceinline__ uint32_t tick(uint32_t x, uint64_t t) {
        return pdm_step<K>(s, HAS_IN ? x : cst, sh, dither ? __ldg(dither + t) : 0u);    // pdm.h:13-77
    }
};

template <int K>
static bool launch_pdm_raw_bulk(cproc_cuda_ctx *ctx, const PdmRawParams &p) {
    if (p.in) {
        PdmRawOp<K, 1> op; op.st = p.st; op.param = p.param; op.dither = p.dither; op.npad = p.npad; op.sh = p.sh;
        return pbulk::launch(ctx, op, p.in, p.out, p.n, p.F);
    }
    PdmRawOp<K, 0> op; op.st = p.st; op.param = p.param; op.dither = p.dither; op.npad = p.npad; op.sh = p.sh;
    return pbulk::launch(ctx, op, p.out, p.out, p.n, p.F);
}

template <int K>
static void launch_pdm_raw_il4(cproc_cuda_ctx *ctx, const PdmRawParams &p) {
    if (p.in) {
        PdmRawOp<K, 1> op; op.st = p.st; op.param = p.param; op.dither = p.dither; op.npad = p.npad; op.sh = p.sh;
        pbulk::launch_interleaved4(ctx, op, p.in, p.out, p.n, p.F);
    } else {
        PdmRawOp<K, 0> op; op.st = p.st; op.param = p.param; op.dither = p.dither; op.npad = p.npad; op.sh = p.sh;
        pbulk::launch_interleaved4(ctx, op, p.out, p.out, p.n, p.F);
    }
}

int launch_pdm(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io) {
    cproc_cuda_ctx *ctx = b->ctx;
    if (!io->out) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "pdm: out is NULL");
    if (io->layout == CPROC_CUDA_TILED) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "pdm: TILED layout not supported");
    if (F == 0) return 0;
    PdmRawParams p;
    p.st = b->d_state; p.param = b->d_param; p.npad = b->npad; p.n = b->n;
    p.in = (const uint32_t *)io->in; p.dither = (const uint32_t *)io->in2; p.out = (uint32_t *)io->out;
    p.F = F; p.sh = b->cfg.out_shift; p.layout = io->layout;
    unsigned grid = (unsigned)ceil_div_u64(p.n, 128);
    if (ctx->planar_bulk && io->layout == CPROC_CUDA_PLANAR) {
        bool staged;
        switch (b->cfg.order) {
        case 1: staged = launch_pdm_raw_bulk<1>(ctx, p); break;
        case 2: staged = launch_pdm_raw_bulk<2>(ctx, p); break;
        case 3: staged = launch_pdm_raw_bulk<3>(ctx, p); break;
        default: staged = launch_pdm_raw_bulk<4>(ctx, p); break;
        }
        if (staged) {
            CK_LAUNCH(ctx, "k_pdm_raw (bulk)");
            return 0;
        }
    }
    if (ctx->planar_bulk && io->layout == CPROC_CUDA_INTERLEAVED && pbulk::usable_interleaved4(p.n, p.in, p.out)) {
        switch (b->cfg.order) {
        case 1: launch_pdm_raw_il4<1>(ctx, p); break;
        case 2: launch_pdm_raw_il4<2>(ctx, p); break;
        case 3: launch_pdm_raw_il4<3>(ctx, p); break;
        default: launch_pdm_raw_il4<4>(ctx, p); break;
        }
        CK_LAUNCH(ctx, "k_pdm_raw (interleaved4)");
        return 0;
    }
    switch (b->cfg.order) {
    case 1: k_pdm_raw<1><<<grid, 128, 0, ctx->stream>>>(p); break;
    case 2: k_pdm_raw<2><<<grid, 128, 0, ctx->stream>>>(p); break;
    case 3: k_pdm_raw<3><<<grid, 128, 0, ctx->stream>>>(p); break;
    default: k_pdm_raw<4><<<grid, 128, 0, ctx->stream>>>(p); break;
    }
    CK_LAUNCH(ctx, "k_pdm_raw");
    return 0;
}

// ---------------------------------------------------------------------------
// pwm_update (mod_pdm.c:167-175): nonlinear phase feedback, serial.
__global__ void k_pwm(uint32_t *phase, const uint32_t *speed, uint64_t n, uint64_t F, uint8_t *out, uint32_t layout) {
    const uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    uint32_t ph = phase[c];
    const uint32_t sp = speed[c];
    for (uint64_t t = 0; t < F; ++t) {
        uint64_t idx = layout == CPROC_CUDA_INTERLEAVED ? t * n + c : c * F + t;
        out[idx] = (uint8_t)(ph >> 16);
        ph = (ph + sp + (ph >> 9)) & 0xFFFFFFu;
    }
    phase[c] = ph;
}

// PLANAR duty bytes through the staging template: one "frame" of the template is a 32-bit word
// = four ticks (duty is 8 bit), so a lane's 64-word tile is 256 ticks of its channel.
struct PwmOp {
    static constexpr int NIN = 0;
    uint32_t *phase; const uint32_t *speed;
    uint32_t ph, sp;
    __device__ __forceinline__ void load(uint64_t i) { ph = phase[i]; sp = speed[i]; }
    __device__ __forceinline__ void store(uint64_t i) { phase[i] = ph; }
    __device__ __forceinline__ uint32_t tick(uint32_t, uint64_t) {
        uint32_t w = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            w |= ((ph >> 16) & 0xFFu) << (8 * k);              // mod_pdm.c:170
            ph = (ph + sp + (ph >> 9)) & 0xFFFFFFu;            // :171-174
        }
        return w;
    }
};

// TILED [F/16][ch][16]: one 128-bit store per 16 ticks, like the PDM v2 duty stream
__global__ void __launch_bounds__(128) k_pwm_tiled(uint32_t *phase, const uint32_t *speed, uint64_t n, uint64_t F, uint8_t *out) {
    const uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    uint32_t ph = phase[c];
    const uint32_t sp = speed[c];
    for (uint64_t g = 0; g < F / 16; ++g) {
        uint32_t w[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            w[q] = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                w[q] |= ((ph >> 16) & 0xFFu) << (8 * k);
                ph = (ph + sp + (ph >> 9)) & 0xFFFFFFu;
            }
        }
        st_v4_stream(out + ((g * n + c) << 4), make_uint4(w[0], w[1], w[2], w[3]));
    }
    phase[c] = ph;
}

int launch_pwm(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io) {
    cproc_cuda_ctx *ctx = b->ctx;
    if (!io->out) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "pwm: out is NULL");
    if (io->layout == CPROC_CUDA_TILED && ((F & 15) || ((uintptr_t)io->out & 15))) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "pwm: TILED needs F %% 16 == 0 and a 16-byte aligned buffer");
    if (F == 0) return 0;
    if (io->layout == CPROC_CUDA_TILED) {
        k_pwm_tiled<<<(unsigned)ceil_div_u64(b->n, 128), 128, 0, ctx->stream>>>(b->d_state, b->d_param, b->n, F, (uint8_t *)io->out);
        CK_LAUNCH(ctx, "k_pwm_tiled");
        return 0;
    }
    PwmOp op; op.phase = b->d_state; op.speed = b->d_param; op.ph = 0; op.sp = 0;
    if (ctx->planar_bulk && io->layout == CPROC_CUDA_PLANAR && F % 16 == 0 && pbulk::launch(ctx, op, (const uint32_t *)io->out, (uint32_t *)io->out, b->n, F / 4)) {
        CK_LAUNCH(ctx, "k_pwm (bulk)");
        return 0;
    }
    k_pwm<<<(unsigned)ceil_div_u64(b->n, 128), 128, 0, ctx->stream>>>(b->d_state, b->d_param, b->n, F, (uint8_t *)io->out, io->layout);
    CK_LAUNCH(ctx, "k_pwm");
    return 0;
}
