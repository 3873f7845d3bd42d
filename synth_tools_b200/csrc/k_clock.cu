// Word clock: the integer-divisor square wave of linux/clock.c:109-120 (one JACK MIDI-clock master in the
// reference; here a batch of clocks).  Per sample:
//     if (phase >= hperiod) { phase -= hperiod; pol ^= 1; }   out[t] = pol;   phase += 1;
// state {int32 phase; int32 pol}, param {int32 hperiod}; out float [inst][F] / [F][inst].  A MIDI clock
// byte goes out where pol turns 1 (clock.c:113-116): the host adapter finds those samples in its block.
// 4 bytes out per sample: HBM-write bound, PLANAR through the staging template of planar_bulk.cuh.
#include "common.cuh"
#include "planar_bulk.cuh"

struct WordClockOp {
    static constexpr int NIN = 0;
    uint32_t *st; const uint32_t *prm; uint64_t npad;
    int32_t phase, pol, h;
    __device__ __forceinline__ void load(uint64_t i) { phase = (int32_t)st[i]; pol = (int32_t)st[npad + i]; h = (int32_t)prm[i]; }
    __device__ __forceinline__ void store(uint64_t i) { st[i] = (uint32_t)phase; st[npad + i] = (uint32_t)pol; }
    __device__ __forceinline__ uint32_t tick(uint32_t, uint64_t) {
        if (phase >= h) { phase = (int32_t)((uint32_t)phase - (uint32_t)h); pol ^= 1; }
        phase = (int32_t)((uint32_t)phase + 1u);
        return __float_as_uint(__int2float_rn(pol));
    }
};

__global__ void __launch_bounds__(128) k_word_clock(WordClockOp op, uint64_t n, uint64_t F, float *out, uint32_t layout) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    op.load(i);
    for (uint64_t t = 0; t < F; ++t)
        out[layout == CPROC_CUDA_INTERLEAVED ? t * n + i : i * F + t] = __uint_as_float(op.tick(0, t));
    op.store(i);
}

int launch_word_clock(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io) {
    cproc_cuda_ctx *ctx = b->ctx;
    if (!io->out) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "word_clock: out is NULL");
    if (io->layout == CPROC_CUDA_TILED) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "word_clock: TILED layout not supported");
    if (F == 0) return 0;
    WordClockOp op; op.st = b->d_state; op.prm = b->d_param; op.npad = b->npad; op.phase = 0; op.pol = 0; op.h = 0;
    if (ctx->planar_bulk && io->layout == CPROC_CUDA_PLANAR && pbulk::launch(ctx, op, (const uint32_t *)io->out, (uint32_t *)io->out, b->n, F)) {
        CK_LAUNCH(ctx, "k_word_clock (planar template)");
        return 0;
    }
    k_word_clock<<<(unsigned)ceil_div_u64(b->n, 128), 128, 0, ctx->stream>>>(op, b->n, F, (float *)io->out, io->layout);
    CK_LAUNCH(ctx, "k_word_clock");
    return 0;
}
