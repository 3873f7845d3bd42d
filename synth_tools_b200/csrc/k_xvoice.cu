// k_xvoice.cu -- extension processors (NOT in the reference; defined by
// oracle/cproc_oracle.c: orc_xvoice_tick, orc_onepole_run).
//
//   voice = phasor_f (acc, cproc.h:140-142, read-then-advance like
//           synth.c:175-177) -> Chamberlin SVF low-pass -> linear AR envelope
//           -> pan.
//
// Every float operation is a single IEEE rounding in the same order as the
// oracle (fmaf == FFMA, explicit __fadd_rn/__fmul_rn so nvcc cannot contract
// differently), so the raw per-voice output is bit-exact against the C oracle.
// The mix is a float sum over voices and therefore order dependent: it is
// reduced in a fixed order (lane tree -> warp rows -> block partials -> final
// pass), deterministic run to run, and compared with tolerance.
#include "common.cuh"
#include "planar_bulk.cuh"
#include "bus_fused.cuh"

struct XVoiceParams {
    uint32_t *st;            // SoA [5][npad]: phase, lp, bp, env, t
    const uint32_t *prm;     // SoA [8][npad]: inc, f, q, attack, release, gate_frames, gl, gr
    uint64_t npad, n, F;
    float *raw;              // PLANAR [inst][F][2] / TILED [F/2][inst][4] or null
    float *partial;          // [n_blocks][2][F] or null
    uint32_t layout;
    float *mix;              // k_xvoice_mix: [2][F]
    uint32_t *done;          // k_xvoice_mix: [2] blocks that left / finalisers done (zero between launches)
    uint32_t n_render_blocks;// k_xvoice_mix: gridDim.x without the finisher block of a pipelined bus
    uint32_t vpt;            // k_xvoice_mix: voices per thread per L2 tile
    uint32_t rows_per_block; // partial rows a block leaves per channel pair for the final reduction (1)
    float *partial_w;        // k_xvoice_mix2: [n_blocks][4 warps][2][F] per-warp rows, summed into the block's row of `partial` when the block is done
};

struct XV {
    uint32_t phase, t, inc, gate;
    float lp, bp, env, f, q, att, rel, gl, gr;
};

// phase += inc on the ALU pipe.  ptxas turns a plain 32-bit add into IMAD.IADD half of the time to "balance" the pipes; here the FMA
// pipe is the busy one (FFMA2 / FADD2 / FMUL2 / I2FP hold it for two cycles each): 24 % of the kernel's stall samples sat on those
// IMADs (profiles/r2_xvoice_mix2_summary.txt).  An add with carry-out can only be an IADD3.
__device__ __forceinline__ void xv_add_alu(uint32_t &x, uint32_t inc) { asm("add.cc.u32 %0, %0, %1;" : "+r"(x) : "r"(inc)); }

// x = (float)(int)phase * 2^-31 is exact (a power-of-two scale of a 24-bit float, no
// underflow), so hp = x - lp (one rounding) is computed as fma(xi, 2^-31, -lp): the
// same bits, one instruction less.
__device__ __forceinline__ void xvoice_svf(XV &v, float &lp_out) {
    const float xi = __int2float_rn((int32_t)v.phase);
    xv_add_alu(v.phase, v.inc);
    const float lp = __fmaf_rn(v.f, v.bp, v.lp);
    float hp = __fmaf_rn(xi, 0x1p-31f, -lp);
    hp = __fmaf_rn(-v.q, v.bp, hp);
    v.bp = __fmaf_rn(v.f, hp, v.bp);
    v.lp = lp;
    lp_out = lp;
}

// Tick with the attack/release decision supplied by the caller (mix kernel: bit k of a
// per-chunk mask, so the frame counter is advanced once per chunk).  Same float
// operations as xvoice_tick except that a -0.0 envelope in release becomes +0.0
// (fmaxf); a -0.0 envelope can only come from an uploaded state.
__device__ __forceinline__ float xvoice_tick_flag(XV &v, bool attack) {
    float lp;
    xvoice_svf(v, lp);
    float e = v.env;
    if (attack) { e = __fadd_rn(e, v.att); if (e > 1.0f) e = 1.0f; }
    else { e = fmaxf(__fsub_rn(e, v.rel), 0.0f); }
    v.env = e;
    return __fmul_rn(lp, e);
}

// Tick of a chunk that lies entirely in the attack or entirely in the release phase, for an
// envelope in [0, 1] and non-negative rates: e' = min(max(e + d, 0), 1) with d = +attack or
// -release is then the same float as the two-branch form (the clamp that does not belong to the
// phase is an identity), three instructions instead of two predicated pairs plus the predicate.
__device__ __forceinline__ float xvoice_tick_uniform(XV &v, float d) {
    float lp;
    xvoice_svf(v, lp);
    const float e = fminf(fmaxf(__fadd_rn(v.env, d), 0.0f), 1.0f);
    v.env = e;
    return __fmul_rn(lp, e);
}

__device__ __forceinline__ float xvoice_tick(XV &v) {
    const float xi = __int2float_rn((int32_t)v.phase);
    v.phase += v.inc;
    const float lp = __fmaf_rn(v.f, v.bp, v.lp);
    float hp = __fmaf_rn(xi, 0x1p-31f, -lp);
    hp = __fmaf_rn(-v.q, v.bp, hp);
    v.bp = __fmaf_rn(v.f, hp, v.bp);
    v.lp = lp;
    float e = v.env;
    if (v.t < v.gate) { e = __fadd_rn(e, v.att); if (e > 1.0f) e = 1.0f; }
    else { e = __fsub_rn(e, v.rel); if (e < 0.0f) e = 0.0f; }
    v.env = e;
    v.t += 1;
    return __fmul_rn(lp, e);
}

#define XV_BLOCK 128
#define XV_WARPS (XV_BLOCK / 32)
#define XV_CHUNK 32

template <bool RAW, bool MIX>
__global__ void __launch_bounds__(XV_BLOCK) k_xvoice(const XVoiceParams p) {
    __shared__ float red[XV_WARPS][2][XV_CHUNK][33];   // [warp][ch][frame][lane]
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool mine = i < p.n;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    XV v = {};
    if (mine) {
        const uint32_t *s = p.st + i; const uint32_t *r = p.prm + i;
        v.phase = s[0]; v.lp = __uint_as_float(s[p.npad]); v.bp = __uint_as_float(s[2 * p.npad]);
        v.env = __uint_as_float(s[3 * p.npad]); v.t = s[4 * p.npad];
        v.inc = r[0]; v.f = __uint_as_float(r[p.npad]); v.q = __uint_as_float(r[2 * p.npad]);
        v.att = __uint_as_float(r[3 * p.npad]); v.rel = __uint_as_float(r[4 * p.npad]); v.gate = r[5 * p.npad];
        v.gl = __uint_as_float(r[6 * p.npad]); v.gr = __uint_as_float(r[7 * p.npad]);
    }
    for (uint64_t t0 = 0; t0 < p.F; t0 += XV_CHUNK) {
        const uint32_t cols = p.F - t0 < XV_CHUNK ? (uint32_t)(p.F - t0) : XV_CHUNK;
        float pl = 0.f, pr = 0.f;
        for (uint32_t k = 0; k < cols; ++k) {
            const float y = xvoice_tick(v);
            const float l = __fmul_rn(v.gl, y), r = __fmul_rn(v.gr, y);
            if (MIX) { red[warp][0][k][lane] = mine ? l : 0.f; red[warp][1][k][lane] = mine ? r : 0.f; }
            if (RAW && mine) {
                const uint64_t t = t0 + k;
                if (p.layout == CPROC_CUDA_TILED) {
                    if (k & 1) st_v4_stream(p.raw + (((t >> 1) * p.n + i) << 2),
                                            make_uint4(__float_as_uint(pl), __float_as_uint(pr), __float_as_uint(l), __float_as_uint(r)));
                    else { pl = l; pr = r; }
                } else {
                    *reinterpret_cast<float2 *>(p.raw + ((i * p.F + t) << 1)) = make_float2(l, r);
                }
            }
        }
        if (MIX) {
            __syncthreads();
            // lane f of warp w sums frame f over the 32 voices of warp w, in lane order
            float sl = 0.f, sr = 0.f;
            if (lane < cols) {
#pragma unroll 8
                for (int j = 0; j < 32; ++j) { sl = __fadd_rn(sl, red[warp][0][lane][j]); sr = __fadd_rn(sr, red[warp][1][lane][j]); }
            }
            __syncthreads();
            if (lane < cols) { red[warp][0][lane][0] = sl; red[warp][1][lane][0] = sr; }
            __syncthreads();
            if (threadIdx.x < 2 * cols) {
                const uint32_t ch = threadIdx.x / cols, f = threadIdx.x % cols;
                float s = 0.f;
#pragma unroll
                for (int w = 0; w < XV_WARPS; ++w) s = __fadd_rn(s, red[w][ch][f][0]);
                p.partial[((uint64_t)blockIdx.x * 2 + ch) * p.F + t0 + f] = s;
            }
            __syncthreads();
        }
    }
    if (mine) {
        uint32_t *s = p.st + i;
        s[0] = v.phase; s[p.npad] = __float_as_uint(v.lp); s[2 * p.npad] = __float_as_uint(v.bp);
        s[3 * p.npad] = __float_as_uint(v.env); s[4 * p.npad] = v.t;
    }
}

// Mix-only render (C4: millions of voices -> one stereo bus).  The SVF is a
// recurrence in time, so a voice stays on one thread; the reduction over voices is
// taken out of the inner loop instead of being paid per voice-sample: a thread keeps
// 2 x 32 bus accumulators (32 frames, left/right) in registers and walks ITS voices
// through the same 32 frames one after the other, so the pan multiply and the mix add
// fuse into one FFMA per channel and nothing crosses lanes until all of the thread's
// voices are done.  Only then: one block reduction per 32 frames (smem columns, fixed
// order) into the block's partial row.
//
// Voice state travels through memory once per 32 frames (13 words in, 5 out per voice): 4.5 GB of DRAM traffic per
// 4 Mi x 512 launch at 3.6 TB/s.  The voices can be walked in TILES of `vpt` voices per thread, all frame chunks of a
// tile before the next tile, so that a tile (vpt = 12: 592 blocks x 128 threads x 12 voices x 72 B = 65 MB) stays in L2
// and DRAM sees every voice once per launch (0.35 GB).  Measured (option xvoice_vpt, tools/xv_time.py): vpt 8 / 12 / 16 /
// 64 = 1.357 / 1.323 / 1.310 / 1.264 ms -- every tile pays its own block reduction per chunk and the kernel is issue
// bound, not bandwidth bound, so the default is one tile (vpt 64).  The loads of the next voice -- across the chunk
// boundary too: the thread's first voice of the next chunk -- are in flight while the current one renders.
//
// The launch finishes its own mix: the last XM chunks' worth of blocks to leave (atomic
// ticket) wait for the stragglers and add the block rows of one 32-frame chunk each, in a
// fixed order, so the result is deterministic run to run; with a mix bus attached they
// push their columns to the peers instead (float sum in rank order, bus_fused.cuh).
#define XM_BLOCK 128
#define XM_CHUNK 32
#define XM_VPT 64
__device__ __forceinline__ void xv_load(XV &v, const XVoiceParams &p, uint64_t i) {
    const uint32_t *s = p.st + i; const uint32_t *r = p.prm + i;
    v.phase = __ldcg(s); v.lp = __uint_as_float(__ldcg(s + p.npad)); v.bp = __uint_as_float(__ldcg(s + 2 * p.npad));
    v.env = __uint_as_float(__ldcg(s + 3 * p.npad)); v.t = __ldcg(s + 4 * p.npad);
    v.inc = __ldcg(r); v.f = __uint_as_float(__ldcg(r + p.npad)); v.q = __uint_as_float(__ldcg(r + 2 * p.npad));
    v.att = __uint_as_float(__ldcg(r + 3 * p.npad)); v.rel = __uint_as_float(__ldcg(r + 4 * p.npad)); v.gate = __ldcg(r + 5 * p.npad);
    v.gl = __uint_as_float(__ldcg(r + 6 * p.npad)); v.gr = __uint_as_float(__ldcg(r + 7 * p.npad));
}
__device__ __forceinline__ uint32_t ld_acquire_gpu_u32(const uint32_t *p) { uint32_t v; asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }

// The launch's own final reduction (shared by both mix kernels): it starts when the last block has left its render, with the whole
// chip waiting, so it is spread wide -- the last n_fin = min(4 n_chunks, blocks) blocks to leave take a QUARTER chunk (16 of its 64
// columns, and every n_fin-th unit) each; a thread adds an eighth of the block rows of one column (four chains, the loads of 16 rows
// in flight), the eight partial sums meet in a fixed order (lane pairs, then the four warps through shared memory).  One thread
// pair per column walking all rows took ~10 us at 443 rows; this form ~3.  With a mix bus attached the finishers push their
// columns to the peers.
#define XM_FIN_UNITS 4                               // units per chunk
__host__ __device__ __forceinline__ uint32_t xm_n_fin(uint32_t n_chunks, uint32_t nb) { return XM_FIN_UNITS * n_chunks < nb ? XM_FIN_UNITS * n_chunks : nb; }
__device__ __forceinline__ void xm_finish(const XVoiceParams &p, const BusFused &bf, const uint32_t n_chunks, uint32_t &tick_s) {
    __shared__ float fin_red[XM_BLOCK / 32][16];
    const uint32_t nb = p.n_render_blocks;
    const uint32_t n_rows = nb * p.rows_per_block;               // partial rows of the launch: one per block, or one per warp (k_xvoice_mix2)
    const uint32_t n_fin = xm_n_fin(n_chunks, nb);
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) tick_s = atomicAdd(p.done, 1u);
    __syncthreads();
    const uint32_t tk = tick_s;
    if (tk < nb - n_fin) return;
    if (threadIdx.x == 0) while (ld_acquire_gpu_u32(p.done) < nb) __nanosleep(64);       // the stragglers are resident: they arrive
    __syncthreads();
    const uint32_t col16 = threadIdx.x & 15u, slice = threadIdx.x >> 4, warp = threadIdx.x >> 5;      // XM_BLOCK == 128: slices 0..7
    const uint32_t b0 = (uint32_t)((uint64_t)n_rows * slice / 8), b1 = (uint32_t)((uint64_t)n_rows * (slice + 1) / 8);
    for (uint32_t u = tk - (nb - n_fin); u < XM_FIN_UNITS * n_chunks; u += n_fin) {
        const uint32_t c = u / XM_FIN_UNITS, colc = (u % XM_FIN_UNITS) * 16u + col16;       // column of the chunk: channel, frame
        const uint64_t t0 = (uint64_t)c * XM_CHUNK;
        const uint32_t cols = p.F - t0 < XM_CHUNK ? (uint32_t)(p.F - t0) : XM_CHUNK;
        const uint32_t ch = colc / XM_CHUNK, f = colc % XM_CHUNK;
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
        if (f < cols) {
            const float *src = p.partial + (uint64_t)ch * p.F + t0 + f;
            uint32_t bq = b0;
#pragma unroll 4
            for (; bq + 4 <= b1; bq += 4) {
                s0 = __fadd_rn(s0, __ldcg(src + (uint64_t)(bq + 0) * 2 * p.F)); s1 = __fadd_rn(s1, __ldcg(src + (uint64_t)(bq + 1) * 2 * p.F));
                s2 = __fadd_rn(s2, __ldcg(src + (uint64_t)(bq + 2) * 2 * p.F)); s3 = __fadd_rn(s3, __ldcg(src + (uint64_t)(bq + 3) * 2 * p.F));
            }
            for (; bq < b1; ++bq) s0 = __fadd_rn(s0, __ldcg(src + (uint64_t)bq * 2 * p.F));
        }
        float s = __fadd_rn(__fadd_rn(s0, s1), __fadd_rn(s2, s3));
        const float o = __shfl_xor_sync(0xFFFFFFFFu, s, 16);       // slices 2w (lanes 0..15) and 2w+1 of warp w
        if ((threadIdx.x & 16u) == 0) fin_red[warp][col16] = __fadd_rn(s, o);
        __syncthreads();
        if (threadIdx.x < 16u && f < cols) {
            s = __fadd_rn(__fadd_rn(fin_red[0][col16], fin_red[1][col16]), __fadd_rn(fin_red[2][col16], fin_red[3][col16]));
            const uint64_t idx = (uint64_t)ch * p.F + t0 + f;
            if (bf.world) bus_emit_word(bf, idx, __float_as_uint(s)); else p.mix[idx] = s;
        }
        __syncthreads();
    }
    __syncthreads();
    if (threadIdx.x == 0 && atomicAdd(p.done + 1, 1u) == n_fin - 1u) { p.done[0] = 0; p.done[1] = 0; __threadfence(); }   // ready for the next launch
    if (bf.world) bus_participant_done(bf);
}

__global__ void __launch_bounds__(XM_BLOCK, 4) k_xvoice_mix(const XVoiceParams p, const BusFused bf) {
    __shared__ float red[2 * XM_CHUNK][XM_BLOCK + 1];
    __shared__ uint32_t tick_s;
    if (blockIdx.x >= p.n_render_blocks) { bus_exchange_block(bf); return; }      // pipelined bus: the previous frame block's exchange
    const uint64_t T = (uint64_t)p.n_render_blocks * XM_BLOCK;
    const uint64_t tid = (uint64_t)blockIdx.x * XM_BLOCK + threadIdx.x;
    const uint32_t n_chunks = (uint32_t)((p.F + XM_CHUNK - 1) / XM_CHUNK);
    for (uint64_t tile0 = 0; tile0 < p.n; tile0 += T * p.vpt) {
        // this thread's voices of the tile: tile0 + tid + j*T, j < nvt
        const uint64_t first = tile0 + tid;
        uint32_t nvt = 0;
        if (first < p.n) { const uint64_t left = (p.n - first + T - 1) / T; nvt = left < p.vpt ? (uint32_t)left : p.vpt; }
        XV nx = {};
        if (nvt) xv_load(nx, p, first);
        for (uint32_t c = 0; c < n_chunks; ++c) {
            const uint64_t t0 = (uint64_t)c * XM_CHUNK;
            const uint32_t cols = p.F - t0 < XM_CHUNK ? (uint32_t)(p.F - t0) : XM_CHUNK;
            float aL[XM_CHUNK], aR[XM_CHUNK];
#pragma unroll
            for (int k = 0; k < XM_CHUNK; ++k) { aL[k] = 0.f; aR[k] = 0.f; }
            for (uint32_t j = 0; j < nvt; ++j) {
                const uint64_t i = first + (uint64_t)j * T;
                XV v = nx;
                // next voice: the following one of this chunk, else the thread's first voice in the next chunk (stored earlier in
                // this chunk, same thread: program order makes the reload see it) -- unless that is this very voice
                const bool wrap = j + 1 == nvt;
                if (!wrap) xv_load(nx, p, i + T);
                else if (nvt > 1 && c + 1 < n_chunks) xv_load(nx, p, first);
                // bit k: tick k of this chunk is in the attack phase, (t + k) mod 2^32 < gate
                uint32_t amask;
                if (v.t <= 0xFFFFFFFFu - XM_CHUNK) {
                    const uint32_t rem = v.t < v.gate ? v.gate - v.t : 0u;
                    amask = rem >= 32u ? 0xFFFFFFFFu : (1u << rem) - 1u;
                } else {                                       // the frame counter wraps inside the chunk
                    amask = 0;
                    for (uint32_t k = 0; k < XM_CHUNK; ++k) amask |= (uint32_t)(v.t + k < v.gate) << k;
                }
                // whole chunk in one phase (sustained or released voices: the steady state of a mix) for every
                // lane still in the loop -> the three-instruction envelope
                // (bit patterns: +0 <= env <= 1 and rates with a clear sign bit exclude NaN and -0.0, for which the
                // extra clamp would not be an identity)
                const bool uni = (amask == 0u || amask == 0xFFFFFFFFu) && __float_as_uint(v.att) <= 0x7F800000u && __float_as_uint(v.rel) <= 0x7F800000u &&
                                 __float_as_uint(v.env) <= 0x3F800000u;
                if (cols == XM_CHUNK && __all_sync(__activemask(), uni)) {
                    const float d = amask ? v.att : -v.rel;
#pragma unroll
                    for (int k = 0; k < XM_CHUNK; ++k) {
                        const float y = xvoice_tick_uniform(v, d);
                        aL[k] = __fmaf_rn(v.gl, y, aL[k]);
                        aR[k] = __fmaf_rn(v.gr, y, aR[k]);
                    }
                } else if (cols == XM_CHUNK) {
#pragma unroll
                    for (int k = 0; k < XM_CHUNK; ++k) {
                        const float y = xvoice_tick_flag(v, (amask >> k) & 1u);
                        aL[k] = __fmaf_rn(v.gl, y, aL[k]);
                        aR[k] = __fmaf_rn(v.gr, y, aR[k]);
                    }
                } else {
#pragma unroll
                    for (int k = 0; k < XM_CHUNK; ++k) {
                        if (k < (int)cols) {
                            const float y = xvoice_tick_flag(v, (amask >> k) & 1u);
                            aL[k] = __fmaf_rn(v.gl, y, aL[k]);
                            aR[k] = __fmaf_rn(v.gr, y, aR[k]);
                        }
                    }
                }
                v.t += cols;
                uint32_t *w = p.st + i;
                __stcg(w, v.phase); __stcg(w + p.npad, __float_as_uint(v.lp)); __stcg(w + 2 * p.npad, __float_as_uint(v.bp));
                __stcg(w + 3 * p.npad, __float_as_uint(v.env)); __stcg(w + 4 * p.npad, v.t);
                if (wrap && nvt == 1) nx = v;                  // the thread's only voice stays in registers
            }
#pragma unroll
            for (int k = 0; k < XM_CHUNK; ++k) { red[k][threadIdx.x] = aL[k]; red[XM_CHUNK + k][threadIdx.x] = aR[k]; }
            __syncthreads();
            {   // column sums: two threads per column (64 rows each, 4 chains), halves combined in a fixed order
                const uint32_t col = threadIdx.x >> 1, half = threadIdx.x & 1u;
                const float *row = &red[col][half * (XM_BLOCK / 2)];
                float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll 4
                for (int j = 0; j < XM_BLOCK / 2; j += 4) {
                    s0 = __fadd_rn(s0, row[j]); s1 = __fadd_rn(s1, row[j + 1]); s2 = __fadd_rn(s2, row[j + 2]); s3 = __fadd_rn(s3, row[j + 3]);
                }
                float s = __fadd_rn(__fadd_rn(s0, s1), __fadd_rn(s2, s3));
                const float o = __shfl_xor_sync(0xFFFFFFFFu, s, 1);
                s = half ? __fadd_rn(o, s) : __fadd_rn(s, o);   // low half + high half on both lanes
                const uint32_t ch = col / XM_CHUNK, f = col % XM_CHUNK;
                if (!half && f < cols) {
                    float *dst = p.partial + ((uint64_t)blockIdx.x * 2 + ch) * p.F + t0 + f;
                    *dst = tile0 ? __fadd_rn(*dst, s) : s;       // tiles accumulate in tile order
                }
            }
            __syncthreads();
        }
    }
    xm_finish(p, bf, n_chunks, tick_s);
}

// ---- mix kernel, second generation: voice PAIRS on the packed fp32 pipe, state tiles resident in shared memory ----------
// (1) Blackwell's fma / add / mul .f32x2 (SASS FFMA2 / FADD2 / FMUL2) work on two floats in an aligned register pair: one
//     instruction slot, the FMA pipe busy for two (tools/ubench_f32x2.cu: 63 /clk/SM against 117 for FFMA, and an ALU-pipe
//     instruction issues beside it for free).  The scalar kernel is ISSUE bound (14.5 instructions per voice-sample at 67 %
//     issue, FMA pipe 45 %, profiles/r2_xvoice_mix_summary.txt): a thread now walks its voices two at a time, the SVF (4),
//     the envelope add (1) and the output multiply (1) of both voices in six packed instructions instead of twelve; every
//     lane of a packed operation is the same single IEEE rounding as the scalar one, so results stay bit-exact per voice.
//     The pipe has no operand negation in PTX, so a chunk works on -lp and -env (exact mirror images: rounding is
//     sign-symmetric; the zero cases are spelled out at the clamp) and flips them back when it stores.
// (2) The scalar kernel moves every voice's state and parameters through L2 / DRAM once per 32-frame chunk (4.4 GB per
//     4 Mi x 512 launch, 18 x the algorithmic bytes).  Here a block owns a contiguous range of voices, cuts it into tiles
//     whose STATE (5 words per voice) sits in shared memory for all the chunks of the launch, and DRAM sees the state once
//     in and once out; the parameters (read-only, 8 words) come through L1 / L2 per chunk.  Ranges are dealt in groups of
//     256 voices (one pair per thread) so that every block has 36 or 37 pair-chunks per thread and chunk at 4 Mi voices.
// Per tile and chunk the block reduces its 2 x 32 accumulators per thread through a 16 KB column buffer (left, then right)
// into its partial row; the launch's final reduction and the bus exchange are those of the first kernel (xm_finish).
#define XM2_BLOCK 128
#ifndef XM2_GMAX
#define XM2_GMAX 14                                  // groups (of 256 voices) per tile: 14 x 5 KB of state, three blocks per SM
#endif
#ifndef XM2_MINB
#define XM2_MINB 3                                   // resident blocks per SM (register cap 168)
#endif
typedef unsigned long long xv2_t;                    // {lo: voice A, hi: voice B}
__device__ __forceinline__ xv2_t xv2_pack(float lo, float hi) { xv2_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ xv2_t xv2_packu(uint32_t lo, uint32_t hi) { xv2_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi)); return r; }
__device__ __forceinline__ float xv2_lo(xv2_t v) { return __uint_as_float((uint32_t)v); }
__device__ __forceinline__ float xv2_hi(xv2_t v) { return __uint_as_float((uint32_t)(v >> 32)); }
__device__ __forceinline__ xv2_t xv2_fma(xv2_t a, xv2_t b, xv2_t c) { xv2_t r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ xv2_t xv2_add(xv2_t a, xv2_t b) { xv2_t r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ xv2_t xv2_mul(xv2_t a, xv2_t b) { xv2_t r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ xv2_t xv2_neg(xv2_t a) { return a ^ 0x8000000080000000ull; }

// explicit shared-space accesses on a 32-bit address (a generic pointer into the dynamic shared array made ptxas rebuild the shared
// window base -- S2R SR_CgaCtaId, UMOV, ULEA -- in front of every pair)
__device__ __forceinline__ uint2 xv_lds64(uint32_t a) { uint2 v; asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a)); return v; }
__device__ __forceinline__ void xv_sts64(uint32_t a, uint2 v) { asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(a), "r"(v.x), "r"(v.y) : "memory"); }

// attack mask of one voice for a chunk (bit k: tick k is in the attack phase) and whether the chunk is uniform
__device__ __forceinline__ uint32_t xv_amask(uint32_t t, uint32_t gate) {
    if (t <= 0xFFFFFFFFu - XM_CHUNK) {
        const uint32_t rem = t < gate ? gate - t : 0u;
        return rem >= 32u ? 0xFFFFFFFFu : (1u << rem) - 1u;
    }
    uint32_t m = 0;                                    // the frame counter wraps inside the chunk
    for (uint32_t k = 0; k < XM_CHUNK; ++k) m |= (uint32_t)(t + k < gate) << k;
    return m;
}

__global__ void __launch_bounds__(XM2_BLOCK, XM2_MINB) k_xvoice_mix2(const XVoiceParams p, const BusFused bf) {
    extern __shared__ __align__(16) uint32_t xm2_tile[];            // [5][256 * ng]: phase, lp, bp, env, t of the tile's voices
    __shared__ uint32_t tick_s;
    if (blockIdx.x >= p.n_render_blocks) { bus_exchange_block(bf); return; }      // pipelined bus: the previous frame block's exchange
    const uint32_t nb = p.n_render_blocks, tid = threadIdx.x;
    const uint32_t n_chunks = (uint32_t)((p.F + XM_CHUNK - 1) / XM_CHUNK);
    const uint64_t G = (p.n + 255) / 256;
    // Blocks with one group more than the others are the LOWEST block indices: the hardware deals blocks to the SMs breadth first, so the
    // uneven last round (a 512 Ki-voice shard: 276 of 443 blocks have a fifth group) is spread two blocks per SM over the SMs instead of
    // three on some and none on others -- that round is latency bound and runs faster with fewer warps per SM.
    const uint64_t g_each = G / nb, g_more = G % nb;
    const uint64_t g_lo = g_each * blockIdx.x + (blockIdx.x < g_more ? blockIdx.x : g_more), g_hi = g_lo + g_each + (blockIdx.x < g_more ? 1 : 0);
    const uint32_t kg = (uint32_t)(g_hi - g_lo), nt = (kg + XM2_GMAX - 1) / XM2_GMAX;
    if (kg == 0)                                                    // more blocks than groups: an all-zero partial row
        for (uint64_t idx = tid; idx < 2 * p.F; idx += XM2_BLOCK) p.partial[(uint64_t)blockIdx.x * 2 * p.F + idx] = 0.0f;
    const xv2_t c31 = xv2_pack(0x1p-31f, 0x1p-31f);
    for (uint32_t ti = 0; ti < nt; ++ti) {
        const uint64_t ga = g_lo + (uint64_t)kg * ti / nt, gb = g_lo + (uint64_t)kg * (ti + 1) / nt;
        const uint32_t ng = (uint32_t)(gb - ga);
        const uint64_t v0 = ga * 256;
        // ---- tile state in: [5][npad] rows -> shared memory.  A thread only ever touches the state of ITS pairs, so the tile is laid out
        // pair-major, 5 x uint2 (40 bytes) per pair: the five accesses of a pair are one base + immediate offsets (no dependent address
        // chain in front of the tick loop), 64-bit accesses at a 40-byte lane stride are conflict free per half-warp, and no barrier is
        // needed between the tile phases.
        const uint32_t tile_s = (uint32_t)__cvta_generic_to_shared(xm2_tile) + tid * 40u;     // this thread's pair 0; pair j: + j * 128 * 40
        // (asynchronous copies: the 5 x ng 8-byte pieces of a thread are all in flight at once -- through registers the groups came one
        // DRAM round trip after the other, ~1 us each, in front of the tile's first tick)
        for (uint32_t j = 0; j < ng; ++j) {
            const uint64_t gi = v0 + 2 * (tid + XM2_BLOCK * j);
#pragma unroll
            for (uint32_t w = 0; w < 5; ++w)                          // npad % 256 == 0: whole groups; [n, npad) is zero
                asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(tile_s + j * (XM2_BLOCK * 40u) + 8 * w), "l"(__cvta_generic_to_global(p.st + (uint64_t)w * p.npad + gi)) : "memory");
        }
        asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
        // (npad is a multiple of 256 for this processor and the rows are zero past n: whole groups, no bounds checks; one 64-bit base per
        // tile and a row pitch in uint2 units keep the address arithmetic of the 8 loads to a handful of instructions -- written as
        // `p.prm + w * npad + gi` with a predicate it was ~60 instructions of IMAD.WIDE / LEA.HI.X per pair and chunk)
        const uint2 *tile_prm = (const uint2 *)(p.prm + v0) + tid;
        const uint64_t row2 = p.npad >> 1;
        auto load_prm = [&](uint32_t j, uint2 (&q)[8]) {
            const uint2 *pp = tile_prm + XM2_BLOCK * j;
#pragma unroll
            for (int w = 0; w < 8; ++w) q[w] = __ldg(pp + (uint64_t)w * row2);
        };
        // a pair's five state words out of the tile; issued one pair ahead like the parameters, so that the shared-memory latency, the
        // attack masks and the path decision of pair j+1 do not sit between two tick loops (profiles/r2_xvoice_mix2_summary.txt: the
        // ~150 instructions around a 32-tick loop took 35 % of the kernel's samples at 2.5 warps per scheduler)
        auto load_st = [&](uint32_t j, uint2 (&st)[5]) {
            const uint32_t sa = tile_s + j * (XM2_BLOCK * 40u);
#pragma unroll
            for (int w = 0; w < 5; ++w) st[w] = xv_lds64(sa + 8 * w);
        };
        uint2 nq[8], nst[5];
        load_prm(0, nq);
        load_st(0, nst);
        for (uint32_t c = 0; c < n_chunks; ++c) {
            const uint64_t t0 = (uint64_t)c * XM_CHUNK;
            const uint32_t cols = p.F - t0 < XM_CHUNK ? (uint32_t)(p.F - t0) : XM_CHUNK;
            float aL[XM_CHUNK], aR[XM_CHUNK];
#pragma unroll
            for (int k = 0; k < XM_CHUNK; ++k) { aL[k] = 0.f; aR[k] = 0.f; }
#pragma unroll 1
            for (uint32_t j = 0; j < ng; ++j) {
                uint2 q[8];
#pragma unroll
                for (int w = 0; w < 8; ++w) q[w] = nq[w];
                uint2 ph = nst[0], slp = nst[1], sbp = nst[2], sen = nst[3], stt = nst[4];
                const uint32_t sp = tile_s + j * (XM2_BLOCK * 40u);
                // the next pair: j + 1, or this thread's first pair in the next chunk (its state was stored earlier in this chunk, by this
                // thread: program order) -- unless that is this very pair (ng == 1: its state stays in registers, below)
                if (j + 1 < ng) { load_prm(j + 1, nq); load_st(j + 1, nst); }
                else if (c + 1 < n_chunks) { load_prm(0, nq); if (ng > 1) load_st(0, nst); }
                const uint32_t mA = xv_amask(stt.x, q[5].x), mB = xv_amask(stt.y, q[5].y);
                // The clamped envelope e' = min(max(e + d, +0), 1), d = +attack or -release, is the two-branch envelope of the oracle
                // whenever the rates have a clear sign bit and +0 <= env <= 1 (bit patterns below; excludes NaN and -0.0): the clamp
                // that does not belong to the phase is an identity.  `sane`: true for both voices of every lane of the warp.
                const bool sane = q[3].x <= 0x7F800000u && q[3].y <= 0x7F800000u && q[4].x <= 0x7F800000u && q[4].y <= 0x7F800000u &&
                                  sen.x <= 0x3F800000u && sen.y <= 0x3F800000u;
                // `uni`: moreover the whole chunk lies in one envelope phase for every voice (sustained or released voices: the
                // steady state of a mix), so d is a chunk constant; otherwise it is selected per tick from the attack mask
                const bool uni = (mA == 0u || mA == 0xFFFFFFFFu) && (mB == 0u || mB == 0xFFFFFFFFu);
                const bool all_sane = __all_sync(0xFFFFFFFFu, sane), all_uni = __all_sync(0xFFFFFFFFu, uni);
                if (cols == XM_CHUNK && all_sane) {
                    uint32_t phA = ph.x, phB = ph.y;
                    const uint32_t incA = q[0].x, incB = q[0].y;
                    const xv2_t f2 = xv2_packu(q[1].x, q[1].y), nf2 = xv2_neg(f2), nq2 = xv2_neg(xv2_packu(q[2].x, q[2].y));
                    xv2_t nlp = xv2_neg(xv2_packu(slp.x, slp.y)), bp = xv2_packu(sbp.x, sbp.y);
                    float neA = -__uint_as_float(sen.x), neB = -__uint_as_float(sen.y);
                    const float glA = __uint_as_float(q[6].x), glB = __uint_as_float(q[6].y), grA = __uint_as_float(q[7].x), grB = __uint_as_float(q[7].y);
                    // one tick of the pair; nd = {-dA, -dB}   (XM2_EXP_*: timing experiments of tools/sweep_xmix2.sh, wrong results)
#ifdef XM2_EXP_NO_I2F
#define XM2_XI(a, b) xv2_packu(a, b)
#else
#define XM2_XI(a, b) xv2_pack(__int2float_rn((int32_t)(a)), __int2float_rn((int32_t)(b)))
#endif
#ifdef XM2_EXP_NO_ENV
#define XM2_ENV(nd)
#else
#define XM2_ENV(nd) const xv2_t sm_ = xv2_add(xv2_pack(neA, neB), nd); \
                        neA = fmaxf(fminf(xv2_lo(sm_), -0.0f), -1.0f); neB = fmaxf(fminf(xv2_hi(sm_), -0.0f), -1.0f);
#endif
#ifdef XM2_EXP_NO_MIX
#define XM2_MIX(k) aL[k & 1] = __fadd_rn(aL[k & 1], yA); aR[k & 1] = __fadd_rn(aR[k & 1], yB);
#else
#define XM2_MIX(k) aL[k] = __fmaf_rn(glA, yA, aL[k]); aR[k] = __fmaf_rn(grA, yA, aR[k]); \
                        aL[k] = __fmaf_rn(glB, yB, aL[k]); aR[k] = __fmaf_rn(grB, yB, aR[k]);
#endif
#define XM2_TICK(k, nd) { \
                        const xv2_t xi = XM2_XI(phA, phB); \
                        xv_add_alu(phA, incA); xv_add_alu(phB, incB); \
                        nlp = xv2_fma(nf2, bp, nlp);                    /* -(lp + f bp) */ \
                        xv2_t hp = xv2_fma(xi, c31, nlp);               /* x - lp */ \
                        hp = xv2_fma(nq2, bp, hp); \
                        bp = xv2_fma(f2, hp, bp); \
                        /* e' = min(max(e + d, +0), 1) mirrored: -e' = max(min(-e - d, -0), -1); a sum that is +0 where the mirror */ \
                        /* image is -0 (e + d == 0) is put right by the clamp at -0 (min(+0, -0) = -0) */ \
                        XM2_ENV(nd) \
                        const xv2_t y = xv2_mul(nlp, xv2_pack(neA, neB));   /* (-lp)(-e) = lp e */ \
                        const float yA = xv2_lo(y), yB = xv2_hi(y); \
                        XM2_MIX(k) }
                    if (all_uni) {
                        const xv2_t nd = xv2_packu(mA ? q[3].x ^ 0x80000000u : q[4].x, mB ? q[3].y ^ 0x80000000u : q[4].y);
#pragma unroll
                        for (int k = 0; k < XM_CHUNK; ++k) XM2_TICK(k, nd)
                    } else {
                        const uint32_t naA = q[3].x ^ 0x80000000u, naB = q[3].y ^ 0x80000000u;       // -attack
#pragma unroll
                        for (int k = 0; k < XM_CHUNK; ++k) {
                            const xv2_t nd = xv2_packu((mA >> k) & 1u ? naA : q[4].x, (mB >> k) & 1u ? naB : q[4].y);
                            XM2_TICK(k, nd)
                        }
                    }
#undef XM2_TICK
#undef XM2_XI
#undef XM2_ENV
#undef XM2_MIX
                    const xv2_t lp = xv2_neg(nlp);
                    ph = make_uint2(phA, phB);
                    slp = make_uint2(__float_as_uint(xv2_lo(lp)), __float_as_uint(xv2_hi(lp)));
                    sbp = make_uint2(__float_as_uint(xv2_lo(bp)), __float_as_uint(xv2_hi(bp)));
                    sen = make_uint2(__float_as_uint(-neA), __float_as_uint(-neB));
                } else {
                    // mixed envelope phases (or a short last chunk): the scalar tick of the first kernel, voice A then voice B
#pragma unroll 1
                    for (int h = 0; h < 2; ++h) {
                        XV v;
                        v.phase = h ? ph.y : ph.x; v.lp = __uint_as_float(h ? slp.y : slp.x); v.bp = __uint_as_float(h ? sbp.y : sbp.x);
                        v.env = __uint_as_float(h ? sen.y : sen.x); v.t = 0; v.gate = 0;
                        v.inc = h ? q[0].y : q[0].x; v.f = __uint_as_float(h ? q[1].y : q[1].x); v.q = __uint_as_float(h ? q[2].y : q[2].x);
                        v.att = __uint_as_float(h ? q[3].y : q[3].x); v.rel = __uint_as_float(h ? q[4].y : q[4].x);
                        v.gl = __uint_as_float(h ? q[6].y : q[6].x); v.gr = __uint_as_float(h ? q[7].y : q[7].x);
                        const uint32_t am = h ? mB : mA;
#pragma unroll
                        for (int k = 0; k < XM_CHUNK; ++k) {
                            if (k < (int)cols) {
                                const float y = xvoice_tick_flag(v, (am >> k) & 1u);
                                aL[k] = __fmaf_rn(v.gl, y, aL[k]);
                                aR[k] = __fmaf_rn(v.gr, y, aR[k]);
                            }
                        }
                        if (h) { ph.y = v.phase; slp.y = __float_as_uint(v.lp); sbp.y = __float_as_uint(v.bp); sen.y = __float_as_uint(v.env); }
                        else { ph.x = v.phase; slp.x = __float_as_uint(v.lp); sbp.x = __float_as_uint(v.bp); sen.x = __float_as_uint(v.env); }
                    }
                }
                stt.x += cols; stt.y += cols;
                xv_sts64(sp, ph); xv_sts64(sp + 8, slp); xv_sts64(sp + 16, sbp); xv_sts64(sp + 24, sen); xv_sts64(sp + 32, stt);
                if (ng == 1) { nst[0] = ph; nst[1] = slp; nst[2] = sbp; nst[3] = sen; nst[4] = stt; }
            }
            // ---- reduction of the chunk, PER WARP and without a block barrier: a butterfly over the lanes that transposes while it adds
            // (stage `st`: a lane keeps the half of its values whose index has bit `st` equal to its own lane bit and receives the partner's
            // copy of that half) leaves lane l with frame l's sum over the warp's 32 lanes -- a fixed order, deterministic.  62 shuffles for
            // the 2 x 32 accumulators, no shared memory; the warps of a block drift apart freely between tile boundaries.  (A column
            // buffer in shared memory with four __syncthreads per chunk was 17 % of the kernel's stall samples for 4 % of its instructions.)
            {
                const uint32_t lane = tid & 31u, warp = tid >> 5;
#pragma unroll
                for (int st = 16; st >= 1; st >>= 1) {
                    const bool up = (lane & st) != 0;
#pragma unroll
                    for (int q = 0; q < st; ++q) {
                        const float sendL = up ? aL[q] : aL[q + st], keepL = up ? aL[q + st] : aL[q];
                        const float sendR = up ? aR[q] : aR[q + st], keepR = up ? aR[q + st] : aR[q];
                        aL[q] = __fadd_rn(keepL, __shfl_xor_sync(0xFFFFFFFFu, sendL, st));
                        aR[q] = __fadd_rn(keepR, __shfl_xor_sync(0xFFFFFFFFu, sendR, st));
                    }
                }
                if (lane < cols) {
                    float *dst = p.partial_w + ((uint64_t)(blockIdx.x * (XM2_BLOCK / 32) + warp) * 2) * p.F + t0 + lane;
                    dst[0] = ti ? __fadd_rn(dst[0], aL[0]) : aL[0];           // tiles accumulate in tile order
                    dst[p.F] = ti ? __fadd_rn(dst[p.F], aR[0]) : aR[0];
                }
            }
        }
        // ---- tile state out
        for (uint32_t j = 0; j < ng; ++j) {
            const uint64_t gi = v0 + 2 * (tid + XM2_BLOCK * j);
#pragma unroll
            for (uint32_t w = 0; w < 5; ++w) {
                const uint2 val = xv_lds64(tile_s + j * (XM2_BLOCK * 40u) + 8 * w);
                uint32_t *dst = p.st + (uint64_t)w * p.npad + gi;
                if (gi + 1 < p.n) __stcs((uint2 *)dst, val);
                else if (gi < p.n) dst[0] = val.x;
            }
        }
    }
    // the block's four warp rows -> its one row for the launch's final reduction (which would otherwise walk four times as many rows
    // at the tail of the launch, with the whole chip waiting: +30 us on a 190 us shard of an 8-GPU render), warps in a fixed order
    if (kg) {
        __syncthreads();
        const float *w0 = p.partial_w + (uint64_t)blockIdx.x * (XM2_BLOCK / 32) * 2 * p.F;
        for (uint64_t idx = tid; idx < 2 * p.F; idx += XM2_BLOCK) {
            float sm = __ldcg(w0 + idx);
#pragma unroll
            for (int r = 1; r < XM2_BLOCK / 32; ++r) sm = __fadd_rn(sm, __ldcg(w0 + (uint64_t)r * 2 * p.F + idx));
            p.partial[(uint64_t)blockIdx.x * 2 * p.F + idx] = sm;
        }
    }
    xm_finish(p, bf, n_chunks, tick_s);
}

// mix[c][t] = SUM_b partial[b][c][t], fixed order, 4 independent chains
__global__ void k_xvoice_final(const float *partial, float *mix, uint64_t n_blocks, uint64_t cols) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= cols) return;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    uint64_t b = 0;
    for (; b + 4 <= n_blocks; b += 4) {
        s0 = __fadd_rn(s0, partial[(b + 0) * cols + i]); s1 = __fadd_rn(s1, partial[(b + 1) * cols + i]);
        s2 = __fadd_rn(s2, partial[(b + 2) * cols + i]); s3 = __fadd_rn(s3, partial[(b + 3) * cols + i]);
    }
    for (; b < n_blocks; ++b) s0 = __fadd_rn(s0, partial[b * cols + i]);
    mix[i] = __fadd_rn(__fadd_rn(s0, s1), __fadd_rn(s2, s3));
}

// ---------------------------------------------------------------------------
// Time-parallel raw render (C5: few thousand variants x hundreds of thousands of
// frames, 8 B of output per variant-frame -> HBM-write bound).  A thread per variant
// would leave the chip idle (2,048 threads), so the time axis is cut into C chunks of
// L frames and every (variant, chunk) pair is a thread.  What a chunk needs at its
// first frame:
//   phase  closed form, phase0 + c*L*inc mod 2^32 (acc, cproc.h:141)         exact
//   t      t0 + c*L                                                           exact
//   env    piecewise linear with clamps; walked in time by one thread per variant,
//          skipping fixed points (e == 1 in attack, e == 0 in release,
//          e + rate == e), same float operations                              exact
//   lp,bp  the SVF is linear time-invariant: s' = A s + B x.  Pass 1 (k_sweep_zsr)
//          runs the recurrence from zero state over each chunk in fp64 (zero-state
//          response z_c); pass 2 (k_sweep_scan) forms A^L by squaring and walks
//          s_{c+1} = A^L s_c + z_c in fp64 -- the associative scan of the affine
//          maps, sequential over the C chunks of a variant because C is small.
// Pass 3 (k_sweep_render) then runs the ordinary bit-exact float tick from each start
// state.  The start states come from exact arithmetic rather than from the float
// trajectory, so the raw output is not bit for bit the sequential path's: per voice it is
// within 1e-5 of the voice's own peak of the fp64 filter, or within twice the sequential
// render's own error where that is larger (measured on a B200: <= 1.3e-6, slow and
// resonant filters included; tests/test_gpu_float_ref.py).  phase, t and env stay bit-exact.
struct SweepParams {
    XVoiceParams x;
    uint64_t L, C;
    uint64_t i0, i1;         // variants [i0, i1) of this launch (variant groups are pipelined over two streams)
    uint64_t zoff, zi1;      // fused render: thread (i, c) also runs the zero-state pass of variant i + zoff (< zi1)
    double2 *z;              // [n][C-1] zero-state response of chunk c
    float2 *s0;              // [C][n]   (lp, bp) at the first frame of chunk c
    float *e0;               // [C][n]   env at the first frame of chunk c
    uint32_t *ph0, *t0;      // [n] snapshot of the initial phase / frame counter
    uint32_t *cst;           // [n] first chunk from which the envelope never changes again (C if none)
    float *est;              // [n] that final envelope value
    double *tab;             // [10 + 6 nlev][n] per-variant segment maps of the closed-form zero-state pass (k_sweep_pre)
    int nlev, closed;
};

// One fp64 tick of the zero-state recurrence on the integer-valued input.
//   lp' = lp + f bp;  bp' = bp + f (x - lp' - q bp), with the x - q bp term off the lp -> bp chain
__device__ __forceinline__ void zsr_tick(uint32_t &phase, uint32_t inc, double f, double nq, double &lp, double &bp) {
    const double x = (double)__int2float_rn((int32_t)phase);              // the float path's x * 2^31, exactly
    phase += inc;
    const double u = fma(nq, bp, x);
    lp = fma(f, bp, lp);
    bp = fma(f, u - lp, bp);
}

// ---- closed-form zero-state response ------------------------------------------------------------
// The SVF tick is s' = A s + b x with A = [[1, f], [-f, 1 - f q - f^2]], b = (0, f), and the input is
// a sawtooth: x_t = x0 + t inc - 2^32 w_t, w_t = number of times the signed phase has wrapped up to
// tick t.  By linearity the zero-state response after L ticks is
//     s_L = P_L x0 + Q_L inc - 2^32 y_L,
//     P_m = sum_{t<m} A^(m-1-t) b        (response to a unit step),
//     Q_m = sum_{t<m} t A^(m-1-t) b      (response to a unit ramp),
// and y is the response to the staircase w_t: constant between wraps, so it advances one whole gap at
// a time, y <- A^g y + j P_g.  Consecutive wraps are k or k+1 ticks apart (k = floor(2^32 / inc)); a
// remainder walk in integer arithmetic says which.  The last stretch up to L has an arbitrary length
// e <= L and is applied from the per-variant table of the maps of 2^i ticks, one step per set bit of e.
// k_sweep_pre builds, per variant: (P_L, Q_L), (A^k, P_k) when k < L, and (A^(2^i), P_(2^i)).
// Cost per (variant, chunk): ~12 fp64 operations per WRAP instead of 4 per TICK (a 4 kHz voice wraps
// every 11 ticks, a 32 Hz voice every 1500), and the tick's int -> float rounding of x (|err| <= 2^-25
// of full scale, zero mean) is replaced by the exact integer: -150 dB, far inside the 120 dB bound.
struct ZSeg { double a11, a12, a21, a22, p1, p2, q1, q2, m; };
// `x` ticks, then `y` ticks
__device__ __forceinline__ ZSeg zseg_then(const ZSeg &x, const ZSeg &y) {
    ZSeg r;
    r.a11 = y.a11 * x.a11 + y.a12 * x.a21; r.a12 = y.a11 * x.a12 + y.a12 * x.a22;
    r.a21 = y.a21 * x.a11 + y.a22 * x.a21; r.a22 = y.a21 * x.a12 + y.a22 * x.a22;
    r.p1 = y.a11 * x.p1 + y.a12 * x.p2 + y.p1; r.p2 = y.a21 * x.p1 + y.a22 * x.p2 + y.p2;
    r.q1 = y.a11 * x.q1 + y.a12 * x.q2 + x.m * y.p1 + y.q1; r.q2 = y.a21 * x.q1 + y.a22 * x.q2 + x.m * y.p2 + y.q2;
    r.m = x.m + y.m;
    return r;
}
// k = floor(2^32 / inc) and rho = 2^32 - k inc, inc > 0
__device__ __forceinline__ void wrap_period(uint32_t inc, uint64_t &k, uint32_t &rho) {
    k = 0xFFFFFFFFu / inc; rho = 0u - (uint32_t)k * inc;
    if (rho == inc) { ++k; rho = 0; }
}
#define ZT_FIXED 10
__global__ void __launch_bounds__(128) k_sweep_pre(const SweepParams p) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, n = p.x.n;
    if (i >= n) return;
    const uint32_t inc = p.x.prm[i];
    const double f = (double)__uint_as_float(p.x.prm[p.x.npad + i]), q = (double)__uint_as_float(p.x.prm[2 * p.x.npad + i]);
    ZSeg lev = {1.0, f, -f, 1.0 - f * q - f * f, 0.0, f, 0.0, 0.0, 1.0};
    const ZSeg id = {1.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    ZSeg sl = id, sk = id;
    uint64_t k = 0; uint32_t rho = 0;
    if (inc) wrap_period(inc, k, rho);
    const bool kuse = inc && k < p.L;
    double *t = p.tab + i;
    for (int l = 0; l < p.nlev; ++l) {
        double *d = t + (uint64_t)(ZT_FIXED + 6 * l) * n;
        d[0] = lev.a11; d[n] = lev.a12; d[2 * n] = lev.a21; d[3 * n] = lev.a22; d[4 * n] = lev.p1; d[5 * n] = lev.p2;
        if ((p.L >> l) & 1) sl = zseg_then(sl, lev);
        if (kuse && ((k >> l) & 1)) sk = zseg_then(sk, lev);
        lev = zseg_then(lev, lev);
    }
    t[0] = sl.p1; t[n] = sl.p2; t[2 * n] = sl.q1; t[3 * n] = sl.q2;
    t[4 * n] = sk.a11; t[5 * n] = sk.a12; t[6 * n] = sk.a21; t[7 * n] = sk.a22; t[8 * n] = sk.p1; t[9 * n] = sk.p2;
}

// zero-state response of full chunk c of variant i, scaled like the ticked pass
__device__ __noinline__ double2 zsr_closed(const SweepParams &p, uint64_t i, uint64_t c) {
    const uint64_t n = p.x.n, L = p.L;
    const uint32_t inc = __ldg(p.x.prm + i);
    const uint32_t ph = p.x.st[i] + (uint32_t)(c * L) * inc;
    const uint32_t u0 = ph ^ 0x80000000u;                       // signed phase + 2^31: wraps when it passes 2^32
    const uint32_t W = (uint32_t)(((uint64_t)u0 + (L - 1) * (uint64_t)inc) >> 32);
    const double *t = p.tab + i;
    double y1 = 0.0, y2 = 0.0;
    if (W) {
        uint64_t at = (uint64_t)(~u0 / inc) + 1;               // tick of the first wrap: smallest t with u0 + t inc >= 2^32
        if (W > 1) {
            uint32_t r = u0 + (uint32_t)at * inc;              // remainder just after a wrap, in [0, inc)
            uint64_t k; uint32_t rho;
            wrap_period(inc, k, rho);
            const double k11 = t[4 * n], k12 = t[5 * n], k21 = t[6 * n], k22 = t[7 * n], pk1 = t[8 * n], pk2 = t[9 * n];
            const double *a = t + (uint64_t)ZT_FIXED * n;        // one tick
            const double a12 = a[n], a21 = a[2 * n], a22 = a[3 * n], b2 = a[5 * n];
            for (uint32_t j = 1; j < W; ++j) {
                const double w = (double)j;
                const double n1 = fma(k11, y1, fma(k12, y2, w * pk1)), n2 = fma(k21, y1, fma(k22, y2, w * pk2));
                y1 = n1; y2 = n2; at += k;
                if (r >= rho) r -= rho;
                else {                                           // k + 1 ticks to the next wrap
                    r = r - rho + inc; at += 1;
                    const double m1 = fma(a12, y2, y1), m2 = fma(a21, y1, fma(a22, y2, w * b2));
                    y1 = m1; y2 = m2;
                }
            }
        }
        const double w = (double)W;
        const double *d = t + (uint64_t)ZT_FIXED * n;
        for (uint64_t e = L - at; e; e >>= 1, d += 6 * n) {
            if (e & 1) {
                const double n1 = fma(d[0], y1, fma(d[n], y2, w * d[4 * n])), n2 = fma(d[2 * n], y1, fma(d[3 * n], y2, w * d[5 * n]));
                y1 = n1; y2 = n2;
            }
        }
    }
    const double x0 = (double)(int32_t)ph, di = (double)inc;
    const double lp = fma(t[0], x0, fma(t[2 * n], di, -4294967296.0 * y1)), bp = fma(t[n], x0, fma(t[3 * n], di, -4294967296.0 * y2));
    return make_double2(lp * 0x1p-31, bp * 0x1p-31);
}

// Closed form, one thread per (variant, chunk) with the LANES OVER THE CHUNKS of one variant: every
// lane of a warp has the same increment, hence the same number of wraps (+-1) and the same table rows
// (broadcast loads) -- no divergence, where lanes over variants pay for the highest note of the 32.
__global__ void __launch_bounds__(128) k_sweep_zsr_closed(const SweepParams p, uint32_t blocks_per_variant) {
    const uint64_t i = p.i0 + blockIdx.x / blocks_per_variant;
    const uint64_t c = (uint64_t)(blockIdx.x % blocks_per_variant) * 128 + threadIdx.x;
    if (c + 1 >= p.C) return;
    p.z[i * (p.C - 1) + c] = zsr_closed(p, i, c);
}

// Zero-state response of every full chunk, fp64.  The SVF is linear, so the recurrence is
// run on the integer-valued input X = (float)(int)phase (what the float path multiplies
// by 2^-31) and the result is scaled by 2^-31 once: one DP multiply less per tick.
__global__ void __launch_bounds__(128) k_sweep_zsr(const SweepParams p) {
    const uint64_t i = p.i0 + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t c = blockIdx.y;
    if (i >= p.i1) return;
    const uint32_t inc = __ldg(p.x.prm + i);
    const double f = (double)__uint_as_float(__ldg(p.x.prm + p.x.npad + i));
    const double nq = -(double)__uint_as_float(__ldg(p.x.prm + 2 * p.x.npad + i));
    uint32_t phase = p.x.st[i] + (uint32_t)(c * p.L) * inc;
    double lp = 0.0, bp = 0.0;
#pragma unroll 4
    for (uint64_t k = 0; k < p.L; ++k) {                        // chunks 0..C-2 are full
        zsr_tick(phase, inc, f, nq, lp, bp);
    }
    p.z[i * (p.C - 1) + c] = make_double2(lp * 0x1p-31, bp * 0x1p-31);
}

// env after `count` more ticks, same operations as xvoice_tick, fixed points skipped
__device__ __forceinline__ void env_advance(float &e, uint32_t &t, uint32_t gate, float att, float rel, uint64_t count) {
    while (count) {
        if (t < gate) {
            float n = __fadd_rn(e, att); if (n > 1.0f) n = 1.0f;
            if (n == e) { const uint64_t left = gate - t, skip = left < count ? left : count; t += (uint32_t)skip; count -= skip; }
            else { e = n; t += 1; count -= 1; }
        } else {
            float n = __fsub_rn(e, rel); if (n < 0.0f) n = 0.0f;
            if (n == e) { const uint64_t left = 0x100000000ull - t, skip = left < count ? left : count; t += (uint32_t)skip; count -= skip; }   // up to the counter wrap
            else { e = n; t += 1; count -= 1; }
        }
    }
}

// Envelope and counters at the chunk starts: one thread per variant walks time (the
// envelope is piecewise linear with clamps, same float operations as xvoice_tick).  The
// walk stops at the first chunk start where the envelope sits on a fixed point that
// nothing can leave before the render ends (release: e - rel == e or clamped at 0, no
// counter wrap ahead; attack: e + att == e or clamped at 1, gate beyond the end): from
// chunk cst[i] on every chunk starts with est[i] and the render kernel needs no table.
__global__ void __launch_bounds__(128) k_sweep_env(const SweepParams p) {
    const uint64_t i = p.i0 + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.i1) return;
    const uint64_t n = p.x.n, npad = p.x.npad;
    float e = __uint_as_float(p.x.st[3 * npad + i]);
    uint32_t t = p.x.st[4 * npad + i];
    const uint32_t gate = p.x.prm[5 * npad + i];
    const float att = __uint_as_float(p.x.prm[3 * npad + i]), rel = __uint_as_float(p.x.prm[4 * npad + i]);
    p.ph0[i] = p.x.st[i]; p.t0[i] = t;
    uint64_t c = 0;
    for (; c < p.C; ++c) {
        const uint64_t remaining = p.x.F - c * p.L;
        bool fixed;
        if (t < gate) { float nx = __fadd_rn(e, att); if (nx > 1.0f) nx = 1.0f; fixed = nx == e && (uint64_t)(gate - t) >= remaining; }
        else { float nx = __fsub_rn(e, rel); if (nx < 0.0f) nx = 0.0f; fixed = nx == e && (uint64_t)t + remaining <= 0x100000000ull; }
        if (fixed) break;
        p.e0[c * n + i] = e;
        if (c + 1 < p.C) env_advance(e, t, gate, att, rel, p.L);
    }
    p.cst[i] = (uint32_t)c; p.est[i] = e;
}

// Filter state at every chunk start: the associative scan of the affine maps
// s -> A^L s + z_c over the chunk axis, one warp per variant.  Lane l owns a run of
// consecutive chunks: it composes its run into one map (P, w), the warp scans the 32
// maps (Kogge-Stone over shuffles, 2x2 fp64 matrices), and the lane walks its run again
// from its start state writing s0[c].  The z loads of a lane are independent, so they
// are all in flight at once (the former per-variant loop paid one L2 round trip per
// chunk).
struct Aff { double p11, p12, p21, p22, w1, w2; };
__device__ __forceinline__ double shfl_up_d(double v, int d) { return __shfl_up_sync(0xFFFFFFFFu, v, d); }
#define SCAN_WARPS 4
__global__ void __launch_bounds__(SCAN_WARPS * 32) k_sweep_scan(const SweepParams p) {
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t i = p.i0 + (uint64_t)blockIdx.x * SCAN_WARPS + (threadIdx.x >> 5);
    if (i >= p.i1) return;                                   // whole warp
    const uint64_t n = p.x.n, npad = p.x.npad;
    const double f = (double)__uint_as_float(p.x.prm[npad + i]), q = (double)__uint_as_float(p.x.prm[2 * npad + i]);
    // one tick: lp' = lp + f bp;  bp' = -f lp + (1 - f q - f^2) bp + f x
    double a11 = 1.0, a12 = f, a21 = -f, a22 = 1.0 - f * q - f * f;
    double m11 = 1.0, m12 = 0.0, m21 = 0.0, m22 = 1.0;            // M = A^L by squaring
    for (uint64_t e = p.L; e; e >>= 1) {
        if (e & 1) {
            const double t11 = m11 * a11 + m12 * a21, t12 = m11 * a12 + m12 * a22, t21 = m21 * a11 + m22 * a21, t22 = m21 * a12 + m22 * a22;
            m11 = t11; m12 = t12; m21 = t21; m22 = t22;
        }
        const double t11 = a11 * a11 + a12 * a21, t12 = a11 * a12 + a12 * a22, t21 = a21 * a11 + a22 * a21, t22 = a21 * a12 + a22 * a22;
        a11 = t11; a12 = t12; a21 = t21; a22 = t22;
    }
    // lane l: chunks [c0, c1); the map of chunk c exists for c < C-1
    const uint64_t K = (p.C + 31) / 32;
    const uint64_t c0 = lane * K < p.C ? lane * K : p.C, c1 = c0 + K < p.C ? c0 + K : p.C;
    Aff t = {1.0, 0.0, 0.0, 1.0, 0.0, 0.0};
    for (uint64_t c = c0; c < c1 && c + 1 < p.C; ++c) {
        const double2 z = p.z[i * (p.C - 1) + c];
        const double w1 = m11 * t.w1 + m12 * t.w2 + z.x, w2 = m21 * t.w1 + m22 * t.w2 + z.y;
        const double p11 = m11 * t.p11 + m12 * t.p21, p12 = m11 * t.p12 + m12 * t.p22;
        const double p21 = m21 * t.p11 + m22 * t.p21, p22 = m21 * t.p12 + m22 * t.p22;
        t.w1 = w1; t.w2 = w2; t.p11 = p11; t.p12 = p12; t.p21 = p21; t.p22 = p22;
    }
    // inclusive scan: t_l <- t_l o t_{l-1} o ... o t_0  (later map applied after the earlier)
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        Aff u;
        u.p11 = shfl_up_d(t.p11, d); u.p12 = shfl_up_d(t.p12, d); u.p21 = shfl_up_d(t.p21, d); u.p22 = shfl_up_d(t.p22, d);
        u.w1 = shfl_up_d(t.w1, d); u.w2 = shfl_up_d(t.w2, d);
        if ((int)lane >= d) {
            const double w1 = t.p11 * u.w1 + t.p12 * u.w2 + t.w1, w2 = t.p21 * u.w1 + t.p22 * u.w2 + t.w2;
            const double p11 = t.p11 * u.p11 + t.p12 * u.p21, p12 = t.p11 * u.p12 + t.p12 * u.p22;
            const double p21 = t.p21 * u.p11 + t.p22 * u.p21, p22 = t.p21 * u.p12 + t.p22 * u.p22;
            t.w1 = w1; t.w2 = w2; t.p11 = p11; t.p12 = p12; t.p21 = p21; t.p22 = p22;
        }
    }
    // exclusive prefix applied to the initial state
    Aff e;
    e.p11 = shfl_up_d(t.p11, 1); e.p12 = shfl_up_d(t.p12, 1); e.p21 = shfl_up_d(t.p21, 1); e.p22 = shfl_up_d(t.p22, 1);
    e.w1 = shfl_up_d(t.w1, 1); e.w2 = shfl_up_d(t.w2, 1);
    const double lp0 = (double)__uint_as_float(p.x.st[npad + i]), bp0 = (double)__uint_as_float(p.x.st[2 * npad + i]);
    double lp = lp0, bp = bp0;
    if (lane) { lp = e.p11 * lp0 + e.p12 * bp0 + e.w1; bp = e.p21 * lp0 + e.p22 * bp0 + e.w2; }
    for (uint64_t c = c0; c < c1; ++c) {
        p.s0[c * n + i] = make_float2((float)lp, (float)bp);
        if (c + 1 < p.C) {
            const double2 z = p.z[i * (p.C - 1) + c];
            const double nl = m11 * lp + m12 * bp + z.x, nb = m21 * lp + m22 * bp + z.y;
            lp = nl; bp = nb;
        }
    }
}

// ZSR: the thread also runs the fp64 zero-state pass of chunk c of variant i + zoff (a
// variant of the group two renders ahead).  The render is HBM-write bound and leaves
// ~40% of the issue slots and the whole DP pipe idle; the zero-state pass is pure
// arithmetic, so inside the same instruction stream it is hidden behind the stores.
template <bool TILED, int ZSR>   // ZSR 1: ticked zero-state pass of a later group beside the render (xvoice_closed = 0)
__global__ void __launch_bounds__(XV_BLOCK) k_sweep_render(const SweepParams p) {
    constexpr int PT = 32;                               // PLANAR: frames staged per pass (256-byte runs per stream; 128-byte runs cost 20% of the bandwidth)
    __shared__ __align__(16) float2 tile[TILED ? 1 : XV_WARPS][TILED ? 1 : 32][TILED ? 1 : PT + 1];   // [warp][stream][frame]
    const uint64_t i = p.i0 + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t c = blockIdx.y, n = p.x.n, npad = p.x.npad, F = p.x.F;
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool mine = i < p.i1;
    const uint64_t f0 = c * p.L, f1 = f0 + p.L < F ? f0 + p.L : F;
    XV v = {};
    if (mine) {
        const uint32_t *r = p.x.prm + i;
        v.inc = r[0]; v.f = __uint_as_float(r[npad]); v.q = __uint_as_float(r[2 * npad]);
        v.att = __uint_as_float(r[3 * npad]); v.rel = __uint_as_float(r[4 * npad]); v.gate = r[5 * npad];
        v.gl = __uint_as_float(r[6 * npad]); v.gr = __uint_as_float(r[7 * npad]);
        v.phase = p.ph0[i] + (uint32_t)f0 * v.inc;
        v.t = p.t0[i] + (uint32_t)f0;
        const float2 s = p.s0[c * n + i];
        v.lp = s.x; v.bp = s.y; v.env = c >= p.cst[i] ? p.est[i] : p.e0[c * n + i];
    }
    // zero-state duty: chunk c of variant j (chunks 0..C-2 are full, the last one needs no response)
    const uint64_t j = i + p.zoff;
    const bool zmine = ZSR != 0 && mine && j < p.zi1 && c + 1 < p.C;
    uint32_t zph = 0, zinc = 0;
    double zf = 0.0, znq = 0.0, zlp = 0.0, zbp = 0.0;
    if (zmine) {
        zinc = __ldg(p.x.prm + j);
        zf = (double)__uint_as_float(__ldg(p.x.prm + npad + j));
        znq = -(double)__uint_as_float(__ldg(p.x.prm + 2 * npad + j));
        zph = p.x.st[j] + (uint32_t)f0 * zinc;
    }
    if (TILED) {                                         // [F/2][inst][2][2]: 16 B per lane, 512 B per warp
        for (uint64_t t = f0; t < f1; t += 2) {
            const float y0 = xvoice_tick(v);
            const float l0 = __fmul_rn(v.gl, y0), r0 = __fmul_rn(v.gr, y0);
            const float y1 = xvoice_tick(v);
            const float l1 = __fmul_rn(v.gl, y1), r1 = __fmul_rn(v.gr, y1);
            if (ZSR == 1) { zsr_tick(zph, zinc, zf, znq, zlp, zbp); zsr_tick(zph, zinc, zf, znq, zlp, zbp); }   // L is even
            if (mine) st_v4_stream(p.x.raw + (((t >> 1) * n + i) << 2),
                                   make_uint4(__float_as_uint(l0), __float_as_uint(r0), __float_as_uint(l1), __float_as_uint(r1)));
        }
    } else {                                             // [inst][F][2]: PT frames staged per warp, rows written as PT*8 B runs
        const uint64_t iw = i - lane;                    // first stream of this warp
        for (uint64_t t = f0; t < f1; t += PT) {
            const uint32_t cols = f1 - t < PT ? (uint32_t)(f1 - t) : PT;
            for (uint32_t k = 0; k < cols; ++k) {
                const float y = xvoice_tick(v);
                tile[warp][lane][k] = make_float2(__fmul_rn(v.gl, y), __fmul_rn(v.gr, y));
                if (ZSR == 1) zsr_tick(zph, zinc, zf, znq, zlp, zbp);
            }
            __syncwarp();
            // PT/2 lanes x 16 B cover the PT frames of one stream; a warp instruction writes 64/PT streams
            constexpr uint32_t LPS = PT / 2, SPI = 32 / LPS;
            const uint32_t sub = lane / LPS, fp = (lane % LPS) * 2;
#pragma unroll 4
            for (uint32_t jj = 0; jj < 32; jj += SPI) {
                const uint32_t sidx = jj + sub;
                if (iw + sidx < p.i1) {
                    float *dst = p.x.raw + (((iw + sidx) * F + t + fp) << 1);
                    if (fp + 1 < cols) {
                        const float2 a = tile[warp][sidx][fp], b2 = tile[warp][sidx][fp + 1];
                        if ((((uintptr_t)dst) & 15) == 0) st_v4_stream(dst, make_uint4(__float_as_uint(a.x), __float_as_uint(a.y), __float_as_uint(b2.x), __float_as_uint(b2.y)));
                        else { *reinterpret_cast<float2 *>(dst) = a; *reinterpret_cast<float2 *>(dst + 2) = b2; }
                    } else if (fp < cols) *reinterpret_cast<float2 *>(dst) = tile[warp][sidx][fp];
                }
            }
            __syncwarp();
        }
    }
    if (zmine) p.z[j * (p.C - 1) + c] = make_double2(zlp * 0x1p-31, zbp * 0x1p-31);
    if (mine && c == p.C - 1) {                          // the last chunk leaves the voice state
        uint32_t *s = p.x.st + i;
        s[0] = v.phase; s[npad] = __float_as_uint(v.lp); s[2 * npad] = __float_as_uint(v.bp);
        s[3 * npad] = __float_as_uint(v.env); s[4 * npad] = v.t;
    }
}

// Variant groups are pipelined with a look-ahead of two: the render of group g (HBM-write
// bound, main stream) also computes the zero-state responses of group g+2; the scan of
// group g+2 (tiny) then runs on the auxiliary high-priority stream beside the render of
// group g+1.  Only the zero-state passes of the first two groups run as kernels of their
// own.  With fewer than three groups the pre-passes simply precede the render.
static int launch_xvoice_scan(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io, uint64_t L, uint64_t groups) {
    cproc_cuda_ctx *ctx = b->ctx;
    const uint64_t n = b->n, C = ceil_div_u64(F, L);
    const size_t bz = sizeof(double2) * (C - 1) * n, bs = sizeof(float2) * C * n, be = sizeof(float) * C * n, bw = sizeof(uint32_t) * n;
    int nlev = 0;
    while ((L >> nlev) != 0) ++nlev;
    const size_t bt = sizeof(double) * n * (ZT_FIXED + 6 * (size_t)nlev);
    const size_t need = bz + bs + be + 4 * bw + bt + 128;
    if (b->cap_scratch < need) {
        if (b->d_scratch) cudaFree(b->d_scratch);
        b->d_scratch = nullptr; b->cap_scratch = 0;
        CK(ctx, cudaMalloc(&b->d_scratch, need));
        b->cap_scratch = need;
    }
    SweepParams p;
    p.x.st = b->d_state; p.x.prm = b->d_param; p.x.npad = b->npad; p.x.n = n; p.x.F = F;
    p.x.raw = (float *)io->out; p.x.layout = io->layout; p.x.partial = nullptr;
    p.L = L; p.C = C; p.zoff = 0; p.zi1 = 0;
    uint8_t *w = (uint8_t *)b->d_scratch;
    p.z = (double2 *)w; w += (bz + 15) & ~(size_t)15;
    p.s0 = (float2 *)w; w += (bs + 15) & ~(size_t)15;
    p.e0 = (float *)w; w += (be + 15) & ~(size_t)15;
    p.ph0 = (uint32_t *)w; w += (bw + 15) & ~(size_t)15;
    p.t0 = (uint32_t *)w; w += (bw + 15) & ~(size_t)15;
    p.cst = (uint32_t *)w; w += (bw + 15) & ~(size_t)15;
    p.est = (float *)w; w += (bw + 15) & ~(size_t)15;
    p.tab = (double *)w; p.nlev = nlev; p.closed = ctx->xvoice_closed;
    if (groups > 8) groups = 8;
    if (groups < 1) groups = 1;
    const uint64_t per = ceil_div_u64(ceil_div_u64(n, groups), 128) * 128;
    groups = ceil_div_u64(n, per);
    const bool piped = groups >= (ctx->xvoice_closed ? 2 : 3) && C > 1;
    // closed-form zero-state pass: cheap enough to stay a kernel of its own; for every group it runs on
    // the auxiliary stream (with its scan) beside the renders of the groups before it
    const bool ahead = piped && ctx->xvoice_closed;
    if (piped && !ctx->aux_stream) {
        int lo = 0, hi = 0;
        CK(ctx, cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CK(ctx, cudaStreamCreateWithPriority(&ctx->aux_stream, cudaStreamNonBlocking, hi));
        for (cudaEvent_t &e : ctx->aux_ev) CK(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    cudaStream_t pre = piped ? ctx->aux_stream : ctx->stream;
    cudaEvent_t *ev_scan = ctx->aux_ev, *ev_render = ctx->aux_ev + 8, ev_fork = ctx->aux_ev[16];
    if (piped) {                                             // fork: the aux stream starts after everything queued so far
        CK(ctx, cudaEventRecord(ev_fork, ctx->stream));
        CK(ctx, cudaStreamWaitEvent(pre, ev_fork, 0));
    }
    auto range = [&](uint64_t g, uint64_t *i0, uint64_t *i1) { *i0 = g * per; *i1 = *i0 + per < n ? *i0 + per : n; };
    p.i0 = 0; p.i1 = n;
    k_sweep_env<<<(unsigned)ceil_div_u64(n, 128), 128, 0, ctx->stream>>>(p);   // only the renders need it: beside the aux-stream passes
    CK_LAUNCH(ctx, "k_sweep_env");
    if (p.closed && C > 1) {
        k_sweep_pre<<<(unsigned)ceil_div_u64(n, 128), 128, 0, pre>>>(p);
        CK_LAUNCH(ctx, "k_sweep_pre");
    }
    // zero-state pass as its own kernel: every group when not pipelined, else the first two
    for (uint64_t g = 0; g < groups; ++g) {
        range(g, &p.i0, &p.i1);
        const unsigned gx = (unsigned)ceil_div_u64(p.i1 - p.i0, 128);
        if (C > 1 && (!piped || ahead || g < 2)) {
            if (p.closed) {
                const uint32_t bpv = (uint32_t)ceil_div_u64(C - 1, 128);
                k_sweep_zsr_closed<<<(unsigned)((p.i1 - p.i0) * bpv), 128, 0, pre>>>(p, bpv);
            } else k_sweep_zsr<<<dim3(gx, (unsigned)(C - 1)), 128, 0, pre>>>(p);
            CK_LAUNCH(ctx, "k_sweep_zsr");
        }
        if (!piped || ahead || g < 2) {
            k_sweep_scan<<<(unsigned)ceil_div_u64(p.i1 - p.i0, SCAN_WARPS), SCAN_WARPS * 32, 0, pre>>>(p);
            CK_LAUNCH(ctx, "k_sweep_scan");
            if (piped) CK(ctx, cudaEventRecord(ev_scan[g], pre));
        }
    }
    for (uint64_t g = 0; g < groups; ++g) {
        range(g, &p.i0, &p.i1);
        const unsigned gx = (unsigned)ceil_div_u64(p.i1 - p.i0, 128);
        const bool duty = piped && !ahead && g + 2 < groups;
        if (duty) { uint64_t z0; range(g + 2, &z0, &p.zi1); p.zoff = z0 - p.i0; } else { p.zoff = 0; p.zi1 = 0; }
        if (piped) CK(ctx, cudaStreamWaitEvent(ctx->stream, ev_scan[g], 0));     // join: start states of this group
        const dim3 grid(gx, (unsigned)C);
        if (io->layout == CPROC_CUDA_TILED) {
            if (duty) k_sweep_render<true, 1><<<grid, XV_BLOCK, 0, ctx->stream>>>(p);
            else k_sweep_render<true, 0><<<grid, XV_BLOCK, 0, ctx->stream>>>(p);
        } else {
            if (duty) k_sweep_render<false, 1><<<grid, XV_BLOCK, 0, ctx->stream>>>(p);
            else k_sweep_render<false, 0><<<grid, XV_BLOCK, 0, ctx->stream>>>(p);
        }
        CK_LAUNCH(ctx, "k_sweep_render");
        if (duty) {                                          // scan of group g+2 beside the render of group g+1
            CK(ctx, cudaEventRecord(ev_render[g], ctx->stream));
            CK(ctx, cudaStreamWaitEvent(pre, ev_render[g], 0));
            SweepParams q = p;
            range(g + 2, &q.i0, &q.i1);
            k_sweep_scan<<<(unsigned)ceil_div_u64(q.i1 - q.i0, SCAN_WARPS), SCAN_WARPS * 32, 0, pre>>>(q);
            CK_LAUNCH(ctx, "k_sweep_scan");
            CK(ctx, cudaEventRecord(ev_scan[g + 2], pre));
        }
    }
    return 0;
}

int launch_xvoice(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io) {
    cproc_cuda_ctx *ctx = b->ctx;
    if (!io->out && !io->mix) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "xvoice: out and mix are both NULL");
    if (io->out && io->layout == CPROC_CUDA_INTERLEAVED) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "xvoice: INTERLEAVED layout not supported");
    if (io->out && io->layout == CPROC_CUDA_TILED && (F & 1)) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "xvoice: TILED needs even F");
    if (F == 0) return 0;
    if (b->cfg.mode == CPROC_CUDA_XVOICE_SCAN && io->out && !io->mix) {
        // variant groups of >= 128; chunk length: enough (variant, chunk) threads per group to
        // fill the chip, multiple of 32 frames
        uint64_t groups = ctx->xvoice_groups > 0 ? (uint64_t)ctx->xvoice_groups : 1;
        if (groups > ceil_div_u64(b->n, 128)) groups = ceil_div_u64(b->n, 128);
        // (one wave of the fused render, 1536 threads per SM, when the groups are pipelined)
        const uint64_t want_threads = groups >= 3 && !ctx->xvoice_closed ? (uint64_t)ctx->n_sm * 1536 : (uint64_t)ctx->n_sm * 2048 * 2;
        uint64_t C = ceil_div_u64(want_threads, ceil_div_u64(b->n, groups));
        if (C > 65535) C = 65535;
        uint64_t L = ceil_div_u64(ceil_div_u64(F, C), 32) * 32;
        if (ctx->xvoice_chunk > 0) L = ceil_div_u64((uint64_t)ctx->xvoice_chunk, 32) * 32;
        if (ceil_div_u64(F, L) > 65535) L = ceil_div_u64(ceil_div_u64(F, 65535), 32) * 32;
        if (L < F) return launch_xvoice_scan(b, F, io, L, groups);
    }
    const bool mix_only = io->mix && !io->out;
    if (b->bus && !mix_only) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "xvoice: with a mix bus attached only the mix is rendered (out must be NULL)");
    // (mix: four resident blocks per SM; a pipelined bus keeps one slot for the block that completes the previous exchange)
    // (second-generation kernel: three blocks per SM, each with a 50 KB state tile; the launch's final reduction waits for the
    // stragglers, so the grid must be co-resident: ask the runtime how many blocks really fit)
    const bool mix2 = mix_only && ctx->xvoice_mix2;
    const size_t mix2_smem = sizeof(uint32_t) * 5 * 256 * XM2_GMAX;
    if (mix2) {
        // (function attributes are per device: set on every launch, like the other staging kernels; the occupancy is cached per context)
        CK(ctx, cudaFuncSetAttribute(k_xvoice_mix2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mix2_smem));
        if (!ctx->xvoice_mix2_per_sm) {
            int occ = 0;
            CK(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_xvoice_mix2, XM2_BLOCK, mix2_smem));
            if (occ < 1) return cproc_set_err(ctx, CPROC_CUDA_ECUDA, "xvoice: k_xvoice_mix2 does not fit an SM");
            ctx->xvoice_mix2_per_sm = occ > XM2_MINB ? XM2_MINB : occ;
        }
    }
    const int mix2_per_sm = ctx->xvoice_mix2_per_sm;
    // Blocks per SM.  A block's work comes in rounds of 256 voices (one pair per thread, all chunks of the launch: ~38 us): 4 Mi voices
    // are 36.9 rounds per block at three blocks per SM (0.3 % lost to the last, uneven round), a 512 Ki-voice shard of an 8-GPU render
    // is 4.62 -> 5 rounds (8 % lost: the residual limiter of the C4 strong-scaling row).  Two blocks per SM do not help (6.94 -> 7
    // rounds of 0.74 of the time: 0.187 against 0.189 ms measured); option xvoice_mix2_blocks is there for the experiment.
    int per_sm = mix2_per_sm;
    if (mix2 && ctx->xvoice_mix2_blocks && ctx->xvoice_mix2_blocks < mix2_per_sm) per_sm = ctx->xvoice_mix2_blocks;
    const uint64_t n_blocks = !mix_only ? ceil_div_u64(b->n, XV_BLOCK)
                            : mix2 ? (uint64_t)ctx->n_sm * per_sm - 1 : (uint64_t)ctx->n_sm * 4 - (b->bus && b->bus_mode == 2 ? 1 : 0);
    XVoiceParams p;
    p.st = b->d_state; p.prm = b->d_param; p.npad = b->npad; p.n = b->n; p.F = F;
    p.raw = (float *)io->out; p.layout = io->layout; p.partial = nullptr;
    p.mix = (float *)io->mix; p.done = nullptr; p.n_render_blocks = (uint32_t)n_blocks;
    p.rows_per_block = 1; p.partial_w = nullptr;
    if (io->mix) {
        size_t need = sizeof(float) * n_blocks * (mix2 ? 1 + XM2_BLOCK / 32 : 1) * 2 * F;
        if (b->cap_mix < need) {
            if (b->d_mix) cudaFree(b->d_mix);
            b->d_mix = nullptr; b->cap_mix = 0;
            CK(ctx, cudaMalloc(&b->d_mix, need));
            b->cap_mix = need;
        }
        p.partial = (float *)b->d_mix;
        if (mix2) p.partial_w = p.partial + n_blocks * 2 * F;
    }
    if (mix_only) {
        if (!b->d_acc) {
            CK(ctx, cudaMalloc(&b->d_acc, 2 * sizeof(uint32_t)));
            CK(ctx, cudaMemsetAsync(b->d_acc, 0, 2 * sizeof(uint32_t), ctx->stream));
            b->cap_acc = 2 * sizeof(uint32_t);
        }
        p.done = b->d_acc;
        p.vpt = ctx->xvoice_vpt > 0 ? (uint32_t)ctx->xvoice_vpt : XM_VPT;
        const uint32_t n_chunks = (uint32_t)ceil_div_u64(F, XM_CHUNK);
        BusFused bf;
        int rc = cproc_bus_fused_begin(b, &bf, 2 * F, 2u, 0u, xm_n_fin(n_chunks, (uint32_t)n_blocks), (int32_t *)io->mix, nullptr);
        if (rc) return rc;
        if (mix2) {
            k_xvoice_mix2<<<(unsigned)n_blocks + (bf.world && bf.mode == 2 ? 1u : 0u), XM2_BLOCK, mix2_smem, ctx->stream>>>(p, bf);
        } else
        k_xvoice_mix<<<(unsigned)n_blocks + (bf.world && bf.mode == 2 ? 1u : 0u), XM_BLOCK, 0, ctx->stream>>>(p, bf);
        CK_LAUNCH(ctx, "k_xvoice_mix");
        return 0;
    }
    if (io->out && io->mix) k_xvoice<true, true><<<(unsigned)n_blocks, XV_BLOCK, 0, ctx->stream>>>(p);
    else k_xvoice<true, false><<<(unsigned)n_blocks, XV_BLOCK, 0, ctx->stream>>>(p);
    CK_LAUNCH(ctx, "k_xvoice");
    if (io->mix) {
        k_xvoice_final<<<(unsigned)ceil_div_u64(2 * F, 128), 128, 0, ctx->stream>>>(p.partial, (float *)io->mix, n_blocks, 2 * F);
        CK_LAUNCH(ctx, "k_xvoice_final");
    }
    return 0;
}

// ---------------------------------------------------------------------------
// one-pole low-pass y = fma(a, x - y, y)
__global__ void k_onepole(float *y, const float *a, uint64_t n, uint64_t F, const float *in, float *out, uint32_t layout) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float s = y[i];
    const float c = a[i];
    for (uint64_t t = 0; t < F; ++t) {
        const uint64_t idx = layout == CPROC_CUDA_INTERLEAVED ? t * n + i : i * F + t;
        s = __fmaf_rn(c, __fsub_rn(in[idx], s), s);
        out[idx] = s;
    }
    y[i] = s;
}

struct OnepoleOp {
    static constexpr int NIN = 1;
    float *y; const float *a;
    float s, c;
    __device__ __forceinline__ void load(uint64_t i) { s = y[i]; c = a[i]; }
    __device__ __forceinline__ void store(uint64_t i) { y[i] = s; }
    __device__ __forceinline__ uint32_t tick(uint32_t x, uint64_t) {
        s = __fmaf_rn(c, __fsub_rn(__uint_as_float(x), s), s);
        return __float_as_uint(s);
    }
};

// ---------------------------------------------------------------------------
// Time-parallel one-pole (few instances, long streams: the block-parallel associative scan of
// the linear recurrence).  y' = y + a (x - y) = (1 - a) y + a x is affine in y, so the stream is
// cut into C chunks of L frames and every (instance, chunk) pair is a thread:
//   pass 1  zero-state response z_c of each full chunk, fp64, same recurrence       (k_onepole_zsr)
//   pass 2  y_{c+1} = (1 - a)^L y_c + z_c, fp64, sequential over the C chunks        (k_onepole_scan)
//   pass 3  the ordinary float tick from each chunk's start state                    (k_onepole_render)
// Start states come from exact arithmetic rather than the float trajectory, so outputs are not bit
// for bit the sequential kernel's: every instance is within 1e-5 of its own peak of the fp64
// recurrence, or within twice the sequential render's error where that is larger (measured on a
// B200: <= 4.7e-6 for 2^-24 <= a <= 1.999; tests/test_gpu_float_ref.py).  The sequential float
// tick stalls where |a (x - y)| < 1/2 ulp(y) (small coefficients) and drifts up to 1.8e-3 of the
// peak from the exact result there; the scan only drifts within one chunk.
struct OnepoleScanParams {
    float *y; const float *a;
    uint64_t n, F, L, C;
    const float *in; float *out;
    uint32_t layout;
    double *z;               // [C-1][n]
    float *y0;               // [C][n]
};
__device__ __forceinline__ uint64_t op_idx(const OnepoleScanParams &p, uint64_t i, uint64_t t) {
    return p.layout == CPROC_CUDA_INTERLEAVED ? t * p.n + i : i * p.F + t;
}
// threads enumerate (chunk, instance) pairs, instance fastest: with few instances the lanes of a
// warp are consecutive chunks of the same stream
__global__ void __launch_bounds__(128) k_onepole_zsr(const OnepoleScanParams p) {
    const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t i = g % p.n, c = g / p.n;
    if (c + 1 >= p.C) return;
    const double a = (double)p.a[i];
    double z = 0.0;
    const uint64_t t0 = c * p.L;
    if (p.layout == CPROC_CUDA_PLANAR && p.L % 4 == 0 && (((uintptr_t)(p.in + i * p.F + t0)) & 15) == 0) {
        const float4 *src = (const float4 *)(p.in + i * p.F + t0);
        for (uint64_t k = 0; k < p.L / 4; ++k) {
            const float4 v = __ldg(src + k);
            z = fma(a, (double)v.x - z, z); z = fma(a, (double)v.y - z, z); z = fma(a, (double)v.z - z, z); z = fma(a, (double)v.w - z, z);
        }
    } else {
        for (uint64_t k = 0; k < p.L; ++k) z = fma(a, (double)__ldg(p.in + op_idx(p, i, t0 + k)) - z, z);
    }
    p.z[c * p.n + i] = z;
}
// One block per instance: thread t owns a run of consecutive chunks, composes its run into one
// affine map (P, w), the block scans the 256 maps (Hillis-Steele in shared memory), and the thread
// walks its run again from its start state writing y0[c].
#define OPS_BLOCK 256
__global__ void __launch_bounds__(OPS_BLOCK) k_onepole_scan(const OnepoleScanParams p) {
    __shared__ double sP[OPS_BLOCK], sW[OPS_BLOCK];
    const uint64_t i = blockIdx.x;
    const uint32_t t = threadIdx.x;
    const double a = (double)p.a[i];
    double m = 1.0, base = 1.0 - a;                       // (1 - a)^L by squaring
    for (uint64_t e = p.L; e; e >>= 1) { if (e & 1) m *= base; base *= base; }
    const uint64_t K = (p.C + OPS_BLOCK - 1) / OPS_BLOCK;
    const uint64_t c0 = (uint64_t)t * K < p.C ? (uint64_t)t * K : p.C, c1 = c0 + K < p.C ? c0 + K : p.C;
    double P = 1.0, w = 0.0;                              // map of chunk c exists for c < C-1
    for (uint64_t c = c0; c < c1 && c + 1 < p.C; ++c) { w = fma(m, w, p.z[c * p.n + i]); P *= m; }
    sP[t] = P; sW[t] = w;
    __syncthreads();
    for (uint32_t d = 1; d < OPS_BLOCK; d <<= 1) {        // inclusive scan: later map applied after the earlier
        double qP = 1.0, qW = 0.0;
        if (t >= d) { qP = sP[t - d]; qW = sW[t - d]; }
        __syncthreads();
        if (t >= d) { sW[t] = fma(sP[t], qW, sW[t]); sP[t] = sP[t] * qP; }
        __syncthreads();
    }
    const double y_init = (double)p.y[i];
    double y = t ? fma(sP[t - 1], y_init, sW[t - 1]) : y_init;
    for (uint64_t c = c0; c < c1; ++c) {
        p.y0[c * p.n + i] = (float)y;
        if (c + 1 < p.C) y = fma(m, y, p.z[c * p.n + i]);
    }
}
__global__ void __launch_bounds__(128) k_onepole_render(const OnepoleScanParams p) {
    const uint64_t g = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t i = g % p.n, c = g / p.n;
    if (c >= p.C) return;
    const float a = p.a[i];
    float s = p.y0[c * p.n + i];
    const uint64_t t0 = c * p.L, t1 = t0 + p.L < p.F ? t0 + p.L : p.F;
    if (p.layout == CPROC_CUDA_PLANAR && (t1 - t0) % 4 == 0 && ((((uintptr_t)(p.in + i * p.F + t0)) | ((uintptr_t)(p.out + i * p.F + t0))) & 15) == 0) {
        const float4 *src = (const float4 *)(p.in + i * p.F + t0);
        float4 *dst = (float4 *)(p.out + i * p.F + t0);
        for (uint64_t k = 0; k < (t1 - t0) / 4; ++k) {
            float4 v = __ldg(src + k);
            s = __fmaf_rn(a, __fsub_rn(v.x, s), s); v.x = s; s = __fmaf_rn(a, __fsub_rn(v.y, s), s); v.y = s;
            s = __fmaf_rn(a, __fsub_rn(v.z, s), s); v.z = s; s = __fmaf_rn(a, __fsub_rn(v.w, s), s); v.w = s;
            __stcs(dst + k, v);
        }
    } else {
        for (uint64_t t = t0; t < t1; ++t) {
            const uint64_t idx = op_idx(p, i, t);
            s = __fmaf_rn(a, __fsub_rn(__ldg(p.in + idx), s), s);
            p.out[idx] = s;
        }
    }
    if (c == p.C - 1) p.y[i] = s;
}

static int launch_onepole_scan(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io, uint64_t L) {
    cproc_cuda_ctx *ctx = b->ctx;
    if (io->in == io->out) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "onepole scan: in place not supported (the input is read twice)");
    const uint64_t n = b->n, C = ceil_div_u64(F, L);
    const size_t bz = sizeof(double) * (C - 1) * n, by = sizeof(float) * C * n, need = bz + by + 64;
    if (b->cap_scratch < need) {
        if (b->d_scratch) cudaFree(b->d_scratch);
        b->d_scratch = nullptr; b->cap_scratch = 0;
        CK(ctx, cudaMalloc(&b->d_scratch, need));
        b->cap_scratch = need;
    }
    OnepoleScanParams p;
    p.y = (float *)b->d_state; p.a = (const float *)b->d_param; p.n = n; p.F = F; p.L = L; p.C = C;
    p.in = (const float *)io->in; p.out = (float *)io->out; p.layout = io->layout;
    p.z = (double *)b->d_scratch; p.y0 = (float *)((uint8_t *)b->d_scratch + ((bz + 15) & ~(size_t)15));
    const unsigned gx = (unsigned)ceil_div_u64(n, 128);
    if (C > 1) { k_onepole_zsr<<<(unsigned)ceil_div_u64(n * (C - 1), 128), 128, 0, ctx->stream>>>(p); CK_LAUNCH(ctx, "k_onepole_zsr"); }
    (void)gx;
    k_onepole_scan<<<(unsigned)n, OPS_BLOCK, 0, ctx->stream>>>(p);
    CK_LAUNCH(ctx, "k_onepole_scan");
    k_onepole_render<<<(unsigned)ceil_div_u64(n * C, 128), 128, 0, ctx->stream>>>(p);
    CK_LAUNCH(ctx, "k_onepole_render");
    return 0;
}

int launch_onepole(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io) {
    cproc_cuda_ctx *ctx = b->ctx;
    if (!io->in || !io->out) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "onepole: in/out is NULL");
    if (io->layout == CPROC_CUDA_TILED) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "onepole: TILED layout not supported");
    if (F == 0) return 0;
    if (b->cfg.mode == CPROC_CUDA_ONEPOLE_SCAN) {
        // chunk length: enough (instance, chunk) threads to fill the chip, at least 64 frames
        const uint64_t C = ceil_div_u64((uint64_t)ctx->n_sm * 2048 * 2, b->n);
        uint64_t L = ceil_div_u64(ceil_div_u64(F, C), 4) * 4;
        if (ctx->xvoice_chunk > 0) L = (uint64_t)ctx->xvoice_chunk;
        if (L < 64 && ctx->xvoice_chunk <= 0) L = 64;
        if (L < F) return launch_onepole_scan(b, F, io, L);
    }
    if (ctx->planar_bulk && io->layout == CPROC_CUDA_PLANAR && pbulk::usable(F, io->in, io->out)) {
        OnepoleOp op; op.y = (float *)b->d_state; op.a = (const float *)b->d_param; op.s = 0.f; op.c = 0.f;
        int rc = pbulk::launch<64, 3>(ctx, op, (const uint32_t *)io->in, (uint32_t *)io->out, b->n, F);
        if (rc) return rc;
        CK_LAUNCH(ctx, "k_onepole (bulk)");
        return 0;
    }
    if (ctx->planar_bulk && io->layout == CPROC_CUDA_INTERLEAVED && pbulk::usable_interleaved4(b->n, io->in, io->out)) {
        OnepoleOp op; op.y = (float *)b->d_state; op.a = (const float *)b->d_param; op.s = 0.f; op.c = 0.f;
        pbulk::launch_interleaved4(ctx, op, (const uint32_t *)io->in, (uint32_t *)io->out, b->n, F);
        CK_LAUNCH(ctx, "k_onepole (interleaved4)");
        return 0;
    }
    k_onepole<<<(unsigned)ceil_div_u64(b->n, 128), 128, 0, ctx->stream>>>((float *)b->d_state, (const float *)b->d_param, b->n, F,
                                                                       (const float *)io->in, (float *)io->out, io->layout);
    CK_LAUNCH(ctx, "k_onepole");
    return 0;
}
