// k_graph.cu -- generated cproc graphs of acc / edge nodes.
//
// Replaces `void cproc_update(w *input, w changed)` (linux/test_cproc.c:13-17,
// stm32f103/bp5_plugin.c:4-9): a straight-line sequence of PROC_COND
// statements (generic/cproc.h:72-77), one tick per call, state in
// function-static structs.  Here: one thread per graph instance, the whole
// node-state vector in registers across the frame block, the node table in
// shared memory, F ticks per launch.
#include "common.cuh"
#include "planar_bulk.cuh"

#define GRAPH_MAX_NODES 16
#define GRAPH_MAX_STATE 48
#define GRAPH_MAX_PARAM 32

struct GraphParams {
    uint32_t *st;                  // SoA [state_words][npad]
    uint64_t npad, n;
    const cproc_cuda_node *nodes;
    uint32_t n_nodes, n_inputs, out_node, state_words;
    const uint32_t *in;            // PLANAR [inst][n_inputs][F] / INTERLEAVED [F][n_inputs][inst]
    const uint32_t *changed;       // [inst][F] / [F][inst] or null
    uint32_t *out;                 // [inst][n_outputs][F] / [F][n_outputs][inst]
    uint64_t F;
    uint32_t layout;
    uint32_t n_outputs;
    uint32_t out_nodes[CPROC_CUDA_GRAPH_MAX_OUTPUTS];
    const uint32_t *prm;           // SoA [param_words][npad]: the nodes' param structs in ANF order
};

// Bus mix of a GRAPH render (io.mix): the second argument of the mix kernels, here and in the generated source (graph_front.cu).
// A mix kernel renders frames [t0, t0 + fc) and writes the sum of every tree group of 32 * wg instances (aligned to the bus
// start) to dst[group][n_outputs][dst_F] at frame dst_t0 + (t - t0).
struct GraphMixParams {
    uint32_t *dst;
    uint64_t t0, fc, dst_F, dst_t0;
    uint32_t wg;                   // warps per tree group (power of two)
    uint32_t outf;                 // bit q: output q is a float (summed with __fadd_rn), else a w (summed mod 2^32)
};

// acc_update (cproc.h:140-142) / edge_update (cproc.h:151-154) on register state
// glide: mod_pdm_pwm.c:129-143 + mod_controlrate.c:28-40 on one parameter (see cproc_cuda.h)
// extension processors: include/cproc_ext.h (x arrives already converted to the input's type: float inputs as float bits)
__device__ __forceinline__ void node_tick(uint32_t type, uint32_t *s, const uint32_t *pr, uint32_t x, uint32_t x2) {
    const uint32_t kind = type & 0xFFu;
    if (kind == CPROC_CUDA_NODE_EDGE) { s[0] = (x != s[1]); s[1] = x; }
    else if (kind == CPROC_CUDA_NODE_PHASOR_F) {
        s[0] = __float_as_uint(__fmul_rn(__int2float_rn((int32_t)s[1]), 4.656612873077392578125e-10f));
        s[1] += pr[0] + x;
    }
    else if (kind == CPROC_CUDA_NODE_SVF) {
        const float f = __uint_as_float(pr[0]), q = __uint_as_float(pr[1]), bp = __uint_as_float(s[1]);
        const float lp = __fmaf_rn(f, bp, __uint_as_float(s[0]));
        float hp = __fsub_rn(__uint_as_float(x), lp);
        hp = __fmaf_rn(-q, bp, hp);
        s[1] = __float_as_uint(__fmaf_rn(f, hp, bp));
        s[0] = __float_as_uint(lp);
    }
    else if (kind == CPROC_CUDA_NODE_ENV) {
        float e = __uint_as_float(s[1]);
        if (s[2] < pr[2]) { e = __fadd_rn(e, __uint_as_float(pr[0])); if (e > 1.0f) e = 1.0f; }
        else { e = __fsub_rn(e, __uint_as_float(pr[1])); if (e < 0.0f) e = 0.0f; }
        s[1] = __float_as_uint(e);
        s[2] += 1u;
        s[0] = __float_as_uint(__fmul_rn(__uint_as_float(x), e));
    }
    else if (kind == CPROC_CUDA_NODE_ONEPOLE) { const float y = __uint_as_float(s[0]); s[0] = __float_as_uint(__fmaf_rn(__uint_as_float(pr[0]), __fsub_rn(__uint_as_float(x), y), y)); }
    else if (kind == CPROC_CUDA_NODE_GAIN) s[0] = __float_as_uint(__fmul_rn(__uint_as_float(pr[0]), __uint_as_float(x)));
    else if (kind == CPROC_CUDA_NODE_ASFLOAT) s[0] = x;
    else if (kind == CPROC_CUDA_NODE_GLIDE_F) {
        const uint32_t L = (type >> 8) & 0xFFu;
        if (s[2] == 0) s[1] = __float_as_uint(__fmul_rn(__fsub_rn(__uint_as_float(x), __uint_as_float(s[0])), 1.0f / (float)(1u << L)));
        s[0] = __float_as_uint(__fadd_rn(__uint_as_float(s[0]), __uint_as_float(s[1])));
        s[2] = (s[2] + 1) & ((1u << L) - 1u);
    }
    else if (kind == CPROC_CUDA_NODE_MUL) s[0] = __float_as_uint(__fmul_rn(__uint_as_float(x), __uint_as_float(x2)));
    else if (kind == CPROC_CUDA_NODE_PDM) {                 // pdm.h:13-77: s[0] = out_q, s[1..K] = s1..sK
        const uint32_t K = (type >> 8) & 7u, sh = (type >> 11) & 31u;
        const uint32_t q = s[K] >> sh;
        const uint32_t a = (q << sh) + (K == 1 ? 0u : x2);
        s[1] += x - a;
        for (uint32_t k = 2; k <= K; ++k) s[k] += s[k - 1] - a;
        s[0] = q;
    }
    else if (kind == CPROC_CUDA_NODE_GLIDE) {
        const uint32_t L = (type >> 8) & 0xFFu;
        if (s[4] == 0) {
            s[0] = s[2]; s[1] = s[3];
            s[2] += s[3] << L;
            s[3] = (uint32_t)((int32_t)(x - s[2]) >> L);
        }
        s[0] += s[1];
        s[4] = (s[4] + 1) & ((1u << L) - 1u);
    }
    else s[0] += x;
}

// Specialisation for the two graphs the reference ships: edge -> acc [-> acc],
// all nodes under one mask bit.  DEPTH = number of acc nodes after the edge.
template <int DEPTH>
__global__ void k_graph_edge_acc(const GraphParams p, uint32_t mask) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    uint32_t e_out = p.st[i], e_last = p.st[p.npad + i], a[DEPTH];
#pragma unroll
    for (int k = 0; k < DEPTH; ++k) a[k] = p.st[(2 + k) * p.npad + i];
    const bool il = p.layout == CPROC_CUDA_INTERLEAVED;
    for (uint64_t t = 0; t < p.F; ++t) {
        const uint64_t idx = il ? t * p.n + i : i * p.F + t;
        const uint32_t x = p.in[idx];
        const uint32_t g = p.changed ? p.changed[idx] : 0xFFFFFFFFu;
        if (g & mask) {
            e_out = (x != e_last); e_last = x;        // n1 = edge(input[0])
            a[0] += e_out;                            // n2 = acc(n1.out)
#pragma unroll
            for (int k = 1; k < DEPTH; ++k) a[k] += a[k - 1];
        }
        p.out[idx] = a[DEPTH - 1];                    // cproc_output(.., nK.out)
    }
    p.st[i] = e_out; p.st[p.npad + i] = e_last;
#pragma unroll
    for (int k = 0; k < DEPTH; ++k) p.st[(2 + k) * p.npad + i] = a[k];
}

__device__ __forceinline__ uint32_t mix_add(uint32_t a, uint32_t b, bool f) {
    return f ? __float_as_uint(__fadd_rn(__uint_as_float(a), __uint_as_float(b))) : a + b;
}

// General table-driven graph.  MIX: frames [m.t0, m.t0 + m.fc) and every frame's sum over each warp's 32 instances (the first
// five levels of the bus tree, lane bit 0 first: a butterfly gives every lane the same bits) to m.dst; out may be NULL.
template <bool MIX>
__global__ void k_graph_table(const GraphParams p, const GraphMixParams m) {
    __shared__ cproc_cuda_node nodes[GRAPH_MAX_NODES];
    __shared__ uint32_t off[GRAPH_MAX_NODES], poff[GRAPH_MAX_NODES], inf[GRAPH_MAX_NODES], outf[GRAPH_MAX_NODES], n_pw;
    if (threadIdx.x == 0) {
        // words per kind: state / param; float-typed first input / float-typed out (cproc_kind_meta in common.cuh, restated for the device)
        const uint8_t sw[CPROC_CUDA_NODE_KINDS] = {1, 2, 5, 0, 2, 2, 3, 1, 1, 1, 3, 1}, pw[CPROC_CUDA_NODE_KINDS] = {0, 0, 0, 0, 1, 2, 3, 1, 1, 0, 0, 0};
        const uint8_t fin[CPROC_CUDA_NODE_KINDS] = {0, 0, 0, 0, 0, 1, 1, 1, 1, 0, 1, 1}, fout[CPROC_CUDA_NODE_KINDS] = {0, 0, 0, 0, 1, 1, 1, 1, 1, 1, 1, 1};
        uint32_t o = 0, q = 0;
        for (uint32_t k = 0; k < p.n_nodes; ++k) {
            nodes[k] = p.nodes[k]; off[k] = o; poff[k] = q;
            const uint32_t kind = nodes[k].type & 0xFFu;
            o += kind == CPROC_CUDA_NODE_PDM ? 1u + ((nodes[k].type >> 8) & 7u) : sw[kind];
            q += pw[kind]; inf[k] = fin[kind]; outf[k] = fout[kind];
        }
        n_pw = q;
    }
    __syncthreads();
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (!MIX && i >= p.n) return;                                 // MIX: every lane takes part in the warp's shuffles
    const bool mine = i < p.n;
    uint32_t s[GRAPH_MAX_STATE];
    uint32_t pr[GRAPH_MAX_PARAM];
    if (mine) {
        for (uint32_t w = 0; w < p.state_words; ++w) s[w] = p.st[w * p.npad + i];
        for (uint32_t w = 0; w < n_pw; ++w) pr[w] = p.prm[w * p.npad + i];
    }
    const bool il = p.layout == CPROC_CUDA_INTERLEAVED;
    const uint64_t t_end = MIX ? m.t0 + m.fc : p.F;
    for (uint64_t t = MIX ? m.t0 : 0; t < t_end; ++t) {
      if (mine) {
        const uint64_t oidx = il ? t * p.n + i : i * p.F + t;
        const uint32_t g = p.changed ? p.changed[oidx] : 0xFFFFFFFFu;
        for (uint32_t k = 0; k < p.n_nodes; ++k) {
            if (!(g & nodes[k].cond_mask)) continue;
            auto fetch = [&](int32_t src, bool want_f) {                 // a w feeding a float input converts by value (cproc.h:75)
                if (src == CPROC_CUDA_SRC_ZERO) return 0u;               // 0u is also +0.0f
                uint32_t v; bool is_f = false;
                if (src >= 0) { v = s[off[src]]; is_f = outf[src] != 0; }
                else { const uint32_t j = (uint32_t)(-(src + 1)); v = p.in[il ? (t * p.n_inputs + j) * p.n + i : (i * p.n_inputs + j) * p.F + t]; }
                return want_f && !is_f ? __float_as_uint(__uint2float_rn(v)) : v;
            };
            const uint32_t x = fetch(nodes[k].src, inf[k] != 0);
            const uint32_t kd = nodes[k].type & 0xFFu;
            const uint32_t x2 = kd == CPROC_CUDA_NODE_PDM ? fetch(nodes[k].src2, false) : kd == CPROC_CUDA_NODE_MUL ? fetch(nodes[k].src2, true) : 0u;
            node_tick(nodes[k].type, s + off[k], pr + poff[k], x, x2);
        }
        if (!MIX || p.out)
            for (uint32_t q = 0; q < p.n_outputs; ++q)
                p.out[il ? (t * p.n_outputs + q) * p.n + i : (i * p.n_outputs + q) * p.F + t] = s[off[p.out_nodes[q]]];
      }
        if (MIX) {
            for (uint32_t q = 0; q < p.n_outputs; ++q) {
                const bool f = (m.outf >> q) & 1u;
                uint32_t v = mine ? s[off[p.out_nodes[q]]] : (f ? 0x80000000u : 0u);    // past n: the tree's -0.0f / 0 padding
#pragma unroll
                for (int b = 1; b < 32; b <<= 1) v = mix_add(v, __shfl_xor_sync(0xFFFFFFFFu, v, b), f);
                if ((threadIdx.x & 31) == 0 && i < p.n)     // lane 0 of a warp with instances: warps past n have no group slot
                    m.dst[((i >> 5) * p.n_outputs + q) * m.dst_F + m.dst_t0 + (t - m.t0)] = v;
            }
        }
    }
    if (mine)
        for (uint32_t w = 0; w < p.state_words; ++w) p.st[w * p.npad + i] = s[w];
}

// One level range of the bus tree above the render kernels' groups: output slot j of bus b is the balanced tree over input
// slots [32 j, 32 j + 32) of that bus, the slots past the bus's last padded with -0.0f / 0 (an exact identity).  src / dst:
// [bus][slot][n_out][frames], src frame stride fc, dst frame stride dst_F at frame offset dst_t0.  The last bus has last_in
// slots, the others gpb_in.  Serves the JIT mix kernels (the level above a block's groups) and the table kernel (above its warps).
__global__ void k_graph_mix_tree(const uint32_t *src, uint32_t *dst, uint64_t n_bus, uint64_t gpb_in, uint64_t last_in, uint64_t gpb_out,
                                 uint32_t n_out, uint64_t fc, uint64_t dst_F, uint64_t dst_t0, uint32_t outf) {
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_bus * gpb_out * n_out * fc) return;
    const uint64_t t = e % fc, q = (e / fc) % n_out, j = (e / (fc * n_out)) % gpb_out, b = e / (fc * n_out * gpb_out);
    const uint64_t m = b == n_bus - 1 ? last_in : gpb_in, k0 = j * 32;
    if (k0 >= m) return;
    const bool f = (outf >> q) & 1u;
    const uint32_t pad = f ? 0x80000000u : 0u;
    uint32_t v[32];
#pragma unroll
    for (int w = 0; w < 32; ++w) v[w] = k0 + w < m ? src[((b * gpb_in + k0 + w) * n_out + q) * fc + t] : pad;
#pragma unroll
    for (int h = 16; h >= 1; h >>= 1)
#pragma unroll
        for (int w = 0; w < h; ++w) v[w] = mix_add(v[2 * w], v[2 * w + 1], f);
    dst[((b * gpb_out + j) * n_out + q) * dst_F + dst_t0 + t] = v[0];
}

// io.mix: the render writes no per-instance stream unless io.out is set too; the tree groups of a render launch are summed
// per bus by k_graph_mix_tree.  Frames go in slices whose partial sums stay under MIX_SCRATCH (mostly L2-resident between
// the two launches); the tree depends on the bus's instance count only, so the slicing does not change a bit.
#define MIX_SCRATCH (64ull << 20)
static int launch_graph_mix(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io, GraphParams &p, cproc_graph_jit *j) {
    cproc_cuda_ctx *ctx = b->ctx;
    const uint64_t n = b->n, vpb = b->cfg.voices_per_bus;
    const uint64_t span = vpb == 0 || vpb >= n ? n : vpb, n_bus = ceil_div_u64(n, span);
    const uint32_t n_out = p.n_outputs;
    uint32_t outf = 0;
    for (uint32_t q = 0; q < n_out; ++q) if (cproc_kind_out_float(b->nodes[b->outs[q]].type)) outf |= 1u << q;
    // tree group of a render launch: a warp (table kernel) or up to a whole block of the generated kernel, aligned to bus starts
    const uint32_t warps = j ? j->mix_warps : 1;
    uint32_t wg = warps;
    while (wg > 1 && n_bus > 1 && span % (32ull * wg)) wg >>= 1;
    const uint64_t g = 32ull * wg, gpb = ceil_div_u64(span, g), last_in = ceil_div_u64(n - (n_bus - 1) * span, g);
    const uint64_t n_groups = (n_bus - 1) * gpb + last_in;
    // scratch per frame: the render's group sums + the first tree level's output (the levels above reuse the first region)
    const uint64_t per_frame = gpb == 1 ? 0 : 4ull * n_out * (n_groups + n_bus * ceil_div_u64(gpb, 32));
    uint64_t fc = F;
    if (per_frame && per_frame * F > MIX_SCRATCH) { fc = MIX_SCRATCH / per_frame / 32 * 32; if (fc < 32) fc = 32; if (fc > F) fc = F; }
    if (per_frame * fc > b->cap_scratch) {
        if (b->d_scratch) cudaFree(b->d_scratch);
        b->d_scratch = nullptr; b->cap_scratch = 0;
        // a period graph captured by cproc_cuda_run (abi.cu) holds the old scratch pointer: capture again
        if (b->rg.exec) { cudaGraphExecDestroy(b->rg.exec); b->rg.exec = nullptr; b->rg.seen = 0; b->rg.F = 0; }
        CK(ctx, cudaMalloc(&b->d_scratch, per_frame * fc));
        b->cap_scratch = per_frame * fc;
    }
    uint32_t *bufA = (uint32_t *)b->d_scratch, *bufB = bufA + n_out * n_groups * fc;
    for (uint64_t t0 = 0; t0 < F; t0 += fc) {
        const uint64_t c = F - t0 < fc ? F - t0 : fc;
        GraphMixParams m;
        m.t0 = t0; m.fc = c; m.wg = wg; m.outf = outf;
        if (gpb == 1) { m.dst = (uint32_t *)io->mix; m.dst_F = F; m.dst_t0 = t0; }
        else { m.dst = bufA; m.dst_F = c; m.dst_t0 = 0; }
        if (j) {
            void *args[] = {&p, &m};
            CK(ctx, cudaLaunchKernel((const void *)j->k_mix, dim3((unsigned)ceil_div_u64(n, 32ull * warps)), dim3(32 * warps), args, 0, ctx->stream));
            ctx->launches++;
        } else {
            k_graph_table<true><<<(unsigned)ceil_div_u64(n, 128), 128, 0, ctx->stream>>>(p, m);
            CK_LAUNCH(ctx, "k_graph_table (mix)");
        }
        uint32_t *src = bufA, *oth = bufB;
        for (uint64_t gin = gpb, lin = last_in; gin > 1;) {
            const uint64_t gout = ceil_div_u64(gin, 32), lout = ceil_div_u64(lin, 32);
            const bool last = gout == 1;
            uint32_t *dst = last ? (uint32_t *)io->mix : oth;
            const uint64_t work = n_bus * gout * n_out * c;
            k_graph_mix_tree<<<(unsigned)ceil_div_u64(work, 256), 256, 0, ctx->stream>>>(src, dst, n_bus, gin, lin, gout, n_out, c, last ? F : c, last ? t0 : 0, outf);
            CK_LAUNCH(ctx, "k_graph_mix_tree");
            oth = src; src = dst; gin = gout; lin = lout;
        }
    }
    return 0;
}

int launch_graph(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io) {
    cproc_cuda_ctx *ctx = b->ctx;
    if ((!io->out && !io->mix) || (!io->in && b->cfg.n_inputs)) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "graph: in/out is NULL");
    if (io->layout == CPROC_CUDA_TILED) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "graph: TILED layout not supported");
    if (io->mix && b->cfg.voices_per_bus % 32)
        return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "graph mix: voices_per_bus %llu is neither 0 nor a multiple of 32", (unsigned long long)b->cfg.voices_per_bus);
    if (io->mix && b->cfg.mode == CPROC_CUDA_GRAPH_SCAN) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "graph mix: not available in the GRAPH_SCAN mode");
    if (F == 0) return 0;
    if (b->cfg.mode == CPROC_CUDA_GRAPH_SCAN && F > 64) return launch_graph_scan(b, F, io);
    GraphParams p;
    p.st = b->d_state; p.npad = b->npad; p.n = b->n; p.nodes = b->d_nodes;
    p.n_nodes = b->cfg.n_nodes; p.n_inputs = b->cfg.n_inputs; p.out_node = b->cfg.out_node;
    p.state_words = b->state_words;
    p.n_outputs = (uint32_t)b->outs.size();
    for (uint32_t q = 0; q < CPROC_CUDA_GRAPH_MAX_OUTPUTS; ++q) p.out_nodes[q] = q < p.n_outputs ? b->outs[q] : 0;
    p.in = (const uint32_t *)io->in; p.changed = (const uint32_t *)io->in2; p.out = (uint32_t *)io->out;
    p.F = F; p.layout = io->layout; p.prm = b->d_param;
    const unsigned grid = (unsigned)ceil_div_u64(p.n, 128);
    // the kernel generated for this graph (graph_front.cu)
    cproc_graph_jit *j = nullptr;
    const bool jit = ctx->graph_jit && cproc_graph_jit_get(b, p.changed != nullptr, &j) == 0;
    if (!jit && (b->nodes.size() > GRAPH_MAX_NODES || b->state_words > GRAPH_MAX_STATE || b->param_words > GRAPH_MAX_PARAM))
        return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "graph: %zu nodes need the NVRTC path, which is unavailable (%s)", b->nodes.size(), b->jit_log.c_str());
    if (io->mix) return launch_graph_mix(b, F, io, p, jit ? j : nullptr);
    if (jit) {
        void *args[] = {&p};
        cudaError_t e;
        CUtensorMap tin, tchg, tout;
        const bool aligned = F % 4 == 0 && ((uintptr_t)p.in & 15) == 0 && ((uintptr_t)p.out & 15) == 0 && (!p.changed || ((uintptr_t)p.changed & 15) == 0);
        const bool vec4 = ctx->graph_vec4 && p.n % 4 == 0 && ((uintptr_t)p.in & 15) == 0 && ((uintptr_t)p.out & 15) == 0 && (!p.changed || ((uintptr_t)p.changed & 15) == 0);
        if (io->layout == CPROC_CUDA_INTERLEAVED && vec4) e = cudaLaunchKernel((const void *)j->k_il4, dim3((unsigned)ceil_div_u64(p.n, 512)), dim3(128), args, 0, ctx->stream);
        else if (io->layout == CPROC_CUDA_INTERLEAVED) e = cudaLaunchKernel((const void *)j->k_il, dim3(grid), dim3(128), args, 0, ctx->stream);
        else if (j->k_pt && aligned && ctx->planar_bulk && pbulk::encode_rows3_u32(&tin, p.n_inputs ? p.in : p.out, F, p.n_inputs ? p.n_inputs : p.n_outputs, p.n) &&
                 pbulk::encode_rows3_u32(&tchg, p.changed ? p.changed : (p.n_inputs ? p.in : p.out), F, 1, p.n) && pbulk::encode_rows3_u32(&tout, p.out, F, p.n_outputs, p.n)) {
            void *targs[] = {&p, &tin, &tchg, &tout};
            e = cudaLaunchKernel((const void *)j->k_pt, dim3((unsigned)ceil_div_u64(p.n, j->pt_block)), dim3(j->pt_block), targs, j->pt_smem, ctx->stream);
        } else e = cudaLaunchKernel((const void *)j->k_ps, dim3(grid), dim3(128), args, 0, ctx->stream);
        ctx->launches++;
        return cproc_check(ctx, e, "graph (jit)");
    }
    // recognise edge -> acc [-> acc] chains under a single mask
    const std::vector<cproc_cuda_node> &nd = b->nodes;
    bool chain = nd.size() >= 2 && nd.size() <= 3 && nd[0].type == CPROC_CUDA_NODE_EDGE && nd[0].src == -1 &&
                 p.n_inputs == 1 && p.n_outputs == 1 && p.out_node == nd.size() - 1;
    for (size_t k = 1; chain && k < nd.size(); ++k)
        chain = nd[k].type == CPROC_CUDA_NODE_ACC && nd[k].src == (int32_t)k - 1 && nd[k].cond_mask == nd[0].cond_mask;
    if (chain && nd.size() == 2) k_graph_edge_acc<1><<<grid, 128, 0, ctx->stream>>>(p, nd[0].cond_mask);
    else if (chain) k_graph_edge_acc<2><<<grid, 128, 0, ctx->stream>>>(p, nd[0].cond_mask);
    else k_graph_table<false><<<grid, 128, 0, ctx->stream>>>(p, GraphMixParams{});
    CK_LAUNCH(ctx, "k_graph");
    return 0;
}
