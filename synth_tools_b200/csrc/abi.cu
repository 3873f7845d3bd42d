// abi.cu -- the C-ABI of libcproc_cuda (include/cproc_cuda.h): contexts,
// batches, reference-layout state upload/download, run dispatch.
#include "common.cuh"
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

static thread_local std::string g_last_err;

int cproc_set_err(cproc_cuda_ctx *ctx, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_err = buf;
    if (ctx) ctx->err = buf;
    return code;
}

int cproc_check(cproc_cuda_ctx *ctx, cudaError_t e, const char *what) {
    if (e == cudaSuccess) return 0;
    int code = e == cudaErrorMemoryAllocation ? CPROC_CUDA_ENOMEM
             : (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) ? CPROC_CUDA_ENODEV
             : CPROC_CUDA_ECUDA;
    return cproc_set_err(ctx, code, "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
}

extern "C" {

int cproc_cuda_abi_version(void) { return CPROC_CUDA_ABI_VERSION; }

int cproc_cuda_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

const char *cproc_cuda_last_error(const cproc_cuda_ctx *ctx) {
    return ctx ? ctx->err.c_str() : g_last_err.c_str();
}

uint64_t cproc_cuda_launch_count(const cproc_cuda_ctx *ctx) { return ctx ? ctx->launches : 0; }

int cproc_cuda_open(int device, void *stream, cproc_cuda_ctx **out) {
    if (!out) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "open: ctx out pointer is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        return cproc_set_err(nullptr, CPROC_CUDA_ENODEV, "open: no CUDA device (%s); this library has no CPU fallback",
                             e == cudaSuccess ? "count is 0" : cudaGetErrorString(e));
    }
    if (device < 0 || device >= n) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "open: device %d out of range [0,%d)", device, n);
    cproc_cuda_ctx *ctx = new cproc_cuda_ctx();
    ctx->device = device;
    int rc;
    if ((rc = cproc_check(ctx, cudaSetDevice(device), "cudaSetDevice"))) { g_last_err = ctx->err; delete ctx; return rc; }
    cudaDeviceProp prop;
    if ((rc = cproc_check(ctx, cudaGetDeviceProperties(&prop, device), "cudaGetDeviceProperties"))) { g_last_err = ctx->err; delete ctx; return rc; }
    if (prop.major < 10) {
        rc = cproc_set_err(nullptr, CPROC_CUDA_ENODEV, "open: device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
        delete ctx; return rc;
    }
    ctx->n_sm = prop.multiProcessorCount;
    if (stream) { ctx->stream = (cudaStream_t)stream; ctx->own_stream = false; }
    else {
        if ((rc = cproc_check(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking), "cudaStreamCreate"))) { g_last_err = ctx->err; delete ctx; return rc; }
        ctx->own_stream = true;
    }
    if ((rc = cproc_check(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking), "cudaStreamCreate(copy)")) ||
        (rc = cproc_check(ctx, cudaEventCreate(&ctx->ev0), "cudaEventCreate")) || (rc = cproc_check(ctx, cudaEventCreate(&ctx->ev1), "cudaEventCreate"))) {
        g_last_err = ctx->err;
        cproc_cuda_close(ctx);
        return rc;
    }
    *out = ctx;
    return 0;
}

int cproc_cuda_close(cproc_cuda_ctx *ctx) {
    if (!ctx) return 0;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->aux_stream) { cudaStreamSynchronize(ctx->aux_stream); cudaStreamDestroy(ctx->aux_stream); }
    for (cudaEvent_t e : ctx->aux_ev) if (e) cudaEventDestroy(e);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    for (uint32_t *j : ctx->d_jump) if (j) cudaFree(j);
    if (ctx->d_sm_rank) cudaFree(ctx->d_sm_rank);
    if (ctx->d_work) cudaFree(ctx->d_work);
    if (ctx->d_jump16) cudaFree(ctx->d_jump16);
    delete ctx;
    return 0;
}

int cproc_cuda_sync(cproc_cuda_ctx *ctx) {
    if (!ctx) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "sync: ctx is NULL");
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

int cproc_cuda_set_option(cproc_cuda_ctx *ctx, const char *name, int64_t value) {
    if (!ctx || !name) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "set_option: NULL argument");
    ctx->opt_epoch++;                                        // captured period graphs (cproc_cuda_run) are re-captured
    if (!strcmp(name, "pdm_block")) { if (value < 32 || value > 128 || (value & 31)) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "pdm_block must be 32, 64, 96 or 128"); ctx->pdm_block = (int)value; }
    else if (!strcmp(name, "pdm_tpb")) { if (value < 0 || value > 2) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "pdm_tpb must be 0 (thread per channel), 1 (thread per bank) or 2 (auto)"); ctx->pdm_tpb = (int)value; }
    else if (!strcmp(name, "pdm_ws")) ctx->pdm_ws = value != 0;
    else if (!strcmp(name, "voice_fpt")) { if (value != 0 && value != 1 && value != 2 && value != 4 && value != 8 && value != 16) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "voice_fpt must be 0, 1, 2, 4, 8 or 16"); ctx->voice_fpt = (int)value; }
    else if (!strcmp(name, "pdm_tlog")) { if (value < 6 || value > 7) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "pdm_tlog must be 6 or 7"); ctx->pdm_tlog = (int)value; }
    else if (!strcmp(name, "pdm_v1_chains")) { if (value != 1 && value != 2) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "pdm_v1_chains must be 1 or 2"); ctx->pdm_v1_chains = (int)value; }
    else if (!strcmp(name, "pdm_planar_bulk")) { if (value < 0 || value > 2) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "pdm_planar_bulk must be 0..2"); ctx->pdm_planar_bulk = value ? 2 : 0; }
    else if (!strcmp(name, "pdm_ctas_per_sm")) { if (value < 1 || value > 8) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "pdm_ctas_per_sm must be 1..8"); ctx->pdm_ctas_per_sm = (int)value; }
    else if (!strcmp(name, "pdm_slice_batches")) { if (value < 2 || value > 65536) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "pdm_slice_batches must be 2..65536"); ctx->pdm_slice_batches = (int)value; }
    else if (!strcmp(name, "grain_blocks_per_sm")) { if (value < 1 || value > 16) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "grain_blocks_per_sm must be 1..16"); ctx->grain_blocks_per_sm = (int)value; }
    else if (!strcmp(name, "planar_bulk")) { if (value != 0 && value != 2) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "planar_bulk must be 0 or 2"); ctx->planar_bulk = (int)value; }
    else if (!strcmp(name, "graph_vec4")) ctx->graph_vec4 = value != 0;
    else if (!strcmp(name, "graph_jit")) ctx->graph_jit = value != 0;
    else if (!strcmp(name, "grain_mix2")) { if (value < 0 || value > 2) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "grain_mix2 must be 0..2"); ctx->grain_mix2 = (int)value; }
    else if (!strcmp(name, "xvoice_chunk")) { if (value < 0) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "xvoice_chunk must be >= 0"); ctx->xvoice_chunk = (int)value; }
    else if (!strcmp(name, "xvoice_vpt")) { if (value < 0 || value > 65536) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "xvoice_vpt must be 0..65536"); ctx->xvoice_vpt = (int)value; }
    else if (!strcmp(name, "xvoice_closed")) ctx->xvoice_closed = value ? 1 : 0;
    else if (!strcmp(name, "xvoice_mix2")) ctx->xvoice_mix2 = value ? 1 : 0;
    else if (!strcmp(name, "xvoice_mix2_blocks")) { if (value < 0 || value > 3) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "xvoice_mix2_blocks must be 0..3"); ctx->xvoice_mix2_blocks = (int)value; }
    else if (!strcmp(name, "run_graph")) { if (value < 0 || value > 3) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "run_graph must be 0..3"); ctx->run_graph = (int)value; }
    else if (!strcmp(name, "xvoice_groups")) { if (value < 0 || value > 8) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "xvoice_groups must be 0..8"); ctx->xvoice_groups = (int)value; }
    else if (!strcmp(name, "pdm_persist")) { if (value < 0 || value > 2) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "pdm_persist must be 0 (never), 1 (auto) or 2 (always)"); ctx->pdm_persist = (int)value; }
    else if (!strcmp(name, "pdm_warps_per_smsp")) { if (value < 1 || value > 4) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "pdm_warps_per_smsp must be 1..4"); ctx->pdm_warps_per_smsp = (int)value; }
    else return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "set_option: unknown option '%s'", name);
    return 0;
}

// ---- batches ----------------------------------------------------------------

static int proc_words(const cproc_cuda_config &c, const std::vector<cproc_cuda_node> &nodes, uint32_t *sw, uint32_t *pw) {
    switch (c.proc) {
    case CPROC_CUDA_GRAPH: {
        uint32_t w = 0, q = 0;
        for (auto &nd : nodes) { w += cproc_node_words(nd.type); q += cproc_node_param_words(nd.type); }
        *sw = w; *pw = q; return 0;
    }
    case CPROC_CUDA_PDM: *sw = c.order; *pw = 1; return 0;
    case CPROC_CUDA_PDM_V1: *sw = 2; *pw = 0; return 0;
    case CPROC_CUDA_PDM_V2: *sw = 5 + c.order; *pw = 0; return 0;
    case CPROC_CUDA_PWM: *sw = 1; *pw = 1; return 0;
    case CPROC_CUDA_VOICE_BANK: *sw = 2; *pw = 0; return 0;
    case CPROC_CUDA_SQUARE_GRAIN: *sw = 1; *pw = 1; return 0;
    case CPROC_CUDA_SQUARE_GRAIN_MIX: *sw = 2; *pw = 4; return 0;
    case CPROC_CUDA_XVOICE: *sw = 5; *pw = 8; return 0;
    case CPROC_CUDA_ONEPOLE: *sw = 1; *pw = 1; return 0;
    case CPROC_CUDA_WORD_CLOCK: *sw = 2; *pw = 1; return 0;
    }
    return -1;
}

int cproc_cuda_alloc(cproc_cuda_ctx *ctx, const cproc_cuda_config *cfg, uint64_t n, cproc_cuda_batch **out) {
    if (!ctx || !cfg || !out) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "alloc: NULL argument");
    *out = nullptr;
    if (n == 0) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "alloc: n_instances is 0");
    cproc_cuda_config c = *cfg;
    std::vector<cproc_cuda_node> nodes;
    std::vector<uint32_t> outs;
    bool pdm_family = c.proc == CPROC_CUDA_PDM || c.proc == CPROC_CUDA_PDM_V1 || c.proc == CPROC_CUDA_PDM_V2;
    if (c.proc == CPROC_CUDA_GRAPH) {
        if (!c.nodes || c.n_nodes == 0 || c.n_nodes > CPROC_CUDA_GRAPH_MAX_NODES) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "alloc: graph needs 1..%d nodes", CPROC_CUDA_GRAPH_MAX_NODES);
        if (c.n_outputs > CPROC_CUDA_GRAPH_MAX_OUTPUTS || (c.n_outputs > 1 && !c.out_nodes)) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "alloc: graph has 1..%d outputs (out_nodes)", CPROC_CUDA_GRAPH_MAX_OUTPUTS);
        if (c.n_outputs > 1) outs.assign(c.out_nodes, c.out_nodes + c.n_outputs); else outs.assign(1, c.n_outputs == 1 && c.out_nodes ? c.out_nodes[0] : c.out_node);
        for (uint32_t o : outs) if (o >= c.n_nodes) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "alloc: graph output node %u of %u", o, c.n_nodes);
        nodes.assign(c.nodes, c.nodes + c.n_nodes);
        for (uint32_t k = 0; k < c.n_nodes; ++k) {
            const cproc_cuda_node &nd = nodes[k];
            if (const char *why = cproc_node_check(nodes.data(), k, c.n_inputs)) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "alloc: node %u (type 0x%x, src %d): %s", k, nd.type, nd.src, why);
        }
    }
    if (pdm_family || c.proc == CPROC_CUDA_PDM_V2) {
        if (c.proc != CPROC_CUDA_PDM_V1 && (c.order < 1 || c.order > 4)) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "alloc: pdm order must be 1..4");
        if (c.proc != CPROC_CUDA_PDM_V1 && c.out_shift > 31) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "alloc: out_shift must be <= 31");
        if (c.proc == CPROC_CUDA_PDM_V2 && c.out_shift < 24) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "alloc: pdm_v2 emits 8-bit duty, out_shift must be >= 24");
        if (c.proc == CPROC_CUDA_PDM_V2 && (c.ctl_div_log < 1 || c.ctl_div_log > 24)) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "alloc: ctl_div_log must be 1..24");
        if (c.proc != CPROC_CUDA_PDM && c.bank_size == 0) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "alloc: bank_size is 0");
    }
    if (c.layout > CPROC_CUDA_TILED) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "alloc: unknown layout %u", c.layout);
    uint32_t sw = 0, pw = 0;
    if (proc_words(c, nodes, &sw, &pw)) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "alloc: unknown processor %u", c.proc);
    if (sw > 5 * CPROC_CUDA_GRAPH_MAX_NODES) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "alloc: graph state too large (%u words)", sw);
    if (pw > CPROC_CUDA_GRAPH_MAX_PARAM_WORDS) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "alloc: graph param record too large (%u words)", pw);

    CK(ctx, cudaSetDevice(ctx->device));
    cproc_cuda_batch *b = new cproc_cuda_batch();
    b->ctx = ctx; b->cfg = c; b->nodes = nodes; b->cfg.nodes = nullptr; b->n = n;
    b->outs = outs; b->cfg.out_nodes = nullptr;
    if (c.proc == CPROC_CUDA_GRAPH) { b->cfg.n_outputs = (uint32_t)outs.size(); b->cfg.out_node = outs[0]; }
    b->state_words = sw; b->param_words = pw;
    bool banked = c.proc == CPROC_CUDA_PDM_V1 || c.proc == CPROC_CUDA_PDM_V2;
    if (banked) {
        if (c.bank_size > n) b->cfg.bank_size = (uint32_t)n;
        b->n_banks = ceil_div_u64(n, b->cfg.bank_size);
        b->npad = b->n_banks * b->cfg.bank_size;
    } else { b->n_banks = 0; b->npad = n; }
    b->npad = (b->npad + 3) & ~3ull;        // rows 16-byte aligned
    if (c.proc == CPROC_CUDA_XVOICE) b->npad = (b->npad + 255) & ~255ull;   // k_xvoice_mix2 walks whole groups of 256 voices without bounds checks (rows are zero past n)
    if (c.proc == CPROC_CUDA_VOICE_BANK) {
        if (b->cfg.voices_per_bus == 0 || b->cfg.voices_per_bus > n) b->cfg.voices_per_bus = n;
        b->n_bus = ceil_div_u64(n, b->cfg.voices_per_bus);
    }
    if (c.proc == CPROC_CUDA_GRAPH) b->n_bus = c.voices_per_bus == 0 ? 1 : ceil_div_u64(n, c.voices_per_bus);   // io.mix checks the value
    int rc = 0;
    do {
        if ((rc = cproc_check(ctx, cudaMalloc(&b->d_state, sizeof(uint32_t) * sw * b->npad), "cudaMalloc(state)"))) break;
        if ((rc = cproc_check(ctx, cudaMemsetAsync(b->d_state, 0, sizeof(uint32_t) * sw * b->npad, ctx->stream), "memset(state)"))) break;
        if (pw) {
            if ((rc = cproc_check(ctx, cudaMalloc(&b->d_param, sizeof(uint32_t) * pw * b->npad), "cudaMalloc(param)"))) break;
            if ((rc = cproc_check(ctx, cudaMemsetAsync(b->d_param, 0, sizeof(uint32_t) * pw * b->npad, ctx->stream), "memset(param)"))) break;
        }
        if (banked) {
            if ((rc = cproc_check(ctx, cudaMalloc(&b->d_prng, sizeof(uint32_t) * b->n_banks), "cudaMalloc(prng)"))) break;
            // xorshift32 must not start at 0: default seed = bank index + 1
            std::vector<uint32_t> seed(b->n_banks);
            for (uint64_t i = 0; i < b->n_banks; ++i) seed[i] = (uint32_t)(i + 1);
            if ((rc = cproc_check(ctx, cudaMemcpyAsync(b->d_prng, seed.data(), sizeof(uint32_t) * b->n_banks, cudaMemcpyHostToDevice, ctx->stream), "memcpy(prng)"))) break;
            if ((rc = cproc_check(ctx, cudaStreamSynchronize(ctx->stream), "sync"))) break;
        }
        if (!nodes.empty()) {
            if ((rc = cproc_check(ctx, cudaMalloc(&b->d_nodes, sizeof(cproc_cuda_node) * nodes.size()), "cudaMalloc(nodes)"))) break;
            if ((rc = cproc_check(ctx, cudaMemcpy(b->d_nodes, nodes.data(), sizeof(cproc_cuda_node) * nodes.size(), cudaMemcpyHostToDevice), "memcpy(nodes)"))) break;
        }
    } while (0);
    if (rc) { cproc_cuda_free(b); return rc; }
    *out = b;
    return 0;
}

int cproc_cuda_free(cproc_cuda_batch *b) {
    if (!b) return 0;
    cudaSetDevice(b->ctx->device);
    cudaStreamSynchronize(b->ctx->stream);
    void *ptrs[] = { b->d_state, b->d_param, b->d_prng, b->d_prng2, b->d_prng_g, b->d_nodes, b->d_in, b->d_in2, b->d_ctl, b->d_out, b->d_out2, b->d_mix, b->d_flags, b->d_scratch, b->d_aux, b->d_acc };
    for (void *q : ptrs) if (q) cudaFree(q);
    for (cproc_graph_jit &j : b->jit) if (j.lib) cudaLibraryUnload(j.lib);
    if (b->rg.exec) cudaGraphExecDestroy(b->rg.exec);
    if (b->rg.h) cudaFreeHost(b->rg.h);
    if (b->st_h) cudaFreeHost(b->st_h);
    delete b;
    return 0;
}

size_t cproc_cuda_state_bytes(const cproc_cuda_batch *b) { return b ? 4u * b->state_words : 0; }
size_t cproc_cuda_param_bytes(const cproc_cuda_batch *b) { return b ? 4u * b->param_words : 0; }

// k_grain_mix2 / k_grain_mix3 carry a grain's trigger state as -1 / 0 / +1 and write back +-0.5; the reference keeps any
// other float (0.3, a subnormal, +-inf; a NaN state never flips and adds 0 to the mix).  Such a state needs k_grain_mix.
static bool grain_state_odd(uint32_t w) {
    return w != 0u && w != 0x80000000u && w != 0x3F000000u && w != 0xBF000000u;
}

// AoS (reference struct layout, any stride) <-> SoA rows on the device.
static int aos_to_dev(cproc_cuda_batch *b, uint32_t *d_rows, uint32_t words, const void *aos, size_t stride) {
    cproc_cuda_ctx *ctx = b->ctx;
    if (!aos) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "upload: source is NULL");
    if (words == 0) return 0;
    if (stride == 0) stride = 4u * words;
    if (stride < 4u * words) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "upload: stride %zu smaller than record (%u bytes)", stride, 4u * words);
    std::vector<uint32_t> soa((size_t)words * b->npad, 0u);
    const uint8_t *src = (const uint8_t *)aos;
    for (uint64_t i = 0; i < b->n; ++i) {
        uint32_t rec[5 * CPROC_CUDA_GRAPH_MAX_NODES + 8];
        memcpy(rec, src + i * stride, 4u * words);
        for (uint32_t w = 0; w < words; ++w) soa[(size_t)w * b->npad + i] = rec[w];
    }
    if (d_rows == b->d_state && b->cfg.proc == CPROC_CUDA_SQUARE_GRAIN_MIX) {
        b->grain_odd_state = false;
        for (uint64_t i = 0; i < b->n; ++i) b->grain_odd_state |= grain_state_odd(soa[i]);
    }
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMemcpyAsync(d_rows, soa.data(), sizeof(uint32_t) * soa.size(), cudaMemcpyHostToDevice, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

int cproc_cuda_upload_state(cproc_cuda_batch *b, const void *aos, size_t stride) {
    if (!b) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "upload_state: batch is NULL");
    return aos_to_dev(b, b->d_state, b->state_words, aos, stride);
}

int cproc_cuda_upload_param(cproc_cuda_batch *b, const void *aos, size_t stride) {
    if (!b) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "upload_param: batch is NULL");
    if (b->param_words == 0) return cproc_set_err(b->ctx, CPROC_CUDA_EINVAL, "upload_param: processor has no param record");
    if (b->cfg.proc == CPROC_CUDA_SQUARE_GRAIN_MIX && aos && (stride == 0 || stride >= 4u * b->param_words)) {
        // pan gains k/64: the mix kernels pack both channels of up to 500 grains into 16-bit halves
        const size_t s = stride ? stride : 4u * b->param_words;
        for (uint64_t i = 0; i < b->n; ++i) {
            uint32_t g[2];
            memcpy(g, (const uint8_t *)aos + i * s + 8, sizeof(g));
            if (g[0] > 64 || g[1] > 64)
                return cproc_set_err(b->ctx, CPROC_CUDA_EINVAL, "upload_param: square_grain_mix grain %llu: gains %u, %u (0..64)", (unsigned long long)i, g[0], g[1]);
        }
    }
    b->aux_dirty = true;
    return aos_to_dev(b, b->d_param, b->param_words, aos, stride);
}

int cproc_cuda_download_state(cproc_cuda_batch *b, void *aos, size_t stride) {
    if (!b) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "download_state: batch is NULL");
    cproc_cuda_ctx *ctx = b->ctx;
    if (!aos) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "download_state: destination is NULL");
    uint32_t words = b->state_words;
    if (stride == 0) stride = 4u * words;
    if (stride < 4u * words) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "download_state: stride too small");
    std::vector<uint32_t> soa((size_t)words * b->npad);
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMemcpyAsync(soa.data(), b->d_state, sizeof(uint32_t) * soa.size(), cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    uint8_t *dst = (uint8_t *)aos;
    for (uint64_t i = 0; i < b->n; ++i) {
        uint32_t rec[5 * CPROC_CUDA_GRAPH_MAX_NODES + 8];
        for (uint32_t w = 0; w < words; ++w) rec[w] = soa[(size_t)w * b->npad + i];
        memcpy(dst + i * stride, rec, 4u * words);
    }
    return 0;
}

int cproc_cuda_upload_bank(cproc_cuda_batch *b, const uint32_t *prng, uint32_t count) {
    if (!b) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "upload_bank: batch is NULL");
    cproc_cuda_ctx *ctx = b->ctx;
    if (!b->d_prng) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "upload_bank: processor has no dither banks");
    if (b->cfg.proc == CPROC_CUDA_PDM_V2 && count >= (1u << b->cfg.ctl_div_log)) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "upload_bank: count %u >= control divider", count);
    CK(ctx, cudaSetDevice(ctx->device));
    if (prng) {
        CK(ctx, cudaMemcpyAsync(b->d_prng, prng, sizeof(uint32_t) * b->n_banks, cudaMemcpyHostToDevice, ctx->stream));
        CK(ctx, cudaStreamSynchronize(ctx->stream));
    }
    b->count = count;
    return 0;
}

int cproc_cuda_download_bank(cproc_cuda_batch *b, uint32_t *prng, uint32_t *count) {
    if (!b) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "download_bank: batch is NULL");
    cproc_cuda_ctx *ctx = b->ctx;
    if (!b->d_prng) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "download_bank: processor has no dither banks");
    CK(ctx, cudaSetDevice(ctx->device));
    if (prng) {
        CK(ctx, cudaMemcpyAsync(prng, b->d_prng, sizeof(uint32_t) * b->n_banks, cudaMemcpyDeviceToHost, ctx->stream));
        CK(ctx, cudaStreamSynchronize(ctx->stream));
    }
    if (count) *count = b->count;
    return 0;
}

// ---- run --------------------------------------------------------------------

} // extern "C"

int cproc_io_bytes(const cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io, cproc_io_sizes *s) {
    const cproc_cuda_config &c = b->cfg;
    const uint64_t n = b->n;
    memset(s, 0, sizeof(*s));
    switch (c.proc) {
    case CPROC_CUDA_GRAPH:
        s->in = 4 * n * c.n_inputs * F; s->in2 = io->in2 ? 4 * n * F : 0; s->out = io->out || !io->mix ? 4 * n * (c.n_outputs ? c.n_outputs : 1) * F : 0;
        s->mix = io->mix ? 4 * b->n_bus * (c.n_outputs ? c.n_outputs : 1) * F : 0; break;
    case CPROC_CUDA_PDM:
        s->in = io->in ? 4 * n * F : 0; s->in2 = io->in2 ? 4 * F : 0; s->out = 4 * n * F; break;
    case CPROC_CUDA_PDM_V1:
        s->in2 = io->in2 ? 4 * b->n_banks * F : 0; s->out = n * (F / 8); break;
    case CPROC_CUDA_PDM_V2:
        s->in2 = io->in2 ? 4 * b->n_banks * F : 0; s->ctl = io->ctl ? 4ull * io->n_ctl * n : 0; s->out = n * F; break;
    case CPROC_CUDA_PWM: s->out = n * F; break;
    case CPROC_CUDA_VOICE_BANK:
        s->out = io->out ? 4 * b->n_bus * F : 0; s->mix = io->mix ? 4 * b->n_bus * F : 0; break;
    case CPROC_CUDA_SQUARE_GRAIN: case CPROC_CUDA_ONEPOLE:
        s->in = 4 * n * F; s->out = 4 * n * F; break;
    case CPROC_CUDA_WORD_CLOCK: s->out = 4 * n * F; break;
    case CPROC_CUDA_SQUARE_GRAIN_MIX:
        s->out = io->out ? 8 * F : 0; s->mix = io->mix ? 8 * F : 0; break;
    case CPROC_CUDA_XVOICE:
        s->out = io->out ? 8 * n * F : 0; s->mix = io->mix ? 8 * F : 0; break;
    default: return -1;
    }
    return 0;
}

extern "C" {

static int dispatch(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io) {
    switch (b->cfg.proc) {
    case CPROC_CUDA_GRAPH: return launch_graph(b, F, io);
    case CPROC_CUDA_PDM: return launch_pdm(b, F, io);
    case CPROC_CUDA_PDM_V1: return launch_pdm_v1(b, F, io);
    case CPROC_CUDA_PDM_V2: return launch_pdm_v2(b, F, io);
    case CPROC_CUDA_PWM: return launch_pwm(b, F, io);
    case CPROC_CUDA_VOICE_BANK: return launch_voice_bank(b, F, io);
    case CPROC_CUDA_SQUARE_GRAIN: return launch_square_grain(b, F, io);
    case CPROC_CUDA_SQUARE_GRAIN_MIX: return launch_square_grain_mix(b, F, io);
    case CPROC_CUDA_XVOICE: return launch_xvoice(b, F, io);
    case CPROC_CUDA_ONEPOLE: return launch_onepole(b, F, io);
    case CPROC_CUDA_WORD_CLOCK: return launch_word_clock(b, F, io);
    }
    return cproc_set_err(b->ctx, CPROC_CUDA_EINVAL, "run: unknown processor");
}

int cproc_cuda_run_dev(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io) {
    if (!b || !io) return cproc_set_err(b ? b->ctx : nullptr, CPROC_CUDA_EINVAL, "run_dev: NULL argument");
    if (io->layout > CPROC_CUDA_TILED) return cproc_set_err(b->ctx, CPROC_CUDA_EINVAL, "run_dev: unknown layout %u", io->layout);
    CK(b->ctx, cudaSetDevice(b->ctx->device));
    return dispatch(b, F, io);
}

static int grow(cproc_cuda_ctx *ctx, void **p, size_t *cap, size_t need) {
    if (need <= *cap) return 0;
    if (*p) cudaFree(*p);
    *p = nullptr; *cap = 0;
    CK(ctx, cudaMalloc(p, need));
    *cap = need;
    return 0;
}

int cproc_cuda_run(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io) {
    if (!b || !io) return cproc_set_err(b ? b->ctx : nullptr, CPROC_CUDA_EINVAL, "run: NULL argument");
    cproc_cuda_ctx *ctx = b->ctx;
    if (io->layout > CPROC_CUDA_TILED) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "run: unknown layout %u", io->layout);
    CK(ctx, cudaSetDevice(ctx->device));
    cproc_io_sizes sz;
    if (cproc_io_bytes(b, F, io, &sz)) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "run: unknown processor");
    if (F == 0) return 0;
    int rc;
    cproc_cuda_io d = *io;
    cudaStream_t st = ctx->stream;
    // ---- small blocks (the JACK / Pd period: a few KB): one CUDA graph per (batch, shape) ----------------------
    // A period of a real-time host is launch-latency bound: pageable H2D + kernels + pageable D2H + sync are 4-6
    // driver calls.  For processors whose kernel arguments depend only on the batch and the shape (not on a
    // per-call counter: the PDM processors carry control_div_count and epochs) the second call with a given shape
    // captures [H2D from pinned staging, the launches of dispatch(), D2H to pinned staging] and every later call
    // is two host memcpys around one cudaGraphLaunch.
    const uint32_t proc = b->cfg.proc;
    const bool graphable = ctx->run_graph && !b->bus && sz.in + sz.in2 + sz.ctl + sz.out + sz.mix <= (256u << 10) &&
        ((proc == CPROC_CUDA_GRAPH && b->cfg.mode != CPROC_CUDA_GRAPH_SCAN) || proc == CPROC_CUDA_VOICE_BANK || proc == CPROC_CUDA_SQUARE_GRAIN ||
         proc == CPROC_CUDA_WORD_CLOCK || proc == CPROC_CUDA_PWM || (proc == CPROC_CUDA_ONEPOLE && b->cfg.mode != CPROC_CUDA_ONEPOLE_SCAN));
    // Zero copy (the kernels work on the pinned staging itself) only where the kernel that will run moves its streams
    // in bulk -- the PLANAR staging kernels (one PCIe round trip per tile) and the voice bank's coalesced stores.  The
    // scalar fallbacks read a word per tick: over PCIe that is a round trip per tick.  An integer mix bus may be
    // accumulated with atomics: device memory only.
    // The graph mix kernel reads and writes per instance and frame: only a mix-only render without input streams qualifies
    // (its group sums go to the batch's device scratch, the bus mix straight to the staging).
    const bool zc_ok = io->layout == CPROC_CUDA_PLANAR && ctx->planar_bulk != 0 &&
        (proc == CPROC_CUDA_VOICE_BANK ? io->mix == nullptr
         : proc == CPROC_CUDA_PWM ? F % 16 == 0
         : proc == CPROC_CUDA_GRAPH && io->mix ? !io->in && !io->in2 && !io->out
         : F % 4 == 0);
    // run_graph 3: no graph and no copies -- direct launches on the pinned staging (one launch + one sync per period)
    if (ctx->run_graph >= 3 && graphable && zc_ok && sz.in + sz.in2 + sz.ctl + sz.out + sz.mix <= (64u << 10)) {
        cproc_cuda_batch::run_graph &g = b->rg;
        const size_t want[5] = {io->in ? sz.in : 0, io->in2 ? sz.in2 : 0, io->ctl ? sz.ctl : 0, io->out ? sz.out : 0, io->mix ? sz.mix : 0};
        size_t off[5], total = 0;
        for (int k = 0; k < 5; ++k) { off[k] = total; total += (want[k] + 255) & ~(size_t)255; }
        if (g.cap < total) {
            if (g.exec) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; g.seen = 0; g.F = 0; }
            CK(ctx, cudaStreamSynchronize(st));
            if (g.h) cudaFreeHost(g.h);
            g.h = nullptr; g.cap = 0;
            CK(ctx, cudaHostAlloc((void **)&g.h, total < 4096 ? 4096 : total, cudaHostAllocDefault));
            g.cap = total < 4096 ? 4096 : total;
        }
        const void *src[3] = {io->in, io->in2, io->ctl};
        for (int k = 0; k < 3; ++k) if (want[k]) memcpy(g.h + off[k], src[k], want[k]);
        if (want[0]) d.in = g.h + off[0];
        if (want[1]) d.in2 = g.h + off[1];
        if (want[2]) d.ctl = g.h + off[2];
        if (want[3]) d.out = g.h + off[3];
        if (want[4]) d.mix = g.h + off[4];
        if ((rc = dispatch(b, F, &d))) return rc;
        if (b->ride_state) CK(ctx, cudaMemcpyAsync(b->st_h, b->d_state, sizeof(uint32_t) * b->state_words * b->npad, cudaMemcpyDeviceToHost, st));
        CK(ctx, cudaStreamSynchronize(st));
        if (want[3]) memcpy(io->out, g.h + off[3], want[3]);
        if (want[4]) memcpy(io->mix, g.h + off[4], want[4]);
        return 0;
    }
    if (graphable) {
        cproc_cuda_batch::run_graph &g = b->rg;
        const size_t want[5] = {io->in ? sz.in : 0, io->in2 ? sz.in2 : 0, io->ctl ? sz.ctl : 0, io->out ? sz.out : 0, io->mix ? sz.mix : 0};
        const bool same = g.F == F && g.layout == io->layout && g.opt_epoch == ctx->opt_epoch && !memcmp(g.sz, want, sizeof(want));
        if (!same) {                                       // new shape: this call runs the ordinary way and warms every lazy allocation
            if (g.exec) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; }
            g.F = F; g.layout = io->layout; g.opt_epoch = ctx->opt_epoch; memcpy(g.sz, want, sizeof(want)); g.seen = 0;
        }
        size_t off[5], total = 0;
        for (int k = 0; k < 5; ++k) { off[k] = total; total += (want[k] + 255) & ~(size_t)255; }
        if (same && g.seen == 1 && !g.exec && g.cap < total) {   // pinned staging; without it the ordinary path stays
            if (g.h) cudaFreeHost(g.h);
            g.h = nullptr; g.cap = 0;
            if (cudaHostAlloc((void **)&g.h, total, cudaHostAllocDefault) == cudaSuccess) g.cap = total;
            else { cudaGetLastError(); g.h = nullptr; g.seen = 2; }
        }
        if (same && g.seen == 1 && !g.exec) {              // second call with this shape: capture
            if (want[0] && (rc = grow(ctx, &b->d_in, &b->cap_in, sz.in))) return rc;
            if (want[1] && (rc = grow(ctx, &b->d_in2, &b->cap_in2, sz.in2))) return rc;
            if (want[2] && (rc = grow(ctx, &b->d_ctl, &b->cap_ctl, sz.ctl))) return rc;
            if (want[3] && (rc = grow(ctx, &b->d_out, &b->cap_out, sz.out))) return rc;
            if (want[4] && (rc = grow(ctx, &b->d_out2, &b->cap_out2, sz.mix))) return rc;
            cudaGraph_t graph = nullptr;
            const uint64_t launches0 = ctx->launches;
            bool ok = cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) == cudaSuccess;
            // run_graph 2: no copy nodes at all -- the kernels read and write the pinned staging itself (pinned host memory
            // is device-addressable at the same address under UVA; a block is a few hundred bytes, one PCIe round trip)
            const bool zc = ctx->run_graph >= 2 && zc_ok;
            if (ok) {
                if (want[0]) { if (zc) d.in = g.h + off[0]; else { ok = ok && cudaMemcpyAsync(b->d_in, g.h + off[0], want[0], cudaMemcpyHostToDevice, st) == cudaSuccess; d.in = b->d_in; } }
                if (want[1]) { if (zc) d.in2 = g.h + off[1]; else { ok = ok && cudaMemcpyAsync(b->d_in2, g.h + off[1], want[1], cudaMemcpyHostToDevice, st) == cudaSuccess; d.in2 = b->d_in2; } }
                if (want[2]) { if (zc) d.ctl = g.h + off[2]; else { ok = ok && cudaMemcpyAsync(b->d_ctl, g.h + off[2], want[2], cudaMemcpyHostToDevice, st) == cudaSuccess; d.ctl = b->d_ctl; } }
                if (want[3]) d.out = zc ? (void *)(g.h + off[3]) : b->d_out;
                if (want[4]) d.mix = zc ? (void *)(g.h + off[4]) : b->d_out2;
                ok = ok && dispatch(b, F, &d) == 0;
                if (want[3] && !zc) ok = ok && cudaMemcpyAsync(g.h + off[3], b->d_out, want[3], cudaMemcpyDeviceToHost, st) == cudaSuccess;
                if (want[4] && !zc) ok = ok && cudaMemcpyAsync(g.h + off[4], b->d_out2, want[4], cudaMemcpyDeviceToHost, st) == cudaSuccess;
                ok = (cudaStreamEndCapture(st, &graph) == cudaSuccess) && ok && graph;
            }
            if (ok) ok = cudaGraphInstantiate(&g.exec, graph, 0) == cudaSuccess;
            if (graph) cudaGraphDestroy(graph);
            g.kernels = (uint32_t)(ctx->launches - launches0);
            ctx->launches = launches0;                     // nothing has run yet: replays count below
            if (!ok) { cudaGetLastError(); g.exec = nullptr; g.seen = 2; ctx->err.clear(); }
            d = *io;
        }
        if (same && g.exec) {
            const void *src[3] = {io->in, io->in2, io->ctl};
            for (int k = 0; k < 3; ++k) if (want[k]) memcpy(g.h + off[k], src[k], want[k]);
            CK(ctx, cudaGraphLaunch(g.exec, st));
            ctx->launches += g.kernels;
            if (b->ride_state) CK(ctx, cudaMemcpyAsync(b->st_h, b->d_state, sizeof(uint32_t) * b->state_words * b->npad, cudaMemcpyDeviceToHost, st));
            CK(ctx, cudaStreamSynchronize(st));
            if (want[3]) memcpy(io->out, g.h + off[3], want[3]);
            if (want[4]) memcpy(io->mix, g.h + off[4], want[4]);
            return 0;
        }
        if (g.seen == 0) g.seen = 1;
    }
    if (io->in && sz.in) {
        if ((rc = grow(ctx, &b->d_in, &b->cap_in, sz.in))) return rc;
        CK(ctx, cudaMemcpyAsync(b->d_in, io->in, sz.in, cudaMemcpyHostToDevice, st));
        d.in = b->d_in;
    }
    if (io->in2 && sz.in2) {
        if ((rc = grow(ctx, &b->d_in2, &b->cap_in2, sz.in2))) return rc;
        CK(ctx, cudaMemcpyAsync(b->d_in2, io->in2, sz.in2, cudaMemcpyHostToDevice, st));
        d.in2 = b->d_in2;
    }
    if (io->ctl && sz.ctl) {
        if ((rc = grow(ctx, &b->d_ctl, &b->cap_ctl, sz.ctl))) return rc;
        CK(ctx, cudaMemcpyAsync(b->d_ctl, io->ctl, sz.ctl, cudaMemcpyHostToDevice, st));
        d.ctl = b->d_ctl;
    }
    if (io->out && sz.out) {
        if ((rc = grow(ctx, &b->d_out, &b->cap_out, sz.out))) return rc;
        d.out = b->d_out;
    }
    void *d_mix_user = nullptr;
    if (io->mix && sz.mix) {
        // the mix staging buffer is separate from the launcher's scratch (d_mix)
        if ((rc = grow(ctx, &b->d_out2, &b->cap_out2, sz.mix))) return rc;
        d_mix_user = b->d_out2;
        d.mix = d_mix_user;
    }
    if ((rc = dispatch(b, F, &d))) return rc;
    if (io->out && sz.out) CK(ctx, cudaMemcpyAsync(io->out, d.out, sz.out, cudaMemcpyDeviceToHost, st));
    if (io->mix && sz.mix) CK(ctx, cudaMemcpyAsync(io->mix, d_mix_user, sz.mix, cudaMemcpyDeviceToHost, st));
    if (b->ride_state) CK(ctx, cudaMemcpyAsync(b->st_h, b->d_state, sizeof(uint32_t) * b->state_words * b->npad, cudaMemcpyDeviceToHost, st));
    CK(ctx, cudaStreamSynchronize(st));
    return 0;
}

// One period of a real-time host whose state lives in the HOST's structs (synth.c: struct voice inside struct synth, note_on /
// note_off write it between periods): records in, render, records out -- as ONE stream sequence with one synchronisation.
// The records travel through a pinned SoA staging buffer owned by the batch (allocated by the first call: warm up before the
// real-time thread exists); nothing is allocated afterwards and the only blocking driver call is the period's own sync.
int cproc_cuda_run_period(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io, void *state_aos, size_t stride) {
    if (!b || !io) return cproc_set_err(b ? b->ctx : nullptr, CPROC_CUDA_EINVAL, "run_period: NULL argument");
    cproc_cuda_ctx *ctx = b->ctx;
    if (!state_aos) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "run_period: state is NULL");
    const uint32_t words = b->state_words;
    if (stride == 0) stride = 4u * words;
    if (words == 0 || stride < 4u * words) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "run_period: stride %zu smaller than the state record (%u bytes)", stride, 4u * words);
    if (F == 0) return 0;
    CK(ctx, cudaSetDevice(ctx->device));
    const size_t bytes = sizeof(uint32_t) * words * b->npad;
    if (!b->st_h) {
        CK(ctx, cudaHostAlloc((void **)&b->st_h, bytes, cudaHostAllocDefault));
        memset(b->st_h, 0, bytes);
    }
    uint8_t *rec = (uint8_t *)state_aos;
    for (uint64_t i = 0; i < b->n; ++i)
        for (uint32_t w = 0; w < words; ++w) memcpy(b->st_h + (size_t)w * b->npad + i, rec + i * stride + 4u * w, 4);
    if (b->cfg.proc == CPROC_CUDA_SQUARE_GRAIN_MIX) {
        b->grain_odd_state = false;
        for (uint64_t i = 0; i < b->n; ++i) b->grain_odd_state |= grain_state_odd(b->st_h[i]);
    }
    CK(ctx, cudaMemcpyAsync(b->d_state, b->st_h, bytes, cudaMemcpyHostToDevice, ctx->stream));
    b->ride_state = true;
    const int rc = cproc_cuda_run(b, F, io);               // ends with the records' D2H copy and the period's one sync
    b->ride_state = false;
    if (rc) return rc;
    for (uint64_t i = 0; i < b->n; ++i)
        for (uint32_t w = 0; w < words; ++w) memcpy(rec + i * stride + 4u * w, b->st_h + (size_t)w * b->npad + i, 4);
    return 0;
}

// Chunked render with the D2H copy of chunk k overlapped with the render of
// chunk k+1 (two device slabs, copy stream + events); the host side trails by
// one chunk and hands finished slabs to on_chunk.
int cproc_cuda_run_stream(cproc_cuda_batch *b, uint64_t F_total, uint64_t F_chunk, const cproc_cuda_io *io,
                          uint32_t ring_chunks, cproc_cuda_chunk_fn on_chunk, void *user) {
    if (!b || !io) return cproc_set_err(b ? b->ctx : nullptr, CPROC_CUDA_EINVAL, "run_stream: NULL argument");
    cproc_cuda_ctx *ctx = b->ctx;
    if (b->cfg.proc != CPROC_CUDA_PDM_V1 && b->cfg.proc != CPROC_CUDA_PDM_V2)
        return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "run_stream: only the PDM processors stream");
    if (F_chunk == 0 || F_total % F_chunk) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "run_stream: F_total must be a multiple of F_chunk");
    if (io->in2) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "run_stream: external dither not supported");
    if (!io->out) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "run_stream: out is NULL");
    if (ring_chunks == 1) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "run_stream: ring_chunks must be 0 or >= 2");
    CK(ctx, cudaSetDevice(ctx->device));
    const uint64_t n_chunks = F_total / F_chunk;
    const uint64_t ring = ring_chunks ? ring_chunks : n_chunks;
    cproc_io_sizes sz;
    cproc_cuda_io probe = *io;
    probe.n_ctl = 0;
    cproc_io_bytes(b, F_chunk, &probe, &sz);
    int rc;
    if ((rc = grow(ctx, &b->d_out, &b->cap_out, sz.out))) return rc;
    if ((rc = grow(ctx, &b->d_out2, &b->cap_out2, sz.out))) return rc;
    const uint32_t div = 1u << b->cfg.ctl_div_log;
    uint64_t rows_done = 0;
    if (io->ctl) {
        size_t need = 4ull * io->n_ctl * b->n;
        if ((rc = grow(ctx, &b->d_ctl, &b->cap_ctl, need))) return rc;
        CK(ctx, cudaMemcpyAsync(b->d_ctl, io->ctl, need, cudaMemcpyHostToDevice, ctx->stream));
    }
    cudaEvent_t done[2], copied[2];
    for (int i = 0; i < 2; ++i) { cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming); cudaEventCreateWithFlags(&copied[i], cudaEventDisableTiming); }
    rc = 0;
    for (uint64_t k = 0; k < n_chunks && !rc; ++k) {
        const int s = (int)(k & 1);
        void *slab = s ? b->d_out2 : b->d_out;
        if (k >= 2) cudaStreamWaitEvent(ctx->stream, copied[s], 0);   // device slab copied out
        cproc_cuda_io d = *io;
        d.out = slab;
        if (io->ctl && b->cfg.proc == CPROC_CUDA_PDM_V2) {
            uint64_t first = b->count == 0 ? 0 : div - b->count;
            uint64_t rows = F_chunk > first ? 1 + (F_chunk - first - 1) / div : 0;
            d.ctl = (const uint32_t *)b->d_ctl + rows_done * b->n;
            d.n_ctl = (uint32_t)(io->n_ctl - rows_done);
            rows_done += rows;
        }
        rc = dispatch(b, F_chunk, &d);
        if (rc) break;
        cudaEventRecord(done[s], ctx->stream);
        cudaStreamWaitEvent(ctx->copy_stream, done[s], 0);
        rc = cproc_check(ctx, cudaMemcpyAsync((uint8_t *)io->out + (k % ring) * sz.out, slab, sz.out, cudaMemcpyDeviceToHost, ctx->copy_stream), "memcpy(D2H chunk)");
        cudaEventRecord(copied[s], ctx->copy_stream);
        if (k >= 1 && !rc) {
            // trail by one chunk: chunk k-1 is (about to be) on the host
            rc = cproc_check(ctx, cudaEventSynchronize(copied[s ^ 1]), "run_stream chunk sync");
            if (!rc && on_chunk) on_chunk(user, k - 1, (const uint8_t *)io->out + ((k - 1) % ring) * sz.out, sz.out);
        }
    }
    cudaStreamSynchronize(ctx->stream);
    cudaError_t e = cudaStreamSynchronize(ctx->copy_stream);
    for (int i = 0; i < 2; ++i) { cudaEventDestroy(done[i]); cudaEventDestroy(copied[i]); }
    if (rc) return rc;
    if ((rc = cproc_check(ctx, e, "run_stream sync"))) return rc;
    if (on_chunk && n_chunks) on_chunk(user, n_chunks - 1, (const uint8_t *)io->out + ((n_chunks - 1) % ring) * sz.out, sz.out);
    return 0;
}

// ---- evented graph driver (mod_cproc_plugin.c:20-38) ---------------------------
static int ev_check(cproc_cuda_batch *b, const char *who) {
    if (!b) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "%s: batch is NULL", who);
    if (b->cfg.proc != CPROC_CUDA_GRAPH) return cproc_set_err(b->ctx, CPROC_CUDA_EINVAL, "%s: not a graph batch", who);
    if (b->ev_in.empty()) b->ev_in.assign((size_t)b->n * b->cfg.n_inputs, 0u);   // w cproc_input[CPROC_NB_INPUTS], static storage: zero
    return 0;
}

int cproc_cuda_graph_set_input(cproc_cuda_batch *b, uint64_t instance, uint32_t i, uint32_t v) {
    int rc;
    if ((rc = ev_check(b, "graph_set_input"))) return rc;
    if (i >= b->cfg.n_inputs) return cproc_set_err(b->ctx, CPROC_CUDA_EINVAL, "graph_set_input: input %u of %u", i, b->cfg.n_inputs);
    if (instance == CPROC_CUDA_ALL_INSTANCES) { for (uint64_t k = 0; k < b->n; ++k) b->ev_in[(size_t)k * b->cfg.n_inputs + i] = v; return 0; }
    if (instance >= b->n) return cproc_set_err(b->ctx, CPROC_CUDA_EINVAL, "graph_set_input: instance %llu of %llu", (unsigned long long)instance, (unsigned long long)b->n);
    b->ev_in[(size_t)instance * b->cfg.n_inputs + i] = v;
    return 0;
}

static int ev_tick(cproc_cuda_batch *b, const uint32_t *changed_rows, uint32_t *out) {
    const uint32_t n_out = b->cfg.n_outputs ? b->cfg.n_outputs : 1;
    b->ev_out.resize((size_t)b->n * n_out);
    cproc_cuda_io io;
    memset(&io, 0, sizeof(io));
    io.in = b->ev_in.data();          // [inst][n_inputs][F = 1]
    io.in2 = changed_rows;            // [inst][F = 1] or NULL (= -1)
    io.out = b->ev_out.data();        // [inst][n_outputs][F = 1]
    io.layout = CPROC_CUDA_PLANAR;
    int rc = cproc_cuda_run(b, 1, &io);
    if (rc) return rc;
    if (out) memcpy(out, b->ev_out.data(), sizeof(uint32_t) * b->ev_out.size());
    return 0;
}

int cproc_cuda_graph_tick(cproc_cuda_batch *b, uint32_t changed, uint32_t *out) {
    int rc;
    if ((rc = ev_check(b, "graph_tick"))) return rc;
    if (changed == 0xFFFFFFFFu) return ev_tick(b, nullptr, out);
    b->ev_chg.assign((size_t)b->n, changed);
    return ev_tick(b, b->ev_chg.data(), out);
}

int cproc_cuda_graph_event(cproc_cuda_batch *b, uint64_t instance, uint32_t i, uint32_t v, uint32_t *out) {
    int rc;
    if ((rc = ev_check(b, "graph_event"))) return rc;
    if (instance >= b->n) return cproc_set_err(b->ctx, CPROC_CUDA_EINVAL, "graph_event: instance %llu of %llu", (unsigned long long)instance, (unsigned long long)b->n);
    if ((rc = cproc_cuda_graph_set_input(b, instance, i, v))) return rc;
    const uint32_t n_out = b->cfg.n_outputs ? b->cfg.n_outputs : 1;
    if (b->n == 1) rc = ev_tick(b, nullptr, nullptr);
    else {                                                   // only the addressed graph ticks: the others see changed = 0
        b->ev_chg.assign((size_t)b->n, 0u);
        b->ev_chg[(size_t)instance] = 0xFFFFFFFFu;
        rc = ev_tick(b, b->ev_chg.data(), nullptr);
    }
    if (rc) return rc;
    if (out) memcpy(out, b->ev_out.data() + (size_t)instance * n_out, sizeof(uint32_t) * n_out);
    return 0;
}

int cproc_cuda_mix_to_float(cproc_cuda_batch *b, const void *imix_dev, float *out_dev, uint64_t count) {
    if (!b || !imix_dev || !out_dev) return cproc_set_err(b ? b->ctx : nullptr, CPROC_CUDA_EINVAL, "mix_to_float: NULL argument");
    cproc_cuda_ctx *ctx = b->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    if (count == 0) return 0;
    const unsigned grid = (unsigned)ceil_div_u64(count, 256);
    if (b->cfg.proc == CPROC_CUDA_VOICE_BANK)
        k_voice_finish<<<grid, 256, 0, ctx->stream>>>((const int32_t *)imix_dev, out_dev, count, b->cfg.mode);
    else if (b->cfg.proc == CPROC_CUDA_SQUARE_GRAIN_MIX)
        k_imix_to_float<<<grid, 256, 0, ctx->stream>>>((const int32_t *)imix_dev, out_dev, count, 0x1p-7f);
    else return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "mix_to_float: processor has no integer mix bus");
    CK_LAUNCH(ctx, "k_mix_to_float");
    return 0;
}

// ---- memory + timing helpers --------------------------------------------------

int cproc_cuda_dev_alloc(cproc_cuda_ctx *ctx, size_t bytes, void **dev) {
    if (!ctx || !dev) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "dev_alloc: NULL argument");
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMalloc(dev, bytes));
    return 0;
}
int cproc_cuda_dev_free(cproc_cuda_ctx *ctx, void *dev) {
    if (!ctx) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "dev_free: ctx is NULL");
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaFree(dev));
    return 0;
}
int cproc_cuda_host_alloc(cproc_cuda_ctx *ctx, size_t bytes, void **pinned) {
    if (!ctx || !pinned) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "host_alloc: NULL argument");
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaHostAlloc(pinned, bytes, cudaHostAllocDefault));
    return 0;
}
int cproc_cuda_host_free(cproc_cuda_ctx *ctx, void *pinned) {
    if (!ctx) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "host_free: ctx is NULL");
    CK(ctx, cudaFreeHost(pinned));
    return 0;
}
int cproc_cuda_memcpy_h2d(cproc_cuda_ctx *ctx, void *dev, const void *host, size_t bytes) {
    if (!ctx) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "memcpy_h2d: ctx is NULL");
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}
int cproc_cuda_memcpy_d2h(cproc_cuda_ctx *ctx, void *host, const void *dev, size_t bytes) {
    if (!ctx) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "memcpy_d2h: ctx is NULL");
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}
int cproc_cuda_memset(cproc_cuda_ctx *ctx, void *dev, int value, size_t bytes) {
    if (!ctx) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "memset: ctx is NULL");
    CK(ctx, cudaSetDevice(ctx->device));
    CK(ctx, cudaMemsetAsync(dev, value, bytes, ctx->stream));
    return 0;
}
int cproc_cuda_timer_start(cproc_cuda_ctx *ctx) {
    if (!ctx) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "timer_start: ctx is NULL");
    CK(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    return 0;
}
int cproc_cuda_timer_stop(cproc_cuda_ctx *ctx, float *ms) {
    if (!ctx || !ms) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "timer_stop: NULL argument");
    CK(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    CK(ctx, cudaEventSynchronize(ctx->ev1));
    CK(ctx, cudaEventElapsedTime(ms, ctx->ev0, ctx->ev1));
    return 0;
}

} // extern "C"
