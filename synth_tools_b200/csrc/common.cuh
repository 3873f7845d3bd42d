// common.cuh -- shared internals of libcproc_cuda (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>
#include "../../include/cproc_cuda.h"

#define CPROC_N_SM 148  // B200

struct cproc_cuda_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;      // render stream (caller's or ours)
    cudaStream_t copy_stream = nullptr; // D2H overlap in run_stream
    cudaStream_t aux_stream = nullptr;  // high-priority side stream (XVOICE_SCAN pre-passes), created on first use
    cudaEvent_t aux_ev[17] = {};        // scan-done[8], render-done[8], fork
    bool own_stream = false;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::string err;
    uint64_t launches = 0;
    // tuning knobs (cproc_cuda_set_option)
    int pdm_block = 64;       // threads per block of the PDM kernels
    int pdm_tpb = 2;          // plain PDM kernels, banks of <= 4: 1 thread per bank, 0 thread per channel (every thread replays its bank's generator), 2 auto
    int pdm_ws = 1;           // PDM v2: 1 = producer / consumer kernel under the dynamic (group, slice) schedule (k_pdm_v2_ws4), 0 = plain thread-per-bank / per-channel kernels
    int pdm_tlog = 7;         // k_pdm_v2_ws4: log2 of the dither batch (ticks per FULL / EMPTY hand-off), 6 or 7
    int pdm_v1_chains = 2;    // v1 thread-per-bank TILED kernels: PRNG chains per lane (1 or 2)
    int pdm_planar_bulk = 2;  // k_pdm_v2_ws4: PLANAR duty rows staged in shared memory and stored as tensor-TMA boxes (0: scattered 16-byte stores)
    int pdm_ctas_per_sm = 4;  // k_pdm_v2_ws4: persistent blocks per SM
    int pdm_slice_batches = 64;   // k_pdm_v2_ws4: ticks per work item, in units of 64 ticks
    uint32_t *d_work = nullptr;   // k_pdm_v2_ws4: work counter + exit counter
    uint32_t *d_sm_rank = nullptr;   // per-SM block arrival counters (producer placement)
    uint32_t *d_jump[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};   // xorshift32 jump LUTs M^(T/2) per batch length 2^(6+i)
    uint32_t *d_jump16 = nullptr;   // M^16 (v1 two-chain PRNG)
    int pdm_persist = 1;      // v1: persistent McNaughton-scheduled kernel when thread == bank (0 never, 1 auto, 2 always)
    int pdm_warps_per_smsp = 1;
    int n_sm = CPROC_N_SM;
    int voice_fpt = 0;        // voice bank: frames per thread (0 = by frame count; 1, 2, 4, 8)
    int grain_blocks_per_sm = 2;
    int grain_mix2 = 2;       // 0: float kernel; 1: register-accumulator / integer-threshold kernel; 2: predicate-state kernel
    int planar_bulk = 2;      // square_grain / pdm_raw / onepole / pwm / word-clock / generated-graph streams: 0 scalar kernels, 2 tensor-TMA staging (PLANAR), k_interleaved4 (INTERLEAVED)
    int graph_vec4 = 1;       // interleaved generated graphs: four instances per thread when n % 4 == 0
    int graph_jit = 1;        // 1: generated graphs are compiled with NVRTC; 0: table-driven kernel
    int xvoice_vpt = 0;       // k_xvoice_mix: voices per thread per L2-resident tile (0 = default)
    int xvoice_mix2_per_sm = 0;   // k_xvoice_mix2: co-resident blocks per SM on this device (occupancy API, cached at the first launch)
    int xvoice_mix2_blocks = 0;   // k_xvoice_mix2: resident blocks per SM (0 = by the round model in launch_xvoice, else 1..3)
    int xvoice_mix2 = 1;      // mix-only XVOICE render: 1 = k_xvoice_mix2 (voice pairs on the packed fp32 pipe, state tiles in shared memory), 0 = k_xvoice_mix
    int xvoice_groups = 0;    // XVOICE_SCAN: variant groups pipelined over the two streams (0 = automatic)
    int xvoice_chunk = 0;     // XVOICE_SCAN: frames per time chunk (0 = automatic)
    uint64_t opt_epoch = 0;   // bumped by every set_option
    int run_graph = 2;        // cproc_cuda_run, small blocks: 0 staged copies, 1 CUDA graph with copy nodes, 2 CUDA graph on pinned staging (zero copy), 3 direct launches on pinned staging
    int xvoice_closed = 1;    // XVOICE_SCAN: zero-state pass in closed form per phase wrap (0: ticked in fp64)
};

// NVRTC-compiled kernels of one graph (graph_front.cu); state 0 = not tried, 1 = ready, 2 = failed
struct cproc_graph_jit {
    int state = 0;
    std::vector<char> cubin;
    cudaLibrary_t lib = nullptr;
    cudaKernel_t k_il = nullptr, k_il4 = nullptr, k_ps = nullptr, k_pt = nullptr, k_mix = nullptr;
    uint32_t pt_block = 0, pt_smem = 0, mix_warps = 0;   // block and shared memory of graph_planar_tma; mix_warps: block of the bus-mix kernel graph_mix, in warps
};

struct cproc_cuda_bus;
struct cproc_cuda_batch {
    cproc_cuda_ctx *ctx = nullptr;
    cproc_cuda_bus *bus = nullptr; uint32_t bus_mode = 0;   // mix bus attached to this batch (cproc_cuda_bus_attach): the render launch exchanges its mix itself
    cproc_cuda_config cfg{};
    std::vector<cproc_cuda_node> nodes;     // copy of cfg.nodes
    std::vector<uint32_t> node_off;         // state word offset per node
    std::vector<uint32_t> outs;             // graph: output nodes, one per output stream (>= 1)
    uint64_t n = 0;                         // instances
    uint64_t npad = 0;                      // SoA row length (>= n)
    uint64_t n_banks = 0;
    uint64_t n_bus = 0;                     // voice bank / graph mix: buses of cfg.voices_per_bus instances
    uint32_t state_words = 0, param_words = 0;
    uint32_t *d_state = nullptr;            // [state_words][npad]
    uint32_t *d_param = nullptr;            // [param_words][npad]
    uint32_t *d_prng = nullptr;             // [n_banks] dither generator state
    uint32_t *d_prng2 = nullptr;            // [n_banks] the other half of the double buffer (a launch reads one, writes the other)
    uint32_t *d_prng_g = nullptr;           // [groups][32] generator state between the time slices of a group (k_pdm_v2_ws4)
    cproc_cuda_node *d_nodes = nullptr;
    uint32_t count = 0;                     // control_div_count
    // staging for host-buffer runs (grown on demand)
    void *d_in = nullptr, *d_in2 = nullptr, *d_ctl = nullptr, *d_out = nullptr, *d_mix = nullptr;
    size_t cap_in = 0, cap_in2 = 0, cap_ctl = 0, cap_out = 0, cap_mix = 0;
    void *d_out2 = nullptr; size_t cap_out2 = 0;   // second slab for run_stream
    uint32_t *d_aux = nullptr; bool aux_dirty = true; uint32_t aux_weird = 0;   // derived parameter rows (grain mix integer thresholds)
    bool grain_odd_state = false;           // grain mix: a state uploaded outside {+-0, +-0.5} (k_grain_mix until the next upload)
    void *d_scratch = nullptr; size_t cap_scratch = 0;   // per-chunk start-state tables (XVOICE_SCAN, GRAPH_SCAN); graph mix: group sums of a frame slice
    uint32_t *d_acc = nullptr; size_t cap_acc = 0;       // voice bank: integer accumulators of a bus split over tiles + tickets; all zero between launches
    unsigned long long *d_flags = nullptr;         // persistent-kernel progress words
    uint64_t n_flags = 0;
    unsigned long long epoch = 0;
    cproc_graph_jit jit[2];                        // [changed stream present]
    std::vector<uint32_t> ev_in, ev_chg, ev_out;   // evented driver (cproc_cuda_graph_set_input / _tick): cproc_input[] per instance, changed, outputs
    std::string jit_log;
    // small host-buffer runs replayed as one CUDA graph (H2D copies, the kernels, D2H copies): abi.cu
    struct run_graph {
        uint64_t F = 0; uint32_t layout = 0; size_t sz[5] = {0, 0, 0, 0, 0};   // key: in, in2, ctl, out, mix bytes (0 = absent)
        uint64_t opt_epoch = 0;                    // ctx->opt_epoch at capture: an option change may select other kernels
        int seen = 0;                              // 1: ran once the ordinary way, 2: capture failed, keep the ordinary way
        cudaGraphExec_t exec = nullptr; uint32_t kernels = 0;
        uint8_t *h = nullptr; size_t cap = 0;      // pinned staging, the five regions back to back
    } rg;
    // cproc_cuda_run_period: the state records ride along with the period (pinned SoA staging, no call of its own)
    uint32_t *st_h = nullptr; bool ride_state = false;
};

int cproc_set_err(cproc_cuda_ctx *ctx, int code, const char *fmt, ...);
int cproc_check(cproc_cuda_ctx *ctx, cudaError_t e, const char *what);

#define CK(ctx, call) do { int _rc = cproc_check((ctx), (call), #call); if (_rc) return _rc; } while (0)
#define CK_LAUNCH(ctx, name) do { (ctx)->launches++; int _rc = cproc_check((ctx), cudaGetLastError(), name); if (_rc) return _rc; } while (0)

// One row per node kind: the field lists of the processor's DEF_PROC structs (cproc.h:134-148 for acc / edge, include/cproc_ext.h for
// the extension processors; glide / pdm: cproc_cuda.h).  *_f: bit k set = field k is a float.  pdm's state is {out, s1..sK}: 1 + K words.
struct cproc_kind_meta {
    const char *name;
    uint32_t n_state; const char *state[5]; uint32_t state_f;
    uint32_t n_param; const char *param[3]; uint32_t param_f;
    uint32_t n_input; const char *input[2]; uint32_t input_f;
    uint32_t n_config; const char *config[1];
};
static const cproc_kind_meta k_cproc_kinds[CPROC_CUDA_NODE_KINDS] = {
    {"acc",      1, {"out"}, 0,                                    0, {nullptr}, 0,                               1, {"in"}, 0,           0, {nullptr}},
    {"edge",     2, {"out", "last"}, 0,                            0, {nullptr}, 0,                               1, {"in"}, 0,           0, {nullptr}},
    {"glide",    5, {"out", "vel0", "pos1", "vel1", "count"}, 0,   0, {nullptr}, 0,                               1, {"in"}, 0,           1, {"div_log"}},
    {"pdm",      5, {"out", "s1", "s2", "s3", "s4"}, 0,            0, {nullptr}, 0,                               2, {"in", "dither"}, 0, 1, {"order_shift"}},
    {"phasor_f", 2, {"out", "phase"}, 1,                           1, {"inc"}, 0,                                 1, {"mod"}, 0,          0, {nullptr}},
    {"svf",      2, {"out", "bp"}, 3,                              2, {"f", "q"}, 3,                              1, {"in"}, 1,           0, {nullptr}},
    {"env",      3, {"out", "env", "t"}, 3,                        3, {"attack", "release", "gate_frames"}, 3,    1, {"in"}, 1,           0, {nullptr}},
    {"onepole",  1, {"out"}, 1,                                    1, {"a"}, 1,                                   1, {"in"}, 1,           0, {nullptr}},
    {"gain",     1, {"out"}, 1,                                    1, {"g"}, 1,                                   1, {"in"}, 1,           0, {nullptr}},
    {"asfloat",  1, {"out"}, 1,                                    0, {nullptr}, 0,                               1, {"in"}, 0,           0, {nullptr}},
    {"glide_f",  3, {"out", "step", "count"}, 3,                   0, {nullptr}, 0,                               1, {"in"}, 1,           1, {"div_log"}},
    {"mul",      1, {"out"}, 1,                                    0, {nullptr}, 0,                               2, {"in", "gain"}, 3,   0, {nullptr}},
};
static inline bool cproc_kind_out_float(uint32_t type) { const uint32_t k = CPROC_CUDA_NODE_KIND(type); return k < CPROC_CUDA_NODE_KINDS && (k_cproc_kinds[k].state_f & 1u); }
static inline uint32_t cproc_node_words(uint32_t type) {   // acc {out}; edge {out, last}; glide {out, vel0, pos1, vel1, count}; pdm {out, s1..sK}; extension processors: cproc_ext.h
    const uint32_t kind = CPROC_CUDA_NODE_KIND(type);
    if (kind == CPROC_CUDA_NODE_PDM) return 1u + (CPROC_CUDA_NODE_ARG(type) & 7u);
    return kind < CPROC_CUDA_NODE_KINDS ? k_cproc_kinds[kind].n_state : 1u;
}
static inline uint32_t cproc_node_param_words(uint32_t type) {
    const uint32_t kind = CPROC_CUDA_NODE_KIND(type);
    return kind < CPROC_CUDA_NODE_KINDS ? k_cproc_kinds[kind].n_param : 0u;
}
// Validity of row k of an ANF table (shared by alloc, the JIT and the patcher); `nodes` = the whole table (source types)
static inline const char *cproc_node_check(const cproc_cuda_node *nodes, uint32_t k, uint32_t n_inputs) {
    const cproc_cuda_node &nd = nodes[k];
    const uint32_t kind = CPROC_CUDA_NODE_KIND(nd.type), arg = CPROC_CUDA_NODE_ARG(nd.type);
    if (kind >= CPROC_CUDA_NODE_KINDS || (nd.type >> 16)) return "unknown node type";
    if ((kind == CPROC_CUDA_NODE_GLIDE || kind == CPROC_CUDA_NODE_GLIDE_F) && (arg < 1 || arg > 24)) return "glide needs a control divider log2 of 1..24";
    if (kind == CPROC_CUDA_NODE_PDM && ((arg & 7u) < 1 || (arg & 7u) > 4)) return "pdm order must be 1..4";
    if (kind != CPROC_CUDA_NODE_GLIDE && kind != CPROC_CUDA_NODE_GLIDE_F && kind != CPROC_CUDA_NODE_PDM && arg) return "this processor takes no config word";
    const cproc_kind_meta &m = k_cproc_kinds[kind];
    for (uint32_t j = 0; j < m.n_input; ++j) {
        const int32_t src = j ? nd.src2 : nd.src;
        if (src == CPROC_CUDA_SRC_ZERO) { if (kind <= CPROC_CUDA_NODE_PDM) return "input not connected"; continue; }   // the reference processors' inputs are always named
        if (src >= (int32_t)k) return j ? "second input reads a node that is not bound yet (ANF)" : "reads a node that is not bound yet (ANF)";
        if (src < 0 && (uint32_t)(-(src + 1)) >= n_inputs) return j ? "second input reads an input stream that does not exist" : "reads an input stream that does not exist";
        if (src >= 0 && cproc_kind_out_float(nodes[src].type) && !((m.input_f >> j) & 1u)) return "a float output feeds an integer input (undefined in C for negative values)";
    }
    return nullptr;
}
static inline uint64_t ceil_div_u64(uint64_t a, uint64_t b) { return (a + b - 1) / b; }

// Element sizes / stream sizes per processor (bytes for F frames).
struct cproc_io_sizes { size_t in, in2, ctl, out, mix; };
int cproc_io_bytes(const cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io, cproc_io_sizes *s);

// Kernel launchers (one translation unit per family).
int launch_graph(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io);
int launch_graph_scan(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io);
int cproc_graph_jit_get(cproc_cuda_batch *b, bool has_changed, cproc_graph_jit **out);
int launch_pdm(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io);
int launch_pdm_v1(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io);
int launch_pdm_v2(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io);
int launch_pwm(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io);
int launch_voice_bank(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io);
int launch_square_grain(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io);
int launch_square_grain_mix(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io);
int launch_xvoice(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io);
int launch_onepole(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io);
int launch_word_clock(cproc_cuda_batch *b, uint64_t F, const cproc_cuda_io *io);

// small conversion kernels shared across translation units
__global__ void k_imix_to_float(const int32_t *imix, float *mix, uint64_t count, float scale);
__global__ void k_voice_finish(const int32_t *isum, float *vec, uint64_t count, uint32_t mode);

// ---- device helpers -------------------------------------------------------
__device__ __forceinline__ uint32_t xorshift32_step(uint32_t x) {
    // uc_tools random_u32 stand-in (parity unpinned): Marsaglia (13,17,5)
    x ^= x << 13;
    x ^= x >> 17;
    x ^= x << 5;
    return x;
}

__device__ __forceinline__ void st_v4_stream(void *p, uint4 v) {
    // write-once output streams: keep them out of L1, evict-first in L2
    asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint4 ld_v4_stream(const void *p) {
    uint4 v;
    asm volatile("ld.global.cs.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}
