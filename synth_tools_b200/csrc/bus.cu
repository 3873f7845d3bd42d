// bus.cu -- the shared stereo mix bus across the GPUs of one box, over NVLink peer memory.
//
// The only exchange step of the path (SURVEY 8e): every rank has rendered the INTEGER mix
// of its shard of the voices (synth.c:169-195: int sum / OR of MSBs; square_grain mix in
// units of 2^-7); the bus is their sum (OR), a few KB, followed by one float scale
// (synth.c:180,194).  With NCCL that is an all-reduce launch plus the conversion kernel;
// here it is ONE kernel per rank: push the local mix into a slot of every peer's bus
// buffer with plain stores through the NVLink peer mapping, publish a flag per peer
// (release, system scope), wait for the peers' flags (acquire), add the slots in rank
// order -- the same order on every rank, although integer sums do not even need it -- and
// write the float bus.  Slots are double buffered by epoch parity, so a fast rank's next
// block cannot overwrite what a slow rank still reads.  One process per GPU: the buffers
// are shared with cudaIpc handles, which the host exchanges over whatever transport it
// has (bench/tests: torch.distributed all_gather).
//
// Two ways to run the exchange: as its own launch (cproc_cuda_bus_allreduce[_begin]: k_bus_allreduce below), or
// as the tail of the render kernel of a batch the bus is attached to (cproc_cuda_bus_attach: bus_fused.cuh).
#include "common.cuh"
#include "bus_fused.cuh"
#include <string.h>

struct cproc_cuda_bus {
    cproc_cuda_ctx *ctx = nullptr;
    int world = 1, rank = 0;
    uint64_t cap = 0;                    // int32 words per slot
    uint8_t *local = nullptr;            // [BUS_NPAR][world][cap] int32, then [BUS_NPAR][world] uint32 flags, status word, ticket, then [2][cap] staging
    // fused exchanges (attach): the reduce of the last pushed epoch still to be done (mode 2)
    uint32_t pend_epoch = 0, pend_op = 0, pend_scale = 0;
    uint64_t pend_count = 0;
    int32_t *pend_imix = nullptr; float *pend_out = nullptr; const uint32_t *pend_stage = nullptr;
    uint32_t launches = 0;               // fused launches so far (staging row parity)
    uint8_t *peer[BUS_MAX_WORLD] = {};   // peer-mapped bases (peer[rank] == local)
    bool connected = false;
    uint32_t epoch = 0;                  // shared by both forms: every rank makes the same sequence of exchanges
    cudaStream_t stream = nullptr;       // high-priority side stream of the overlapped form
    cudaEvent_t ev_in[2] = {}, ev_done[2] = {};
    bool pending[2] = {false, false};
};

struct BusParams {
    int world, rank;
    uint64_t cap, count;
    uint32_t epoch, op, scale;
    int32_t *slots[BUS_MAX_WORLD];
    uint32_t *flags[BUS_MAX_WORLD];
    uint32_t *status;
    int32_t *imix;
    float *out;
};

static size_t bus_flag_off(int world, uint64_t cap) { return sizeof(int32_t) * BUS_NPAR * world * cap; }
static size_t bus_stage_off(int world, uint64_t cap) { return bus_flag_off(world, cap) + sizeof(uint32_t) * (BUS_NPAR * world + 4); }   // flags, status, ticket, pad
static size_t bus_bytes(int world, uint64_t cap) { return bus_stage_off(world, cap) + sizeof(uint32_t) * 2 * cap; }                       // + two staging rows (mode 2)

__device__ __forceinline__ void st_release_sys(uint32_t *p, uint32_t v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t *p) { uint32_t v; asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }

__global__ void __launch_bounds__(256) k_bus_allreduce(const BusParams p) {
    const uint32_t par = p.epoch & (BUS_NPAR - 1);
    const uint64_t my_slot = ((uint64_t)par * p.world + p.rank) * p.cap;
    // 1. push: my mix into slot[rank] of every rank (NVLink stores; the own copy is local)
    for (int q = 0; q < p.world; ++q) {
        int32_t *dst = p.slots[q] + my_slot;
        for (uint64_t i = threadIdx.x; i < p.count; i += blockDim.x) dst[i] = p.imix[i];
    }
    __threadfence_system();
    __syncthreads();
    if ((int)threadIdx.x < p.world) st_release_sys(p.flags[threadIdx.x] + par * p.world + p.rank, p.epoch);
    // 2. wait for every rank's push into MY buffer
    __shared__ uint32_t failed;
    if (threadIdx.x == 0) failed = 0;
    __syncthreads();
    if ((int)threadIdx.x < p.world) {
        const uint32_t *f = p.flags[p.rank] + par * p.world + threadIdx.x;
        const long long t0 = clock64();
        while (ld_acquire_sys(f) != p.epoch) {
            if (clock64() - t0 > 20000000000ll) { failed = 1; break; }       // ~10 s: a rank never arrived
            __nanosleep(200);
        }
    }
    __syncthreads();
    if (failed) { if (threadIdx.x == 0) *p.status = p.epoch; return; }
    // 3. reduce in rank order, scale once (synth.c:180 / :194; grain mix 2^-7)
    const int32_t *mine = p.slots[p.rank] + (uint64_t)par * p.world * p.cap;
    for (uint64_t i = threadIdx.x; i < p.count; i += blockDim.x) {
        uint32_t acc = 0;
        if (p.op == 2) {                                   // float bus (extension voices): fixed rank order, one rounding per add
            float fa = 0.0f;
            for (int q = 0; q < p.world; ++q) fa = __fadd_rn(fa, __int_as_float(mine[(uint64_t)q * p.cap + i]));
            acc = __float_as_uint(fa);
        } else {
            for (int q = 0; q < p.world; ++q) {
                const uint32_t v = (uint32_t)mine[(uint64_t)q * p.cap + i];
                acc = p.op ? (acc | v) : (acc + v);
            }
        }
        p.imix[i] = (int32_t)acc;
        if (p.out) {
            float f;
            if (p.scale == 2) f = __uint2float_rn(acc) * 0x1p-32f;
            else if (p.scale == 3) f = __int2float_rn((int32_t)acc) * 0x1p-7f;
            else f = __int2float_rn((int32_t)acc) * 0x1p-32f;
            p.out[i] = f;
        }
    }
}

extern "C" {

int cproc_cuda_bus_create(cproc_cuda_ctx *ctx, uint64_t max_words, int world, int rank, cproc_cuda_bus **out) {
    if (!ctx || !out) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "bus_create: NULL argument");
    *out = nullptr;
    if (world < 1 || world > BUS_MAX_WORLD || rank < 0 || rank >= world || max_words == 0)
        return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "bus_create: world 1..%d, 0 <= rank < world, max_words > 0", BUS_MAX_WORLD);
    CK(ctx, cudaSetDevice(ctx->device));
    cproc_cuda_bus *b = new cproc_cuda_bus();
    b->ctx = ctx; b->world = world; b->rank = rank; b->cap = (max_words + 3) & ~3ull;
    const size_t bytes = bus_bytes(world, b->cap);
    int rc = cproc_check(ctx, cudaMalloc(&b->local, bytes), "cudaMalloc(bus)");
    if (!rc) rc = cproc_check(ctx, cudaMemset(b->local, 0, bytes), "memset(bus)");
    if (rc) { if (b->local) cudaFree(b->local); delete b; return rc; }
    b->peer[rank] = b->local;
    b->connected = world == 1;
    *out = b;
    return 0;
}

size_t cproc_cuda_bus_handle_bytes(void) { return sizeof(cudaIpcMemHandle_t); }

// the handle of this rank's buffer, to be sent to every other rank
int cproc_cuda_bus_handle(cproc_cuda_bus *b, void *handle) {
    if (!b || !handle) return cproc_set_err(b ? b->ctx : nullptr, CPROC_CUDA_EINVAL, "bus_handle: NULL argument");
    CK(b->ctx, cudaSetDevice(b->ctx->device));
    cudaIpcMemHandle_t h;
    CK(b->ctx, cudaIpcGetMemHandle(&h, b->local));
    memcpy(handle, &h, sizeof(h));
    return 0;
}

// handles: world x cproc_cuda_bus_handle_bytes(), in rank order (the own entry is ignored)
int cproc_cuda_bus_connect(cproc_cuda_bus *b, const void *handles) {
    if (!b || !handles) return cproc_set_err(b ? b->ctx : nullptr, CPROC_CUDA_EINVAL, "bus_connect: NULL argument");
    cproc_cuda_ctx *ctx = b->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    for (int q = 0; q < b->world; ++q) {
        if (q == b->rank || b->peer[q]) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, (const uint8_t *)handles + (size_t)q * sizeof(h), sizeof(h));
        void *ptr = nullptr;
        int rc = cproc_check(ctx, cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess), "cudaIpcOpenMemHandle (NVLink peer mapping of the mix bus)");
        if (rc) return rc;
        b->peer[q] = (uint8_t *)ptr;
    }
    b->connected = true;
    return 0;
}

// In place on device memory, asynchronous on the context stream.  op: 0 wrap-around sum, 1 OR,
// 2 float sum in rank order (the words are float bits: the float mix of the extension voices).
// scale: 0 none (out_dev may be NULL), 1 saw (float)(int)x * 2^-32, 2 square (float)(unsigned)x * 2^-32,
// 3 grain mix (float)x * 2^-7.  Every rank of the bus must make the same sequence of calls.
static int bus_launch(cproc_cuda_bus *b, int32_t *imix_dev, float *out_dev, uint64_t count, uint32_t op, uint32_t scale, cudaStream_t st);

int cproc_cuda_bus_allreduce(cproc_cuda_bus *b, int32_t *imix_dev, float *out_dev, uint64_t count, uint32_t op, uint32_t scale) {
    if (!b) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "bus_allreduce: bus is NULL");
    return bus_launch(b, imix_dev, out_dev, count, op, scale, b->ctx->stream);
}

// Overlapped form: the exchange of block k runs on the bus's own high-priority stream, ordered
// after everything queued on the context stream so far, while the context stream goes on with
// the render of block k+1 (into the other mix buffer).  `slot` (0/1) names the buffer pair in
// use; _wait(slot) makes the context stream wait for that slot's last exchange -- call it before
// the buffers of the slot are written again or read on the context stream.
int cproc_cuda_bus_allreduce_begin(cproc_cuda_bus *b, uint32_t slot, int32_t *imix_dev, float *out_dev, uint64_t count, uint32_t op, uint32_t scale) {
    if (!b || slot > 1) return cproc_set_err(b ? b->ctx : nullptr, CPROC_CUDA_EINVAL, "bus_allreduce_begin: bad bus / slot");
    cproc_cuda_ctx *ctx = b->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    if (!b->stream) {
        int lo = 0, hi = 0;
        CK(ctx, cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CK(ctx, cudaStreamCreateWithPriority(&b->stream, cudaStreamNonBlocking, hi));
        for (int i = 0; i < 2; ++i) { CK(ctx, cudaEventCreateWithFlags(&b->ev_in[i], cudaEventDisableTiming)); CK(ctx, cudaEventCreateWithFlags(&b->ev_done[i], cudaEventDisableTiming)); }
    }
    CK(ctx, cudaEventRecord(b->ev_in[slot], ctx->stream));
    CK(ctx, cudaStreamWaitEvent(b->stream, b->ev_in[slot], 0));
    int rc = bus_launch(b, imix_dev, out_dev, count, op, scale, b->stream);
    if (rc) return rc;
    CK(ctx, cudaEventRecord(b->ev_done[slot], b->stream));
    b->pending[slot] = true;
    return 0;
}

int cproc_cuda_bus_wait(cproc_cuda_bus *b, uint32_t slot) {
    if (!b || slot > 1) return cproc_set_err(b ? b->ctx : nullptr, CPROC_CUDA_EINVAL, "bus_wait: bad bus / slot");
    if (!b->pending[slot]) return 0;
    CK(b->ctx, cudaStreamWaitEvent(b->ctx->stream, b->ev_done[slot], 0));
    b->pending[slot] = false;
    return 0;
}

static int bus_launch(cproc_cuda_bus *b, int32_t *imix_dev, float *out_dev, uint64_t count, uint32_t op, uint32_t scale, cudaStream_t st) {
    if (!b || !imix_dev) return cproc_set_err(b ? b->ctx : nullptr, CPROC_CUDA_EINVAL, "bus_allreduce: NULL argument");
    cproc_cuda_ctx *ctx = b->ctx;
    if (!b->connected) return cproc_set_err(ctx, CPROC_CUDA_ESTATE, "bus_allreduce: bus not connected (cproc_cuda_bus_connect)");
    if (count > b->cap) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "bus_allreduce: %llu words, bus holds %llu", (unsigned long long)count, (unsigned long long)b->cap);
    if (op > 2 || scale > 3 || (scale && !out_dev) || (op == 2 && scale)) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "bus_allreduce: bad op / scale");
    if (count == 0) return 0;
    CK(ctx, cudaSetDevice(ctx->device));
    BusParams p;
    memset(&p, 0, sizeof(p));
    p.world = b->world; p.rank = b->rank; p.cap = b->cap; p.count = count;
    p.epoch = ++b->epoch; p.op = op; p.scale = scale;
    if (p.epoch == 0) p.epoch = b->epoch = BUS_NPAR;          // flags start at 0; keep the parity sequence
    const size_t flag_off = bus_flag_off(b->world, b->cap);
    for (int q = 0; q < b->world; ++q) { p.slots[q] = (int32_t *)b->peer[q]; p.flags[q] = (uint32_t *)(b->peer[q] + flag_off); }
    p.status = (uint32_t *)(b->local + flag_off) + BUS_NPAR * b->world;
    p.imix = imix_dev; p.out = scale ? out_dev : nullptr;
    k_bus_allreduce<<<1, 256, 0, st>>>(p);
    CK_LAUNCH(ctx, "k_bus_allreduce");
    return 0;
}

// 0 = every exchange so far completed; otherwise the epoch at which a peer failed to arrive (after a sync)
int cproc_cuda_bus_status(cproc_cuda_bus *b, uint32_t *failed_epoch) {
    if (!b || !failed_epoch) return cproc_set_err(b ? b->ctx : nullptr, CPROC_CUDA_EINVAL, "bus_status: NULL argument");
    cproc_cuda_ctx *ctx = b->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    const size_t flag_off = bus_flag_off(b->world, b->cap);
    CK(ctx, cudaMemcpyAsync(failed_epoch, (uint32_t *)(b->local + flag_off) + BUS_NPAR * b->world, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return 0;
}

// ---- the exchange as the tail of the render kernel (bus_fused.cuh) -------------------------------------------

__global__ void __launch_bounds__(256) k_bus_finish(const BusFused bf) { bus_exchange_block(bf); }

static void bus_fill(const cproc_cuda_bus *b, BusFused *bf) {
    memset(bf, 0, sizeof(*bf));
    bf->world = b->world; bf->rank = b->rank; bf->cap = b->cap;
    const size_t flag_off = bus_flag_off(b->world, b->cap);
    for (int q = 0; q < b->world; ++q) { bf->slots[q] = (int32_t *)b->peer[q]; bf->flags[q] = (uint32_t *)(b->peer[q] + flag_off); }
    bf->status = (uint32_t *)(b->local + flag_off) + BUS_NPAR * b->world;
    bf->ticket = bf->status + 1;
}

int cproc_cuda_bus_attach(cproc_cuda_bus *bus, cproc_cuda_batch *batch, uint32_t mode) {
    if (!batch) return cproc_set_err(bus ? bus->ctx : nullptr, CPROC_CUDA_EINVAL, "bus_attach: batch is NULL");
    cproc_cuda_ctx *ctx = batch->ctx;
    if (!bus || mode == 0) { batch->bus = nullptr; batch->bus_mode = 0; return 0; }
    if (mode > 2) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "bus_attach: mode must be 0 (detach), 1 (reduce inside the render launch) or 2 (pipelined)");
    if (bus->ctx != ctx) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "bus_attach: bus and batch belong to different contexts");
    if (!bus->connected) return cproc_set_err(ctx, CPROC_CUDA_ESTATE, "bus_attach: bus not connected (cproc_cuda_bus_connect)");
    const uint32_t proc = batch->cfg.proc;
    if (proc != CPROC_CUDA_VOICE_BANK && proc != CPROC_CUDA_XVOICE && proc != CPROC_CUDA_SQUARE_GRAIN_MIX)
        return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "bus_attach: only the voice bank, the xvoice mix and the square_grain mix exchange their bus in the render launch");
    batch->bus = bus; batch->bus_mode = mode;
    return 0;
}

}  // extern "C"

int cproc_bus_fused_begin(cproc_cuda_batch *b, BusFused *bf, uint64_t count, uint32_t op, uint32_t scale, uint32_t n_pushers,
                          int32_t *imix_out, float *float_out) {
    cproc_cuda_bus *bus = b->bus;
    if (!bus) { memset(bf, 0, sizeof(*bf)); return 0; }
    cproc_cuda_ctx *ctx = b->ctx;
    if (count > bus->cap) return cproc_set_err(ctx, CPROC_CUDA_EINVAL, "run: the mix is %llu words, the attached bus holds %llu", (unsigned long long)count, (unsigned long long)bus->cap);
    bus_fill(bus, bf);
    bf->mode = b->bus_mode;
    uint32_t epoch = ++bus->epoch;
    if (epoch == 0) epoch = bus->epoch = BUS_NPAR;
    if (bf->mode == 1) {
        if (bus->pend_epoch) return cproc_set_err(ctx, CPROC_CUDA_ESTATE, "run: a pipelined exchange is pending on this bus (cproc_cuda_bus_flush first)");
        bf->epoch = epoch; bf->participants = n_pushers;
        bf->fin_epoch = epoch; bf->fin_op = op; bf->fin_scale = scale; bf->fin_count = count; bf->fin_imix = imix_out; bf->fin_out = float_out;
    } else {
        uint32_t *stage = (uint32_t *)(bus->local + bus_stage_off(bus->world, bus->cap)) + (size_t)(bus->launches++ & 1u) * bus->cap;
        bf->stage = stage;
        bf->fin_epoch = bus->pend_epoch; bf->fin_op = bus->pend_op; bf->fin_scale = bus->pend_scale; bf->fin_count = bus->pend_count;
        bf->fin_imix = bus->pend_imix; bf->fin_out = bus->pend_out; bf->fin_stage = bus->pend_stage;
        bus->pend_epoch = epoch; bus->pend_op = op; bus->pend_scale = scale; bus->pend_count = count; bus->pend_imix = imix_out; bus->pend_out = float_out;
        bus->pend_stage = stage;
    }
    return 0;
}

extern "C" {

// mode 2: complete the exchange of the last rendered block (asynchronous on the context stream)
int cproc_cuda_bus_flush(cproc_cuda_bus *bus) {
    if (!bus) return cproc_set_err(nullptr, CPROC_CUDA_EINVAL, "bus_flush: bus is NULL");
    cproc_cuda_ctx *ctx = bus->ctx;
    if (!bus->pend_epoch) return 0;
    CK(ctx, cudaSetDevice(ctx->device));
    BusFused bf;
    bus_fill(bus, &bf);
    bf.mode = 2;
    bf.fin_epoch = bus->pend_epoch; bf.fin_op = bus->pend_op; bf.fin_scale = bus->pend_scale; bf.fin_count = bus->pend_count;
    bf.fin_imix = bus->pend_imix; bf.fin_out = bus->pend_out; bf.fin_stage = bus->pend_stage;
    bus->pend_epoch = 0;
    k_bus_finish<<<1, 256, 0, ctx->stream>>>(bf);
    CK_LAUNCH(ctx, "k_bus_finish");
    return 0;
}

int cproc_cuda_bus_destroy(cproc_cuda_bus *b) {
    if (!b) return 0;
    cudaSetDevice(b->ctx->device);
    cudaStreamSynchronize(b->ctx->stream);
    if (b->stream) {
        cudaStreamSynchronize(b->stream); cudaStreamDestroy(b->stream);
        for (int i = 0; i < 2; ++i) { cudaEventDestroy(b->ev_in[i]); cudaEventDestroy(b->ev_done[i]); }
    }
    for (int q = 0; q < b->world; ++q) if (q != b->rank && b->peer[q]) cudaIpcCloseMemHandle(b->peer[q]);
    if (b->local) cudaFree(b->local);
    delete b;
    return 0;
}

}  // extern "C"
