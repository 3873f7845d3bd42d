"""Every launch that bench.py and tools/bench_configs.py time, checked at the shape it is timed at.

The other suites check small shapes against the oracle; tests/test_gpu_fullsize.py checks BASELINE
shapes.  The launches the benchmark times run longer, run more work items per launch and write above
byte offsets those tests never reach.  Here each one is rendered at its timed shape into torch device
buffers (the library runs on torch's stream, so torch operations and library launches stay in order)
and checked twice:

- against a second kernel or schedule of the library that renders the same thing, whole output
  buffers compared on the device;
- against the CPU oracle on a subset of independent units (banks, instances), bit for bit: the first
  units, the ragged last group or warp, units that write above 2^31 / 2^32 bytes and a seeded sample.
  Only the sampled units are copied to the host.

The inputs differ across the whole instance range (per-instance states and parameters on top of a
repeated input chunk), so a launch that wrote instance i mod 2^k in place of instance i is visible.

The headline C2 step is rendered once, launch for launch as bench.py renders it, by a module fixture;
test_bench_dump_matches_the_oracle then runs the unmodified bench.py and checks what its
--dump-outputs writes against that render.
"""
import contextlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import bench
from oracle import pyoracle as po
from tests.test_gpu_parity import V2_DEFAULTS, pack_bits
from tools import bench_configs

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# the options these tests change, at their defaults (synth_tools_b200/csrc/common.cuh)
DEFAULTS = dict(V2_DEFAULTS, pdm_persist=1, pdm_v1_chains=2, planar_bulk=2, graph_jit=1)
MAX_REPORTED = 8                                  # mismatches listed per check


@pytest.fixture(scope="module")
def gpu():
    """torch on cuda:0 with a non-default stream, and a library context on that stream (as bench.py opens it)."""
    import torch
    import synth_tools_b200 as st
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    prev = torch.cuda.current_stream(dev)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    ctx = st.Context(0, stream.cuda_stream)
    po.set_threads(os.cpu_count() or 1)
    try:
        yield _Gpu(torch, st, ctx, dev)
    finally:
        ctx.close()
        torch.cuda.set_stream(prev)
        torch.cuda.empty_cache()


class _Gpu:
    def __init__(self, torch, st, ctx, dev):
        self.torch, self.st, self.ctx, self.dev = torch, st, ctx, dev

    def empty(self, n, dtype):
        return self.torch.empty(n, dtype=dtype, device=self.dev)

    def put(self, a):
        """host numpy -> device tensor (unsigned words travel as the signed type of the same width)"""
        a = np.ascontiguousarray(a)
        if a.dtype == np.uint32:
            a = a.view(np.int32)
        return self.torch.from_numpy(a).to(self.dev)

    def done(self):
        self.ctx.sync()
        self.torch.cuda.synchronize()
        self.torch.cuda.empty_cache()


@contextlib.contextmanager
def options(ctx, **kv):
    """set library options for the body; put every one back to its default afterwards"""
    try:
        for k, v in kv.items():
            ctx.set_option(k, v)
        yield
    finally:
        for k in kv:
            ctx.set_option(k, DEFAULTS[k])


def same(torch, a, b):
    """two device buffers hold the same bytes (compared as 64-bit words where the shapes allow)"""
    if a.is_contiguous() and b.is_contiguous() and a.dtype == b.dtype and a.numel() * a.element_size() % 8 == 0:
        return a.shape == b.shape and torch.equal(a.view(torch.int64), b.view(torch.int64))
    return torch.equal(a, b)


def mismatch(got, want, units):
    """the first units (by their global index) whose rows differ"""
    bad = np.nonzero((got.reshape(len(units), -1) != want.reshape(len(units), -1)).any(axis=1))[0]
    return [int(units[j]) for j in bad[:MAX_REPORTED]]


def sample_units(n, groups, seed, count):
    """first units, the given ranges (ragged ends, units above a byte offset), a seeded random sample; sorted, unique"""
    r = np.random.default_rng(seed)
    parts = [np.arange(a, min(b, n)) for a, b in groups] + [r.choice(n, size=count, replace=False)]
    return np.unique(np.concatenate(parts)).astype(np.int64)


# =====================================================================================================================
# 1. The headline C2 step (bench.py run_native), launch for launch
N_CH, F_CHUNK, N_LAUNCH, BANK, CTL = bench.N_CH, bench.F_CHUNK, bench.F_TOTAL // bench.F_CHUNK, bench.BANK, bench.CTL_LOG
ROWS = F_CHUNK >> CTL                             # setpoint rows per launch
RENDERS = {                                       # a name -> the options of that render
    "default": {},                                # what bench.py times: k_pdm_v2_ws4 <K=2, CW=3, TLOG=7>, 64-batch slices, 4 blocks / SM
    "thread_per_bank": {"pdm_ws": 0},             # k_pdm_v2_simple: no work items, no scheduling code in common with ws4
    # 64-tick batches, 24-batch slices (86 per launch, the last one 8 batches long), one block per SM: ~400 rounds of the grid
    "ws4_t64_s24_c1": {"pdm_tlog": 6, "pdm_slice_batches": 24, "pdm_ctas_per_sm": 1},
}


def written(a):
    """an array as bench.write_outputs stores it: 8- and 16-bit integers as float32, wider integers as float64"""
    a = np.asarray(a)
    return a.astype(np.float32 if a.dtype.kind == "f" or a.dtype.itemsize <= 2 else np.float64)


def headline_units(n_banks):
    """the oracle's banks: those of bench's dump channels, banks 0..31, the last (ragged, 64-channel) work group from
    channel 65,472 on, whose last bank holds one channel (65,535).  Returns (banks, their channels, the dump channels)."""
    dump = bench.dump_channels(N_CH)
    banks = np.unique(np.concatenate([dump // BANK, np.arange(32), np.arange(65472 // BANK, n_banks)]))
    chans = np.concatenate([np.arange(BANK * b, min(BANK * b + BANK, N_CH)) for b in banks])
    return banks, chans, dump


def setpoint_rows(sp64, chans, r0, n):
    """rows r0 .. r0+n-1 of bench's setpoint table for the given channels: row r is block r // 64 of the 64 distinct rows,
    rolled by r // 64 along the channel axis (np.roll semantics)"""
    r = np.arange(r0, r0 + n)
    return np.ascontiguousarray(sp64[(r % 64)[:, None], (chans[None, :] - (r // 64)[:, None]) % N_CH])


class V2Oracle:
    """oracle.pdm_v2_run on a compacted set of banks with its state carried from call to call, cut into parts (whole banks,
    the ragged bank last) that run side by side, one thread and one state array each: one OpenMP call over all the banks
    shares cache lines of the channel records between threads and runs slower than a single thread."""

    def __init__(self, oracle, chan, prng, bank, parts):
        self.oracle, self.bank, self.count = oracle, bank, 0
        cuts = [int(c) for c in np.linspace(0, len(prng), min(parts, len(prng)) + 1)]
        self.parts = [(chan[bank * b0:bank * b1].copy(), prng[b0:b1].copy(), bank * b0, min(bank * b1, len(chan)))
                      for b0, b1 in zip(cuts[:-1], cuts[1:])]
        self.pool = ThreadPoolExecutor(len(self.parts), initializer=po.set_threads, initargs=(1,))

    def submit(self, sp_rows, F, out):
        """render the next F ticks into out [channels][F]; returns the futures (wait with .wait())"""
        def run(part):
            ch, pr, c0, c1 = part
            return self.oracle.pdm_v2_run(ch, 2, c1 - c0, self.bank, pr, None, 0x3FF, self.count, CTL, 24,
                                          np.ascontiguousarray(sp_rows[:, c0:c1]), F, out=out[c0:c1])[1]
        return [self.pool.submit(run, part) for part in self.parts]

    def wait(self, futures):
        counts = {f.result() for f in futures}
        assert len(counts) == 1, counts
        self.count = counts.pop()

    def state(self):
        return np.concatenate([p[0] for p in self.parts]), np.concatenate([p[1] for p in self.parts])

    def close(self):
        self.pool.shutdown()


class HeadlineStep:
    pass


@pytest.fixture(scope="module")
def headline(gpu, oracle):
    """bench.py's step (128 launches of 131,072 ticks, 65,536 channels, setpoints rolled per 64-row block) rendered
    three times, each render on its own batch and slab, compared on the device after every launch and against the
    oracle on the sampled banks.  Records the mismatches and builds the arrays bench.dump_native writes."""
    torch, st, ctx = gpu.torch, gpu.st, gpu.ctx
    res = HeadlineStep()
    res.gpu_fail, res.oracle_fail = [], []
    batches, slabs, orc = {}, {}, None
    try:
        sp64 = po.pdm_setpoints(N_CH, 64, seed_base=1)
        sp_dev = torch.empty((bench.F_TOTAL >> CTL, N_CH), dtype=torch.int32, device=gpu.dev)
        sp64_d = gpu.put(sp64)
        for r in range(0, sp_dev.shape[0], 64):
            sp_dev[r:r + 64] = torch.roll(sp64_d, shifts=r // 64, dims=1)
        for fill, name in enumerate(RENDERS):
            b = ctx.batch(st.PDM_V2, N_CH, order=2, bank_size=BANK, ctl_div_log=CTL, out_shift=24, dither_mask=0x3FF, layout=st.TILED)
            batches[name] = b
            b.upload_bank((np.arange(b.n_banks) + 1).astype(np.uint32), 0)
            slabs[name] = gpu.empty(N_CH * F_CHUNK, torch.uint8).fill_(0x11 * (fill + 1))
        n_banks = batches["default"].n_banks
        state0 = batches["default"].download_state()           # the state a batch is allocated with
        for name, b in batches.items():
            assert np.array_equal(b.download_state(), state0), name
        banks, chans, dump = headline_units(n_banks)
        n = len(chans)
        assert chans[-1] == N_CH - 1 and N_CH % BANK == 1           # the ragged one-channel bank closes the compacted set
        orc = V2Oracle(oracle, state0[chans], (banks + 1).astype(np.uint32), BANK, os.cpu_count() or 1)
        sel = torch.from_numpy(chans).to(gpu.dev)
        want = np.zeros((n, F_CHUNK), np.uint8)
        dump_pos = np.searchsorted(chans, dump)
        arrays = {"duty_channels": dump}
        for k in range(N_LAUNCH):
            pending = orc.submit(setpoint_rows(sp64, chans, ROWS * k, ROWS), F_CHUNK, want)     # on the host, beside the renders
            ctl = sp_dev.data_ptr() + 4 * N_CH * ROWS * k
            for name, opts in RENDERS.items():
                with options(ctx, **opts):
                    batches[name].run_dev(F_CHUNK, ctl=ctl, n_ctl=ROWS, out=slabs[name].data_ptr())
            for name in RENDERS:
                if name != "default" and not same(torch, slabs["default"], slabs[name]):
                    res.gpu_fail.append("launch %d: %s slab differs from the default render" % (k, name))
            tiles = slabs["default"].view(F_CHUNK // 16, N_CH, 16)     # TILED [t/16][ch][16]
            got = tiles.index_select(1, sel).permute(1, 0, 2).reshape(n, F_CHUNK).cpu().numpy()
            orc.wait(pending)
            if not np.array_equal(got, want):
                res.oracle_fail.append("launch %d: duty of channels %s differs from the oracle" % (k, mismatch(got, want, chans)))
            if k >= N_LAUNCH - 2:
                name = "prev_launch" if k == N_LAUNCH - 2 else "last_launch"
                arrays[name + "_duty"] = got[dump_pos, -bench.DUMP_TICKS:].copy()
                total = torch.zeros(N_CH, dtype=torch.int64, device=gpu.dev)
                for r in range(0, F_CHUNK // 16, 128):
                    total += tiles[r:r + 128].sum(dim=(0, 2), dtype=torch.int64)
                arrays[name + "_duty_sum"] = total.cpu().numpy()
                if not np.array_equal(arrays[name + "_duty_sum"][chans], got.sum(axis=1, dtype=np.int64)):
                    res.oracle_fail.append("launch %d: device duty sums of the sampled channels differ from their duty" % k)
        chan, prng = orc.state()
        ends = {name: (b.download_state(), *b.download_bank()) for name, b in batches.items()}
        s0, p0, c0 = ends["default"]
        for name, (s, p, c) in ends.items():
            if not (np.array_equal(s, s0) and np.array_equal(p, p0) and c == c0):
                res.gpu_fail.append("end of step: %s channel state / bank PRNG / count differ from the default render" % name)
        if not np.array_equal(s0[chans], chan):
            res.oracle_fail.append("end of step: channel state of %s differs from the oracle" % mismatch(s0[chans], chan, chans))
        if not (np.array_equal(p0[banks], prng) and c0 == orc.count):
            res.oracle_fail.append("end of step: bank PRNG / count (%d vs %d) differ from the oracle" % (c0, orc.count))
        arrays["channel_state"] = s0
        arrays["bank_prng"] = p0
        arrays["bank_count"] = np.array([c0], np.uint32)
        res.arrays = {k: written(v) for k, v in arrays.items()}
        res.n_sampled_banks, res.n_sampled_channels = len(banks), n
    finally:
        if orc is not None:
            orc.close()
        for b in batches.values():
            b.free()
        slabs.clear()
        sp_dev = sp64_d = tiles = sel = total = None
        gpu.done()
    return res


def test_headline_step_renders_agree_launch_for_launch(headline):
    """The default k_pdm_v2_ws4 schedule, the thread-per-bank kernel and ws4 with 64-tick batches in 86 slices per launch
    (the last one ragged) on a one-block-per-SM grid write identical 8 GiB slabs at every one of the step's 128 launches,
    and end the step with the same channel state, bank PRNG and count for all 65,536 channels."""
    assert not headline.gpu_fail, headline.gpu_fail[:MAX_REPORTED]


def test_headline_step_matches_the_oracle(headline):
    """The sampled banks (bench's 256 dump channels, banks 0..31, the ragged last work group and the one-channel last bank):
    their full 131,072-tick duty streams equal the oracle's at every launch, the oracle carrying their state from launch
    to launch, and so do their channel state, bank PRNG and count at the end of the step."""
    assert headline.n_sampled_banks >= 54 and headline.n_sampled_channels >= 160
    assert not headline.oracle_fail, headline.oracle_fail[:MAX_REPORTED]


# =====================================================================================================================
# 2. bench.py --dump-outputs against the render above
def test_bench_dump_matches_the_oracle(headline, tmp_path):
    """The unmodified bench.py, one step without warm-up: every array --dump-outputs writes equals the one built from the
    render that test_headline_step_* check launch for launch against the oracle and against two other kernels.  This pins
    bench's own TILED window gather and its int32 partial duty sums as well."""
    assert not headline.gpu_fail and not headline.oracle_fail, "the headline render itself failed its checks"
    out = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "1", "--warmup", "0",
           "--no-other-configs", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, cwd=str(tmp_path), capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stderr[-4000:]
    names = sorted(p[:-4] for p in os.listdir(out) if p.endswith(".npy"))
    assert names == sorted(headline.arrays), names
    for name, want in headline.arrays.items():
        got = np.load(out / (name + ".npy"))
        assert got.dtype == want.dtype and got.shape == want.shape, (name, got.dtype, got.shape)
        assert np.array_equal(got, want), name


# =====================================================================================================================
# 3. The other timed rows (tools/bench_configs.py) at their bench shapes
def test_c2_layout_bench_shape(gpu, oracle):
    """c2_layout: 65,536 channels x 32,768 ticks, banks of 3, a setpoint row every 4096 ticks, distinct bank PRNG words.
    PLANAR (k_pdm_v2_ws4 PL=2, tensor-TMA boxes) and INTERLEAVED (PL=1, block tiles) equal the TILED render transposed
    (2 GiB each, on the device); the oracle reproduces the sampled banks, the ragged last group (64 channels) included."""
    torch, st, ctx = gpu.torch, gpu.st, gpu.ctx
    N, F, L = 65536, 32768, 12
    rows = F >> L
    nb = (N + 2) // 3
    sp = np.random.default_rng(6).integers(0x40000000, 0xC0000000, (rows, N), dtype=np.uint32)
    prng0 = (np.arange(nb, dtype=np.uint64) * 2654435761 + 12345).astype(np.uint32) | np.uint32(1)
    sp_d = gpu.put(sp)
    outs, ends = {}, {}
    try:
        state0 = None
        for layout in ("TILED", "PLANAR", "INTERLEAVED"):
            b = ctx.batch(st.PDM_V2, N, order=2, bank_size=3, ctl_div_log=L, out_shift=24, dither_mask=0x3FF, layout=getattr(st, layout))
            try:
                state0 = b.download_state() if state0 is None else state0
                b.upload_bank(prng0, 0)
                outs[layout] = gpu.empty(N * F, torch.uint8).fill_(len(outs) + 1)
                b.run_dev(F, ctl=sp_d.data_ptr(), n_ctl=rows, out=outs[layout].data_ptr())
                ends[layout] = (b.download_state(), *b.download_bank())
            finally:
                b.free()
        planar = outs["TILED"].view(F // 16, N, 16).permute(1, 0, 2).reshape(N, F)
        assert same(torch, outs["PLANAR"].view(N, F), planar)
        assert torch.equal(outs["INTERLEAVED"].view(F, N), planar.t())
        s0, p0, c0 = ends["TILED"]
        for layout, (s, p, c) in ends.items():
            assert np.array_equal(s, s0) and np.array_equal(p, p0) and c == c0, layout
        banks = sample_units(nb, [(0, 32), (21000, 21040), (65472 // 3, nb)], 31, 64)
        chans = np.concatenate([np.arange(3 * b, min(3 * b + 3, N)) for b in banks])
        chan, pr = state0[chans].copy(), prng0[banks].copy()
        want, cnt = oracle.pdm_v2_run(chan, 2, len(chans), 3, pr, None, 0x3FF, 0, L, 24, np.ascontiguousarray(sp[:, chans]), F)
        got = outs["PLANAR"].view(N, F).index_select(0, torch.from_numpy(chans).to(gpu.dev)).cpu().numpy()
        assert np.array_equal(got, want), mismatch(got, want, chans)
        assert np.array_equal(s0[chans], chan) and np.array_equal(p0[banks], pr) and c0 == cnt
    finally:
        outs.clear()
        sp_d = planar = None
        gpu.done()


V1_RENDERS = [{"pdm_persist": 0, "pdm_v1_chains": 2}, {"pdm_persist": 2, "pdm_v1_chains": 2},
              {"pdm_persist": 0, "pdm_v1_chains": 1}, {"pdm_persist": 2, "pdm_v1_chains": 1}]


def test_c2_v1_bench_shape(gpu, oracle):
    """c2_v1: the carry-bit PDM, 65,536 channels x 524,288 ticks, banks of 2, TILED packed bits (4 GiB).  The plain and the
    persistent (McNaughton-scheduled) kernels, each with one and two PRNG chains per lane, write identical slabs and end
    in the same state; the oracle reproduces the sampled banks."""
    torch, st, ctx = gpu.torch, gpu.st, gpu.ctx
    N, F, bank = 65536, 512 * 1024, 2
    nb = N // bank
    rng = np.random.default_rng(2)
    ch0 = rng.integers(0x40000000, 0xC0000000, (N, 2), dtype=np.uint32)
    ch0[:, 1] = rng.integers(0, 2**32, N, dtype=np.uint32)
    prng0 = rng.integers(1, 2**32, nb, dtype=np.uint32)
    outs, ends = [], []
    try:
        for opts in V1_RENDERS:
            b = ctx.batch(st.PDM_V1, N, bank_size=bank, dither_mask=0x0FFFFFFF, layout=st.TILED)
            try:
                b.upload_state(ch0); b.upload_bank(prng0)
                out = gpu.empty(N * F // 8, torch.uint8).fill_(len(outs) + 1)
                with options(ctx, **opts):
                    b.run_dev(F, out=out.data_ptr())
                ends.append((b.download_state(), b.download_bank()[0]))
                if outs:
                    assert same(torch, outs[0], out), opts
                    assert np.array_equal(ends[0][0], ends[-1][0]) and np.array_equal(ends[0][1], ends[-1][1]), opts
                    out = None
                else:
                    outs.append(out)
            finally:
                b.free()
        banks = sample_units(nb, [(0, 16), (nb - 16, nb)], 32, 48)
        chans = np.concatenate([np.arange(bank * b, bank * b + bank) for b in banks])
        ca, pa = ch0[chans].copy(), prng0[banks].copy()
        want = pack_bits(oracle.pdm_v1_run(ca, len(chans), bank, pa, None, 0x0FFFFFFF, F))
        words = outs[0].view(torch.int32).view(F // 128, N, 4)                  # TILED [t/128][ch][4 words]
        got = words.index_select(1, torch.from_numpy(chans).to(gpu.dev)).permute(1, 0, 2).reshape(len(chans), F // 32)
        got = got.cpu().numpy().view(np.uint32)
        assert np.array_equal(got, want), mismatch(got, want, chans)
        assert np.array_equal(ends[0][0][chans], ca) and np.array_equal(ends[0][1][banks], pa)
    finally:
        outs.clear()
        out = words = got = None
        gpu.done()


def test_pdm_raw_bench_shape(gpu, oracle):
    """pdm_raw: pdm2_update (order 2, shift 24) on 1 Mi channels x 1,024 ticks, 4 GiB in and 4 GiB out.  PLANAR through
    tensor-TMA staging (planar_bulk 2) and through the scalar k_pdm_raw (planar_bulk 0) write identical streams, and the
    INTERLEAVED render (k_interleaved4) is their transpose.  The input repeats bench's 16,384-row chunk; the channels
    differ through their integrator states, so the oracle on the sampled channels sees every channel's own output."""
    torch, st, ctx = gpu.torch, gpu.st, gpu.ctx
    N, F, order = 1024 * 1024, 1024, 2
    rng = np.random.default_rng(10)
    chunk = rng.integers(0, 2**32, (16384, F), dtype=np.uint32)
    s0 = rng.integers(0, 2**32, (N, order), dtype=np.uint32)
    bufs, ends = {}, {}
    try:
        bufs["in"] = gpu.put(chunk).repeat(N // 16384, 1)                      # [ch][F]
        bufs["in_il"] = bufs["in"].t().contiguous()                             # [F][ch]
        for name, layout, mode in (("planar_tma", "PLANAR", 2), ("planar_scalar", "PLANAR", 0), ("interleaved", "INTERLEAVED", 2)):
            b = ctx.batch(st.PDM, N, order=order, out_shift=24, layout=getattr(st, layout))
            try:
                b.upload_state(s0)
                bufs[name] = gpu.empty(N * F, torch.int32).fill_(len(bufs))
                inp = bufs["in_il" if layout == "INTERLEAVED" else "in"]
                with options(ctx, planar_bulk=mode):
                    b.run_dev(F, inp=inp.data_ptr(), out=bufs[name].data_ptr())
                ends[name] = b.download_state()
            finally:
                b.free()
        assert same(torch, bufs["planar_tma"], bufs["planar_scalar"])
        assert torch.equal(bufs["interleaved"].view(F, N).t(), bufs["planar_tma"].view(N, F))
        for name, s in ends.items():
            assert np.array_equal(s, ends["planar_tma"]), name
        # rows above byte offset 2^31 start at channel 2^19 (4 KiB per row); the INTERLEAVED ticks >= 512 of every channel
        units = sample_units(N, [(0, 64), ((1 << 19) - 32, (1 << 19) + 32), (N - 64, N)], 33, 192)
        sa = s0[units].copy()
        want = oracle.pdm_run(order, sa, len(units), F, np.ascontiguousarray(chunk[units % 16384]), None, 24, None)
        got = bufs["planar_tma"].view(N, F).index_select(0, torch.from_numpy(units).to(gpu.dev)).cpu().numpy().view(np.uint32)
        assert np.array_equal(got, want), mismatch(got, want, units)
        assert np.array_equal(ends["planar_tma"][units], sa)
    finally:
        bufs.clear()
        inp = None
        gpu.done()


def _graph_jit_ran(b):
    log = b.jit_log
    assert "not found" not in log and "failed" not in log, log


BP5_TEXT = """#define CPROC_NB_INPUTS 1
    void cproc_update(w *input, w g) {
        PROC_COND(g&0b1, n1, edge, NULL, NULL, .in = input[0]);
        PROC_COND(g&0b1, n2, acc, NULL, NULL, .in = n1.out);
        PROC_COND(g&0b1, n3, acc, NULL, NULL, .in = n2.out);
        cproc_output(3, n3.out); }"""                  # stm32f103/bp5_plugin.c, as tools/bench_configs.graph_bp5 parses it


def test_graph_bp5_bench_shape(gpu, oracle):
    """graph_bp5: the generated edge -> acc -> acc graph, 4 Mi instances x 256 ticks, 4 GiB per stream.  The NVRTC kernels
    (PLANAR with tensor-TMA staging and the scalar graph_planar_simple, INTERLEAVED) and the library's own chain kernel (graph_jit 0)
    agree on the device; the oracle reproduces instances around 2^20 and 2^21 and the last ones up to 2^22 - 1 (PLANAR rows
    above 3 GiB from 2^22 - 2^20 on; INTERLEAVED ticks >= 128 above 2 GiB).  Every instance starts from its own state."""
    torch, st, ctx = gpu.torch, gpu.st, gpu.ctx
    rows, n_in, out_node, _ = st.graph_parse(BP5_TEXT)
    assert [r[:2] for r in rows] == [r[:2] for r in po.GRAPH_BP5]
    N, F = 4 * 1024 * 1024, 256
    rng = np.random.default_rng(8)
    chunk = rng.integers(0, 2, (65536, F), dtype=np.uint32)
    sw = sum(po.node_words(r[0]) for r in rows)
    s0 = rng.integers(0, 2**32, (N, sw), dtype=np.uint32)
    bufs, ends = {}, {}
    try:
        bufs["in"] = gpu.put(chunk).repeat(N // 65536, 1)                      # [inst][1][F]
        bufs["in_il"] = bufs["in"].t().contiguous()                             # [F][1][inst]
        for name, layout, opts in (("jit_tma", "PLANAR", {"planar_bulk": 2}), ("jit_simple", "PLANAR", {"planar_bulk": 0}),
                                   ("jit_il", "INTERLEAVED", {}), ("chain_kernel", "PLANAR", {"graph_jit": 0})):
            with options(ctx, **opts):
                b = ctx.batch(st.GRAPH, N, nodes=rows, n_inputs=n_in, out_node=out_node, layout=getattr(st, layout))
                try:
                    b.upload_state(s0)
                    bufs[name] = gpu.empty(N * F, torch.int32).fill_(len(bufs))
                    b.run_dev(F, inp=bufs["in_il" if layout == "INTERLEAVED" else "in"].data_ptr(), out=bufs[name].data_ptr())
                    if "graph_jit" not in opts:
                        _graph_jit_ran(b)
                    ends[name] = b.download_state()
                finally:
                    b.free()
        for name in ("jit_simple", "chain_kernel"):
            assert same(torch, bufs["jit_tma"], bufs[name]), name
        assert torch.equal(bufs["jit_il"].view(F, N).t(), bufs["jit_tma"].view(N, F))
        for name, s in ends.items():
            assert np.array_equal(s, ends["jit_tma"]), name
        units = sample_units(N, [(0, 32), ((1 << 20) - 32, (1 << 20) + 32), ((1 << 21) - 32, (1 << 21) + 32),
                                 (N - (1 << 20), N - (1 << 20) + 32), (N - 64, N)], 34, 128)
        sa = s0[units].copy()
        want = oracle.graph_run(rows, n_in, out_node, sa, len(units), F, np.ascontiguousarray(chunk[units % 65536]).reshape(-1, 1, F))
        got = bufs["jit_tma"].view(N, F).index_select(0, torch.from_numpy(units).to(gpu.dev)).cpu().numpy().view(np.uint32)
        assert np.array_equal(got, want), mismatch(got, want, units)
        assert np.array_equal(ends["jit_tma"][units], sa)
    finally:
        bufs.clear()
        gpu.done()


def test_graph_voice_bench_shape(gpu, oracle):
    """graph_voice: the C4 voice as a generated graph (phasor_f -> svf -> env -> 2 x gain), 2 Mi instances x 512 ticks, no
    input, 8 GiB of float output.  The generated PLANAR and INTERLEAVED renders equal k_xvoice's raw PLANAR output for the
    same records bit for bit over all 8 GiB, with the same final state; the oracle (graph_run_ext) reproduces the sampled
    instances, those from 2^20 on included (PLANAR rows above 4 GiB; INTERLEAVED ticks >= 256 above 4 GiB)."""
    torch, st, ctx = gpu.torch, gpu.st, gpu.ctx
    g = st.graph_parse_ex(bench_configs.VOICE_GRAPH_TEXT)
    N, F = 2 * 1024 * 1024, 512
    stt, prm = bench_configs.xvoice_records(np.random.default_rng(12), N)
    gst = np.zeros((N, 9), np.uint32)
    gst[:, 1] = stt[:, 0]
    outs = g["out_nodes"]
    assert len(outs) == 2
    bufs, ends = {}, {}
    try:
        for name, layout in (("planar", "PLANAR"), ("interleaved", "INTERLEAVED")):
            b = ctx.batch(st.GRAPH, N, nodes=g["rows"], n_inputs=0, out_node=outs, layout=getattr(st, layout))
            try:
                b.upload_state(gst); b.upload_param(prm)
                bufs[name] = gpu.empty(2 * N * F, torch.int32).fill_(len(bufs) + 1)
                b.run_dev(F, out=bufs[name].data_ptr())
                _graph_jit_ran(b)
                ends[name] = b.download_state()
            finally:
                b.free()
        b = ctx.batch(st.XVOICE, N, layout=st.PLANAR)
        try:
            b.upload_state(stt); b.upload_param(prm)
            bufs["xvoice"] = gpu.empty(2 * N * F, torch.int32).fill_(3)
            b.run_dev(F, out=bufs["xvoice"].data_ptr())
            xst = b.download_state()
        finally:
            b.free()
        raw = bufs["xvoice"].view(N, F, 2)                                      # k_xvoice PLANAR raw [voice][F][L, R]
        assert torch.equal(bufs["planar"].view(N, 2, F).permute(0, 2, 1), raw)   # graph PLANAR [inst][out][F]
        assert torch.equal(bufs["interleaved"].view(F, 2, N).permute(2, 0, 1), raw)   # graph INTERLEAVED [F][out][inst]
        assert np.array_equal(ends["planar"], ends["interleaved"])
        assert np.array_equal(ends["planar"][:, [1, 2, 3, 5, 6]], xst)          # phase, lp, bp, env, t
        units = sample_units(N, [(0, 32), ((1 << 20) - 16, (1 << 20) + 48), (N - 64, N)], 35, 64)
        sa = gst[units].copy()
        want = oracle.graph_run_ext(g["rows"], 0, outs, sa, np.ascontiguousarray(prm[units]), len(units), F)
        got = bufs["planar"].view(N, 2 * F).index_select(0, torch.from_numpy(units).to(gpu.dev)).cpu().numpy().view(np.uint32)
        assert np.array_equal(got, want.reshape(len(units), 2 * F)), mismatch(got, want, units)
        assert np.array_equal(ends["planar"][units], sa)
    finally:
        bufs.clear()
        raw = None
        gpu.done()


@pytest.mark.parametrize("masked", [False, True], ids=["every_tick", "changed_and_masks"])
def test_c1_long_bench_shape(gpu, oracle, masked):
    """c1_long: the test_cproc chain (edge -> acc), ONE instance x 16 Mi ticks through the time-parallel scan
    (CPROC_CUDA_GRAPH_SCAN): 262,144 chunks of 64 ticks, so every k_gs_scan thread folds 1,024 chunks.  The whole stream
    and the state equal the oracle and the serial graph kernel.  `changed_and_masks` adds a changed stream (with a long
    stretch where nothing executes) and different masks on the two nodes: the masked branches of k_gs_reduce / k_gs_apply."""
    torch, st, ctx = gpu.torch, gpu.st, gpu.ctx
    N, F = 1, 16 * 1024 * 1024
    rng = np.random.default_rng(9)
    inp = rng.integers(0, 2, (N, 1, F), dtype=np.uint32)
    inp[:, :, ::17] = rng.integers(0, 2**32, inp[:, :, ::17].shape, dtype=np.uint32)
    rows = [(st.NODE_EDGE, -1, 1), (st.NODE_ACC, 0, 2 if masked else 1)]
    s0 = rng.integers(0, 2**32, (N, 3), dtype=np.uint32)
    changed = None
    if masked:
        changed = rng.integers(0, 4, (N, F), dtype=np.uint32)
        changed[:, F // 3:F // 3 + 200000] = 0
    sa = s0.copy()
    want = oracle.graph_run(rows, 1, 1, sa, N, F, inp, changed)
    bufs, ends = {}, {}
    try:
        bufs["in"] = gpu.put(inp)
        if masked:
            bufs["changed"] = gpu.put(changed)
        for name, mode in (("scan", 1), ("serial", 0)):
            b = ctx.batch(st.GRAPH, N, nodes=rows, mode=mode)
            try:
                b.upload_state(s0)
                bufs[name] = gpu.empty(N * F, torch.int32).fill_(mode + 1)
                l0 = ctx.launches
                b.run_dev(F, inp=bufs["in"].data_ptr(), in2=bufs["changed"].data_ptr() if masked else None, out=bufs[name].data_ptr())
                if mode == 1:
                    assert ctx.launches - l0 >= 3 * len(rows)                   # reduce, scan, apply per node
                ends[name] = b.download_state()
            finally:
                b.free()
        assert same(torch, bufs["scan"], bufs["serial"])
        got = bufs["scan"].cpu().numpy().view(np.uint32).reshape(N, F)
        if not np.array_equal(got, want):
            bad = np.nonzero(got[0] != want[0])[0]
            pytest.fail("scan output differs from the oracle at %d ticks, first %s" % (len(bad), bad[:MAX_REPORTED].tolist()))
        assert np.array_equal(ends["scan"], sa) and np.array_equal(ends["serial"], sa)
    finally:
        bufs.clear()
        gpu.done()
