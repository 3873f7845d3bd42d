"""GPU parity at the BASELINE.json shapes.  The units of every configuration are
independent (banks / grains / voices / variants), so the oracle can be run on a SUBSET of
them with the same inputs and must reproduce exactly the bytes the full-size launch wrote for
those units; on top of that, size-independent properties: the same render through different
kernels gives the same checksum, a split run equals one run, integer mixes are linear over a
partition of the voices, PDM duty averages to the setpoint."""
import zlib

import numpy as np
import pytest

from oracle import pyoracle as po

pytestmark = pytest.mark.gpu
rng = np.random.default_rng(77)


@pytest.fixture(scope="module")
def st():
    import synth_tools_b200 as st_
    return st_


@pytest.fixture(scope="module")
def ctx(st):
    c = st.Context(0)
    yield c
    c.close()


def _note_incs(orc, n, lo, hi):
    tab = np.array([orc.note_to_inc(k) for k in range(128)], np.uint32)
    return tab[rng.integers(lo, hi, n)]


def test_c2_pdm_v2_full_launch_shape(st, ctx, oracle):
    """65,536 channels x 65,536 ticks (one launch of the headline bench), banks of 3, a setpoint
    row every 4096 ticks.  (1) the oracle on banks 0..31, 10,000..10,031 and the last 32 banks
    (with the ragged last bank) reproduces their duty bytes, state and PRNG words exactly;
    (2) k_pdm_v2_ws4 with 128-tick and with 64-tick dither batches and the plain thread-per-bank kernel
    write identical slabs (CRC of all 4 GiB); (3) mean duty tracks the glided setpoint."""
    N, F, L = 65536, 65536, 12
    nb = (N + 2) // 3
    rows = F >> L
    sp = po.pdm_setpoints(N, rows)
    prng0 = (np.arange(nb, dtype=np.uint64) * 2654435761 + 12345).astype(np.uint32) | np.uint32(1)
    d_out = ctx.dev_alloc(N * F)
    d_sp = ctx.dev_alloc(sp.nbytes); ctx.h2d(d_sp, sp)
    host = np.zeros(N * F, np.uint8)
    crcs = {}
    keep = None
    for name, opts in (("t128", {"pdm_ws": 1, "pdm_tlog": 7}), ("t64", {"pdm_ws": 1, "pdm_tlog": 6}), ("plain", {"pdm_ws": 0})):
        for k, v in opts.items():
            ctx.set_option(k, v)
        b = ctx.batch(st.PDM_V2, N, order=2, bank_size=3, ctl_div_log=L, layout=st.TILED)
        b.upload_bank(prng0, 0)
        b.run_dev(F, ctl=d_sp, n_ctl=rows, out=d_out)
        ctx.d2h(host, d_out)
        state, (prng1, cnt) = b.download_state(), b.download_bank()
        crcs[name] = (zlib.crc32(host), zlib.crc32(state.tobytes()), zlib.crc32(prng1.tobytes()), cnt)
        if name == "t128":
            keep = (host.reshape(F // 16, N, 16).copy(), state, prng1)
        b.free()
        ctx.set_option("pdm_ws", 1); ctx.set_option("pdm_tlog", 7)
    assert crcs["t128"] == crcs["t64"] == crcs["plain"], crcs
    tiled, state, prng1 = keep
    for b0 in (0, 10000, nb - 32):
        c0, c1 = 3 * b0, min(N, 3 * (b0 + 32))
        n = c1 - c0
        chan = np.zeros((n, 7), np.uint32)
        pr = prng0[b0:b0 + 32].copy()
        want, _ = oracle.pdm_v2_run(chan, 2, n, 3, pr, None, 0x3FF, 0, L, 24, np.ascontiguousarray(sp[:, c0:c1]), F)
        got = tiled[:, c0:c1, :].transpose(1, 0, 2).reshape(n, F)
        assert np.array_equal(got, want), b0
        assert np.array_equal(state[c0:c1], chan) and np.array_equal(prng1[b0:b0 + 32], pr), b0
    # density: over the last control period the line has converged to within one step of the setpoint
    duty = tiled[-(1 << L) // 16:, :4096, :].astype(np.float64).mean(axis=(0, 2))
    target = sp[-2, :4096].astype(np.float64) / 2**24          # line[0] of the last period glides towards row -2
    prev = sp[-3, :4096].astype(np.float64) / 2**24
    lo, hi = np.minimum(target, prev) - 1.0, np.maximum(target, prev) + 1.0
    assert np.all((duty >= lo) & (duty <= hi))
    ctx.dev_free(d_out); ctx.dev_free(d_sp)


def test_c2_split_run_equals_one_run(st, ctx):
    """Property at full channel count: 16 launches of 4096 ticks == 1 launch of 65,536 ticks."""
    N, F, L = 65536, 65536, 12
    rows = F >> L
    sp = po.pdm_setpoints(N, rows)
    d_sp = ctx.dev_alloc(sp.nbytes); ctx.h2d(d_sp, sp)
    d_out = ctx.dev_alloc(N * F)
    res = []
    for pieces in (1, 16):
        b = ctx.batch(st.PDM_V2, N, order=2, bank_size=3, ctl_div_log=L, layout=st.TILED)
        f = F // pieces
        for k in range(pieces):
            b.run_dev(f, ctl=d_sp + 4 * N * (f >> L) * k, n_ctl=f >> L, out=d_out + N * f * k)
        host = np.zeros(N * F, np.uint8)
        ctx.d2h(host, d_out)
        res.append((zlib.crc32(host), zlib.crc32(b.download_state().tobytes()), zlib.crc32(b.download_bank()[0].tobytes())))
        b.free()
    assert res[0] == res[1]
    ctx.dev_free(d_out); ctx.dev_free(d_sp)


@pytest.mark.parametrize("layout", ["PLANAR", "INTERLEAVED"])
def test_c3a_square_grain_full_size(st, ctx, oracle, layout):
    """1 Mi grains x 256 frames, every output word against the oracle (2 x 1 GiB)."""
    N, F = 1024 * 1024, 256
    inp = rng.uniform(-1, 1, (N, F)).astype(np.float32)
    th = rng.uniform(0.05, 0.5, (N, 1)).astype(np.float32)
    s0 = rng.choice(np.array([0.0, 0.5, -0.5], np.float32), (N, 1))
    sa = s0[:, 0].copy()
    want = oracle.square_grain_run(sa, th[:, 0].copy(), N, F, inp)
    il = layout == "INTERLEAVED"
    b = ctx.batch(st.SQUARE_GRAIN, N, layout=getattr(st, layout))
    b.upload_state(s0); b.upload_param(th)
    out = np.zeros((F, N) if il else (N, F), np.float32)
    b.run(F, inp=np.ascontiguousarray(inp.T) if il else inp, out=out)
    assert np.array_equal((out.T if il else out).view(np.uint32), want.view(np.uint32))
    assert np.array_equal(b.download_state().view(np.float32)[:, 0], sa)
    b.free()


def test_c3b_square_grain_mix_full_size(st, ctx, oracle):
    """1 Mi grains x 256 frames, integer stereo mix: exact against the oracle, and linear over a
    partition of the grains (mix(all) == mix(first half) + mix(second half), bit for bit)."""
    N, F = 1024 * 1024, 256
    state = rng.choice(np.array([0.0, 0.5, -0.5], np.float32), N)
    th = rng.uniform(0.05, 0.5, N).astype(np.float32)
    phase = rng.integers(0, 2**32, N, dtype=np.uint32)
    inc = _note_incs(oracle, N, 36, 97)
    gl = rng.integers(0, 65, N).astype(np.uint8); gr = (64 - gl).astype(np.uint8)
    sa, pa = state.copy(), phase.copy()
    want_i, want_f = oracle.square_grain_mix_run(sa, th, pa, inc, gl, gr, N, F)

    def render(sl):
        n = sl.stop - sl.start
        b = ctx.batch(st.SQUARE_GRAIN_MIX, n)
        s_rec = np.zeros((n, 2), np.uint32); s_rec[:, 0] = state[sl].view(np.uint32); s_rec[:, 1] = phase[sl]
        p_rec = np.zeros((n, 4), np.uint32); p_rec[:, 0] = th[sl].view(np.uint32); p_rec[:, 1] = inc[sl]; p_rec[:, 2] = gl[sl]; p_rec[:, 3] = gr[sl]
        b.upload_state(s_rec); b.upload_param(p_rec)
        out = np.zeros((2, F), np.float32); mix = np.zeros((2, F), np.int32)
        b.run(F, out=out, mix=mix)
        s1 = b.download_state()
        b.free()
        return mix, out, s1

    mix, out, s1 = render(slice(0, N))
    assert np.array_equal(mix, want_i) and np.array_equal(out.view(np.uint32), want_f.view(np.uint32))
    assert np.array_equal(s1[:, 0].view(np.float32), sa) and np.array_equal(s1[:, 1], pa)
    ma, _, _ = render(slice(0, N // 2)); mb, _, _ = render(slice(N // 2, N))
    assert np.array_equal(ma + mb, mix)


@pytest.mark.parametrize("mode", [0, 1])
def test_c4p_voice_bank_full_size(st, ctx, oracle, mode):
    """4 Mi reference voices x 512 frames on one bus (sum_tick_saw / sum_tick_square): the integer
    mix, the float vector and every phase exactly; the mix is linear (saw) / an OR (square) over a
    partition of the voices -- what the multi-GPU all-reduce relies on."""
    N, F = 4 * 1024 * 1024, 512
    v = np.zeros((N, 2), np.uint32)
    v[:, 0] = _note_incs(oracle, N, 0, 128)
    v[::97, 0] = 0                                        # silent voices (note off, synth.c:173)
    v[:, 1] = rng.integers(0, 2**32, N, dtype=np.uint32)
    va = v.copy()
    want_i, want_f = oracle.voice_bank_run(va, N, N, mode, F)

    def render(sl):
        n = sl.stop - sl.start
        b = ctx.batch(st.VOICE_BANK, n, voices_per_bus=0, mode=mode)
        b.upload_state(np.ascontiguousarray(v[sl]))
        vec = np.zeros((1, F), np.float32); mix = np.zeros((1, F), np.int32)
        b.run(F, out=vec, mix=mix)
        s1 = b.download_state()
        b.free()
        return mix, vec, s1

    mix, vec, s1 = render(slice(0, N))
    assert np.array_equal(mix.view(np.uint32), np.asarray(want_i).reshape(1, F).view(np.uint32))
    assert np.array_equal(vec.view(np.uint32), np.asarray(want_f).reshape(1, F).view(np.uint32))
    assert np.array_equal(s1, va)
    ma, _, _ = render(slice(0, N // 3)); mb, _, _ = render(slice(N // 3, N))
    comb = (ma.view(np.uint32) | mb.view(np.uint32)) if mode == 1 else (ma.view(np.uint32) + mb.view(np.uint32))
    assert np.array_equal(comb, mix.view(np.uint32))


def test_c4_xvoice_mix_full_size_properties(st, ctx, oracle):
    """4 Mi voices x 512 frames, float stereo mix.  The voices are independent, so (1) the final
    state of EVERY voice must equal the oracle's for a 64 Ki subset rendered alone (bit-exact
    tick), (2) the mix of the subset alone is within the stated tolerance of the oracle's, and
    (3) the full mix equals the sum of the mixes of two halves within float summation noise."""
    N, F = 4 * 1024 * 1024, 512
    prm = np.zeros(N, po.xvoice_param_dtype)
    prm["inc"] = _note_incs(oracle, N, 24, 109)
    prm["f"] = rng.uniform(0.01, 0.3, N); prm["q"] = rng.uniform(0.5, 2.0, N)
    prm["env_attack"] = rng.uniform(1e-3, 1e-1, N); prm["env_release"] = rng.uniform(1e-3, 1e-2, N)
    prm["gate_frames"] = rng.integers(0, 400, N)
    prm["gl"] = rng.uniform(0, 1, N); prm["gr"] = 1.0 - prm["gl"]
    s0 = np.zeros(N, po.xvoice_state_dtype)
    s0["phase"] = rng.integers(0, 2**32, N, dtype=np.uint32)

    def render(sl):
        n = sl.stop - sl.start
        b = ctx.batch(st.XVOICE, n)
        b.upload_state(np.ascontiguousarray(s0[sl]).view(np.uint32).reshape(n, 5))
        b.upload_param(np.ascontiguousarray(prm[sl]).view(np.uint32).reshape(n, 8))
        mix = np.zeros((2, F), np.float32)
        b.run(F, mix=mix)
        s1 = b.download_state().view(po.xvoice_state_dtype).reshape(n)
        b.free()
        return mix, s1

    mix, s1 = render(slice(0, N))
    sub = slice(1_000_000, 1_000_000 + 65536)
    sa = s0[sub].copy()                                  # the oracle advances its state in place
    _, want_mix = oracle.xvoice_run(sa, np.ascontiguousarray(prm[sub]), 65536, F)
    assert np.array_equal(s1[sub].view(np.uint32), sa.view(np.uint32))
    msub, ssub = render(sub)
    assert np.array_equal(ssub.view(np.uint32), sa.view(np.uint32))
    w64, g64 = np.asarray(want_mix, np.float64).reshape(2, F), msub.astype(np.float64)
    assert np.abs(g64 - w64).max() <= 1e-5 * np.abs(w64).max()
    assert 10 * np.log10((w64 ** 2).sum() / max(((g64 - w64) ** 2).sum(), 1e-300)) >= 120.0
    ma, _ = render(slice(0, N // 2)); mb, _ = render(slice(N // 2, N))
    both = ma.astype(np.float64) + mb.astype(np.float64)
    assert np.abs(mix.astype(np.float64) - both).max() <= 1e-5 * np.abs(both).max()


@pytest.mark.parametrize("layout", ["TILED", "PLANAR"])
def test_c5_sweep_full_shard(st, ctx, oracle, layout):
    """2,048 variants x 480,000 frames (one GPU's shard of the 16,384-variant sweep, 7.9 GB of
    output).  The oracle renders 48 variants spread over the 8 pipeline groups sequentially;
    their rows of the time-parallel render must agree within 1e-5 of peak / 120 dB SNR -- on this
    grid (f 0.01..0.3, q 0.5..2) the sequential render is itself within ~1e-6 of the exact filter --
    with phase / frame counter / envelope bit-exact.  (The per-voice contract against the fp64 filter,
    slow and resonant settings included: tests/test_gpu_float_ref.py.)"""
    N, F = 2048, 480000
    prm = np.zeros(N, po.xvoice_param_dtype)
    prm["inc"] = oracle.note_to_inc(45)
    fg, qg = np.meshgrid(np.linspace(0.01, 0.3, 64), np.linspace(0.5, 2.0, 32))     # cutoff x resonance grid
    prm["f"] = fg.reshape(-1); prm["q"] = qg.reshape(-1)
    prm["env_attack"] = 0.01; prm["env_release"] = 1e-4; prm["gate_frames"] = 240000
    prm["gl"] = 0.75; prm["gr"] = 0.25
    s0 = np.zeros(N, po.xvoice_state_dtype)
    pick = np.sort(np.concatenate([np.arange(g * 256, g * 256 + 3) for g in range(8)] + [np.arange(g * 256 + 253, g * 256 + 256) for g in range(8)]))
    sa = np.ascontiguousarray(s0[pick])
    want_raw, _ = oracle.xvoice_run(sa, np.ascontiguousarray(prm[pick]), len(pick), F)
    want = np.asarray(want_raw).reshape(len(pick), F, 2)
    b = ctx.batch(st.XVOICE, N, layout=getattr(st, layout), mode=st.XVOICE_SCAN)
    b.upload_state(s0.view(np.uint32).reshape(N, 5)); b.upload_param(prm.view(np.uint32).reshape(N, 8))
    d_out = ctx.dev_alloc(8 * N * F)
    b.run_dev(F, out=d_out)
    got_state = b.download_state().view(po.xvoice_state_dtype).reshape(N)
    for k in ("phase", "t"):
        assert np.array_equal(got_state[k][pick], sa[k])
    assert np.array_equal(got_state["env"][pick].view(np.uint32), sa["env"].view(np.uint32))
    if layout == "PLANAR":
        got = np.zeros((len(pick), F, 2), np.float32)
        for j, i in enumerate(pick):
            ctx.d2h(got[j], d_out + 8 * F * int(i))
    else:                                                  # [F/2][inst][2][2]: the whole slab, then the picked columns
        slab = np.zeros((F // 2, N, 2, 2), np.float32)
        ctx.d2h(slab, d_out)
        got = slab[:, pick].transpose(1, 0, 2, 3).reshape(len(pick), F, 2)
        del slab
    w64, g64 = want.astype(np.float64), got.astype(np.float64)
    peak = np.abs(w64).max()
    assert peak > 0.01
    assert np.abs(g64 - w64).max() <= 1e-5 * peak
    assert 10 * np.log10((w64 ** 2).sum() / max(((g64 - w64) ** 2).sum(), 1e-300)) >= 120.0
    b.free(); ctx.dev_free(d_out)
