"""Bus mix of generated cproc graphs (io.mix of a CPROC_CUDA_GRAPH batch).

The mix of output q on bus b is a balanced pairwise tree over the bus's instances in index order: the instance count
padded to a power of two with -0.0f (0 for a `w` output), then level 1 adds instances (2m, 2m+1), level 2 those pair
sums, and so on (include/cproc_cuda.h).  Float outputs add with one binary32 rounding per add, `w` outputs mod 2^32.
Because the tree is fixed, every test here compares bit for bit against `model_mix`, a numpy statement of that tree
applied to the oracle's raw per-instance outputs (themselves bit-identical to the GPU's raw streams); a NaN only has
to be a NaN on both sides.  The CPU tests check the model; the GPU tests carry the `gpu` mark one by one.
"""
import os

import numpy as np
import pytest

from oracle import pyoracle as po
from synth_tools_b200 import abi
from tests.test_gpu_float_ref import _contrib_sums, _dyadic_voices, _mix_device, _n_sm, _xvoice_voices, gamma, mix_depth
from tools import bench_configs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TEXTS = {nm: open(os.path.join(ROOT, "tests", "golden", nm + ".cproc")).read() for nm in ("ext_voice", "ext_gain", "ext_chain")}
NEG0 = np.uint32(0x80000000)


# ------------------------------------------------------------------------------------------------ the model
def tree_sum(x, isf):
    """The documented tree over axis 0 of uint32 words x (float bits when isf)."""
    m = x.shape[0]
    P = 1 << (m - 1).bit_length()
    v = np.concatenate([x, np.full((P - m,) + x.shape[1:], NEG0 if isf else 0, np.uint32)])
    v = v.view(np.float32) if isf else v
    with np.errstate(all="ignore"):
        while len(v) > 1:
            v = v[0::2] + v[1::2]
    return v[0].view(np.uint32) if isf else v[0]


def n_bus(N, vpb):
    return 1 if vpb == 0 else -(-N // vpb)


def model_mix(raw, outf, vpb):
    """raw uint32 [N][n_out][F] -> mix uint32 [n_bus][n_out][F]; bus = instance // vpb (vpb 0: one bus)."""
    N, n_out, F = raw.shape
    span = N if vpb == 0 or vpb >= N else vpb
    mix = np.zeros((n_bus(N, vpb), n_out, F), np.uint32)
    for b in range(mix.shape[0]):
        seg = raw[b * span:(b + 1) * span]
        for q in range(n_out):
            mix[b, q] = tree_sum(seg[:, q], bool(outf[q]))
    return mix


def out_float(g):
    """Output q is a float when its node kind outputs a float (whatever statement named it)."""
    return np.array([(g["rows"][k][0] & 0xFF) >= po.NODE_PHASOR_F for k in g["out_nodes"]], bool)


def assert_mix_equal(got, want, outf, what):
    f = np.asarray(outf, bool)
    assert np.array_equal(got[:, ~f], want[:, ~f]), (what, "w outputs")
    a, b = got[:, f].view(np.float32), want[:, f].view(np.float32)
    same = (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))
    bad = np.argwhere(~same)
    assert bad.size == 0, (what, len(bad), [(tuple(int(x) for x in i), float(a[tuple(i)]), float(b[tuple(i)])) for i in bad[:4]])


def f32(x):
    return np.array(x, np.float32).view(np.uint32)


def test_tree_differs_from_serial_sum():
    u = 2.0 ** -24
    x = f32([1.0, u, u, u])
    assert tree_sum(x, True).view(np.float32) == np.float32(1.0 + 2 * u)      # (1 + u) + (u + u): the pair of halves survives
    serial = np.float32(0)
    for v in x.view(np.float32):
        serial = np.float32(serial + v)
    assert serial == np.float32(1.0)                                          # 1 + u ties to 1, three times
    x = f32([1e8, 1.0, -1e8, 1.0])
    assert tree_sum(x, True).view(np.float32) == 0.0                          # (1e8 + 1) + (-1e8 + 1) = 1e8 - 1e8
    assert np.float32(np.float32(np.float32(np.float32(1e8) + 1) - np.float32(1e8)) + 1) == 1.0
    x = f32([3.0, 5.0, 7.0])                                                  # padded to 4: (3 + 5) + (7 + -0)
    assert tree_sum(x, True).view(np.float32) == 15.0


def test_tree_identities():
    for v in (0.0, -0.0, 1.5, -2.0 ** -149, np.inf, -np.inf):
        assert tree_sum(f32([v]), True) == f32(v)                           # a one-instance bus is its output, -0 included
    assert tree_sum(f32([-0.0] * 5), True) == NEG0                           # an all -0 bus gives -0
    assert tree_sum(f32([-0.0, 0.0]), True) == 0
    assert np.isnan(tree_sum(f32([1.0, np.nan, 2.0]), True).view(np.float32))
    w = np.array([0xFFFFFFFF, 2, 0x80000000, 0x80000000], np.uint32)
    assert tree_sum(w, False) == 1                                            # mod 2^32
    raw = np.arange(2 * 3 * 4 * 5, dtype=np.uint32).reshape(4 * 5, 2, 3)
    m = model_mix(raw, [False, False], 8)                                     # 20 instances, buses of 8: 8 + 8 + 4
    assert m.shape == (3, 2, 3) and np.array_equal(m[2], raw[16:].sum(axis=0, dtype=np.uint32))


def test_jit_source_has_mix_kernel_and_no_ftz():
    for nm, text in TEXTS.items():
        g = abi.graph_parse_ex(text)
        src = abi.graph_jit_source(g["rows"], g["n_inputs"], g["out_nodes"], has_changed=nm == "ext_chain")
        assert "graph_mix(" in src and "__shfl_xor_sync" in src and ".ftz" not in src.lower(), nm
        mask = sum(1 << q for q, f in enumerate(out_float(g)) if f)
        assert "#define GRAPH_OUTF 0x%xu" % mask in src, nm


# ------------------------------------------------------------------------------------------------ records
def records(rng, g, N):
    """Random state (phasor phases, float state in [-1, 1], counters) and params (the text's initialisers, with
    per-instance increments, filters, envelopes and gains)."""
    rows = g["rows"]
    sw = sum(po.node_words(r[0]) for r in rows)
    st0 = np.zeros((N, sw), np.uint32)
    prm = np.tile(g["param_init"], (N, 1))
    o = p = 0
    for r in rows:
        k = r[0] & 0xFF
        if k == po.NODE_PHASOR_F:
            st0[:, o + 1] = rng.integers(0, 2**32, N, dtype=np.uint32)
            prm[:, p] = rng.integers(1 << 22, 1 << 28, N, dtype=np.uint32)
        elif k in (po.NODE_SVF, po.NODE_ONEPOLE):
            st0[:, o:o + po.node_words(r[0])] = rng.uniform(-1, 1, (N, po.node_words(r[0]))).astype(np.float32).view(np.uint32)
            if k == po.NODE_SVF:
                prm[:, p:p + 2] = np.stack([rng.uniform(0.01, 0.3, N), rng.uniform(0.5, 2.0, N)], axis=1).astype(np.float32).view(np.uint32)
        elif k == po.NODE_ENV:
            prm[:, p:p + 2] = np.stack([rng.uniform(1e-3, 0.1, N), rng.uniform(1e-3, 1e-2, N)], axis=1).astype(np.float32).view(np.uint32)
            prm[:, p + 2] = rng.integers(0, 400, N, dtype=np.uint32)
        elif k == po.NODE_GAIN:
            prm[:, p] = rng.uniform(-1, 1, N).astype(np.float32).view(np.uint32)
        elif k in (po.NODE_ACC, po.NODE_EDGE):
            st0[:, o] = rng.integers(0, 2**32, N, dtype=np.uint32)
        o += po.node_words(r[0])
        p += {po.NODE_PHASOR_F: 1, po.NODE_SVF: 2, po.NODE_ENV: 3, po.NODE_ONEPOLE: 1, po.NODE_GAIN: 1}.get(k, 0)
    return st0, np.ascontiguousarray(prm) if prm.shape[1] else None


def streams(rng, nm, N, F):
    """Input streams [N][n_in][F] and the changed stream [N][F] (ext_chain only) of a golden graph."""
    if nm == "ext_voice":
        return rng.integers(0, 1 << 20, (N, 1, F), dtype=np.uint32), None
    if nm == "ext_gain":
        return rng.uniform(-1, 1, (N, 1, F)).astype(np.float32).view(np.uint32), None
    inp = np.stack([rng.integers(0, 3, (N, F)), rng.integers(0, 1 << 20, (N, F))], axis=1).astype(np.uint32)
    return inp, rng.integers(0, 4, (N, F)).astype(np.uint32)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def st():
    import synth_tools_b200 as st_
    return st_


@pytest.fixture(scope="module")
def ctx(st):
    c = st.Context(0)
    yield c
    c.close()


def render(st, ctx, g, st0, prm, N, F, vpb, layout, inp=None, chg=None, want_out=False, slices=None):
    """Mix (and out, when asked) of F frames rendered through cproc_cuda_run in the given frame slices; the final state."""
    il = layout == st.INTERLEAVED
    n_out = len(g["out_nodes"])
    b = ctx.batch(st.GRAPH, N, nodes=g["rows"], n_inputs=g["n_inputs"], out_node=g["out_nodes"], layout=layout, voices_per_bus=vpb)
    mixes, outs = [], []
    try:
        b.upload_state(st0)
        if prm is not None:
            b.upload_param(prm)
        for a, c in slices or [(0, F)]:
            Fk = c - a
            mix = np.full((n_bus(N, vpb), n_out, Fk), 0xDEADBEEF, np.uint32)
            out = np.zeros((Fk, n_out, N) if il else (N, n_out, Fk), np.uint32) if want_out else None
            x = None if inp is None else np.ascontiguousarray(inp[:, :, a:c].transpose(2, 1, 0) if il else inp[:, :, a:c])
            y = None if chg is None else np.ascontiguousarray(chg[:, a:c].T if il else chg[:, a:c])
            b.run(Fk, inp=x, in2=y, out=out, mix=mix)
            mixes.append(mix)
            if want_out:
                outs.append(np.ascontiguousarray(out.transpose(2, 1, 0)) if il else out)
        state = b.download_state()
    finally:
        b.free()
    return np.concatenate(mixes, axis=2), (np.concatenate(outs, axis=2) if want_out else None), state


NS = [1, 31, 32, 33, 1000, 148 * 128 + 333]
FS = [1, 63, 64, 512, 1000]
VPBS = [0, 32, 64, 96]


@pytest.mark.gpu
@pytest.mark.parametrize("jit", [1, 0], ids=["generated", "table"])
@pytest.mark.parametrize("F", FS)
@pytest.mark.parametrize("N", NS)
@pytest.mark.parametrize("nm", sorted(TEXTS))
def test_graph_mix_bit_exact(st, ctx, oracle, nm, N, F, jit):
    """The GPU mix equals the tree over the oracle's raw outputs, bit for bit, for PLANAR and INTERLEAVED inputs and
    buses of 0 (all), 32, 64 and 96 instances; the final state equals the oracle's.  Both the generated kernel and the
    table-driven one (graph_jit = 0, the path without libnvrtc)."""
    rng = np.random.default_rng(N * 1009 + F)
    g = abi.graph_parse_ex(TEXTS[nm])
    st0, prm = records(rng, g, N)
    inp, chg = streams(rng, nm, N, F)
    sa = st0.copy()
    raw = oracle.graph_run_ext(g["rows"], g["n_inputs"], g["out_nodes"], sa, prm, N, F, inp, chg)
    outf = out_float(g)
    try:
        ctx.set_option("graph_jit", jit)
        for vpb in VPBS:
            want = model_mix(raw, outf, vpb)
            for layout in (st.PLANAR, st.INTERLEAVED):
                mix, _, state = render(st, ctx, g, st0, prm, N, F, vpb, layout, inp, chg)
                assert_mix_equal(mix, want, outf, (nm, N, F, vpb, layout))
                assert np.array_equal(state, sa), (nm, N, F, vpb, layout)
    finally:
        ctx.set_option("graph_jit", 1)


@pytest.mark.gpu
@pytest.mark.parametrize("jit", [1, 0], ids=["generated", "table"])
@pytest.mark.parametrize("N", [1, 31, 32, 33, 95, 97, 129, 1000])
@pytest.mark.parametrize("vpb", [0, 32, 64])
def test_graph_mix_writes_nothing_past_the_mix(st, ctx, oracle, N, vpb, jit):
    """run_dev into a device buffer followed by a canary region: the mix fills [n_bus][n_outputs][F] exactly and not a
    word past it, whatever the launch's last block holds beyond n (the instance count rarely fills it); the mix is the
    model's."""
    F = 40
    rng = np.random.default_rng(N + 7 * vpb)
    g = abi.graph_parse_ex(bench_configs.VOICE_GRAPH_TEXT)
    st0, prm = records(rng, g, N)
    sa = st0.copy()
    want = model_mix(oracle.graph_run_ext(g["rows"], 0, g["out_nodes"], sa, prm, N, F), out_float(g), vpb)
    words, canary = want.size, 8 * 2 * F * 4
    host = np.full(words + canary, 0xC0FFEE11, np.uint32)
    d = ctx.dev_alloc(host.nbytes)
    b = ctx.batch(st.GRAPH, N, nodes=g["rows"], n_inputs=0, out_node=g["out_nodes"], voices_per_bus=vpb)
    try:
        ctx.set_option("graph_jit", jit)
        b.upload_state(st0); b.upload_param(prm)
        ctx.h2d(d, host)
        b.run_dev(F, mix=d)
        ctx.sync()
        ctx.d2h(host, d)
        assert np.all(host[words:] == 0xC0FFEE11), (N, vpb, int(np.argmax(host[words:] != 0xC0FFEE11)))
        assert_mix_equal(host[:words].reshape(want.shape), want, out_float(g), (N, vpb))
        assert np.array_equal(b.download_state(), sa)
    finally:
        ctx.set_option("graph_jit", 1)
        b.free()
        ctx.dev_free(d)


@pytest.mark.gpu
@pytest.mark.parametrize("nm", sorted(TEXTS))
@pytest.mark.parametrize("layout", [0, 1])
def test_graph_mix_with_out(st, ctx, oracle, nm, layout):
    """out + mix: out is bit for bit what an out-only render writes, and so is the final state."""
    N, F, vpb = 1000, 203, 96
    rng = np.random.default_rng(77)
    g = abi.graph_parse_ex(TEXTS[nm])
    st0, prm = records(rng, g, N)
    inp, chg = streams(rng, nm, N, F)
    il = layout == st.INTERLEAVED
    b = ctx.batch(st.GRAPH, N, nodes=g["rows"], n_inputs=g["n_inputs"], out_node=g["out_nodes"], layout=layout)
    try:
        b.upload_state(st0)
        b.upload_param(prm)
        n_out = len(g["out_nodes"])
        out = np.zeros((F, n_out, N) if il else (N, n_out, F), np.uint32)
        b.run(F, inp=np.ascontiguousarray(inp.transpose(2, 1, 0) if il else inp), in2=None if chg is None else np.ascontiguousarray(chg.T if il else chg), out=out)
        want_state = b.download_state()
    finally:
        b.free()
    want_out = np.ascontiguousarray(out.transpose(2, 1, 0)) if il else out
    mix, got_out, state = render(st, ctx, g, st0, prm, N, F, vpb, layout, inp, chg, want_out=True)
    assert np.array_equal(got_out, want_out)
    assert np.array_equal(state, want_state)
    assert_mix_equal(mix, model_mix(want_out, out_float(g), vpb), out_float(g), nm)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", [0, 1])
def test_graph_mix_options(st, ctx, oracle, layout):
    """graph_jit 0/1 (generated kernel / table-driven kernel), graph_vec4 0/1 and planar_bulk 0/2 give the same bits."""
    N, F, vpb = 333, 100, 64
    rng = np.random.default_rng(5)
    g = abi.graph_parse_ex(TEXTS["ext_chain"])
    st0, prm = records(rng, g, N)
    inp, chg = streams(rng, "ext_chain", N, F)
    sa = st0.copy()
    want = model_mix(oracle.graph_run_ext(g["rows"], g["n_inputs"], g["out_nodes"], sa, prm, N, F, inp, chg), out_float(g), vpb)
    try:
        for jit in (1, 0):
            for vec4 in (1, 0):
                for pb in (0, 2):
                    ctx.set_option("graph_jit", jit); ctx.set_option("graph_vec4", vec4); ctx.set_option("planar_bulk", pb)
                    mix, _, state = render(st, ctx, g, st0, prm, N, F, vpb, layout, inp, chg)
                    assert_mix_equal(mix, want, out_float(g), (jit, vec4, pb))
                    assert np.array_equal(state, sa), (jit, vec4, pb)
    finally:
        ctx.set_option("graph_jit", 1); ctx.set_option("graph_vec4", 1); ctx.set_option("planar_bulk", 2)


@pytest.mark.gpu
@pytest.mark.parametrize("nm", sorted(TEXTS))
@pytest.mark.parametrize("jit", [1, 0])
def test_graph_mix_split_renders(st, ctx, nm, jit):
    """F frames in one call equal the same frames in several calls: the mixes concatenated, the state identical."""
    N, F, vpb = 1000, 300, 32
    rng = np.random.default_rng(11)
    g = abi.graph_parse_ex(TEXTS[nm])
    st0, prm = records(rng, g, N)
    inp, chg = streams(rng, nm, N, F)
    try:
        ctx.set_option("graph_jit", jit)
        for layout in (st.PLANAR, st.INTERLEAVED):
            whole, _, s1 = render(st, ctx, g, st0, prm, N, F, vpb, layout, inp, chg)
            parts, _, s2 = render(st, ctx, g, st0, prm, N, F, vpb, layout, inp, chg, slices=[(0, 1), (1, 64), (64, 65), (65, 200), (200, 300)])
            assert np.array_equal(whole, parts) and np.array_equal(s1, s2), (layout,)
    finally:
        ctx.set_option("graph_jit", 1)


@pytest.mark.gpu
@pytest.mark.parametrize("nm", ["voice", "ext_voice"])
def test_graph_mix_host_buffers_period_shape(st, ctx, nm):
    """The JACK period shape (16 parts x 64 voices x 64 frames): cproc_cuda_run under run_graph 0..3 (staged copies,
    CUDA graph with copy nodes, CUDA graph on pinned staging, direct launches) and cproc_cuda_run_period give the bits of
    cproc_cuda_run_dev, period after period (the first call of a shape runs the ordinary way, the second captures)."""
    N, F, vpb, periods = 16 * 64, 64, 64, 4
    rng = np.random.default_rng(3)
    g = abi.graph_parse_ex(bench_configs.VOICE_GRAPH_TEXT if nm == "voice" else TEXTS[nm])
    st0, prm = records(rng, g, N)
    n_in, n_out = g["n_inputs"], len(g["out_nodes"])
    inps = [rng.integers(0, 1 << 20, (N, n_in, F), dtype=np.uint32) if n_in else None for _ in range(periods)]
    b = ctx.batch(st.GRAPH, N, nodes=g["rows"], n_inputs=n_in, out_node=g["out_nodes"], voices_per_bus=vpb)
    d_mix = ctx.dev_alloc(4 * N // vpb * n_out * F)
    d_in = ctx.dev_alloc(4 * N * max(n_in, 1) * F)
    try:
        b.upload_param(prm)
        b.upload_state(st0)
        want = []
        for k in range(periods):
            if n_in:
                ctx.h2d(d_in, inps[k])
            b.run_dev(F, inp=d_in if n_in else None, mix=d_mix)
            m = np.zeros((N // vpb, n_out, F), np.uint32)
            ctx.d2h(m, d_mix)
            want.append(m)
        want_state = b.download_state()
        for rg in range(4):
            ctx.set_option("run_graph", rg)
            b.upload_state(st0)
            for k in range(periods):
                m = np.full((N // vpb, n_out, F), 0xDEADBEEF, np.uint32)
                b.run(F, inp=inps[k], mix=m)
                assert np.array_equal(m, want[k]), (rg, k)
            assert np.array_equal(b.download_state(), want_state), rg
        ctx.set_option("run_graph", 2)
        state = st0.copy()
        for k in range(periods):
            m = np.full((N // vpb, n_out, F), 0xDEADBEEF, np.uint32)
            b.run_period(F, state, inp=inps[k], mix=m)
            assert np.array_equal(m, want[k]), ("run_period", k)
        assert np.array_equal(state, want_state)
    finally:
        ctx.set_option("run_graph", 2)
        ctx.dev_free(d_mix); ctx.dev_free(d_in)
        b.free()


def voice_graph_records(s0, prm):
    """XVOICE records -> the voice graph's {osc.out, osc.phase, flt.out, flt.bp, amp.out, amp.env, amp.t, l.out, r.out} and
    its param record (the same eight words in the same order)."""
    N = len(s0)
    gst = np.zeros((N, 9), np.uint32)
    gst[:, 1] = s0["phase"]; gst[:, 2] = s0["lp"].view(np.uint32); gst[:, 3] = s0["bp"].view(np.uint32)
    gst[:, 5] = s0["env"].view(np.uint32); gst[:, 6] = s0["t"]
    return gst, np.ascontiguousarray(prm.view(np.uint32).reshape(N, 8))


def voice_mix(st, ctx, s0, prm, F, vpb=0):
    g = abi.graph_parse_ex(bench_configs.VOICE_GRAPH_TEXT)
    gst, gp = voice_graph_records(s0, prm)
    mix, _, state = render(st, ctx, g, gst, gp, len(s0), F, vpb, st.PLANAR)
    return mix, state


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["random", "cancelling"])
def test_graph_mix_error_bound(st, ctx, oracle, case):
    """About 1 Mi voices on one bus: |mix[t] - S[t]| <= gamma_d sum_v |c_v[t]| with d = log2 of the padded bus size
    (each leaf-to-root path of the tree has d roundings).  Cancelling: pairs of equal voices with opposite gains, S = 0."""
    rng = np.random.default_rng(21)
    N, F = (1 << 20) - 3, 64
    s0, prm = _xvoice_voices(oracle, N, F, rng.uniform(0.01, 0.3, N), rng.uniform(0.5, 2.0, N), quiet=0.1)
    if case == "cancelling":
        h = N // 2
        for k in s0.dtype.names:
            s0[k][h:2 * h] = s0[k][:h]
        for k in prm.dtype.names:
            prm[k][h:2 * h] = prm[k][:h]
        prm["gl"][h:2 * h] = -prm["gl"][:h]; prm["gr"][h:2 * h] = -prm["gr"][:h]
    S, A, sa = _contrib_sums(oracle, s0, prm, F)
    mix, state = voice_mix(st, ctx, s0, prm, F)
    kept = [1, 2, 3, 5, 6]                                               # the words the XVOICE record holds too
    assert np.array_equal(state[:, kept], voice_graph_records(sa, prm)[0][:, kept])
    d = (N - 1).bit_length()
    err = np.abs(mix[0].view(np.float32).astype(np.float64) - S)
    assert np.all(err <= gamma(d) * A), (d, float((err - gamma(d) * A).max()))


@pytest.mark.gpu
@pytest.mark.parametrize("N,F", [(1000, 512), (148 * 4 * 128 + 333, 96)])
def test_graph_mix_against_xvoice(st, ctx, oracle, N, F):
    """The voice graph's mix and XVOICE's mix (k_xvoice_mix2) of the same voices are each within their gamma_d of the exact
    sum; on dyadic voices (every partial sum exact in binary32) the two are bit-identical and equal the exact sum."""
    rng = np.random.default_rng(N)
    s0, prm = _xvoice_voices(oracle, N, F, rng.uniform(0.01, 0.3, N), rng.uniform(0.5, 2.0, N), quiet=0.1)
    S, A, _ = _contrib_sums(oracle, s0, prm, F)
    gm, _ = voice_mix(st, ctx, s0, prm, F)
    xm, _ = _mix_device(st, ctx, s0, prm, F, "mix2")
    dg, dx = (N - 1).bit_length(), mix_depth("mix2", N, _n_sm())
    assert np.all(np.abs(gm[0].view(np.float32).astype(np.float64) - S) <= gamma(dg) * A)
    assert np.all(np.abs(xm.astype(np.float64) - S) <= gamma(dx) * A)
    s0, prm = _dyadic_voices(N, F)
    S, _, _ = _contrib_sums(oracle, s0, prm, F)
    gm, _ = voice_mix(st, ctx, s0, prm, F)
    xm, _ = _mix_device(st, ctx, s0, prm, F, "mix2")
    assert np.array_equal(gm[0].view(np.float32), xm) and np.array_equal(xm.astype(np.float64), S)


@pytest.mark.gpu
def test_graph_mix_full_shape(st, ctx, oracle):
    """4 Mi voices x 512 frames, mix only, buses of 4096: a sample of buses equals the tree over the oracle's outputs
    of those buses' voices, bit for bit, and so do their final states."""
    N, F, vpb = 4 * 1024 * 1024, 512, 4096
    g = abi.graph_parse_ex(bench_configs.VOICE_GRAPH_TEXT)
    stt, prm = bench_configs.xvoice_records(np.random.default_rng(12), N)
    gst = np.zeros((N, 9), np.uint32)
    gst[:, 1] = stt[:, 0]
    mix, _, state = render(st, ctx, g, gst, prm, N, F, vpb, st.PLANAR)
    for bus in (0, 1, 517, N // vpb - 1):
        sl = slice(bus * vpb, (bus + 1) * vpb)
        sa = gst[sl].copy()
        raw = oracle.graph_run_ext(g["rows"], 0, g["out_nodes"], sa, np.ascontiguousarray(prm[sl]), vpb, F)
        assert_mix_equal(mix[bus:bus + 1], model_mix(raw, out_float(g), 0), out_float(g), bus)
        assert np.array_equal(state[sl], sa), bus


@pytest.mark.gpu
def test_graph_mix_errors(st, ctx):
    """voices_per_bus neither 0 nor a multiple of 32, the GRAPH_SCAN mode and the TILED layout are rejected with a message
    when io.mix is set -- alloc accepts them, as before -- and nothing is written."""
    g = abi.graph_parse_ex(TEXTS["ext_voice"])
    N, F = 100, 64
    inp = np.zeros((N, 1, F), np.uint32)
    chain = [(po.NODE_EDGE, -1, 1), (po.NODE_ACC, 0, 1)]
    cases = [(dict(nodes=g["rows"], out_node=g["out_nodes"], voices_per_bus=48), st.PLANAR, "voices_per_bus"),
             (dict(nodes=g["rows"], out_node=g["out_nodes"], voices_per_bus=1), st.INTERLEAVED, "voices_per_bus"),
             (dict(nodes=chain, mode=1), st.PLANAR, "GRAPH_SCAN"),
             (dict(nodes=g["rows"], out_node=g["out_nodes"]), st.TILED, "TILED")]
    for kw, layout, what in cases:
        b = ctx.batch(st.GRAPH, N, n_inputs=1, **kw)
        try:
            s0 = b.download_state()
            n_out = len(kw.get("out_node", [0]))
            for dev in (False, True):
                mix = np.full((4, n_out, F), 0xDEADBEEF, np.uint32)
                with pytest.raises(abi.CprocCudaError) as e:
                    if dev:
                        d_in, d_mix = ctx.dev_alloc(inp.nbytes), ctx.dev_alloc(mix.nbytes)
                        try:
                            ctx.h2d(d_mix, mix)
                            try:
                                b.run_dev(F, inp=d_in, mix=d_mix, layout=layout)
                            finally:
                                ctx.sync()
                                ctx.d2h(mix, d_mix)
                        finally:
                            ctx.dev_free(d_in); ctx.dev_free(d_mix)
                    else:
                        b.run(F, inp=inp, mix=mix, layout=layout)
                assert e.value.code == abi.EINVAL and what in str(e.value), (what, str(e.value))
                assert np.all(mix == 0xDEADBEEF), what
            assert np.array_equal(b.download_state(), s0), what
        finally:
            b.free()
