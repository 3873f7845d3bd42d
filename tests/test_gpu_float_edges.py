"""The float processors at the edges of IEEE binary32: signed zeros, subnormals, FLT_MIN / FLT_MAX, infinities, NaNs
with different payloads, and thresholds the square_grain phasor lands on exactly.

cproc_cuda.h promises every float processor bit-identical to its C definition compiled with -ffp-contract=off, with
one exception: a NaN result may be the GPU's canonical NaN where an x86 host keeps the operand's payload.
`same_float` is that rule, and nothing looser.

CPU: the comparison and the value pool test themselves; the oracle equals the reference's own code at these values
(square_grain_proc also against an independent restatement); no float instruction of the built library, nor of the
source generated for a graph, flushes subnormals to zero.  GPU: every sequential float path -- raw square_grain, the
three square_grain mix generations with and without a fused bus, the one-pole, the extension voice raw and mixed,
and the extension graph nodes in every kernel the front end can pick -- equals the oracle under `same_float`, final
state included.  The GPU tests carry the `gpu` mark one by one."""
import ctypes as C
import glob
import itertools
import os
import re
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from oracle import pyoracle as po

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OBJ = os.path.join(ROOT, "synth_tools_b200", "build")
rng = np.random.default_rng(20261022)
M32 = 0xFFFFFFFF


def f32(bits):
    return np.uint32(bits).view(np.float32)


# ------------------------------------------------------------------------------------------------ value pool
# name -> bit pattern.  The multiples of 2^-31 are the values (float)(int32)phase * 2^-31 takes next to zero.
POOL = {
    "+0": 0x00000000, "-0": 0x80000000,
    "+min subnormal": 0x00000001, "-min subnormal": 0x80000001,
    "+max subnormal": 0x007FFFFF, "-max subnormal": 0x807FFFFF,
    "+FLT_MIN": 0x00800000, "-FLT_MIN": 0x80800000,
    "+2^-31": 0x30000000, "-2^-31": 0xB0000000, "+2*2^-31": 0x30800000, "-3*2^-31": 0xB0C00000, "+5*2^-31": 0x31200000,
    "+0.5": 0x3F000000, "-0.5": 0xBF000000, "+1": 0x3F800000, "-1": 0xBF800000,
    "1-ulp": 0x3F7FFFFF, "1+ulp": 0x3F800001,
    "+FLT_MAX": 0x7F7FFFFF, "-FLT_MAX": 0xFF7FFFFF, "+inf": 0x7F800000, "-inf": 0xFF800000,
    "+qNaN": 0x7FC00000, "-qNaN": 0xFFC00000, "+qNaN payload": 0x7FC12345, "-qNaN payload": 0xFFD00001, "NaN all ones": 0x7FFFFFFF,
}
POOL_BITS = np.array(list(POOL.values()), np.uint32)
POOL_F = POOL_BITS.view(np.float32)
POOL_FINITE = POOL_F[np.isfinite(POOL_F)]
SUBNORMALS = POOL_F[(POOL_F != 0) & (np.abs(POOL_F) < np.float32(1.1754944e-38))]


def pool_draw(shape, finite=False):
    return rng.choice(POOL_FINITE if finite else POOL_F, shape).astype(np.float32)


# ------------------------------------------------------------------------------------------------ comparison
def float_mismatch(got, want, strict=False, zero_sign=True):
    """None when got equals want word for word, where two NaNs count as equal (any payloads, any signs) unless
    `strict`, and +0 equals -0 only when `zero_sign` is False; else a message naming the first differing index and
    both bit patterns."""
    g = np.ascontiguousarray(got)
    w = np.ascontiguousarray(want)
    if g.shape != w.shape:
        return "shape %s, want %s" % (g.shape, w.shape)
    gb, wb = g.view(np.uint32).reshape(-1), w.view(np.uint32).reshape(-1)
    ok = gb == wb
    gf, wf = gb.view(np.float32), wb.view(np.float32)
    if not strict:
        ok |= np.isnan(gf) & np.isnan(wf)
    if not zero_sign:
        ok |= (gf == 0) & (wf == 0)
    if ok.all():
        return None
    i = int(np.argmin(ok))
    return "%d of %d words differ; first at index %s: got 0x%08x (%r), want 0x%08x (%r)" % (
        int((~ok).sum()), ok.size, tuple(int(k) for k in np.unravel_index(i, g.shape)), int(gb[i]), float(gf[i]), int(wb[i]), float(wf[i]))


def same_float(got, want, what="", **kw):
    m = float_mismatch(got, want, **kw)
    assert m is None, "%s: %s" % (what, m)


def test_same_float_is_bitwise_except_nan():
    a = np.array([0.0, 1.0, -2.5], np.float32)
    same_float(a, a.copy())
    assert float_mismatch(np.array([0.0], np.float32), np.array([-0.0], np.float32))
    assert float_mismatch(f32(0x3F800000).reshape(1), f32(0x3F800001).reshape(1))
    assert float_mismatch(f32(0x00000001).reshape(1), np.zeros(1, np.float32))        # a flushed subnormal
    nan1, nan2 = f32(0x7FC00000).reshape(1), f32(0xFFD00001).reshape(1)
    assert float_mismatch(nan1, nan2) is None                                          # the header's one exception
    assert float_mismatch(nan1, nan2, strict=True)
    assert float_mismatch(nan1, np.array([np.inf], np.float32))
    assert float_mismatch(np.array([0.0], np.float32), np.array([-0.0], np.float32), zero_sign=False) is None
    assert float_mismatch(np.zeros(3, np.float32), np.zeros(4, np.float32))
    m = float_mismatch(np.array([[1, 2], [3, 4]], np.float32), np.array([[1, 2], [3, 5]], np.float32))
    assert "(1, 1)" in m and "0x40400000" not in m and "0x40800000" in m and "0x40a00000" in m


def test_value_pool():
    assert len(set(POOL_BITS.tolist())) == len(POOL_BITS)
    f = POOL_F
    assert np.sum((f == 0) & ~np.signbit(f)) == 1 and np.sum((f == 0) & np.signbit(f)) == 1
    assert len(SUBNORMALS) == 4 and set(np.signbit(SUBNORMALS).tolist()) == {False, True}
    assert f32(0x00000001) == np.float32(2.0 ** -149) and f32(0x00800000) == np.finfo(np.float32).tiny
    assert f32(0x7F7FFFFF) == np.finfo(np.float32).max and np.isposinf(f32(0x7F800000)) and np.isneginf(f32(0xFF800000))
    assert f32(0x30000000) == np.float32(2.0 ** -31) and f32(0xB0C00000) == np.float32(-3 * 2.0 ** -31)
    assert f32(0x3F800001) == np.nextafter(np.float32(1), np.float32(2))
    assert f32(0x3F7FFFFF) == np.nextafter(np.float32(1), np.float32(0))
    nans = POOL_BITS[np.isnan(f)]
    assert len(nans) >= 4 and len(set(nans.tolist())) == len(nans) and {n >> 31 for n in nans.tolist()} == {0, 1}
    assert all(n & 0x00400000 for n in nans.tolist())                                 # quiet NaNs only
    for k in (1, 2, 3, 5):                                                             # the phasor's read-out near 0
        x = np.float32(np.float32(k) * np.float32(2.0 ** -31))
        assert x in np.abs(f)


# ------------------------------------------------------------------------------------------------ CPU: oracle vs reference
def square_grain_restated(state, th, inp):
    """synth_tools.c:85-100 restated with numpy's IEEE comparisons: out = state; flip on the two-branch rule."""
    s = np.asarray(state, np.float32).copy()
    out = np.empty_like(inp)
    for i in range(inp.shape[1]):
        out[:, i] = s
        v = inp[:, i]
        down = (s >= 0) & (v < -th)
        up = ~down & (s < 0) & (v > th)
        s = np.where(down, np.float32(-0.5), np.where(up, np.float32(0.5), s))
    return out, s


def _grain_edge_inputs(N, F):
    st = pool_draw(N)
    th = pool_draw(N)
    th[::3] = rng.uniform(0.05, 0.5, len(th[::3])).astype(np.float32)
    inp = rng.uniform(-1, 1, (N, F)).astype(np.float32)
    pick = rng.random((N, F))
    inp = np.where(pick < 0.3, pool_draw((N, F)), inp)
    inp = np.where((pick >= 0.3) & (pick < 0.5), th[:, None], inp)
    inp = np.where((pick >= 0.5) & (pick < 0.7), -th[:, None], inp)
    return st, th, np.ascontiguousarray(inp, np.float32)


@pytest.fixture(scope="module")
def libref():
    """The reference's own code (oracle/_ref/libref.so), where its sources are present to build it."""
    if not po.have_ref():
        pytest.skip("the reference's sources are not present: oracle/_ref/libref.so cannot be built")
    return po.Ref()


def test_square_grain_oracle_vs_restatement_at_edge_values(oracle):
    N, F = 97, 300
    st, th, inp = _grain_edge_inputs(N, F)
    sa = st.copy()
    out = oracle.square_grain_run(sa, th, N, F, inp)
    want, s1 = square_grain_restated(st, th, inp)
    same_float(out, want, "out", strict=True)
    same_float(sa, s1, "state", strict=True)
    assert np.isnan(st).any() and np.isnan(th).any() and (inp == th[:, None]).any()


def test_square_grain_oracle_vs_ref_at_edge_values(oracle, libref):
    N, F = 97, 300
    st, th, inp = _grain_edge_inputs(N, F)
    sa, sb = st.copy(), st.copy()
    a = oracle.square_grain_run(sa, th, N, F, inp)
    b = libref.square_grain_run(sb, th, N, F, inp)
    same_float(a, b, "out", strict=True)
    same_float(sa, sb, "state", strict=True)


# Extension graphs at edge values.  Which words of a node's state / param record are floats (include/cproc_ext.h).
STATE_FLOAT = {po.NODE_ACC: [0], po.NODE_EDGE: [0, 0], po.NODE_PHASOR_F: [1, 0], po.NODE_SVF: [1, 1], po.NODE_ENV: [1, 1, 0],
               po.NODE_ONEPOLE: [1], po.NODE_GAIN: [1], po.NODE_ASFLOAT: [1], po.NODE_GLIDE_F: [1, 1, 0], po.NODE_MUL: [1]}
PARAM_FLOAT = {po.NODE_PHASOR_F: [0], po.NODE_SVF: [1, 1], po.NODE_ENV: [1, 1, 0], po.NODE_ONEPOLE: [1], po.NODE_GAIN: [1]}


def edge_ext_graph(r, n_nodes, n_inputs, masks):
    """A random table over acc / edge and all eight float kinds (tests/test_graph_ext.py), where asfloat may read any
    word: an input stream or an integer node."""
    from tests.test_graph_ext import random_ext_graph
    rows = random_ext_graph(r, n_nodes, n_inputs, masks=masks)
    for k, row in enumerate(rows):
        if row[0] & 0xFF == po.NODE_ASFLOAT and row[1] != po.SRC_ZERO:
            cands = [-(j + 1) for j in range(n_inputs)] + [j for j in range(k) if (rows[j][0] & 0xFF) < po.NODE_PHASOR_F]
            rows[k] = (row[0], int(r.choice(cands)), row[2])
    return rows


def edge_ext_records(r, rows, N, n_inputs, F):
    """Pool-drawn float words in state, params and inputs; env gates of 0xFFFFFFFF with t near the wrap; glide_f with
    in - out = +-inf.  Returns (state, param or None, inputs, float mask of the state words)."""
    sw = sum(po.node_words(x[0]) for x in rows)
    st0 = r.integers(0, 2**32, (N, sw), dtype=np.uint32)
    fmask = np.zeros(sw, bool)
    o = 0
    for x in rows:
        kind = x[0] & 0xFF
        for k, isf in enumerate(STATE_FLOAT[kind]):
            fmask[o + k] = isf
            if isf:
                st0[:, o + k] = pool_draw(N).view(np.uint32)
                st0[::2, o + k] = r.uniform(-1, 1, len(st0[::2])).astype(np.float32).view(np.uint32)
        if kind == po.NODE_ENV:
            st0[:, o + 2] = r.choice(np.array([0, 5, M32 - 40, M32 - 3, M32], np.uint32), N)
        if kind == po.NODE_GLIDE_F:
            st0[:, o + 2] = r.integers(0, 1 << ((x[0] >> 8) & 0xFF), N, dtype=np.uint32)   # count below the divider
        o += po.node_words(x[0])
    cols = []
    for x in rows:
        kind = x[0] & 0xFF
        for k, isf in enumerate(PARAM_FLOAT.get(kind, [])):
            if isf:
                c = pool_draw(N)
                c[::2] = r.uniform(0.001, 0.9, len(c[::2])).astype(np.float32)
                cols.append(c.view(np.uint32))
            elif kind == po.NODE_ENV:
                cols.append(r.choice(np.array([0, 1, 7, M32 - 1, M32], np.uint32), N))
            else:
                cols.append(r.integers(0, 2**32, N, dtype=np.uint32))
    prm = np.ascontiguousarray(np.stack(cols, axis=1)) if cols else None
    inp = np.where(r.random((N, n_inputs, F)) < 0.5, pool_draw((N, n_inputs, F)),
                   r.uniform(-2, 2, (N, n_inputs, F)).astype(np.float32)).astype(np.float32).view(np.uint32)
    inp = np.ascontiguousarray(inp)
    inp[:, 0, ::7] = r.integers(0, 2**32, inp[:, 0, ::7].shape, dtype=np.uint32)      # any word at all
    # glide_f with in - out = +-inf: out = -+FLT_MAX (or inf) against pool inputs of the opposite sign
    o = 0
    for x in rows:
        if x[0] & 0xFF == po.NODE_GLIDE_F:
            st0[1::3, o] = f32(0xFF7FFFFF).view(np.uint32)
            st0[2::5, o] = f32(0x7F800000).view(np.uint32)
        o += po.node_words(x[0])
    return st0, prm, inp, fmask


def out_float_mask(rows, outs):
    return np.array([(rows[q][0] & 0xFF) >= po.NODE_PHASOR_F for q in outs], bool)


def assert_ext_equal(got, want, st_got, st_want, rows, outs, fmask, what):
    om = out_float_mask(rows, outs)
    assert np.array_equal(got[:, ~om], want[:, ~om]), (what, "integer outputs", rows)
    same_float(got[:, om].view(np.float32), want[:, om].view(np.float32), "%s: float outputs of %s" % (what, rows))
    assert np.array_equal(st_got[:, ~fmask], st_want[:, ~fmask]), (what, "integer state words", rows)
    same_float(st_got[:, fmask].view(np.float32), st_want[:, fmask].view(np.float32), "%s: float state words of %s" % (what, rows))


def every_float_kind_graph():
    """asfloat -> onepole, phasor_f -> svf -> env -> gain -> glide_f, mul (gain x glide_f); acc and edge on input 1."""
    rows = [(po.NODE_ASFLOAT, -1, M32), (po.NODE_PHASOR_F, po.SRC_ZERO, M32), (po.NODE_SVF, 0, M32), (po.NODE_ENV, 2, M32),
            (po.NODE_ONEPOLE, 3, M32), (po.NODE_GAIN, 4, M32), (po.node_glide_f(2), 5, M32), (po.NODE_MUL, 5, M32, 6),
            (po.NODE_EDGE, -2, M32), (po.NODE_ACC, 8, M32), (po.NODE_ONEPOLE, 0, M32)]
    return rows, 2, [7, 1, 9, 10]


@pytest.mark.parametrize("seed", range(4))
def test_ext_oracle_vs_def_proc_bodies_at_edge_values(oracle, libref, seed):
    r = np.random.default_rng(300 + seed)
    N, F, n_in = 7, 150, 2
    rows = every_float_kind_graph()[0] if seed == 0 else edge_ext_graph(r, int(r.integers(2, 14)), n_in, masks=seed % 2 == 1)
    outs = every_float_kind_graph()[2] if seed == 0 else list(range(len(rows)))[-4:]
    st0, prm, inp, fmask = edge_ext_records(r, rows, N, n_in, F)
    chg = r.integers(0, 8, (N, F)).astype(np.uint32) if seed % 2 == 1 else None
    sa, sb = st0.copy(), st0.copy()
    a = oracle.graph_run_ext(rows, n_in, outs, sa, prm, N, F, inp, chg)
    b = libref.graph_run_ext(rows, n_in, outs, sb, prm, N, F, inp, chg)
    assert_ext_equal(a, b, sa, sb, rows, outs, fmask, "oracle vs DEF_PROC")


# ------------------------------------------------------------------------------------------------ CPU: no flush to zero
FLOAT_OP = re.compile(r"\b(FADD2|FMUL2|FFMA2|FADD|FMUL|FFMA|FMNMX|FSETP)((?:\.[A-Z0-9_]+)*)")


def ftz_in_sass(text):
    """(float instructions, those carrying .FTZ) of a cuobjdump -sass listing."""
    n, bad = 0, []
    for line in text.splitlines():
        for m in FLOAT_OP.finditer(line):
            n += 1
            if "FTZ" in m.group(2).split("."):
                bad.append(line.strip())
    return n, bad


def test_ftz_parser():
    n, bad = ftz_in_sass("/*0010*/ FFMA.FTZ R1, R2, R3, R4 ;\n/*0020*/ FADD R1, R2, R3 ;\n/*0030*/ @P0 FSETP.GT.FTZ.AND P0, PT, R1, R2, PT ;\n"
                         "/*0040*/ FMUL2 R2, R4.F32x2.HI_LO, R6.F32 ;\n/*0050*/ FMNMX.FTZ R1, R1, R2, !PT ;\n/*0060*/ IMAD R1, R2, R3, R4 ;")
    assert n == 5 and len(bad) == 3


def test_no_float_instruction_of_the_library_flushes_subnormals():
    """-ftz=true (or --use_fast_math) would make every float processor flush subnormal operands and results to zero,
    which the C definitions do not do."""
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    objs = sorted(glob.glob(os.path.join(OBJ, "*.o")))
    if not objs:
        pytest.skip("no objects under synth_tools_b200/build (python synth_tools_b200/build.py keeps them there)")
    counts, bad = {}, []
    for o in objs:
        out = subprocess.run(["cuobjdump", "-sass", o], capture_output=True, text=True, check=True).stdout
        n, b = ftz_in_sass(out)
        counts[os.path.basename(o)] = n
        bad += ["%s: %s" % (os.path.basename(o), x) for x in b[:5]]
    for o in ("k_grain.o", "k_xvoice.o", "k_graph.o", "bus.o"):                       # the float processors are there
        assert counts.get(o, 0) > 0, (o, counts)
    assert not bad, bad


def test_generated_graph_source_does_not_flush_subnormals():
    """The NVRTC source of a graph with every float kind, compiled with the options of graph_front.cu: no .ftz in its
    PTX, no .FTZ in its SASS."""
    from synth_tools_b200 import abi
    from tests.test_graph_front import _nvrtc
    nv = _nvrtc()
    if nv is None:
        pytest.skip("libnvrtc not present")
    rows, n_in, outs = every_float_kind_graph()
    src = abi.graph_jit_source(rows, n_in, outs, True)

    def compile_(arch, get_size, get):
        prog = C.c_void_p()
        assert nv.nvrtcCreateProgram(C.byref(prog), src.encode(), b"cproc_graph.cu", 0, None, None) == 0
        opts = (C.c_char_p * 4)(arch, b"-std=c++17", b"-lineinfo", b"-default-device")
        assert nv.nvrtcCompileProgram(prog, 4, opts) == 0
        sz = C.c_size_t()
        assert getattr(nv, get_size)(prog, C.byref(sz)) == 0
        buf = C.create_string_buffer(sz.value)
        assert getattr(nv, get)(prog, buf) == 0
        nv.nvrtcDestroyProgram(C.byref(prog))
        return buf.raw
    ptx = compile_(b"--gpu-architecture=compute_100a", "nvrtcGetPTXSize", "nvrtcGetPTX").decode(errors="replace")
    assert re.search(r"\b(add|sub|mul|fma)\.(rn\.)?f32\b", ptx), "no float arithmetic in the PTX"
    assert ".ftz" not in ptx
    if shutil.which("cuobjdump") is None:
        return
    cubin = compile_(b"--gpu-architecture=sm_100a", "nvrtcGetCUBINSize", "nvrtcGetCUBIN")
    with tempfile.TemporaryDirectory() as d:
        p = os.path.join(d, "graph.cubin")
        with open(p, "wb") as f:
            f.write(cubin)
        n, bad = ftz_in_sass(subprocess.run(["cuobjdump", "-sass", p], capture_output=True, text=True, check=True).stdout)
    assert n > 0 and not bad, bad[:5]


# ------------------------------------------------------------------------------------------------ GPU fixtures
@pytest.fixture(scope="module")
def st():
    import synth_tools_b200 as st_
    return st_


@pytest.fixture(scope="module")
def ctx(st):
    c = st.Context(0)
    yield c
    c.close()


def _n_sm():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ------------------------------------------------------------------------------------------------ GPU: square_grain raw
@pytest.mark.gpu
@pytest.mark.parametrize("inplace", [False, True], ids=["out-of-place", "in-place"])
@pytest.mark.parametrize("layout,N,F", [("PLANAR", 300, 256), ("PLANAR", 300, 203), ("INTERLEAVED", 256, 100), ("INTERLEAVED", 301, 77)])
@pytest.mark.parametrize("bulk", [0, 2])
def test_square_grain_edges(st, ctx, oracle, bulk, layout, N, F, inplace):
    """Raw square_grain on every stream path (planar_bulk 0 or 2; F and N multiples of 4 or not), two blocks.  The outputs
    are copies of the state, so the comparison is bitwise, NaN payloads included."""
    s0, th, _ = _grain_edge_inputs(N, F)
    il = layout == "INTERLEAVED"
    ctx.set_option("planar_bulk", bulk)
    b = ctx.batch(st.SQUARE_GRAIN, N, layout=st.INTERLEAVED if il else st.PLANAR)
    d_in = ctx.dev_alloc(4 * N * F)
    d_out = d_in if inplace else ctx.dev_alloc(4 * N * F)
    try:
        b.upload_state(s0.reshape(N, 1).copy())
        b.upload_param(th.reshape(N, 1).copy())
        sa = s0.copy()
        for blk in range(2):
            _, _, inp = _grain_edge_inputs(N, F)
            want = oracle.square_grain_run(sa, th, N, F, inp)
            ctx.h2d(d_in, np.ascontiguousarray(inp.T) if il else inp)
            b.run_dev(F, inp=d_in, out=d_out)
            ctx.sync()
            got = np.zeros((F, N) if il else (N, F), np.float32)
            ctx.d2h(got, d_out)
            same_float(got.T if il else got, want, "block %d out" % blk, strict=True)
            same_float(b.download_state().view(np.float32)[:, 0], sa, "block %d state" % blk, strict=True)
    finally:
        ctx.set_option("planar_bulk", 2)
        ctx.dev_free(d_in)
        if not inplace:
            ctx.dev_free(d_out)
        b.free()


# ------------------------------------------------------------------------------------------------ GPU: square_grain mix
TIE = 0x3F000001                         # 0.5 + 2^-24: (float)x rounds to it or away from it for x near 2^30 + 128
TH_NONNEG = [0.25, f32(0x30000000), f32(0x30C00000), f32(TIE), 0.0, -0.0, f32(0x00000001), f32(0x00800000), 1.0, 1.5,
             np.inf, np.nan, 0.5]
TH_SETS = {"nonneg": TH_NONNEG,
           "neg": TH_NONNEG + [-0.25, f32(0x80000001), -1.0],             # both flip conditions can hold: k_grain_mix2
           "unrep": TH_NONNEG + [-0.25, -1.5, -np.inf]}                   # no integer threshold exists: k_grain_mix
ST_REF = [0.0, -0.0, 0.5, -0.5]
ST_SETS = {"ref": ST_REF, "edge": ST_REF + [0.3, f32(0x00000001), np.inf, -np.inf, np.nan, f32(0xFFD00001)]}
# (phase, inc): phases that land exactly on +-th * 2^31 (0.25, 2^-31, 3 * 2^-31), walk through the rounding ties of
# (float)x around +-(2^30 + 128), cross the wrap at 2^31, or are arbitrary
PHASE_INC = [(0, 1 << 24), ((-3) & M32, 1), ((-(1 << 29) - (8 << 24)) & M32, 1 << 24), ((1 << 30) + 60, 1),
             ((-(1 << 30) - 200) & M32, 1), (0x7FFFFFF0, 1), (0x12345678, 39370533)]
GAINS = [(0, 64), (64, 0), (64, 64), (0, 0), (17, 47)]


def grain_mix_grains(th_set, st_set):
    combos = list(itertools.product(TH_SETS[th_set], ST_SETS[st_set], PHASE_INC))
    N = len(combos)
    th = np.array([c[0] for c in combos], np.float32)
    state = np.array([c[1] for c in combos], np.float32)
    phase = np.array([c[2][0] for c in combos], np.uint32)
    inc = np.array([c[2][1] for c in combos], np.uint32)
    g = np.array([GAINS[i % len(GAINS)] for i in range(N)], np.uint8)
    return [state, th, phase, inc, g[:, 0].copy(), g[:, 1].copy()]


def grain_mix_batch(st, ctx, g):
    state, th, phase, inc, gl, gr = g
    N = state.size
    b = ctx.batch(st.SQUARE_GRAIN_MIX, N)
    s_rec = np.zeros((N, 2), np.uint32); s_rec[:, 0] = state.view(np.uint32); s_rec[:, 1] = phase
    p_rec = np.zeros((N, 4), np.uint32)
    p_rec[:, 0] = th.view(np.uint32); p_rec[:, 1] = inc; p_rec[:, 2] = gl; p_rec[:, 3] = gr
    b.upload_state(s_rec)
    b.upload_param(p_rec)
    return b


@pytest.mark.gpu
@pytest.mark.parametrize("F", [256, 131])
@pytest.mark.parametrize("st_set", ["ref", "edge"])
@pytest.mark.parametrize("th_set", ["nonneg", "neg", "unrep"])
@pytest.mark.parametrize("bus_mode", [0, 1, 2], ids=["no-bus", "bus1", "bus2"])
@pytest.mark.parametrize("gen", [0, 1, 2])
def test_square_grain_mix_edges(st, ctx, oracle, gen, bus_mode, th_set, st_set, F):
    """Every generation (grain_mix2 0..2), without a bus and with a fused world-1 bus, two consecutive blocks: the int32
    mix, the float out and the final state (value and phase) equal the oracle at exact threshold ties, signed zero,
    subnormal, infinite and NaN thresholds, and states other than {+-0, +-0.5}."""
    g = grain_mix_grains(th_set, st_set)
    ctx.set_option("grain_mix2", gen)
    b = grain_mix_batch(st, ctx, g)
    bus = None
    d = [ctx.dev_alloc(8 * F) for _ in range(4)]
    try:
        wants = []
        if bus_mode:
            bus = st.Bus(ctx, 2 * F, 1, 0)
            bus.attach(b, bus_mode)
        for blk in range(2):
            wants.append(oracle.square_grain_mix_run(g[0], g[1], g[2], g[3], g[4], g[5], g[0].size, F))
            if bus_mode:
                b.run_dev(F, mix=d[2 * blk], out=d[2 * blk + 1])
            else:
                mix, out = np.zeros((2, F), np.int32), np.zeros((2, F), np.float32)
                b.run(F, mix=mix, out=out)
                ctx.h2d(d[2 * blk], mix); ctx.h2d(d[2 * blk + 1], out)
        if bus:
            bus.flush()
        ctx.sync()
        if bus:
            assert bus.status() == 0
        for blk, (w_i, w_f) in enumerate(wants):
            mix, out = np.zeros((2, F), np.int32), np.zeros((2, F), np.float32)
            ctx.d2h(mix, d[2 * blk]); ctx.d2h(out, d[2 * blk + 1])
            bad = np.argwhere(mix != w_i)
            assert bad.size == 0, ("block %d mix" % blk, len(bad), [(int(c), int(t), int(mix[c, t]), int(w_i[c, t])) for c, t in bad[:4]])
            same_float(out, w_f, "block %d out" % blk)
        s = b.download_state()
        same_float(s[:, 0].view(np.float32), g[0], "final state")
        assert np.array_equal(s[:, 1], g[2]), "final phase"
    finally:
        if bus:
            bus.detach(b); bus.destroy()
        for p in d:
            ctx.dev_free(p)
        b.free()
        ctx.set_option("grain_mix2", 2)


@pytest.mark.gpu
@pytest.mark.parametrize("gen", [1, 2])
@pytest.mark.parametrize("state,gains", [(0.5, (64, 64)), (-0.5, (64, 0))])
def test_square_grain_mix_packing_bound(st, ctx, gen, state, gains):
    """The 16-bit halves of the packed per-thread accumulators at their bound: one block per SM and 500 grains per
    thread, every grain at full gain 64 and never flipping (threshold +inf), so every mix word is exactly +-64 N."""
    n_sm = _n_sm()
    N, F = n_sm * 128 * 500, 64
    ctx.set_option("grain_mix2", gen)
    ctx.set_option("grain_blocks_per_sm", 1)
    b = ctx.batch(st.SQUARE_GRAIN_MIX, N)
    try:
        s_rec = np.zeros((N, 2), np.uint32); s_rec[:, 0] = np.float32(state).view(np.uint32)
        s_rec[:, 1] = rng.integers(0, 2**32, N, dtype=np.uint32)
        p_rec = np.zeros((N, 4), np.uint32)
        p_rec[:, 0] = np.float32(np.inf).view(np.uint32); p_rec[:, 1] = rng.integers(0, 2**32, N, dtype=np.uint32)
        p_rec[:, 2], p_rec[:, 3] = gains
        b.upload_state(s_rec); b.upload_param(p_rec)
        mix, out = np.zeros((2, F), np.int32), np.zeros((2, F), np.float32)
        b.run(F, mix=mix, out=out)
        sign = 1 if state > 0 else -1
        want = np.array([[sign * gains[0] * N] * F, [sign * gains[1] * N] * F], np.int64)
        assert np.array_equal(mix.astype(np.int64), want), (mix[:, :3], want[:, :3])
        same_float(out, (want.astype(np.float32) * np.float32(2.0 ** -7)).astype(np.float32), "out")
        s = b.download_state()
        assert np.all(s[:, 0] == s_rec[:, 0])
        assert np.array_equal(s[:, 1], s_rec[:, 1] + np.uint32(F) * p_rec[:, 1])
    finally:
        b.free()
        ctx.set_option("grain_blocks_per_sm", 2)
        ctx.set_option("grain_mix2", 2)


@pytest.mark.gpu
def test_square_grain_mix_gain_range(st, ctx):
    """Pan gains are k/64, k <= 64: a larger gain would overflow the packed accumulators silently, so it is refused."""
    N = 10
    b = ctx.batch(st.SQUARE_GRAIN_MIX, N)
    try:
        for gl, gr in [(65, 0), (0, 65), (1 << 15, 1), (0, 0xFFFFFFFF)]:
            p = np.zeros((N, 4), np.uint32)
            p[:, 2] = 64; p[:, 3] = 64
            p[N - 1, 2], p[N - 1, 3] = gl, gr
            with pytest.raises(st.CprocCudaError) as e:
                b.upload_param(p)
            assert e.value.code == st.abi.EINVAL
        p = np.zeros((N, 5), np.uint32)                                              # stride: the fifth word is not a gain
        p[:, 2] = 64; p[:, 3] = 64; p[:, 4] = 1000
        b.upload_param(p, stride=20)
    finally:
        b.free()


# ------------------------------------------------------------------------------------------------ GPU: one-pole
OP_COEFS = [0.0, -0.0, f32(0x00000001), 2.0 ** -24, 0.5, 1.0, 2.0, 3.0, np.inf, np.nan]
OP_KINDS = ["pool", "overflow", "uniform", "subnormal", "decay tail"]


def onepole_edge_inputs(N, F):
    a = np.zeros(N, np.float32); y0 = pool_draw(N); x = np.zeros((N, F), np.float32)
    kinds = []
    for i in range(N):
        a[i] = OP_COEFS[i % len(OP_COEFS)]
        kind = OP_KINDS[(i // len(OP_COEFS)) % len(OP_KINDS)]
        kinds.append(kind)
        if kind == "pool":
            x[i] = pool_draw(F)
        elif kind == "overflow":
            x[i] = np.where(np.arange(F) % 2 == 0, f32(0x7F7FFFFF), f32(0xFF7FFFFF))
            y0[i] = f32(0xFF7FFFFF)
        elif kind == "uniform":
            x[i] = rng.uniform(-1, 1, F)
        elif kind == "subnormal":
            x[i] = rng.choice(SUBNORMALS, F)
        else:                                                   # 1e-37 halves through the subnormals to exactly 0
            a[i], y0[i] = 0.5, 1e-37
    return a, y0, x, kinds


@pytest.mark.gpu
@pytest.mark.parametrize("layout,N,F", [("PLANAR", 52, 256), ("PLANAR", 53, 203), ("INTERLEAVED", 52, 160), ("INTERLEAVED", 53, 77)])
@pytest.mark.parametrize("bulk", [0, 2])
def test_onepole_edges(st, ctx, oracle, bulk, layout, N, F):
    """Sequential one-pole on every stream path: coefficients 0, -0, subnormal, 2^-24, 0.5, 1, 2, 3 (unstable: to inf,
    then NaN), inf, NaN; pool inputs, overflowing inputs, subnormal inputs and a decay through the subnormal range to
    exactly 0 (a render that flushed subnormals would reach 0 some 23 frames early)."""
    a, y0, x, kinds = onepole_edge_inputs(N, F)
    il = layout == "INTERLEAVED"
    ctx.set_option("planar_bulk", bulk)
    b = ctx.batch(st.ONEPOLE, N, layout=st.INTERLEAVED if il else st.PLANAR)
    try:
        b.upload_state(y0.reshape(N, 1).copy()); b.upload_param(a.reshape(N, 1).copy())
        ya = y0.copy()
        for blk in range(2):
            want = oracle.onepole_run(ya, a.copy(), N, F, x)
            got = np.zeros((F, N) if il else (N, F), np.float32)
            b.run(F, inp=np.ascontiguousarray(x.T) if il else x, out=got)
            same_float(got.T if il else got, want, "block %d out" % blk)
            same_float(b.download_state().view(np.float32)[:, 0], ya, "block %d state" % blk)
            if blk == 0:
                tail = want[kinds.index("decay tail")]
                assert np.any((tail != 0) & (np.abs(tail) < np.finfo(np.float32).tiny)) and tail[-1] == 0
            x = x[:, ::-1].copy()
    finally:
        ctx.set_option("planar_bulk", 2)
        b.free()


# ------------------------------------------------------------------------------------------------ GPU: extension voice
def _choice(vals, N):
    return np.array(vals, np.float64)[rng.integers(0, len(vals), N)]


def xvoice_edge_voices(N, F):
    sub, msub = float(f32(0x00000001)), float(f32(0x807FFFFF))
    prm = np.zeros(N, po.xvoice_param_dtype)
    prm["inc"] = rng.integers(0, 2**32, N, dtype=np.uint32)
    prm["f"] = _choice([0.0, 0.1, sub, 0.5, 1.0], N)
    prm["q"] = _choice([0.0, 0.7, 2.0, -0.0], N)
    prm["env_attack"] = _choice([0.0, -0.0, np.inf, -0.1, 0.25, sub, 2.0 ** -24], N)
    prm["env_release"] = _choice([0.0, -0.0, np.inf, -0.1, 0.25, sub, 2.0 ** -24], N)
    prm["gate_frames"] = rng.choice(np.array([0, 10, M32 - 20, 0xFFFFFFF0, M32], np.uint32), N)
    prm["gl"] = _choice([0.0, -0.0, -1.0, sub, 1.0, 0.5], N)
    prm["gr"] = _choice([0.0, -0.0, -1.0, sub, 1.0, 0.5], N)
    s0 = np.zeros(N, po.xvoice_state_dtype)
    s0["phase"] = rng.integers(0, 2**32, N, dtype=np.uint32)
    s0["lp"] = _choice([0.0, -0.0, sub, msub, 0.5, -1.0, 3e38], N)
    s0["bp"] = _choice([0.0, -0.0, sub, msub, 0.25, -0.5], N)
    s0["env"] = _choice([0.0, -0.0, 1.0, sub, float(f32(0x007FFFFF)), 0.5, float(f32(0x3F7FFFFF))], N)
    s0["t"] = rng.choice(np.array([0, 7, M32 - F // 2, M32 - 40, M32 - 1, M32], np.uint32), N)
    return s0, prm


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["PLANAR", "TILED"])
@pytest.mark.parametrize("N,F", [(300, 130), (1000, 64)])
def test_xvoice_raw_edges(st, ctx, oracle, layout, N, F):
    """Raw sequential XVOICE: subnormal lp / bp / env, env exactly 1 and -0, rates of +-0, inf and negative values,
    f = 0 and q = 0, gains of +-0, -1 and a subnormal, and frame counters that wrap inside a chunk."""
    s0, prm = xvoice_edge_voices(N, F)
    b = ctx.batch(st.XVOICE, N, layout=getattr(st, layout))
    try:
        b.upload_state(s0.view(np.uint32).reshape(N, 5)); b.upload_param(prm.view(np.uint32).reshape(N, 8))
        sa = s0.copy()
        for blk in range(2):
            want, _ = oracle.xvoice_run(sa, prm.copy(), N, F, want_mix=False)
            raw = np.zeros(N * F * 2, np.float32)
            b.run(F, out=raw)
            got = raw.reshape(F // 2, N, 2, 2).transpose(1, 0, 2, 3).reshape(N, F, 2) if layout == "TILED" else raw.reshape(N, F, 2)
            same_float(got, want, "block %d raw" % blk)
            s = b.download_state().view(po.xvoice_state_dtype).reshape(N)
            assert np.array_equal(s["phase"], sa["phase"]) and np.array_equal(s["t"], sa["t"])
            for k in ("lp", "bp", "env"):
                same_float(s[k].copy(), sa[k].copy(), "block %d state %s" % (blk, k))
    finally:
        b.free()


XV_MIX_N = 148 * 4 * 128 + 333
XV_SOUNDING = {
    "subnormal": dict(lp=float(f32(0x00000005)), env=1.0, gl=1.0, gr=-0.5),      # gr * y rounds a subnormal
    "overflow": dict(lp=3e38, env=1.0, gl=2.0, gr=-2.0),                          # +-inf
    "nan": dict(lp=np.inf, env=0.0, gl=1.0, gr=1.0),                              # inf * 0
    "normal": dict(lp=0.375, env=0.5, gl=0.75, gr=f32(0x00000001)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("pos", [0, 1, 255, 256, 40001, XV_MIX_N - 1])
@pytest.mark.parametrize("kind", list(XV_SOUNDING))
@pytest.mark.parametrize("bus_mode", [0, 1, 2], ids=["no-bus", "bus1", "bus2"])
@pytest.mark.parametrize("gen", [1, 0], ids=["mix2", "mix1"])
def test_xvoice_mix_one_sounding_voice(st, ctx, oracle, gen, bus_mode, kind, pos):
    """Every voice but one is silent (env 0, rates 0, f = 0, finite lp / bp, nonzero gains): adding their exact zeros
    does not round, so the mix is the sounding voice's gl * y and gr * y bit for bit -- at pair lanes A and B, in other
    tiles and blocks, through the packed FFMA2 / FMUL2 path, with subnormal, infinite and NaN products.  Zeros in the
    mix are compared without their sign."""
    N, F = XV_MIX_N, 64
    prm = np.zeros(N, po.xvoice_param_dtype)
    prm["inc"] = rng.integers(0, 2**32, N, dtype=np.uint32)
    prm["q"] = rng.uniform(0, 2, N)
    prm["gate_frames"] = rng.integers(0, 2 * F, N)
    prm["gl"] = rng.uniform(-1, 1, N); prm["gr"] = rng.uniform(-1, 1, N)
    s0 = np.zeros(N, po.xvoice_state_dtype)
    s0["phase"] = rng.integers(0, 2**32, N, dtype=np.uint32)
    s0["lp"] = rng.choice(np.array([0.0, -0.0, 0.5, -0.25, float(f32(0x80000001))], np.float32), N)
    s0["bp"] = rng.uniform(-1, 1, N)
    s0["t"] = rng.integers(0, 2**32, N, dtype=np.uint32)
    v = XV_SOUNDING[kind]
    prm["gate_frames"][pos] = M32; s0["t"][pos] = 0
    s0["lp"][pos] = v["lp"]; s0["env"][pos] = v["env"]; prm["gl"][pos] = v["gl"]; prm["gr"][pos] = v["gr"]
    sa = s0.copy()
    wants = []
    for _ in range(2):
        one = sa[pos:pos + 1].copy()
        raw, _ = oracle.xvoice_run(one, prm[pos:pos + 1].copy(), 1, F, want_mix=False)
        oracle.xvoice_run(sa, prm.copy(), N, F, want_raw=False, want_mix=False)
        wants.append(np.ascontiguousarray(raw[0].T))
    ctx.set_option("xvoice_mix2", gen)
    b = ctx.batch(st.XVOICE, N)
    bus = None
    d_mix = [ctx.dev_alloc(8 * F) for _ in range(2)]
    try:
        b.upload_state(s0.view(np.uint32).reshape(N, 5)); b.upload_param(prm.view(np.uint32).reshape(N, 8))
        if bus_mode:
            bus = st.Bus(ctx, 2 * F, 1, 0)
            bus.attach(b, bus_mode)
        for k in range(2):
            b.run_dev(F, mix=d_mix[k])
        if bus:
            bus.flush()
        ctx.sync()
        if bus:
            assert bus.status() == 0
        for k in range(2):
            mix = np.zeros((2, F), np.float32)
            ctx.d2h(mix, d_mix[k])
            same_float(mix, wants[k], "block %d mix" % k, zero_sign=False)
        s = b.download_state().view(po.xvoice_state_dtype).reshape(N)
        assert np.array_equal(s["phase"], sa["phase"]) and np.array_equal(s["t"], sa["t"])
        for k in ("lp", "bp", "env"):
            # (k_xvoice_mix2: the sign of a zero lp, test_xvoice_mix2_lp_zero_sign)
            same_float(s[k].copy(), sa[k].copy(), "state " + k, zero_sign=not (gen == 1 and k == "lp"))
    finally:
        if bus:
            bus.detach(b); bus.destroy()
        for p in d_mix:
            ctx.dev_free(p)
        b.free()
        ctx.set_option("xvoice_mix2", 1)


@pytest.mark.gpu
@pytest.mark.xfail(strict=True, reason="k_xvoice_mix2 runs the filter on -lp; round-to-nearest makes an exact cancellation +0 "
                                       "whatever the operands' signs, so where lp + f bp cancels it stores -0 for the definition's +0")
def test_xvoice_mix2_lp_zero_sign(st, ctx, oracle):
    """lp = +0, f = 0, bp = -0.5: lp' = fmaf(0, -0.5, +0) = -0 + +0 = +0 every tick.  The packed kernel computes
    -lp' = fma(-0, -0.5, -0) = +0 + -0 = +0 and stores lp' = -0.  Only the sign of a zero differs: every later tick
    and every nonzero output agree (test_xvoice_mix_one_sounding_voice)."""
    N, F = 256, 64
    prm = np.zeros(N, po.xvoice_param_dtype)
    prm["inc"] = rng.integers(0, 2**32, N, dtype=np.uint32); prm["q"] = 0.5; prm["gl"] = 1.0; prm["gr"] = 1.0
    s0 = np.zeros(N, po.xvoice_state_dtype)
    s0["bp"] = -0.5
    sa = s0.copy()
    oracle.xvoice_run(sa, prm.copy(), N, F, want_raw=False, want_mix=False)
    assert np.all(sa["lp"].view(np.uint32) == 0)
    ctx.set_option("xvoice_mix2", 1)
    b = ctx.batch(st.XVOICE, N)
    try:
        b.upload_state(s0.view(np.uint32).reshape(N, 5)); b.upload_param(prm.view(np.uint32).reshape(N, 8))
        b.run(F, mix=np.zeros((2, F), np.float32))
        s = b.download_state().view(po.xvoice_state_dtype).reshape(N)
        same_float(s["lp"].copy(), sa["lp"].copy(), "state lp")
    finally:
        b.free()


# ------------------------------------------------------------------------------------------------ GPU: extension graphs
# kernel -> (layout, N, F, planar_bulk, graph_jit): how the front end is steered to it (k_graph.cu launch_graph)
GRAPH_KERNELS = {"graph_planar_tma": (0, 300, 256, 2, 1),
                 "graph_planar_simple": (0, 131, 203, 2, 1), "graph_interleaved4": (1, 256, 100, 2, 1),
                 "graph_interleaved": (1, 301, 77, 2, 1), "table": (0, 131, 96, 2, 0)}


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(4))
@pytest.mark.parametrize("kernel", list(GRAPH_KERNELS))
def test_ext_graph_edges(ctx, oracle, kernel, seed):
    """Random tables over all eight float kinds plus acc and edge (seed 0: a chain through every float kind) with
    pool-drawn states, params and inputs, env gates at 0xFFFFFFFF with t near the wrap, glide_f steps of +-inf; every
    kernel the front end can pick."""
    from tests.test_graph_ext import run_cuda_graph
    layout, N, F, bulk, jit = GRAPH_KERNELS[kernel]
    r = np.random.default_rng(400 + seed)
    n_in = 2
    if seed == 0:
        rows, n_in, outs = every_float_kind_graph()
    else:
        rows = edge_ext_graph(r, int(r.integers(2, 14 if jit == 0 else 20)), n_in, masks=seed % 2 == 1)
        outs = list(range(len(rows)))[-3:]
    st0, prm, inp, fmask = edge_ext_records(r, rows, N, n_in, F)
    chg = r.integers(0, 8, (N, F)).astype(np.uint32) if seed % 2 == 1 else None
    sa = st0.copy()
    want = oracle.graph_run_ext(rows, n_in, outs, sa, prm, N, F, inp, chg)
    ctx.set_option("graph_jit", jit); ctx.set_option("planar_bulk", bulk)
    try:
        got, st1, log = run_cuda_graph(ctx, rows, n_in, outs, st0, prm, N, F, inp, chg, layout)
    finally:
        ctx.set_option("graph_jit", 1); ctx.set_option("planar_bulk", 2)
    if jit:
        assert "not found" not in log and "failed" not in log and "error" not in log, log
    assert_ext_equal(got, want, st1, sa, rows, outs, fmask, kernel)
