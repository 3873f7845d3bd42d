"""Extension processors as cproc processors (SURVEY 8 a-X): phasor_f, svf, env, onepole, gain, asfloat are DEF_PROC
definitions (include/cproc_ext.h) against the reference's generic/cproc.h:89-103, graph node kinds of the front end,
the JIT, the table kernel and the patcher.

CPU: the header compiles against the real cproc.h (oracle/_ref), the oracle's restatement equals the DEF_PROC bodies
bit for bit, the graph TEXT compiled as C equals the parsed node table run by the oracle, the voice graph equals the
fused extension voice (orc_xvoice_tick).  GPU: the CUDA graph path equals the oracle bit for bit in every layout and
kernel variant, and the voice graph equals k_xvoice's raw output."""
import os

import numpy as np
import pytest

from oracle import pyoracle as po
from synth_tools_b200 import abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VOICE_TEXT = open(os.path.join(ROOT, "tests", "golden", "ext_voice.cproc")).read()
CHAIN_TEXT = open(os.path.join(ROOT, "tests", "golden", "ext_chain.cproc")).read()
GAIN_TEXT = open(os.path.join(ROOT, "tests", "golden", "ext_gain.cproc")).read()
EXT_KINDS = [po.NODE_PHASOR_F, po.NODE_SVF, po.NODE_ENV, po.NODE_ONEPOLE, po.NODE_GAIN, po.NODE_ASFLOAT, po.NODE_GLIDE_F, po.NODE_MUL]
IN_FLOAT = {po.NODE_SVF, po.NODE_ENV, po.NODE_ONEPOLE, po.NODE_GAIN, po.NODE_GLIDE_F, po.NODE_MUL}
F32 = lambda x: np.float32(x).view(np.uint32)


def random_ext_graph(rng, n_nodes, n_inputs, with_int_nodes=True, masks=False):
    """A random valid ANF table over acc / edge and the extension kinds, with a param record per instance drawn by
    `random_params`."""
    rows = []
    for k in range(n_nodes):
        kind = int(rng.choice([po.NODE_ACC, po.NODE_EDGE] + EXT_KINDS * 2)) if with_int_nodes else int(rng.choice(EXT_KINDS))
        want_f = kind in IN_FLOAT
        cands = [-(j + 1) for j in range(n_inputs)]
        for j, r in enumerate(rows):
            src_f = (r[0] & 0xFF) >= po.NODE_PHASOR_F
            if want_f or not src_f:                              # a float .out never feeds a w input
                cands.append(j)
        if kind == po.NODE_ASFLOAT:
            cands = [-2]                                         # input[1] carries float bits; arbitrary words would decode to NaNs, whose
                                                                 # payloads x86 propagates and the GPU canonicalises (cproc_cuda.h)
        if kind >= po.NODE_PHASOR_F and rng.random() < 0.15:
            cands = [po.SRC_ZERO]
        if not cands:
            kind, cands = po.NODE_PHASOR_F, [po.SRC_ZERO]
        mask = int(rng.choice([1, 2, 3, 6, 0xFFFFFFFF])) if masks else 0xFFFFFFFF
        if kind == po.NODE_GLIDE_F:
            rows.append((po.node_glide_f(int(rng.integers(1, 7))), int(rng.choice(cands)), mask))
        elif kind == po.NODE_MUL:                                # two float inputs
            rows.append((kind, int(rng.choice(cands)), mask, int(rng.choice(cands))))
        else:
            rows.append((kind, int(rng.choice(cands)), mask))
    return rows


def random_params(rng, rows, N):
    cols = []
    for r in rows:
        kind = r[0] & 0xFF
        if kind == po.NODE_PHASOR_F:
            cols.append(rng.integers(0, 2**28, N, dtype=np.uint32))
        elif kind == po.NODE_SVF:
            cols += [rng.uniform(0.01, 0.3, N).astype(np.float32).view(np.uint32), rng.uniform(0.5, 2.0, N).astype(np.float32).view(np.uint32)]
        elif kind == po.NODE_ENV:
            cols += [rng.uniform(1e-3, 1e-1, N).astype(np.float32).view(np.uint32), rng.uniform(1e-3, 1e-2, N).astype(np.float32).view(np.uint32),
                     rng.integers(0, 60, N, dtype=np.uint32)]
        elif kind == po.NODE_ONEPOLE:
            cols.append(rng.uniform(0.001, 0.9, N).astype(np.float32).view(np.uint32))
        elif kind == po.NODE_GAIN:
            cols.append(rng.uniform(-1.5, 1.5, N).astype(np.float32).view(np.uint32))
    if not cols:
        return None
    return np.ascontiguousarray(np.stack(cols, axis=1))


def state_words(rows):
    return sum(po.node_words(r[0]) for r in rows)


# ---- CPU --------------------------------------------------------------------------------------------------------

def test_ext_structs_compile_against_the_reference_cproc_h(ref):
    """DEF_PROC_STRUCTS (cproc.h:99-103) of include/cproc_ext.h: struct sizes = the word counts every layer uses
    (GNU C: an empty field list gives size 0, like acc_config)."""
    want = {po.NODE_PHASOR_F: (8, 4, 4), po.NODE_SVF: (8, 8, 4), po.NODE_ENV: (12, 12, 4), po.NODE_ONEPOLE: (4, 4, 4),
            po.NODE_GAIN: (4, 4, 4), po.NODE_ASFLOAT: (4, 0, 4), po.NODE_GLIDE_F: (12, 0, 4), po.NODE_MUL: (4, 0, 8)}
    assert ref.ext_sizeof(24) == 4                               # glide_f_config {w div_log}
    for kind, (s, p, i) in want.items():
        k = kind - po.NODE_PHASOR_F
        assert (ref.ext_sizeof(3 * k), ref.ext_sizeof(3 * k + 1), ref.ext_sizeof(3 * k + 2)) == (s, p, i), kind
        assert po.node_words(kind) * 4 == s and po.node_param_words(kind) * 4 == p
    classes = {c["name"]: c for c in abi.patch_classes()}
    assert classes["svf"]["param"] == ["f", "q"] and classes["svf"]["state"] == ["out", "bp"] and classes["svf"]["input"] == ["in"]
    assert classes["env"]["param"] == ["attack", "release", "gate_frames"] and classes["env"]["state"] == ["out", "env", "t"]
    assert classes["phasor_f"]["param"] == ["inc"] and classes["phasor_f"]["input"] == ["mod"] and classes["phasor_f"]["state"] == ["out", "phase"]
    assert classes["onepole"]["param"] == ["a"] and classes["gain"]["param"] == ["g"] and classes["asfloat"]["param"] == []
    assert [c["name"] for c in abi.patch_classes()][:5] == ["acc", "edge", "glide", "input", "pdm"]      # ABI 2 class numbers kept


@pytest.mark.parametrize("seed", range(6))
def test_ext_oracle_restatement_equals_the_def_proc_bodies(ref, oracle, seed):
    rng = np.random.default_rng(100 + seed)
    N, F, n_in = 5, 200, 2
    rows = random_ext_graph(rng, int(rng.integers(1, 12)), n_in, masks=seed % 2 == 1)
    prm = random_params(rng, rows, N)
    inp = rng.integers(0, 2**32, (N, n_in, F), dtype=np.uint32)
    inp[:, 1] = rng.uniform(-1, 1, (N, F)).astype(np.float32).view(np.uint32)       # float bits for asfloat
    chg = rng.integers(0, 8, (N, F)).astype(np.uint32) if seed % 2 == 1 else None
    outs = list(range(len(rows)))[-4:]
    sa = np.zeros((N, state_words(rows)), np.uint32); sb = sa.copy()
    a = oracle.graph_run_ext(rows, n_in, outs, sa, prm, N, F, inp, chg)
    b = ref.graph_run_ext(rows, n_in, outs, sb, prm, N, F, inp, chg)
    assert np.array_equal(a, b) and np.array_equal(sa, sb), rows


def test_graph_text_compiled_as_c_equals_the_parsed_table(ref, oracle):
    """tests/golden/ext_voice.cproc and ext_chain.cproc: the SAME text compiled with the reference's PROC / PROC_COND
    macros (oracle/ref/ref_ext_voice.c) and parsed by cproc_cuda_graph_parse + run by the oracle."""
    rng = np.random.default_rng(5)
    F = 700
    r = ref.private_copy()                                       # node state is function-static: one instance per loaded copy
    # voice: input[0] = pitch modulation
    g = abi.graph_parse_ex(VOICE_TEXT)
    assert g["out_is_float"] == [True, True] and g["out_indices"] == [0, 1] and g["n_inputs"] == 1
    assert [x[0] for x in g["rows"]] == [po.NODE_PHASOR_F, po.NODE_SVF, po.NODE_ENV, po.NODE_GAIN, po.NODE_GAIN]
    assert g["param_init"].tolist() == [39370533, F32(0.1), F32(0.7), F32(0.01), F32(0.002), 300, F32(0.75), F32(0.25)]
    mod = rng.integers(0, 1 << 22, (1, 1, F)).astype(np.uint32)
    want = r.ext_text_run(0, np.ascontiguousarray(mod[0]), None, F, 2)
    st = np.zeros((1, state_words(g["rows"])), np.uint32)
    got = oracle.graph_run_ext(g["rows"], 1, g["out_nodes"], st, g["param_init"].reshape(1, -1).copy(), 1, F, mod)
    assert np.array_equal(got[0], want)
    assert np.abs(want.view(np.float32)).max() > 0.05
    # chain: masked subgraphs, w -> float conversion by value (gain of the edge counter), three outputs of mixed type
    g = abi.graph_parse_ex(CHAIN_TEXT)
    assert g["out_is_float"] == [False, True, True] and g["out_indices"] == [2, 3, 4] and g["n_inputs"] == 2
    assert g["rows"][4] == (po.NODE_GAIN, 1, 2) and g["rows"][2] == (po.NODE_PHASOR_F, -2, 2)
    inp = np.zeros((1, 2, F), np.uint32)
    inp[0, 0] = rng.integers(0, 2, F); inp[0, 1] = rng.integers(0, 1 << 20, F)
    chg = rng.integers(0, 4, (1, F)).astype(np.uint32)
    want = r.ext_text_run(1, np.ascontiguousarray(inp[0]), np.ascontiguousarray(chg[0]), F, 3)
    st = np.zeros((1, state_words(g["rows"])), np.uint32)
    got = oracle.graph_run_ext(g["rows"], 2, g["out_nodes"], st, g["param_init"].reshape(1, -1).copy(), 1, F, inp, chg)
    assert np.array_equal(got[0], want)
    assert want[0].max() > 10 and np.array_equal(want[2].view(np.float32)[-1], np.float32(0.5) * np.float32(want[0][-1]))
    # gain: a control-rate gain amount through glide_f, applied by mul (doc/combinators.org:28-34)
    g = abi.graph_parse_ex(GAIN_TEXT)
    assert g["rows"] == [(po.NODE_PHASOR_F, po.SRC_ZERO, 0xFFFFFFFF), (po.NODE_ASFLOAT, -1, 0xFFFFFFFF), (po.node_glide_f(6), 1, 0xFFFFFFFF),
                         (po.NODE_MUL, 0, 0xFFFFFFFF, 2)] and g["n_inputs"] == 1 and g["out_is_float"] == [True]
    amt = np.repeat(rng.uniform(0, 1, F // 64 + 1).astype(np.float32), 64)[:F].view(np.uint32).reshape(1, 1, F).copy()
    want = r.ext_text_run(2, np.ascontiguousarray(amt[0]), None, F, 1)
    st = np.zeros((1, state_words(g["rows"])), np.uint32)
    got = oracle.graph_run_ext(g["rows"], 1, g["out_nodes"], st, g["param_init"].reshape(1, -1).copy(), 1, F, amt)
    assert np.array_equal(got[0], want)
    a = amt.view(np.float32)[0, 0]                               # ramp.out after 700 ticks: 60 of the 64 steps from the target of tick 576 to that of tick 640
    assert abs(float(st[0, 3:4].view(np.float32)[0]) - (float(a[576]) + (float(a[640]) - float(a[576])) * 60 / 64)) < 1e-3


def voice_graph_and_records(rng, N):
    """phasor_f -> svf -> env -> gain x 2 with no external input, and the same voices as XVOICE records."""
    rows = [(po.NODE_PHASOR_F, po.SRC_ZERO, 0xFFFFFFFF), (po.NODE_SVF, 0, 0xFFFFFFFF), (po.NODE_ENV, 1, 0xFFFFFFFF),
            (po.NODE_GAIN, 2, 0xFFFFFFFF), (po.NODE_GAIN, 2, 0xFFFFFFFF)]
    xp = np.zeros(N, po.xvoice_param_dtype)
    xp["inc"] = rng.integers(1 << 20, 1 << 28, N); xp["f"] = rng.uniform(0.01, 0.3, N); xp["q"] = rng.uniform(0.5, 2.0, N)
    xp["env_attack"] = rng.uniform(1e-3, 1e-1, N); xp["env_release"] = rng.uniform(1e-3, 1e-2, N); xp["gate_frames"] = rng.integers(0, 400, N)
    xp["gl"] = rng.uniform(0, 1, N); xp["gr"] = np.float32(1) - xp["gl"]
    xs = np.zeros(N, po.xvoice_state_dtype)
    xs["phase"] = rng.integers(0, 2**32, N, dtype=np.uint32)
    prm = np.ascontiguousarray(xp.view(np.uint32).reshape(N, 8))           # inc | f q | attack release gate | gl | gr: the same order
    gst = np.zeros((N, 9), np.uint32)
    gst[:, 1] = xs["phase"]                                                # {osc.out, osc.phase, flt.out, flt.bp, amp.out, amp.env, amp.t, l.out, r.out}
    return rows, prm, gst, xs, xp


def test_voice_graph_equals_the_fused_extension_voice(oracle):
    """The graph phasor_f -> svf -> env -> gain x 2 IS the extension voice of CPROC_CUDA_XVOICE (orc_xvoice_tick):
    same raw stereo output and same final state, bit for bit."""
    rng = np.random.default_rng(8)
    N, F = 37, 512
    rows, prm, gst, xs, xp = voice_graph_and_records(rng, N)
    got = oracle.graph_run_ext(rows, 0, [3, 4], gst, prm, N, F)
    raw, _ = oracle.xvoice_run(xs, xp, N, F, want_raw=True, want_mix=False)
    assert np.array_equal(got.view(np.float32).transpose(0, 2, 1), raw.reshape(N, F, 2))
    assert np.array_equal(gst[:, 1], xs["phase"]) and np.array_equal(gst[:, 2].view(np.float32), xs["lp"])
    assert np.array_equal(gst[:, 3].view(np.float32), xs["bp"]) and np.array_equal(gst[:, 5].view(np.float32), xs["env"]) and np.array_equal(gst[:, 6], xs["t"])


@pytest.mark.parametrize("text,what", [
    ("PROC(a, svf, NULL, NULL, .in = input[0]); cproc_output_f(0, a.out);", "needs a param record"),
    ("PROC(a, svf, NULL, &p, .in = input[0]); cproc_output(0, a.out);", "cproc_output_f"),
    ("PROC(a, acc, NULL, NULL, .in = input[0]); cproc_output_f(0, a.out);", "use cproc_output"),
    ("PROC(a, phasor_f, NULL, &p); PROC(b, acc, NULL, NULL, .in = a.out); cproc_output(0, b.out);", "is a float"),
    ("PROC(a, svf, NULL, (&(svf_param){ .f = 0.1f, .r = 2 }), .in = input[0]); cproc_output_f(0, a.out);", "no member 'r'"),
    ("PROC(a, svf, NULL, (&(gain_param){ .g = 1 }), .in = input[0]); cproc_output_f(0, a.out);", "svf_param"),
    ("PROC(a, svf, &cfg, &p, .in = input[0]); cproc_output_f(0, a.out);", "expected NULL"),
    ("PROC(a, gain, NULL, &p, .mod = input[0]); cproc_output_f(0, a.out);", "'.in = ...'"),
    ("PROC(a, asfloat, NULL, &p, .in = input[0]); cproc_output_f(0, a.out);", "expected NULL"),
    ("PROC(a, biquad, NULL, NULL, .in = input[0]); cproc_output(0, a.out);", "unknown processor"),
    ("PROC(a, acc, NULL, NULL, .in = input[4294967295]); cproc_output(0, a.out);", "out of range"),
])
def test_ext_parse_errors(text, what):
    with pytest.raises(abi.CprocCudaError) as e:
        abi.graph_parse_ex(text)
    assert e.value.code == abi.EINVAL and what in str(e.value), str(e.value)


def test_ext_parse_forms():
    g = abi.graph_parse_ex("PROC(o, phasor_f, NULL, &o_p); PROC(y, onepole, NULL, (&(onepole_param){ .a = 0.25 }), .in = o.out); cproc_output_f(7, y.out);")
    assert g["rows"] == [(po.NODE_PHASOR_F, po.SRC_ZERO, 0xFFFFFFFF), (po.NODE_ONEPOLE, 0, 0xFFFFFFFF)]
    assert g["n_inputs"] == 0 and g["param_init"].tolist() == [0, F32(0.25)] and g["out_indices"] == [7]
    src = abi.graph_jit_source(g["rows"], 0, g["out_nodes"])
    assert "#define GRAPH_NIN 0" in src and "__fmaf_rn(__uint_as_float(P.p1)" in src and "P.p0 + 0u" in src
    g = abi.graph_parse_ex("#define CPROC_NB_INPUTS 3\nPROC(x, asfloat, NULL, NULL, .in = input[2]); PROC(y, gain, NULL, &gp, .in = x.out); PROC(z, gain, NULL, &gq, .in = input[0]); cproc_output_f(0, y.out); cproc_output_f(1, z.out);")
    assert g["n_inputs"] == 3 and g["rows"][2] == (po.NODE_GAIN, -1, 0xFFFFFFFF)
    src = abi.graph_jit_source(g["rows"], 3, g["out_nodes"])
    assert "__uint2float_rn((x)[0])" in src                       # a w into a float input converts by value
    # the table is checked again where it enters the library: a float output must not feed an integer input
    with pytest.raises(abi.CprocCudaError) as e:
        abi.graph_jit_source([(po.NODE_PHASOR_F, po.SRC_ZERO, 1), (po.NODE_ACC, 0, 1)], 1, 1)
    assert "float output feeds an integer input" in str(e.value)
    with pytest.raises(abi.CprocCudaError) as e:
        abi.graph_jit_source([(po.NODE_ACC, po.SRC_ZERO, 1)], 1, 0)
    assert "not connected" in str(e.value)


# ---- GPU --------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def ctx():
    import synth_tools_b200 as st
    c = st.Context(0)
    yield c
    c.close()


def run_cuda_graph(ctx, rows, n_in, outs, st0, prm, N, F, inp, chg, layout):
    import synth_tools_b200 as st
    b = ctx.batch(st.GRAPH, N, nodes=rows, n_inputs=n_in, out_node=outs, layout=layout)
    b.upload_state(st0)
    if prm is not None:
        b.upload_param(prm)
    il = layout == st.INTERLEAVED
    out = np.zeros((F, len(outs), N) if il else (N, len(outs), F), np.uint32)
    b.run(F, inp=None if inp is None else np.ascontiguousarray(inp.transpose(2, 1, 0) if il else inp),
          in2=None if chg is None else np.ascontiguousarray(chg.T if il else chg), out=out)
    st1 = b.download_state()
    log = b.jit_log
    b.free()
    return (np.ascontiguousarray(out.transpose(2, 1, 0)) if il else out), st1, log


@pytest.mark.gpu
@pytest.mark.parametrize("jit", [1, 0])
@pytest.mark.parametrize("layout,N,F", [(0, 300, 256), (0, 131, 203), (0, 64, 64), (1, 256, 100), (1, 301, 77)])
@pytest.mark.parametrize("seed", range(4))
def test_gpu_ext_graphs_bit_exact(ctx, oracle, seed, layout, N, F, jit):
    rng = np.random.default_rng(1000 + seed)
    n_in = 2
    rows = random_ext_graph(rng, int(rng.integers(1, 9)), n_in, masks=seed % 2 == 1)
    prm = random_params(rng, rows, N)
    inp = rng.integers(0, 2**32, (N, n_in, F), dtype=np.uint32)
    inp[:, 1] = rng.uniform(-1, 1, (N, F)).astype(np.float32).view(np.uint32)
    chg = rng.integers(0, 8, (N, F)).astype(np.uint32) if seed % 2 == 1 else None
    outs = list(range(len(rows)))[-3:]
    st0 = rng.integers(0, 2**32, (N, state_words(rows)), dtype=np.uint32)
    o = 0
    for r in rows:                                               # float state words start as finite floats
        w = po.node_words(r[0])
        if (r[0] & 0xFF) >= po.NODE_PHASOR_F:
            st0[:, o] = rng.uniform(-1, 1, N).astype(np.float32).view(np.uint32)
            if (r[0] & 0xFF) in (po.NODE_SVF, po.NODE_ENV, po.NODE_GLIDE_F):
                st0[:, o + 1] = rng.uniform(0, 1, N).astype(np.float32).view(np.uint32)
        o += w
    sa = st0.copy()
    want = oracle.graph_run_ext(rows, n_in, outs, sa, prm, N, F, inp, chg)
    ctx.set_option("graph_jit", jit)
    try:
        got, st1, log = run_cuda_graph(ctx, rows, n_in, outs, st0, prm, N, F, inp, chg, layout)
    finally:
        ctx.set_option("graph_jit", 1)
    assert np.array_equal(got, want), (rows, log)
    assert np.array_equal(st1, sa)
    if jit:
        assert "not found" not in log and "failed" not in log and "error" not in log, log


@pytest.mark.gpu
@pytest.mark.parametrize("layout,N,F", [(0, 4096 + 37, 512), (0, 1000, 130), (1, 4096, 512), (1, 999, 64)])
def test_gpu_voice_graph_bit_identical_to_xvoice_kernel(ctx, oracle, layout, N, F):
    """VERDICT r1 next #4: phasor_f -> svf -> env (-> pan gains) written as graph nodes renders bit-identically to
    k_xvoice's raw output -- and to the oracle.  No external input stream (n_inputs = 0)."""
    import synth_tools_b200 as st
    rng = np.random.default_rng(77)
    rows, prm, gst, xs, xp = voice_graph_and_records(rng, N)
    got, st1, log = run_cuda_graph(ctx, rows, 0, [3, 4], gst, prm, N, F, None, None, layout)
    b = ctx.batch(st.XVOICE, N)
    b.upload_state(np.ascontiguousarray(xs.view(np.uint32).reshape(N, 5))); b.upload_param(prm)
    raw = np.zeros((N, F, 2), np.float32)
    b.run(F, out=raw, layout=st.PLANAR)
    xst = b.download_state()
    b.free()
    assert np.array_equal(got.view(np.float32).transpose(0, 2, 1).view(np.uint32), raw.view(np.uint32)), log
    assert np.array_equal(st1[:, [1, 2, 3, 5, 6]], xst)            # phase, lp, bp, env, t
    sa = gst.copy()
    want = oracle.graph_run_ext(rows, 0, [3, 4], sa, prm, N, F)
    assert np.array_equal(got, want) and np.array_equal(st1, sa)


@pytest.mark.gpu
def test_gpu_graph_text_to_render(ctx, oracle):
    """The .cproc texts end to end on the GPU: parse -> alloc -> param record from the text's literals -> render."""
    import synth_tools_b200 as st
    rng = np.random.default_rng(9)
    for text, n_out in ((VOICE_TEXT, 2), (CHAIN_TEXT, 3), (GAIN_TEXT, 1)):
        g = st.graph_parse_ex(text)
        N, F = 500, 384
        n_in = g["n_inputs"]
        inp = rng.integers(0, 1 << 20, (N, n_in, F)).astype(np.uint32)
        if n_in == 2:
            inp[:, 0] = rng.integers(0, 2, (N, F))
        if text is GAIN_TEXT:
            inp[:, 0] = rng.uniform(0, 1, (N, F)).astype(np.float32).view(np.uint32)
        chg = rng.integers(0, 4, (N, F)).astype(np.uint32) if n_in == 2 else None
        prm = np.ascontiguousarray(np.tile(g["param_init"], (N, 1)))
        prm[:, 0] = rng.integers(1 << 20, 1 << 27, N)             # per-instance pitch
        st0 = np.zeros((N, state_words(g["rows"])), np.uint32)
        sa = st0.copy()
        want = oracle.graph_run_ext(g["rows"], n_in, g["out_nodes"], sa, prm, N, F, inp, chg)
        for layout in (st.PLANAR, st.INTERLEAVED):
            got, st1, log = run_cuda_graph(ctx, g["rows"], n_in, g["out_nodes"], st0, prm, N, F, inp, chg, layout)
            assert np.array_equal(got, want) and np.array_equal(st1, sa), (layout, log)


@pytest.mark.gpu
def test_gpu_patcher_with_extension_classes(ctx, oracle):
    """The dynamic patcher (mod_bpmodular.c RPC tree) builds osc -> svf -> gain node by node, sets params through
    inst/<node>/param/<k>/set (kind 0) and ticks; params survive the rebuilds."""
    import synth_tools_b200 as st
    N, F = 64, 96
    p = st.Patch(ctx, N, 1)
    i0 = p.apply("input", config=0)
    osc = p.apply("phasor_f", i0)
    for inst in range(N):
        p.set(osc, 0, 1000003 * (inst + 1), inst, kind=p.PARAM)
    flt = p.apply("svf", osc)
    for inst in range(N):
        p.set(flt, 0, int(F32(0.05 + 0.001 * inst)), inst, kind=p.PARAM); p.set(flt, 1, int(F32(0.9)), inst, kind=p.PARAM)
    p.output(flt)
    rng = np.random.default_rng(3)
    inp = rng.integers(0, 1 << 16, (N, 1, F)).astype(np.uint32)
    out1 = np.zeros((N, F), np.uint32)
    p.tick(F, inp=inp, out=out1)
    g = p.apply("gain", flt)                                       # grow the patch: state and params are carried over
    for inst in range(N):
        p.set(g, 0, int(F32(0.5)), inst, kind=p.PARAM)
    p.output(g)
    out2 = np.zeros((N, F), np.uint32)
    p.tick(F, inp=inp, out=out2)
    assert p.get(osc, 0, 5, kind=p.PARAM) == 1000003 * 6 and p.get(flt, 1, 9, kind=p.PARAM) == int(F32(0.9))
    rows = [(po.NODE_PHASOR_F, -1, 0xFFFFFFFF), (po.NODE_SVF, 0, 0xFFFFFFFF)]
    prm = np.zeros((N, 3), np.uint32)
    prm[:, 0] = 1000003 * (np.arange(N) + 1)
    prm[:, 1] = np.array([F32(0.05 + 0.001 * i) for i in range(N)], np.uint32); prm[:, 2] = F32(0.9)
    s = np.zeros((N, 4), np.uint32)
    w1 = oracle.graph_run_ext(rows, 1, [1], s, prm, N, F, inp)
    assert np.array_equal(out1, w1[:, 0])
    rows2 = rows + [(po.NODE_GAIN, 1, 0xFFFFFFFF)]
    prm2 = np.concatenate([prm, np.full((N, 1), F32(0.5), np.uint32)], axis=1)
    s2 = np.concatenate([s, np.zeros((N, 1), np.uint32)], axis=1)
    w2 = oracle.graph_run_ext(rows2, 1, [2], s2, np.ascontiguousarray(prm2), N, F, inp)
    assert np.array_equal(out2, w2[:, 0])
    with pytest.raises(abi.CprocCudaError):
        p.apply("acc", flt)                                        # float .out into a w input
    p.close()


@pytest.mark.parametrize("which", ["voice", "chain", "gain", "free", "random"])
def test_ext_generated_source_compiles_for_sm_100a_without_a_diagnostic(which):
    """The JIT path without a device: the source the library generates for graphs with extension processors (also
    with no input stream at all) compiles with NVRTC exactly as graph_front.cu compiles it, with an empty log."""
    import ctypes as C
    from tests.test_graph_front import _nvrtc
    rng = np.random.default_rng(12)
    if which == "gain":
        g = abi.graph_parse_ex(GAIN_TEXT); rows, n_in, outs, chg = g["rows"], g["n_inputs"], g["out_nodes"], False
    elif which == "voice":
        g = abi.graph_parse_ex(VOICE_TEXT); rows, n_in, outs, chg = g["rows"], g["n_inputs"], g["out_nodes"], False
    elif which == "chain":
        g = abi.graph_parse_ex(CHAIN_TEXT); rows, n_in, outs, chg = g["rows"], g["n_inputs"], g["out_nodes"], True
    elif which == "free":
        rows, _, _, _, _ = voice_graph_and_records(rng, 1); n_in, outs, chg = 0, [3, 4], False
    else:
        rows = random_ext_graph(rng, 40, 3, masks=True); n_in, outs, chg = 3, [39, 5, 17], True
    src = abi.graph_jit_source(rows, n_in, outs, chg)
    nv = _nvrtc()
    if nv is None:
        pytest.skip("libnvrtc not present")
    prog = C.c_void_p()
    assert nv.nvrtcCreateProgram(C.byref(prog), src.encode(), b"cproc_graph.cu", 0, None, None) == 0
    opts = (C.c_char_p * 4)(b"--gpu-architecture=sm_100a", b"-std=c++17", b"-lineinfo", b"-default-device")
    rc = nv.nvrtcCompileProgram(prog, 4, opts)
    ls = C.c_size_t()
    nv.nvrtcGetProgramLogSize(prog, C.byref(ls))
    log = C.create_string_buffer(ls.value)
    nv.nvrtcGetProgramLog(prog, log)
    assert rc == 0 and ls.value <= 1, log.value.decode()
    nv.nvrtcDestroyProgram(C.byref(prog))
