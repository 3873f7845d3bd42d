"""The float paths that are not bit-exact by construction -- the time-parallel one-pole and XVOICE renders and the
XVOICE float mix -- against float64 references of the OPERATION (not the float32 sequential render), instance by
instance and frame by frame, at the settings where float recurrences go wrong: slow poles, resonant filters,
quiet instances next to loud ones, cancelling mixes.

The references below are plain float64 loops over time, vectorised over instances; their self-tests run without a
GPU.  The GPU tests carry the `gpu` mark one by one.

Comparison rule of the scan renders (per instance i):
    scale_i  = max_t |ref64_i|                       (floored at SILENT for an instance that never sounds)
    e_scan,i = max_t |scan_i - ref64_i|,  e_seq,i the same for the sequential render (itself bit-exact vs the oracle)
    e_scan,i <= max(1e-5 scale_i, C_SEQ e_seq,i)
The time-parallel render must be near the exact operation AND never meaningfully worse than the sequential render
it replaces.  Where the float32 recurrence stalls (|a (x - y)| < 1/2 ulp(y): a one-pole smoother with a small
coefficient) the sequential render drifts from the exact result by more than 1e-5 of the peak; the scan restarts
every chunk from an fp64 state and drifts only within one chunk.

C_SEQ = 2: the scan's error at frame t is (1) the rounding of its chunk start state to float32, at most 1/2 ulp of
each state word -- one tick's worth of the rounding the sequential render makes every tick -- propagated by the
same stable filter, plus (2) the float recurrence's own rounding over the at most L ticks since that chunk start,
the same operations on the same inputs the sequential render performs over F >= L ticks.  Each part is at most
what the sequential render accumulates, so e_scan <= 2 e_seq wherever the 1e-5 floor does not already hold.
"""
import numpy as np
import pytest

from oracle import pyoracle as po

rng = np.random.default_rng(20261020)

C_SEQ = 2.0
REL = 1e-5
SILENT = 1e-30
U = 2.0 ** -24                                       # unit roundoff of binary32


@pytest.fixture(scope="module")
def st():
    import synth_tools_b200 as st_
    return st_


@pytest.fixture(scope="module")
def ctx(st):
    c = st.Context(0)
    yield c
    c.close()


# ------------------------------------------------------------------------------------------------ fp64 references
def onepole_ref64(y0, a, x):
    """y <- y + a (x - y) in float64 on the float32 inputs and coefficients.  y0, a: [N]; x: [N][F].
    Returns (y [N][F], final y [N])."""
    y = np.asarray(y0, np.float32).astype(np.float64)
    a64 = np.asarray(a, np.float32).astype(np.float64)
    xt = np.ascontiguousarray(np.asarray(x, np.float32).T).astype(np.float64)     # [F][N]: one row per tick
    out = np.empty_like(xt)
    for t in range(xt.shape[0]):
        y = y + a64 * (xt[t] - y)
        out[t] = y
    return out.T, y


def svf_ref64(s0, prm, F):
    """The XVOICE filter in float64: x_t = (float)(int32)phase * 2^-31 (exact: phase is 32 bits wide, the float has 24),
    lp <- lp + f bp; bp <- bp + f (x - lp - q bp), from the state's float32 lp / bp with the float32 f / q.
    Returns (lp [N][F], final lp [N], final bp [N], max |lp| [N], max |bp| [N]) -- the maxima over the start and every tick."""
    N = len(s0)
    phase = np.array(s0["phase"], np.uint32)
    inc = np.array(prm["inc"], np.uint32)
    f = prm["f"].astype(np.float64); q = prm["q"].astype(np.float64)
    lp = s0["lp"].astype(np.float64); bp = s0["bp"].astype(np.float64)
    lpm, bpm = np.abs(lp), np.abs(bp)
    lps = np.empty((F, N))
    for t in range(F):
        x = phase.view(np.int32).astype(np.float32).astype(np.float64) * 2.0 ** -31
        phase += inc                                 # uint32: wraps like the accumulator
        lp = lp + f * bp
        bp = bp + f * (x - lp - q * bp)
        lps[t] = lp
        np.maximum(bpm, np.abs(bp), out=bpm)
    np.maximum(lpm, np.abs(lps).max(axis=0) if F else lpm, out=lpm)
    return lps.T, lp, bp, lpm, bpm


def oracle_env(oracle, s0, prm, F):
    """The envelope of every voice and tick, [N][F] float32, from the oracle: the same voices with f = 0, lp = 1, bp = 0,
    gl = 1 render lp * env * gl = env exactly (the filter holds lp at 1; the envelope does not depend on it)."""
    s = s0.copy(); s["lp"] = 1.0; s["bp"] = 0.0
    p = prm.copy(); p["f"] = 0.0; p["q"] = 0.0; p["gl"] = 1.0; p["gr"] = 1.0
    raw, _ = oracle.xvoice_run(s, p, len(s0), F, want_mix=False)
    return raw[:, :, 0]


def xvoice_ref64(oracle, s0, prm, F):
    """Raw XVOICE output in float64: lp from svf_ref64, env from the oracle (bit-exact by contract), out = lp env g.
    Returns (out [N][F][2], final lp, final bp, max |lp|, max |bp|)."""
    lp, lpf, bpf, lpm, bpm = svf_ref64(s0, prm, F)
    y = lp * oracle_env(oracle, s0, prm, F).astype(np.float64)
    out = np.stack([y * prm["gl"].astype(np.float64)[:, None], y * prm["gr"].astype(np.float64)[:, None]], axis=2)
    return out, lpf, bpf, lpm, bpm


def svf_stable(f, q):
    """Strict stability of the Chamberlin map s' = A s + b x, A = [[1, f], [-f, 1 - f q - f^2]]: with tr A = 2 - f q - f^2
    and det A = 1 - f q, both eigenvalues lie inside the unit circle iff (Jury) |det A| < 1, 1 - tr + det = f^2 > 0 and
    1 + tr + det = 4 - 2 f q - f^2 > 0, i.e. f > 0, 0 < f q < 2 and f^2 + 2 f q < 4.  (q = 0 is the undamped oscillator,
    det A = 1: not stable.)"""
    f, q = float(np.float32(f)), float(np.float32(q))
    return f > 0 and 0 < f * q < 2 and f * f + 2 * f * q < 4


# ------------------------------------------------------------------------------------------------ reference self-tests
def test_onepole_ref64_step_response():
    """Unit step from rest: y_t = 1 - (1 - a)^(t+1) (t = 0 is the first output)."""
    F = 5000
    a = np.array([2.0 ** -24, 1e-6, 1e-3, 0.5, 1.5, 1.999], np.float32)
    y, yf = onepole_ref64(np.zeros(len(a)), a, np.ones((len(a), F), np.float32))
    t = np.arange(1, F + 1)
    want = 1.0 - (1.0 - a.astype(np.float64)[:, None]) ** t
    assert np.abs(y - want).max() <= 1e-12
    assert np.array_equal(yf, y[:, -1])


def test_svf_ref64_lowpass_dc_gain():
    """A constant input (inc = 0) settles to lp = x: the low-pass has DC gain 1, for slow and fast, damped and resonant
    settings of the stable region."""
    fq = [(0.01, 0.5), (0.3, 2.0), (0.9, 0.5), (0.05, 0.05), (0.3, 0.005)]
    N = len(fq)
    s0 = np.zeros(N, po.xvoice_state_dtype)
    s0["phase"] = np.array([0x40000000, 0xC0000000, 0x10000000, 0x7FFFFFFF, 0x80000000], np.uint32)
    prm = np.zeros(N, po.xvoice_param_dtype)
    prm["f"] = [f for f, _ in fq]; prm["q"] = [q for _, q in fq]
    assert all(svf_stable(f, q) for f, q in fq)
    lp, lpf, bpf, _, _ = svf_ref64(s0, prm, 60000)
    x = s0["phase"].view(np.int32).astype(np.float64) * 2.0 ** -31
    assert np.abs(lpf - x).max() <= 1e-9 and np.abs(bpf).max() <= 1e-9
    assert np.array_equal(lp[:, -1], lpf)


def test_svf_stable_region():
    assert svf_stable(1e-3, 5e-3) and svf_stable(0.9, 0.5) and svf_stable(0.3, 2.0)
    assert not svf_stable(0.01, 0.0) and not svf_stable(0.9, 2.0) and not svf_stable(0.0, 1.0)
    # the region is what the eigenvalues say
    for f in (1e-3, 0.01, 0.3, 0.9, 1.2):
        for q in (0.0, 5e-3, 0.05, 0.5, 2.0, 3.0):
            f32, q32 = float(np.float32(f)), float(np.float32(q))
            A = np.array([[1.0, f32], [-f32, 1.0 - f32 * q32 - f32 * f32]])
            assert svf_stable(f, q) == (np.abs(np.linalg.eigvals(A)).max() < 1.0 - 1e-12), (f, q)


def test_onepole_ref64_near_oracle(oracle):
    """Benign coefficients and inputs: the float32 oracle stays within a few float32 ulps per tick of the fp64 recurrence."""
    N, F = 40, 3000
    a = rng.uniform(0.01, 0.5, N).astype(np.float32)
    x = (rng.uniform(-1, 1, (N, F)) + np.sin(np.arange(F) * 0.003)).astype(np.float32)
    y0 = rng.uniform(-1, 1, N).astype(np.float32)
    ya = y0.copy()
    want = oracle.onepole_run(ya, a.copy(), N, F, x)
    ref, yf = onepole_ref64(y0, a, x)
    err = np.abs(want.astype(np.float64) - ref).max(axis=1) / np.abs(ref).max(axis=1)
    # a stable one-pole forgets old rounding: the error is a few roundings of the last ~1/a ticks
    assert err.max() <= 8 * U, err.max()
    assert (np.abs(ya - yf) / np.abs(ref).max(axis=1)).max() <= 8 * U


def test_xvoice_ref64_near_oracle(oracle):
    """Benign filters: the oracle's raw output stays within a few float32 ulps per tick of the fp64 reference."""
    N, F = 48, 2000
    s0, prm = _xvoice_voices(oracle, N, F, f=rng.uniform(0.05, 0.3, N), q=rng.uniform(0.5, 2.0, N))
    sa = s0.copy()
    want, _ = oracle.xvoice_run(sa, prm, N, F, want_mix=False)
    ref, lpf, bpf, lpm, bpm = xvoice_ref64(oracle, s0, prm, F)
    scale = np.maximum(np.abs(ref).reshape(N, -1).max(axis=1), SILENT)
    err = np.abs(want.astype(np.float64) - ref).reshape(N, -1).max(axis=1) / scale
    # the damped filter forgets in ~1/(f q) ticks; per tick four roundings of the SVF, two products after it
    assert err.max() <= 64 * U, err.max()
    assert (np.abs(sa["lp"] - lpf) / lpm).max() <= 64 * U and (np.abs(sa["bp"] - bpf) / bpm).max() <= 64 * U


# ------------------------------------------------------------------------------------------------ comparison rule
def per_instance(scan, seq, ref):
    """Per-instance errors against the fp64 reference, [N][...] arrays: (e_scan, e_seq, scale)."""
    N = ref.shape[0]
    ref = ref.reshape(N, -1)
    scale = np.maximum(np.abs(ref).max(axis=1), SILENT) if ref.shape[1] else np.full(N, SILENT)
    e_scan = np.abs(scan.reshape(N, -1).astype(np.float64) - ref).max(axis=1)
    e_seq = np.abs(seq.reshape(N, -1).astype(np.float64) - ref).max(axis=1)
    return e_scan, e_seq, scale


def assert_rule(e_scan, e_seq, scale, what, labels=None):
    bound = np.maximum(REL * scale, C_SEQ * e_seq)
    bad = np.nonzero(~(e_scan <= bound))[0]
    if bad.size:
        rows = ["  %s: e_scan %.3g  e_seq %.3g  scale %.3g (e_scan/scale %.3g, e_seq/scale %.3g)"
                % (labels[i] if labels is not None else i, e_scan[i], e_seq[i], scale[i], e_scan[i] / scale[i], e_seq[i] / scale[i])
                for i in bad[:12]]
        pytest.fail("%s: %d of %d instances outside max(1e-5 scale, %g e_seq):\n%s" % (what, bad.size, len(e_scan), C_SEQ, "\n".join(rows)))


def report(what, labels, e_scan, e_seq, scale):
    """Worst e_scan / e_seq relative to the instance's scale per label (printed: `pytest -s` shows the measured numbers)."""
    rows = {}
    for i, lab in enumerate(labels):
        r = rows.setdefault(lab, [0.0, 0.0])
        r[0] = max(r[0], e_scan[i] / scale[i]); r[1] = max(r[1], e_seq[i] / scale[i])
    print("\n[%s]" % what)
    for lab, (es, eq) in rows.items():
        print("  %-34s e_scan/scale %.2e   e_seq/scale %.2e" % (lab, es, eq))


# ------------------------------------------------------------------------------------------------ one-pole
OP_A = [2.0 ** -24, 1e-6, 1e-4, 1e-3, 0.5, 1.5, 1.999]
OP_KINDS = ["step 1", "step 1e4", "decay from +1", "decay from -1", "noise + slow sine", "tiny"]
OP_COMBOS = [(a, k) for a in OP_A for k in OP_KINDS]


def _onepole_inputs(N, F):
    """Instance i: coefficient and input kind OP_COMBOS[...] (every combination once N >= 42)."""
    pick = np.arange(N) % len(OP_COMBOS) if N >= len(OP_COMBOS) else rng.choice(len(OP_COMBOS), N, replace=False)
    a = np.zeros(N, np.float32); y0 = np.zeros(N, np.float32); x = np.zeros((N, F), np.float32)
    t = np.arange(F)
    labels = []
    for i, c in enumerate(pick):
        ai, kind = OP_COMBOS[c]
        a[i] = ai
        labels.append("a=%.4g %s" % (ai, kind))
        if kind == "step 1":
            x[i] = 1.0
        elif kind == "step 1e4":
            x[i] = 1e4
        elif kind == "decay from +1":
            y0[i] = 1.0
        elif kind == "decay from -1":
            y0[i] = -1.0
        elif kind == "noise + slow sine":
            x[i] = rng.uniform(-1, 1, F) + 3.0 * np.sin(2 * np.pi * t / 7919.0)
            y0[i] = rng.uniform(-1e3, 1e3)                       # a large initial state
        else:
            x[i] = rng.uniform(-1, 1, F) * 1e-20
            y0[i] = rng.uniform(-1, 1) * 1e-20
    return a, y0, x, labels


def _onepole_device(st, ctx, mode, layout, y0, a, x, chunk=0):
    """Render x through a ONEPOLE batch; layout PLANAR / INTERLEAVED through host buffers, "PLANAR+1": device buffers whose
    rows start one float past a 16-byte boundary of a larger allocation (the kernels' unaligned branches).
    Returns (out [N][F], final y [N])."""
    N, F = x.shape
    ctx.set_option("xvoice_chunk", chunk)
    b = ctx.batch(st.ONEPOLE, N, layout=st.INTERLEAVED if layout == "INTERLEAVED" else st.PLANAR, mode=mode)
    try:
        b.upload_state(np.ascontiguousarray(y0, np.float32).reshape(N, 1))
        b.upload_param(np.ascontiguousarray(a, np.float32).reshape(N, 1))
        if layout == "PLANAR+1":
            nb = 4 * (N * F + 8)
            d_in, d_out = ctx.dev_alloc(nb), ctx.dev_alloc(nb)
            try:
                ctx.h2d(d_in + 4, np.ascontiguousarray(x))
                b.run_dev(F, inp=d_in + 4, out=d_out + 4, layout=st.PLANAR)
                ctx.sync()
                out = np.zeros((N, F), np.float32)
                ctx.d2h(out, d_out + 4)
            finally:
                ctx.dev_free(d_in); ctx.dev_free(d_out)
        elif layout == "INTERLEAVED":
            o = np.zeros((F, N), np.float32)
            b.run(F, inp=np.ascontiguousarray(x.T), out=o)
            out = o.T
        else:
            out = np.zeros((N, F), np.float32)
            b.run(F, inp=np.ascontiguousarray(x), out=out)
        yf = b.download_state().view(np.float32)[:, 0].copy()
    finally:
        b.free()
        ctx.set_option("xvoice_chunk", 0)
    return out, yf


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["PLANAR", "INTERLEAVED", "PLANAR+1"])
@pytest.mark.parametrize("N", [1, 3, 130])
@pytest.mark.parametrize("F,chunk", [(65, 64), (40000, 0), (40000, 96), (9999, 50), (3001, 7), (20000, 33)])
def test_onepole_scan_vs_fp64(st, ctx, oracle, layout, N, F, chunk):
    """ONEPOLE_SCAN per instance against the fp64 recurrence, at stalling (a = 2^-24 .. 1e-3), fast and overshooting
    (a = 1.5, 1.999) coefficients, on steps, decays, noise with large initial states and tiny inputs; F = L + 1, F not a
    multiple of L, C > 256 chunks (several per thread of the scan), chunk lengths that are not multiples of 4.  The
    sequential render of the same run is bit-exact against the oracle."""
    a, y0, x, labels = _onepole_inputs(N, F)
    ya = y0.copy()
    want = oracle.onepole_run(ya, a.copy(), N, F, x)
    seq, yseq = _onepole_device(st, ctx, 0, layout, y0, a, x)
    assert np.array_equal(seq.view(np.uint32), want.view(np.uint32))
    assert np.array_equal(yseq.view(np.uint32), ya.view(np.uint32))
    scan, yscan = _onepole_device(st, ctx, 1, layout, y0, a, x, chunk)
    ref, yref = onepole_ref64(y0, a, x)
    e_scan, e_seq, scale = per_instance(scan, seq, ref)
    report("one-pole N=%d F=%d chunk=%d %s" % (N, F, chunk, layout), labels, e_scan, e_seq, scale)
    assert_rule(e_scan, e_seq, scale, "one-pole output", labels)
    assert_rule(np.abs(yscan.astype(np.float64) - yref), np.abs(yseq.astype(np.float64) - yref), scale, "one-pole final state", labels)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1], ids=["SEQ", "SCAN"])
@pytest.mark.parametrize("layout", ["PLANAR", "INTERLEAVED", "PLANAR+1"])
@pytest.mark.parametrize("F,chunk", [(3001, 50), (40000, 0), (1000, 96)])
def test_onepole_exact_coefficients(st, ctx, oracle, mode, layout, F, chunk):
    """a = 0 holds y0 forever; a = 1 on dyadic inputs (k/256, |k| < 2^15, and a dyadic y0) makes y = x exactly: every
    fp32 and fp64 operation of both renders is exact there, so SEQ and SCAN must reproduce it bit for bit."""
    N = 6
    a = np.array([0, 0, 0, 1, 1, 1], np.float32)
    y0 = np.array([rng.uniform(-1e6, 1e6), 0.1, -3e-9, 0.5, -2.0, 17.25], np.float32)
    x = rng.uniform(-1e3, 1e3, (N, F)).astype(np.float32)
    x[3:] = (rng.integers(-(1 << 15) + 1, 1 << 15, (3, F)) / 256.0).astype(np.float32)
    out, yf = _onepole_device(st, ctx, mode, layout, y0, a, x, chunk)
    assert np.array_equal(out[:3].view(np.uint32), np.repeat(y0[:3, None], F, axis=1).view(np.uint32))
    assert np.array_equal(out[3:].view(np.uint32), x[3:].view(np.uint32))
    assert np.array_equal(yf.view(np.uint32), np.concatenate([y0[:3], x[3:, -1]]).view(np.uint32))


# ------------------------------------------------------------------------------------------------ XVOICE scan
def _xvoice_voices(oracle, N, F, f, q, lp_range=0.5, quiet=0.0):
    """Voices with the given f / q (arrays), random notes, phases, states (lp, bp in +-lp_range), envelopes crossing their
    gates inside the render, and pan gains; a `quiet` fraction of them at gl = gr = 1e-3 (next to loud ones)."""
    prm = np.zeros(N, po.xvoice_param_dtype)
    prm["inc"] = [oracle.note_to_inc(int(n)) for n in rng.integers(12, 109, N)]
    prm["f"] = f; prm["q"] = q
    prm["env_attack"] = rng.uniform(1e-4, 1e-1, N); prm["env_release"] = rng.uniform(2e-5, 1e-2, N)
    prm["gate_frames"] = rng.integers(0, F + F // 4 + 1, N)
    prm["gl"] = rng.uniform(0.3, 1.0, N); prm["gr"] = 1.0 - prm["gl"] + 0.1
    prm["gr"][::5] = prm["gl"][::5]
    nq = int(round(quiet * N))
    if nq:
        idx = rng.choice(N, nq, replace=False)
        prm["gl"][idx] = 1e-3; prm["gr"][idx] = 1e-3
    s0 = np.zeros(N, po.xvoice_state_dtype)
    s0["phase"] = rng.integers(0, 2**32, N, dtype=np.uint32)
    s0["lp"] = rng.uniform(-lp_range, lp_range, N); s0["bp"] = rng.uniform(-lp_range, lp_range, N)
    s0["env"] = rng.uniform(0, 1, N); s0["t"] = rng.integers(0, 100, N)
    return s0, prm


def _xvoice_device(st, ctx, s0, prm, F, layout, mode, chunk=0, groups=0, closed=1):
    """Raw render of the voices ([N][F][2]) and the final state."""
    N = len(s0)
    ctx.set_option("xvoice_chunk", chunk); ctx.set_option("xvoice_groups", groups); ctx.set_option("xvoice_closed", closed)
    b = ctx.batch(st.XVOICE, N, layout=getattr(st, layout), mode=mode)
    try:
        b.upload_state(s0.view(np.uint32).reshape(N, 5)); b.upload_param(prm.view(np.uint32).reshape(N, 8))
        raw = np.zeros(N * F * 2, np.float32)
        b.run(F, out=raw)
        got = raw.reshape(F // 2, N, 2, 2).transpose(1, 0, 2, 3).reshape(N, F, 2) if layout == "TILED" else raw.reshape(N, F, 2)
        state = b.download_state().view(po.xvoice_state_dtype).reshape(N).copy()
    finally:
        b.free()
        ctx.set_option("xvoice_chunk", 0); ctx.set_option("xvoice_groups", 0); ctx.set_option("xvoice_closed", 1)
    return got, state


def _xvoice_scan_check(st, ctx, oracle, s0, prm, F, layout, labels, chunk=0, groups=0, closed=1, what="xvoice"):
    N = len(s0)
    sa = s0.copy()
    want, _ = oracle.xvoice_run(sa, prm, N, F, want_mix=False)
    seq, sseq = _xvoice_device(st, ctx, s0, prm, F, layout, st.XVOICE_SEQ)
    assert np.array_equal(seq.view(np.uint32), want.view(np.uint32))
    assert np.array_equal(sseq.view(np.uint32), sa.view(np.uint32))
    scan, sscan = _xvoice_device(st, ctx, s0, prm, F, layout, st.XVOICE_SCAN, chunk, groups, closed)
    for k in ("phase", "t", "env"):
        assert np.array_equal(sscan[k].view(np.uint32), sa[k].view(np.uint32)), k
    ref, lpf, bpf, lpm, bpm = xvoice_ref64(oracle, s0, prm, F)
    e_scan, e_seq, scale = per_instance(scan, seq, ref)
    report("%s F=%d %s chunk=%d groups=%d closed=%d" % (what, F, layout, chunk, groups, closed), labels, e_scan, e_seq, scale)
    assert_rule(e_scan, e_seq, scale, what + " output", labels)
    for k, fin, m in (("lp", lpf, lpm), ("bp", bpf, bpm)):
        assert_rule(np.abs(sscan[k].astype(np.float64) - fin), np.abs(sa[k].astype(np.float64) - fin), np.maximum(m, SILENT),
                    what + " final " + k, labels)


SVF_F = [1e-3, 0.01, 0.3, 0.9]
SVF_Q = [0.0, 5e-3, 0.05, 0.5, 2.0]
SVF_GRID = [(f, q) for f in SVF_F for q in SVF_Q if svf_stable(f, q)]


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["PLANAR", "TILED"])
@pytest.mark.parametrize("groups,chunk", [(0, 0), (3, 96)])
@pytest.mark.parametrize("closed", [1, 0])
def test_xvoice_scan_filter_grid(st, ctx, oracle, layout, groups, chunk, closed):
    """XVOICE_SCAN over the stable part of f x q = {1e-3, 0.01, 0.3, 0.9} x {0, 5e-3, 0.05, 0.5, 2} (slow, resonant and
    fast filters), initial lp / bp up to +-4, a third of the voices quiet (gl = gr = 1e-3) beside loud ones: per voice
    within max(1e-5 of its own peak, C_SEQ x the sequential render's error) of the fp64 reference."""
    V, F = 24, 6000
    N = V * len(SVF_GRID)
    f = np.repeat([g[0] for g in SVF_GRID], V); q = np.repeat([g[1] for g in SVF_GRID], V)
    s0, prm = _xvoice_voices(oracle, N, F, f, q, lp_range=4.0, quiet=1 / 3)
    labels = ["f=%g q=%g%s" % (f[i], q[i], " quiet" if prm["gl"][i] == np.float32(1e-3) else "") for i in range(N)]
    _xvoice_scan_check(st, ctx, oracle, s0, prm, F, layout, labels, chunk, groups, closed, "svf grid")


@pytest.mark.gpu
@pytest.mark.parametrize("closed", [1, 0])
@pytest.mark.parametrize("layout,groups", [("TILED", 3), ("PLANAR", 0)])
def test_xvoice_scan_slow_filter_increments(st, ctx, oracle, closed, layout, groups):
    """Every kind of increment (none, one wrap per 2^32 ticks, powers of two, past 2^31, gaps of k and k + 1 ticks) at
    the slow filter f = 1e-3, where the closed-form zero-state pass cancels large terms (P x0 + Q inc - 2^32 y), for both
    zero-state forms."""
    special = np.array([0, 1, 2, 3, 1 << 20, 1 << 24, (1 << 24) + 1, (1 << 24) - 1, 3 << 28, 1 << 31, (1 << 31) + 5, (1 << 31) - 1,
                        0xFFFFFFFF, 0xFFFFFFFE, 0x12345678, 0x9ABCDEF0, 0x55555555, 0x55555556, 0x00F00F00, 715827883], np.uint32)
    qs = [5e-3, 0.05, 0.5, 2.0]
    F = 8192
    N = len(special) * len(qs) * 4
    q = np.tile(np.repeat(qs, len(special)), 4)
    s0, prm = _xvoice_voices(oracle, N, F, np.full(N, 1e-3), q, lp_range=4.0, quiet=0.25)
    prm["inc"] = np.tile(special, len(qs) * 4)
    labels = ["q=%g inc=%#x" % (q[i], prm["inc"][i]) for i in range(N)]
    _xvoice_scan_check(st, ctx, oracle, s0, prm, F, layout, labels, 96, groups, closed, "slow svf increments")


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["PLANAR", "TILED"])
def test_xvoice_scan_long_render(st, ctx, oracle, layout):
    """2^18 frames (8192 chunks) for a handful of voices, slow and resonant filters among them."""
    fq = [(1e-3, 5e-3), (1e-3, 0.05), (0.01, 5e-3), (0.01, 0.5), (0.3, 0.05), (0.9, 0.5), (1e-3, 2.0), (0.3, 2.0)]
    N, F = len(fq), 1 << 18
    s0, prm = _xvoice_voices(oracle, N, F, [g[0] for g in fq], [g[1] for g in fq], lp_range=4.0)
    prm["gl"][3] = prm["gr"][3] = 1e-3
    labels = ["f=%g q=%g" % g for g in fq]
    _xvoice_scan_check(st, ctx, oracle, s0, prm, F, layout, labels, what="long render")


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["PLANAR", "TILED"])
@pytest.mark.parametrize("closed", [1, 0])
def test_xvoice_scan_frozen_filter_is_exact(st, ctx, oracle, layout, closed):
    """f = 0: lp and bp never change, the zero-state responses are exactly zero and the chunk start states are the initial
    state -- SEQ and SCAN render the oracle's output bit for bit."""
    N, F = 200, 4096
    s0, prm = _xvoice_voices(oracle, N, F, np.zeros(N), rng.uniform(0, 2, N), lp_range=4.0, quiet=0.2)
    s0["lp"][s0["lp"] == 0] = 0.5
    sa = s0.copy()
    want, _ = oracle.xvoice_run(sa, prm, N, F, want_mix=False)
    for mode in (st.XVOICE_SEQ, st.XVOICE_SCAN):
        got, state = _xvoice_device(st, ctx, s0, prm, F, layout, mode, 96, 0, closed)
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), mode
        assert np.array_equal(state.view(np.uint32), sa.view(np.uint32)), mode


# ------------------------------------------------------------------------------------------------ XVOICE mix
# Per-frame bound.  Every mix word is a sum tree over the voices' contributions c_v = gl y (or gr y); with d the most
# roundings on any leaf-to-root path, |mix - sum c| <= gamma_d sum |c|, gamma_d = d u / (1 - d u), u = 2^-24 (Higham,
# Accuracy and Stability of Numerical Algorithms, 2nd ed., (4.4)).  The mix kernels fuse the pan product into their
# first add (fma(gl, y, acc)) where the reference rounds it (c = fl(gl y)): one more u, so d counts it.  The paths:
#   raw + mix (k_xvoice<RAW, MIX> + k_xvoice_final): a lane adds the 32 voices of its warp in order (31 roundings), the 4
#     warp rows meet in order (3), k_xvoice_final adds the nb = ceil(N / 128) block rows in 4 chains (<= ceil(nb / 4) + 3)
#     and combines the chains (2)
#   k_xvoice_mix: a thread's voices of a tile in one register (<= min(ceil(N / T), 64)), tiles add into the block row (one
#     each), the block's 128 rows in two halves of 4 chains of 16 (15 + 2 + 1 = 18), then xm_finish below; nb = 4 n_sm
#     blocks of 128 threads (T = 128 nb)
#   k_xvoice_mix2: a thread's voice PAIRS, two fmas per pair into the same accumulator (2 kg, kg <= ceil(ceil(N / 256) / nb)
#     groups of a block), one add per further tile, the warp butterfly (5), the block's 4 warp rows (3), then xm_finish;
#     nb = 3 n_sm - 1
#   xm_finish: 8 slices of the nb block rows, 4 chains each (<= ceil(ceil(nb / 8) / 4) + 3), chains combined (2), slice
#     pairs (1), the 4 warps (2)
# plus 2 for the float sum in rank order of a mix bus (world 1: an add of zero at most).
def _ceil(a, b):
    return -(-a // b)


def mix_depth(path, N, n_sm):
    fin = lambda nb: _ceil(_ceil(nb, 8), 4) + 3 + 2 + 1 + 2
    if path == "raw":
        nb = _ceil(N, 128)
        d = 31 + 3 + _ceil(nb, 4) + 3 + 2
    elif path == "mix1":
        nb = 4 * n_sm
        T = 128 * nb
        d = min(_ceil(N, T), 64) + _ceil(N, T * 64) + 18 + fin(nb)
    else:
        nb = 3 * n_sm - 1
        kg = _ceil(_ceil(N, 256), nb)
        d = 2 * kg + _ceil(kg, 14) + 5 + 3 + fin(nb)
    return d + 1 + 2


def gamma(d):
    return d * U / (1 - d * U)


def _n_sm():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _mix_device(st, ctx, s0, prm, F, path, split=False):
    """Mix [2][F] of the voices through one of the three paths ("raw": raw + mix kernel, "mix1" / "mix2": the mix-only
    generations), optionally as two calls of 32 and F - 32 frames; returns (mix, final state)."""
    N = len(s0)
    ctx.set_option("xvoice_mix2", 1 if path == "mix2" else 0)
    b = ctx.batch(st.XVOICE, N)
    try:
        b.upload_state(s0.view(np.uint32).reshape(N, 5)); b.upload_param(prm.view(np.uint32).reshape(N, 8))
        parts = []
        for Fk in ([32, F - 32] if split else [F]):
            mix = np.zeros((2, Fk), np.float32)
            b.run(Fk, out=np.zeros(N * Fk * 2, np.float32) if path == "raw" else None, mix=mix)
            parts.append(mix)
        state = b.download_state().view(po.xvoice_state_dtype).reshape(N).copy()
    finally:
        b.free()
        ctx.set_option("xvoice_mix2", 1)
    return np.concatenate(parts, axis=1), state


def _contrib_sums(oracle, s0, prm, F, slab=1 << 17):
    """S[c][t] = sum_v c_v[t] and A[c][t] = sum_v |c_v[t]| in float64 from the oracle's per-voice (bit-exact) outputs,
    rendered in slabs of voices; also the oracle's final state."""
    N = len(s0)
    sa = s0.copy()
    S = np.zeros((2, F)); A = np.zeros((2, F))
    for v0 in range(0, N, slab):
        s = sa[v0:v0 + slab]
        raw, _ = oracle.xvoice_run(s, prm[v0:v0 + slab].copy(), len(s), F, want_mix=False)
        sa[v0:v0 + slab] = s
        r = raw.astype(np.float64)
        S += r.sum(axis=0).T; A += np.abs(r).sum(axis=0).T
    return S, A, sa


MIX_PATHS = ["mix2", "mix1", "raw"]


@pytest.mark.gpu
@pytest.mark.parametrize("path", MIX_PATHS)
@pytest.mark.parametrize("case,N,F", [("random", 1000, 512), ("random", 148 * 4 * 128 + 333, 96), ("cancelling", 1000, 200),
                                      ("cancelling", 148 * 3 * 256 + 2, 64), ("half-period pairs", 2000, 300)])
def test_xvoice_mix_per_frame_bound(st, ctx, oracle, path, case, N, F):
    """|mix[t] - S[t]| <= gamma_d sum_v |c_v[t]| frame by frame, d from the kernel's reduction tree (mix_depth).  In the
    cancelling cases the peak of the mix is tiny or zero, so a bound relative to it would say nothing: voices come in
    pairs with the same filter and state and opposite gains (S = 0 exactly), with gl = gr, or with the same increment and
    phases 2^31 apart (a half period: the odd harmonics cancel)."""
    s0, prm = _xvoice_voices(oracle, N, F, rng.uniform(0.01, 0.3, N), rng.uniform(0.5, 2.0, N), quiet=0.1)
    if case == "cancelling":
        h = N // 2
        for k in s0.dtype.names:
            s0[k][h:2 * h] = s0[k][:h]
        for k in prm.dtype.names:
            prm[k][h:2 * h] = prm[k][:h]
        prm["gr"][:h] = prm["gl"][:h]
        prm["gl"][h:2 * h] = -prm["gl"][:h]; prm["gr"][h:2 * h] = -prm["gr"][:h]
    elif case == "half-period pairs":
        h = N // 2
        for k in prm.dtype.names:
            prm[k][h:2 * h] = prm[k][:h]
        s0["phase"][h:2 * h] = s0["phase"][:h] + np.uint32(1 << 31)
        s0["lp"][h:2 * h] = s0["lp"][:h]; s0["bp"][h:2 * h] = s0["bp"][:h]
        s0["env"][h:2 * h] = s0["env"][:h]; s0["t"][h:2 * h] = s0["t"][:h]
    S, A, sa = _contrib_sums(oracle, s0, prm, F)
    mix, state = _mix_device(st, ctx, s0, prm, F, path)
    assert np.array_equal(state.view(np.uint32), sa.view(np.uint32))
    d = mix_depth(path, N, _n_sm())
    err = np.abs(mix.astype(np.float64) - S)
    bound = gamma(d) * A
    worst = np.unravel_index(np.argmax(err - bound), err.shape)
    assert np.all(err <= bound), (path, d, worst, float(err[worst]), float(bound[worst]), float(S[worst]))
    print("\n[mix %s %s N=%d F=%d] d=%d  max err/sum|c| %.2e (gamma_d %.2e)  max |S| %.3g  max sum|c| %.3g"
          % (path, case, N, F, d, (err / np.maximum(A, SILENT)).max(), gamma(d), np.abs(S).max(), A.max()))


# Exact mix.  f = 0 holds lp at lp0; env moves in quarters (attack, release, env0 multiples of 1/4, clamps at 0 and 1);
# lp0 is +-1/2 or +-1, the gains are nonzero multiples of 2^-b in [-1, 1].  Every contribution c = g (lp0 env) is then a
# multiple of 2^-m, m = 3 + b, with |c| <= 1.  While N max|c| < 2^(24 - m), every partial sum of any order is a multiple
# of 2^-m below 2^(24 - m) in magnitude -- an integer of fewer than 24 bits times a power of two, exact in binary32 -- so
# every reduction order gives the exact sum.  b is the largest (up to 6) that keeps the bound for the voice count.
def _dyadic_voices(N, F):
    b = 0
    while b < 6 and N * 2 ** (3 + b + 1) < 2 ** 24:
        b += 1
    m = 3 + b
    assert N * 1.0 < 2.0 ** (24 - m)
    prm = np.zeros(N, po.xvoice_param_dtype)
    prm["inc"] = rng.integers(0, 2**32, N, dtype=np.uint32)
    prm["f"] = 0.0; prm["q"] = rng.uniform(0, 2, N)
    prm["env_attack"] = rng.choice([0.25, 0.5], N); prm["env_release"] = rng.choice([0.25, 0.5], N)
    prm["gate_frames"] = rng.integers(1, F + 1, N)                    # every voice's gate falls inside the render
    k = 2 ** b
    for g in ("gl", "gr"):
        v = rng.integers(1, k + 1, N) * rng.choice([-1, 1], N)
        prm[g] = v / float(k)
    s0 = np.zeros(N, po.xvoice_state_dtype)
    s0["phase"] = rng.integers(0, 2**32, N, dtype=np.uint32)
    s0["lp"] = rng.choice([-1.0, -0.5, 0.5, 1.0], N); s0["bp"] = rng.uniform(-1, 1, N)
    s0["env"] = rng.integers(0, 5, N) / 4.0
    return s0, prm


EXACT_NF = [(1, 96), (255, 96), (256, 96), (257, 96), (148 * 4 * 128 + 333, 96), (148 * 3 * 256 * 12 + 257, 96),
            (1000, 1), (1000, 31), (1000, 32), (1000, 33), (1000, 96), (1000, 513)]
# (the raw + mix path writes every voice's output as well: 1 GB for 1.4 M voices x 96 frames -- it runs the rest)
EXACT_CASES = [(p, N, F) for p in MIX_PATHS for N, F in EXACT_NF if p != "raw" or N * F <= 1 << 24]


@pytest.mark.gpu
@pytest.mark.parametrize("path,N,F", EXACT_CASES)
def test_xvoice_mix_exact(st, ctx, oracle, path, N, F):
    """Dyadic voices (see _dyadic_voices): the mix must equal the exact sum of the oracle's per-voice outputs, whole and
    as a split run (32 + rest).  A dropped, doubled or mistimed voice changes it by an exact, nonzero amount."""
    s0, prm = _dyadic_voices(N, F)
    S, _, sa = _contrib_sums(oracle, s0, prm, F)
    mix, state = _mix_device(st, ctx, s0, prm, F, path)
    assert np.array_equal(state.view(np.uint32), sa.view(np.uint32))
    bad = np.argwhere(mix.astype(np.float64) != S)
    assert bad.size == 0, (len(bad), [(int(c), int(t), float(mix[c, t]), float(S[c, t])) for c, t in bad[:6]])
    if F > 32:
        mix2, state2 = _mix_device(st, ctx, s0, prm, F, path, split=True)
        assert np.array_equal(mix2.astype(np.float64), S)
        assert np.array_equal(state2.view(np.uint32), sa.view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("gen", [1, 0], ids=["mix2", "mix1"])
@pytest.mark.parametrize("bus_mode", [1, 2])
@pytest.mark.parametrize("N,F", [(257, 96), (148 * 4 * 128 + 333, 64)])
def test_xvoice_mix_exact_fused_bus(st, ctx, oracle, gen, bus_mode, N, F):
    """The mix exchanged in the render launch (cproc_cuda_bus_attach, world 1, float sum): three consecutive blocks of
    dyadic voices, each mix equal to the exact sum; mode 2 completes the last exchange in bus_flush."""
    s0, prm = _dyadic_voices(N, 3 * F)
    sums, sa = [], s0.copy()
    for _ in range(3):
        S, _, sa = _contrib_sums(oracle, sa, prm, F)
        sums.append(S)
    ctx.set_option("xvoice_mix2", gen)
    b = ctx.batch(st.XVOICE, N)
    bus = st.Bus(ctx, 2 * F, 1, 0)
    d_mix = [ctx.dev_alloc(8 * F) for _ in range(3)]
    try:
        b.upload_state(s0.view(np.uint32).reshape(N, 5)); b.upload_param(prm.view(np.uint32).reshape(N, 8))
        bus.attach(b, bus_mode)
        for k in range(3):
            b.run_dev(F, mix=d_mix[k])
        bus.flush()
        ctx.sync()
        assert bus.status() == 0
        for k in range(3):
            mix = np.zeros((2, F), np.float32)
            ctx.d2h(mix, d_mix[k])
            assert np.array_equal(mix.astype(np.float64), sums[k]), k
        assert np.array_equal(b.download_state().view(np.uint32), sa.view(np.uint32).reshape(N, 5))
        bus.detach(b)
    finally:
        for p in d_mix:
            ctx.dev_free(p)
        bus.destroy(); b.free()
        ctx.set_option("xvoice_mix2", 1)
