"""Pin the oracle (oracle/cproc_oracle.c) against the reference's own code
compiled unmodified (oracle/_ref/libref.so) and against the regression anchors
recorded in SURVEY.md section 8c.  CPU only."""
import numpy as np
import pytest

from oracle import pyoracle as po

rng = np.random.default_rng(1234)


def test_struct_sizes(ref):
    # SURVEY 8c: sizeof(acc_state)=4, edge_state=8, acc_input=4, acc_config=0, acc_param=0
    assert [ref.sizeof(i) for i in range(7)] == [4, 4, 0, 0, 8, 4, 4]
    assert [ref.pdm_sizeof(k) for k in (1, 2, 3, 4)] == [4, 8, 12, 16]
    assert ref.synth_sizeof(0) == 8 and ref.synth_sizeof(1) == 1024


def test_test_cproc_anchor(ref, oracle):
    """linux/test_cproc.c graph: inputs 0,1,1,0,0,1,0,1,1,1,0 -> n2.out = 0,1,1,2,2,3,4,5,5,5,6.
    The reference keeps its state in function statics, so load a private copy."""
    r = ref.private_copy()
    seq = [0, 1, 1, 0, 0, 1, 0, 1, 1, 1, 0]
    got = [r.test_cproc_tick(x, 1) for x in seq]
    assert [g[0] for g in got] == [2] * len(seq)          # cproc_output(2, ...)
    assert [g[1] for g in got] == [0, 1, 1, 2, 2, 3, 4, 5, 5, 5, 6]
    # masked ticks (g&1 == 0) leave the graph untouched but still report n2.out
    assert r.test_cproc_tick(1, 0)[1] == 6
    assert r.test_cproc_tick(1, 2)[1] == 6
    assert r.test_cproc_tick(1, 3)[1] == 7
    # the oracle's table form of the same graph, same sequence
    full = np.array(seq + [1, 1, 1], np.uint32)[None, :]
    ch = np.array([1] * len(seq) + [0, 2, 3], np.uint32)[None, :]
    st = np.zeros((1, 3), np.uint32)
    out = oracle.graph_run(po.GRAPH_TEST_CPROC, 1, 1, st, 1, full.shape[1], full, ch)
    assert out[0].tolist() == [0, 1, 1, 2, 2, 3, 4, 5, 5, 5, 6, 6, 6, 7]


@pytest.mark.parametrize("rows", [po.GRAPH_TEST_CPROC, po.GRAPH_BP5,
                                  [(po.NODE_ACC, -1, 1), (po.NODE_ACC, -2, 2), (po.NODE_EDGE, 1, 4), (po.NODE_ACC, 2, 3)]])
def test_graph_oracle_vs_ref(ref, oracle, rows):
    N, F = 37, 211
    n_in = max(1, max(-s for _, s, _ in rows))
    inp = rng.integers(0, 3, (N, n_in, F), dtype=np.uint32)
    inp[::5] = rng.integers(0, 2**32, inp[::5].shape, dtype=np.uint32)
    changed = rng.integers(0, 8, (N, F), dtype=np.uint32)
    sw = sum(2 if t == po.NODE_EDGE else 1 for t, _, _ in rows)
    s0 = rng.integers(0, 2**32, (N, sw), dtype=np.uint32)
    for ch in (None, changed):
        sa, sb = s0.copy(), s0.copy()
        a = oracle.graph_run(rows, n_in, len(rows) - 1, sa, N, F, inp, ch)
        b = ref.graph_run(rows, n_in, len(rows) - 1, sb, N, F, inp, ch)
        assert np.array_equal(a, b) and np.array_equal(sa, sb)


@pytest.mark.parametrize("order", [1, 2, 3, 4])
def test_pdm_kat_and_ref(ref, oracle, order):
    # SURVEY 8c anchor: pdm*_update(0x60000000, sh=24, dither=0) -> 0, 96, 96, ...
    st = np.zeros((1, order), np.uint32)
    out = oracle.pdm_run(order, st, 1, 8, None, np.array([0x60000000], np.uint32), 24, None)
    assert out[0, 0] == 0
    if order == 1:
        assert out[0, 1:].tolist() == [96] * 7
    N, F = 19, 1000
    for sh in (24, 31, 16, 28):
        inp = rng.integers(0, 2**32, (N, F), dtype=np.uint32)
        dith = rng.integers(0, 2**10, F, dtype=np.uint32)
        s0 = rng.integers(0, 2**32, (N, order), dtype=np.uint32)
        sa, sb = s0.copy(), s0.copy()
        a = oracle.pdm_run(order, sa, N, F, inp, None, sh, dith)
        b = ref.pdm_run(order, sb, N, F, inp, None, sh, dith)
        assert np.array_equal(a, b) and np.array_equal(sa, sb)
        cst = rng.integers(0x40000000, 0xC0000000, N, dtype=np.uint32)
        a = oracle.pdm_run(order, sa, N, F, None, cst, sh, None)
        b = ref.pdm_run(order, sb, N, F, None, cst, sh, None)
        assert np.array_equal(a, b) and np.array_equal(sa, sb)


@pytest.mark.parametrize("order,bank", [(2, 3), (1, 1), (3, 2), (4, 5), (2, 64)])
def test_pdm_v2_oracle_vs_ref(ref, oracle, order, bank):
    """v2 ISR restatement around the real pdmK_update (ref) vs the oracle."""
    N, F, ctl = 23, 3000, 8
    nb = (N + bank - 1) // bank
    chan0 = rng.integers(0, 2**32, (N, 5 + order), dtype=np.uint32)
    prng0 = rng.integers(1, 2**32, nb, dtype=np.uint32)
    n_rows = F // (1 << ctl) + 2
    sp = po.pdm_setpoints(N, n_rows)
    for count0, setp, dext in ((0, sp, None), (77, None, None), (255, sp, rng.integers(0, 2**32, (nb, F), dtype=np.uint32))):
        ca, cb, pa, pb = chan0.copy(), chan0.copy(), prng0.copy(), prng0.copy()
        da, na = oracle.pdm_v2_run(ca, order, N, bank, pa, dext, 0x3FF, count0, ctl, 24, setp, F)
        db, nb_ = ref.pdm_v2_run(cb, order, N, bank, pb, dext, 0x3FF, count0, ctl, 24, setp, F)
        assert np.array_equal(da, db) and np.array_equal(ca, cb) and np.array_equal(pa, pb) and na == nb_
        assert na == (count0 + F) % (1 << ctl)


@pytest.mark.parametrize("count0,with_setpoints", [(0, True), (1234, True), (4095, False), (0, False)])
def test_pdm_v2_oracle_vs_the_firmware_isr(ref, oracle, count0, with_setpoints):
    """The REAL stm32f103/mod_pdm_pwm.c + mod_controlrate.c, compiled against a hosted hardware stand-in
    (oracle/ref/ref_v2_isr.c): TIM3 ISR called once per tick, duty captured at hw_multi_pwm_duty().  The oracle's
    v2 channel (glide, PDM_COPY_LINE at the control boundary, pdm_update_line, dither & 0x3FF, out_shift 24,
    the divider) must agree on every duty byte and on the whole final state over 5+ control periods."""
    nb, size, L = ref.v2_isr_config()
    assert (nb, size, L) == (3, 28, 12)                         # PDM_FOR_CHANNELS c(0) c(1) c(2); struct channel; CONTROL_DIV_LOG
    F = 5 * 4096 + 777
    chan0 = rng.integers(0, 2**32, (nb, 7), dtype=np.uint32)
    prng0 = int(rng.integers(1, 2**32))
    sp = rng.integers(0x40000000, 0xC0000000, (F // 4096 + 2, nb), dtype=np.uint32) if with_setpoints else None
    ca, cb = chan0.copy(), chan0.copy()
    pa = np.array([prng0], np.uint32)
    da, na = oracle.pdm_v2_run(ca, 2, nb, 3, pa, None, 0x3FF, count0, L, 24, sp, F)
    db, pb, nb_ = ref.v2_isr_run(cb, prng0, count0, sp, F)
    assert np.array_equal(da, db)
    assert np.array_equal(ca, cb) and int(pa[0]) == pb and na == nb_ == (count0 + F) % 4096


def test_word_clock_oracle_vs_ref(ref, oracle):
    """linux/clock.c:108-120 compiled from the reference (the loop only; JACK glue excluded) vs the restatement,
    two consecutive blocks; the MIDI clock bytes leave at the samples where the polarity turns 1."""
    hp = np.array([1, 2, 3, 8, 62, 500, 0, 7], np.int32)
    N, F = len(hp), 3000
    s0 = np.zeros((N, 2), np.int32); s0[:, 0] = rng.integers(0, 100, N); s0[:, 1] = rng.integers(0, 2, N)
    sa, sb = s0.copy(), s0.copy()
    for blk in range(2):
        prev = int(sb[4, 1])
        a = oracle.word_clock_run(sa, hp, N, F)
        b, ev = ref.word_clock_run(sb, hp, N, F, ev_clock=4)
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)) and np.array_equal(sa, sb)
        pol = np.concatenate([[prev], a[4].astype(np.int64)])
        assert np.array_equal(ev, np.flatnonzero((pol[1:] == 1) & (pol[:-1] != 1)))


def test_pwm_update_oracle_vs_ref(ref, oracle):
    """stm32f103/mod_pdm.c:159-175 (pwm_update and its globals) compiled from the reference vs the restatement."""
    N, F = 64, 5000
    ph = rng.integers(0, 1 << 24, N, dtype=np.uint32); sp = rng.integers(0, 1 << 16, N, dtype=np.uint32)
    sp[0] = 256 * 13                                         # the firmware's default speed (:160)
    pa, pb = ph.copy(), ph.copy()
    a = oracle.pwm_run(pa, sp.copy(), N, F)
    b = ref.pwm_run(pb, sp.copy(), N, F)
    assert np.array_equal(a, b) and np.array_equal(pa, pb)


def test_v2_mean_tracks_setpoint(oracle):
    """Domain property: after the glide settles the mean duty equals setpoint/2^24."""
    N, F = 8, 1 << 16
    chan = np.zeros((N, 7), np.uint32)
    sp = np.linspace(0x40000000, 0xC0000000, N).astype(np.uint32)
    chan[:, 0] = sp
    prng = np.arange(1, 4, dtype=np.uint32)
    duty, _ = oracle.pdm_v2_run(chan, 2, N, 3, prng, None, 0x3FF, 0, 12, 24, None, F)
    tail = duty[:, -(1 << 14):].astype(np.float64).mean(axis=1)
    assert np.allclose(tail, sp / 2.0**24, atol=0.05)


def test_note_table(ref, oracle):
    golden12 = [594573364, 629928536, 667386036, 707070875, 749115497, 793660223,
                840853716, 890853479, 943826384, 999949221, 1059409296, 1122405051]
    assert ref.note_tab12().tolist() == golden12          # SURVEY a-9
    t = ref.note_table()
    assert t[69] == 39370533 and t[60] == 23409859 and t[0] == 731558
    assert [oracle.note_to_inc(n) for n in range(128)] == t.tolist()
    assert oracle.note_to_inc(128 + 69) == t[69]          # note & 127 (synth.c:119)


def test_synth_anchor(ref, oracle):
    # SURVEY 8c: notes 69,60,127,0 on -> first 8 saw-mix samples
    vec, voices = ref.synth_play([69, 60, 127, 0], 8)
    want = [0.0, float.fromhex("0x1.1abeap-6"), float.fromhex("-0x1.ca82bep-6"), float.fromhex("-0x1.5f883ap-7"),
            float.fromhex("0x1.abea1p-8"), float.fromhex("0x1.85b924p-6"), float.fromhex("-0x1.5f883ap-6"),
            float.fromhex("-0x1.132662p-8")]
    assert vec.tolist() == want
    v = np.zeros((64, 2), np.uint32)
    v[:4, 0] = [oracle.note_to_inc(n) for n in (69, 60, 127, 0)]
    _, ovec = oracle.voice_bank_run(v, 64, 64, po.MIX_SAW, 8)
    assert ovec[0].tolist() == want
    assert np.array_equal(v, voices)


@pytest.mark.parametrize("mode", [po.MIX_SAW, po.MIX_SQUARE])
def test_voice_bank_oracle_vs_ref(ref, oracle, mode):
    n_synth, F = 9, 300
    v0 = np.zeros((n_synth * 64, 2), np.uint32)
    v0[:, 1] = rng.integers(0, 2**32, n_synth * 64, dtype=np.uint32)
    notes = rng.integers(0, 128, n_synth * 64)
    tab = ref.note_table()
    v0[:, 0] = np.where(rng.random(n_synth * 64) < 0.7, tab[notes], 0)
    v0[64:128, 0] = 0x7FFFFFFF        # loud: forces int wrap in the saw sum
    va, vb = v0.copy(), v0.copy()
    _, a = oracle.voice_bank_run(va, n_synth * 64, 64, mode, F)
    b = ref.voice_bank_run(vb, n_synth, mode, F)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32)) and np.array_equal(va, vb)


def test_square_grain_oracle_vs_ref(ref, oracle):
    N, F = 33, 257
    inp = rng.uniform(-1, 1, (N, F)).astype(np.float32)
    th = rng.uniform(0.05, 0.5, N).astype(np.float32)
    th[0] = 0.0
    st0 = rng.choice(np.array([0.0, 0.5, -0.5], np.float32), N)
    sa, sb = st0.copy(), st0.copy()
    a = oracle.square_grain_run(sa, th, N, F, inp)
    b = ref.square_grain_run(sb, th, N, F, inp)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32)) and np.array_equal(sa, sb)
    # in-place (Pd aliases in/out): same answer
    io = inp.copy()
    sc = st0.copy()
    ref.square_grain_run(sc, th, N, F, io, io)
    assert np.array_equal(io, a) and np.array_equal(sc, sa)
    assert set(np.unique(a)) <= {0.0, 0.5, -0.5}


def test_v1_carry_properties(oracle):
    """v1 is ARM asm in the reference (mod_pdm.c:214-244): check the restatement
    against an independent 64-bit formulation of add-with-carry."""
    N, F, bank = 11, 500, 2
    nb = (N + bank - 1) // bank
    ch = np.zeros((N, 2), np.uint32)
    ch[:, 0] = rng.integers(0, 2**32, N, dtype=np.uint32)
    ch[:, 1] = rng.integers(0, 2**32, N, dtype=np.uint32)
    dext = rng.integers(0, 2**32, (nb, F), dtype=np.uint32)
    c0 = ch.copy()
    bits = oracle.pdm_v1_run(ch, N, bank, None, dext, 0x0FFFFFFF, F)
    acc = c0[:, 1].astype(np.uint64)
    for t in range(F):
        d = (dext[np.arange(N) // bank, t] & 0x0FFFFFFF).astype(np.uint64)
        x = (c0[:, 0].astype(np.uint64) + d) & 0xFFFFFFFF
        s = acc + x
        assert np.array_equal(bits[:, t], (s >> 32).astype(np.uint8))
        acc = s & 0xFFFFFFFF
    assert np.array_equal(ch[:, 1], acc.astype(np.uint32))
    # pulse density == setpoint / 2^32 without dither
    ch2 = np.zeros((1, 2), np.uint32); ch2[0, 0] = 0x60000000
    b2 = oracle.pdm_v1_run(ch2, 1, 1, None, np.zeros((1, 4096), np.uint32), 0, 4096)
    assert b2.sum() == 4096 * 3 // 8


def test_xorshift_and_pwm(oracle):
    r, s = oracle.xorshift32(1)
    assert r == s == 270369               # Marsaglia xorshift32 (13,17,5), x0 = 1
    r, s = oracle.xorshift32(2463534242)
    assert r == 723471715
    ph = np.array([0, 0x123456], np.uint32); sp = np.array([256 * 13, 5000], np.uint32)
    duty = oracle.pwm_run(ph, sp, 2, 1000)
    p = [0, 0x123456]
    for t in range(1000):
        for i in range(2):
            assert duty[i, t] == (p[i] >> 16)
            p[i] = (p[i] + int(sp[i]) + (p[i] >> 9)) & 0xFFFFFF
    assert ph.tolist() == p


def test_pixi_lfo_bank_vs_acc(ref, oracle):
    """a-20: stm32f103/pixi.c:279,282-285 compiled from the reference against the oracle's acc under a 12-bit mask."""
    rng = np.random.default_rng(3)
    for adc0 in [0, 37, 2048, 4095, 51234]:
        dac = rng.integers(0, 0x1000, 12).astype(np.uint16)
        st = dac.astype(np.uint32).reshape(12, 1).copy()
        trace = ref.pixi_lfo_run(dac, adc0, 500)
        inp = np.full((12, 1, 500), adc0 >> 5, np.uint32)
        out = oracle.graph_run([(po.NODE_ACC, -1, 0xFFFFFFFF)], 1, 0, st, 12, 500, inp)
        assert np.array_equal((out & 0xFFF).T, trace.astype(np.uint32))
        assert np.array_equal(st[:, 0] & 0xFFF, dac.astype(np.uint32))


@pytest.mark.parametrize("n_ch,pin0", [(2, 0), (3, 5), (8, 2), (16, 16), (32, 0)])
def test_v1_restatement_against_the_arm_instruction_model(oracle, n_ch, pin0):
    """SURVEY 8 a-14 (ARM inline asm, no ARM toolchain here: restated).  Two independent readings of `adds` + `rrx`
    (mod_pdm.c:214-244) must agree: the add-with-carry restatement behind every v1 parity test (carry = a < x, bits laid out
    per channel over time) and oracle/arm_v1_model.c (AddWithCarry's 33-bit sum, RRX through the C flag, ONE shift register
    per tick over the MCU's channels and the GPIO alignment shift of pdm_update, :254-275)."""
    rng = np.random.default_rng(n_ch)
    F = 2000
    ch = np.zeros((n_ch, 2), np.uint32)
    ch[:, 0] = rng.integers(0, 2**32, n_ch, dtype=np.uint32)
    ch[0, 0] = 0xFFFFFFFF                                       # setpoint + dither wraps
    ch[:, 1] = rng.integers(0, 2**32, n_ch, dtype=np.uint32)
    seed = 2463534242
    a = ch.copy()
    gpio, rng1 = oracle.arm_v1_mcu_run(a, pin0, seed, 0x0FFFFFFF, F)
    b = ch.copy()
    prng = np.array([seed], np.uint32)
    bits = oracle.pdm_v1_run(b, n_ch, n_ch, prng, None, 0x0FFFFFFF, F)     # one bank = the MCU's channels, one dither word per tick
    assert np.array_equal(a, b) and rng1 == int(prng[0])
    for c in range(n_ch):
        assert np.array_equal((gpio >> np.uint32(pin0 + c)) & 1, bits[c].astype(np.uint32)), c
    if pin0 + n_ch < 32:
        assert not np.any(gpio >> np.uint32(pin0 + n_ch))       # nothing above the last channel's pin
