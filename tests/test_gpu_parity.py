"""GPU parity: every CUDA path, called through the C-ABI (ctypes over
libcproc_cuda.so), against the CPU oracle on the same seeded inputs.
Integer / index / exactly-representable float work is compared bit for bit."""
import numpy as np
import pytest

from oracle import pyoracle as po

pytestmark = pytest.mark.gpu

rng = np.random.default_rng(20261018)


@pytest.fixture(scope="module")
def st():
    import synth_tools_b200 as st_
    return st_


@pytest.fixture(scope="module")
def ctx(st):
    c = st.Context(0)
    yield c
    c.close()


def tiled16_to_planar(a, N, F):
    return a.reshape(F // 16, N, 16).transpose(1, 0, 2).reshape(N, F)


def pack_bits(bits):
    """[N][F] 0/1 -> uint32 words [N][F/32], sample t at bit t&31."""
    N, F = bits.shape
    return np.packbits(bits.reshape(N, F // 32, 32), axis=2, bitorder="little").view("<u4").reshape(N, F // 32)


# --------------------------------------------------------------------------- v2
def _v2_case(st, ctx, oracle, order, bank, N, F, layout, count0, use_setp, use_dext, ctl=6, opts=None, split=None):
    nb = (N + bank - 1) // bank
    chan0 = rng.integers(0, 2**32, (N, 5 + order), dtype=np.uint32)
    prng0 = rng.integers(1, 2**32, nb, dtype=np.uint32)
    n_rows = F // (1 << ctl) + 2
    sp = po.pdm_setpoints(N, n_rows) if use_setp else None
    dext = rng.integers(0, 2**32, (nb, F), dtype=np.uint32) if use_dext else None
    ca, pa = chan0.copy(), prng0.copy()
    want, want_cnt = oracle.pdm_v2_run(ca, order, N, bank, pa, dext, 0x3FF, count0, ctl, 24, sp, F)
    for k, v in (opts or {}).items():
        ctx.set_option(k, v)
    b = ctx.batch(st.PDM_V2, N, order=order, bank_size=bank, ctl_div_log=ctl, out_shift=24, dither_mask=0x3FF, layout=layout)
    try:
        b.upload_state(chan0)
        b.upload_bank(prng0, count0)
        if split is None:
            out = np.zeros(N * F, np.uint8)
            b.run(F, in2=dext, ctl=sp, out=out)
            got = tiled16_to_planar(out, N, F) if layout == st.TILED else out.reshape(F, N).T if layout == st.INTERLEAVED else out.reshape(N, F)
        else:
            # the same render in several calls must continue seamlessly (checkpoint semantics)
            assert dext is None
            got = np.zeros((N, F), np.uint8)
            t = 0
            row = 0
            cnt = count0
            for f in split:
                o = np.zeros(N * f, np.uint8)
                first = 0 if cnt == 0 else (1 << ctl) - cnt
                rows = 1 + (f - first - 1) // (1 << ctl) if f > first else 0
                b.run(f, ctl=None if sp is None else np.ascontiguousarray(sp[row:row + max(rows, 1)]), out=o)
                got[:, t:t + f] = tiled16_to_planar(o, N, f) if layout == st.TILED else o.reshape(N, f)
                t += f
                row += rows
                cnt = (cnt + f) % (1 << ctl)
            assert t == F
        assert np.array_equal(got, want)
        assert np.array_equal(b.download_state(), ca)
        p, c = b.download_bank()
        assert c == want_cnt
        if not use_dext:
            assert np.array_equal(p, pa)
    finally:
        b.free()
        for k, v in V2_DEFAULTS.items():
            ctx.set_option(k, v)


V2_DEFAULTS = {"pdm_tpb": 2, "pdm_block": 64, "pdm_ws": 1, "pdm_tlog": 7, "pdm_ctas_per_sm": 4,
               "pdm_slice_batches": 64, "pdm_planar_bulk": 2}


@pytest.mark.parametrize("order", [1, 2, 3, 4])
@pytest.mark.parametrize("bank", [1, 2, 3, 4, 7])
def test_pdm_v2_orders_banks(st, ctx, oracle, order, bank):
    """F not a whole dither batch: the plain thread-per-bank / thread-per-channel kernels."""
    _v2_case(st, ctx, oracle, order, bank, N=203, F=48, layout=st.TILED, count0=0, use_setp=True, use_dext=False, ctl=4)
    _v2_case(st, ctx, oracle, order, bank, N=203, F=512, layout=st.TILED, count0=0, use_setp=True, use_dext=False)


@pytest.mark.parametrize("layout", ["PLANAR", "TILED"])
@pytest.mark.parametrize("tpb,ws", [(0, 0), (1, 0), (1, 1)])
@pytest.mark.parametrize("blk", [32, 128])
def test_pdm_v2_layouts_and_mappings(st, ctx, oracle, layout, tpb, ws, blk):
    _v2_case(st, ctx, oracle, 2, 3, N=1000, F=1024, layout=getattr(st, layout), count0=16, use_setp=True,
             use_dext=False, opts={"pdm_tpb": tpb, "pdm_block": blk, "pdm_ws": ws})


@pytest.mark.parametrize("order", [1, 2, 3, 4])
@pytest.mark.parametrize("bank", [1, 2, 3, 4, 7, 33])
@pytest.mark.parametrize("planar_bulk", [0, 2])
def test_pdm_v2_ws4_planar_paths(st, ctx, oracle, order, bank, planar_bulk):
    """PLANAR duty rows out of k_pdm_v2_ws4 both ways -- scattered 16-byte stores, tensor-TMA boxes per warp (64-tick batches) --
    over ragged channel counts, straddling banks and a ragged last slice."""
    _v2_case(st, ctx, oracle, order, bank, N=2999, F=128 * 7, layout=st.PLANAR, count0=128, use_setp=True,
             use_dext=False, ctl=8, opts={"pdm_ctas_per_sm": 1, "pdm_slice_batches": 4, "pdm_planar_bulk": planar_bulk})


@pytest.mark.parametrize("order", [1, 2, 3, 4])
@pytest.mark.parametrize("bank", [1, 2, 3, 4, 5, 7, 33])
@pytest.mark.parametrize("layout", ["PLANAR", "TILED"])
def test_pdm_v2_ws4_orders_banks(st, ctx, oracle, order, bank, layout):
    """k_pdm_v2_ws4 for every order and bank sizes on both sides of the aligned / unaligned split (banks of 1..4 are a
    consumer warp each; larger banks straddle groups of 128 channels), ragged channel count, the counter starting
    inside a control period (3 batches of 64 into a period of 4)."""
    _v2_case(st, ctx, oracle, order, bank, N=2999, F=64 * 12, layout=getattr(st, layout), count0=192, use_setp=True,
             use_dext=False, ctl=8, opts={"pdm_ctas_per_sm": 1, "pdm_slice_batches": 4})


@pytest.mark.parametrize("order", [1, 2, 3, 4])
@pytest.mark.parametrize("bank", [1, 2, 3, 4, 7, 33])
def test_pdm_v2_ws4_interleaved_tiles(st, ctx, oracle, order, bank):
    """INTERLEAVED duty [tick][ch] (the order the ISR emits) through k_pdm_v2_ws4's shared-memory tiles: every order, aligned and
    straddling banks, slices of two batches with a ragged last slice, the counter starting inside a control period; then a channel
    count that is not whole sixteens, which must take the conformance kernel and give the same bytes."""
    _v2_case(st, ctx, oracle, order, bank, N=16 * 191, F=128 * 7, layout=st.INTERLEAVED, count0=128, use_setp=True,
             use_dext=False, ctl=8, opts={"pdm_ctas_per_sm": 1, "pdm_slice_batches": 4})
    if order == 2:
        _v2_case(st, ctx, oracle, order, bank, N=32 * 95 + 5, F=128 * 3, layout=st.INTERLEAVED, count0=0, use_setp=True, use_dext=False, ctl=7)
        _v2_case(st, ctx, oracle, order, bank, N=32 * 20, F=128 * 40, layout=st.INTERLEAVED, count0=0, use_setp=True, use_dext=False, ctl=9,
                 split=None, opts={"pdm_ctas_per_sm": 4, "pdm_slice_batches": 64})


@pytest.mark.parametrize("tlog", [6, 7])
@pytest.mark.parametrize("layout", ["PLANAR", "TILED"])
@pytest.mark.parametrize("order,bank", [(2, 3), (3, 2), (4, 9), (1, 1)])
def test_pdm_v2_ws4_batches_and_schedule(st, ctx, oracle, tlog, layout, order, bank):
    """Both batch lengths; dynamic (group, slice) schedule: more groups than persistent blocks (148 x 1), slices of 512
    ticks with a ragged last slice, setpoint rows latched inside slices, the counter starting inside a control period."""
    _v2_case(st, ctx, oracle, order, bank, N=32 * bank * 150 + 5 if bank <= 4 else 128 * 150 + 5, F=256 * 9, layout=getattr(st, layout), count0=256,
             use_setp=True, use_dext=False, ctl=9, opts={"pdm_tlog": tlog, "pdm_ctas_per_sm": 1, "pdm_slice_batches": 8})


@pytest.mark.parametrize("mask", [0x3FF, 0xFFFF, 0x00FFFFFF, 0, 0x01000001])
def test_pdm_v2_dither_masks(st, ctx, oracle, mask):
    """Dither below bit 24 takes the one-LOP3 quantiser step; a mask that reaches the output byte takes the literal form."""
    N, F, bank = 777, 64 * 6, 3
    chan0 = rng.integers(0, 2**32, (N, 7), dtype=np.uint32)
    prng0 = rng.integers(1, 2**32, (N + bank - 1) // bank, dtype=np.uint32)
    sp = po.pdm_setpoints(N, F // 64 + 2)
    ca, pa = chan0.copy(), prng0.copy()
    want, _ = oracle.pdm_v2_run(ca, 2, N, bank, pa, None, mask, 0, 6, 24, sp, F)
    b = ctx.batch(st.PDM_V2, N, order=2, bank_size=bank, ctl_div_log=6, out_shift=24, dither_mask=mask, layout=st.PLANAR)
    b.upload_state(chan0); b.upload_bank(prng0, 0)
    out = np.zeros((N, F), np.uint8)
    b.run(F, ctl=sp, out=out)
    assert np.array_equal(out, want) and np.array_equal(b.download_state(), ca) and np.array_equal(b.download_bank()[0], pa)
    b.free()


@pytest.mark.parametrize("ctas,slice_b,F", [(4, 2, 64 * 8), (4, 3, 64 * 8), (2, 4, 64 * 8), (4, 64, 64 * 128)])
def test_pdm_v2_ws4_c2_shape(st, ctx, oracle, ctas, slice_b, F):
    """The C2 channel count (65,536 channels = 683 groups for 148 x ctas blocks)."""
    _v2_case(st, ctx, oracle, 2, 3, N=65536, F=F, layout=st.TILED, count0=0, use_setp=True, use_dext=False, ctl=7,
             opts={"pdm_ctas_per_sm": ctas, "pdm_slice_batches": slice_b})


@pytest.mark.parametrize("slice_b,F,bulk", [(4, 64 * 9, 2), (4, 64 * 16, 2), (8, 64 * 22, 2), (4, 64 * 10, 2), (12, 64 * 38, 2),
                                             (3, 64 * 16, 2), (4, 64 * 16, 0)])
def test_pdm_v2_ws4_planar_rows(st, ctx, oracle, slice_b, F, bulk):
    """PLANAR duty rows: tensor-TMA boxes of 128 ticks x 32 channels (whole boxes only: F % 128 == 0, else scattered
    16-byte stores), odd slice lengths rounded to whole boxes, ragged channel count (rows clipped by the tensor map)."""
    _v2_case(st, ctx, oracle, 2, 3, N=96 * 150 + 5, F=F, layout=st.PLANAR, count0=64, use_setp=True, use_dext=False, ctl=8,
             opts={"pdm_ctas_per_sm": 1, "pdm_slice_batches": slice_b, "pdm_planar_bulk": bulk})


def test_pdm_v2_ws4_split_runs(st, ctx, oracle):
    """Consecutive launches (work counter, epochs, progress words and the double-buffered generator state are reused)."""
    _v2_case(st, ctx, oracle, 2, 3, N=96 * 150 + 5, F=64 * 22, layout=st.TILED, count0=0, use_setp=True, use_dext=False,
             ctl=7, split=[64 * 5, 64 * 4, 64 * 9, 64 * 4], opts={"pdm_ctas_per_sm": 1, "pdm_slice_batches": 2})
    _v2_case(st, ctx, oracle, 3, 7, N=1000, F=64 * 9, layout=st.PLANAR, count0=0, use_setp=True, use_dext=False,
             ctl=6, split=[64, 16, 48, 64 * 5, 64 * 2])


@pytest.mark.parametrize("N,bank,layout,F", [(1 << 20, 3, "INTERLEAVED", 48), (1 << 20, 7, "TILED", 64), (1 << 20, 4096, "TILED", 64),
                                             ((1 << 20) + 11, 4096, "PLANAR", 40), (1 << 20, 1 << 20, "TILED", 64),
                                             (400000, 400000, "INTERLEAVED", 32), (1 << 20, 7, "TILED", 48)])
def test_pdm_v2_banks_wider_than_a_block(st, ctx, oracle, N, bank, layout, F):
    """A bank that spans blocks (or the whole batch: one dither word for every channel) is replayed by every block
    that holds one of its channels; the generator state is double buffered so that no block sees another's
    write-back.  >= 1 Mi channels: more blocks than one resident wave.  Covers k_pdm_v2_any (INTERLEAVED, ragged F),
    the thread-per-channel kernel (F % 64 != 0) and k_pdm_v2_ws4 (unaligned groups)."""
    _v2_case(st, ctx, oracle, 2, bank, N=N, F=F, layout=getattr(st, layout), count0=0, use_setp=True, use_dext=False, ctl=5)


def test_pdm_v2_external_dither(st, ctx, oracle):
    _v2_case(st, ctx, oracle, 2, 3, N=100, F=256, layout=st.TILED, count0=0, use_setp=False, use_dext=True)
    _v2_case(st, ctx, oracle, 3, 2, N=64, F=160, layout=st.PLANAR, count0=32, use_setp=True, use_dext=True)


def test_pdm_v2_ragged(st, ctx, oracle):
    """F / count not multiples of 16, single channel, bank larger than N."""
    _v2_case(st, ctx, oracle, 2, 3, N=10, F=77, layout=st.PLANAR, count0=5, use_setp=True, use_dext=False)
    _v2_case(st, ctx, oracle, 2, 3, N=1, F=1, layout=st.PLANAR, count0=63, use_setp=True, use_dext=False)
    _v2_case(st, ctx, oracle, 4, 64, N=5, F=100, layout=st.PLANAR, count0=0, use_setp=False, use_dext=False)
    _v2_case(st, ctx, oracle, 2, 3, N=33, F=130, layout=st.PLANAR, count0=3, use_setp=False, use_dext=True)


def test_pdm_v2_split_runs(st, ctx, oracle):
    _v2_case(st, ctx, oracle, 2, 3, N=96, F=640, layout=st.TILED, count0=0, use_setp=True, use_dext=False, split=[64, 16, 320, 240])
    _v2_case(st, ctx, oracle, 2, 3, N=50, F=200, layout=st.PLANAR, count0=7, use_setp=True, use_dext=False, split=[1, 9, 100, 90])


def test_pdm_v2_reference_config(st, ctx, oracle):
    """The firmware configuration itself: 3 channels, PDM_ORDER 2, control divider
    4096, dither mask 0x3FF, zero-initialised state, setpoints as pdm_init
    (mod_pdm_pwm.c:147-161)."""
    N, F = 3, 3 * 4096
    chan = np.zeros((N, 7), np.uint32)
    chan[:, 0] = [2000000000, 0x40000000, 0x40000000]
    prng = np.array([2463534242], np.uint32)
    ca, pa = chan.copy(), prng.copy()
    want, _ = oracle.pdm_v2_run(ca, 2, N, 3, pa, None, 0x3FF, 0, 12, 24, None, F)
    b = ctx.batch(st.PDM_V2, N, order=2, bank_size=3, ctl_div_log=12)
    b.upload_state(chan); b.upload_bank(prng, 0)
    out = np.zeros((N, F), np.uint8)
    b.run(F, out=out)
    assert np.array_equal(out, want) and np.array_equal(b.download_state(), ca)
    b.free()


def test_pdm_v2_errors(st, ctx):
    with pytest.raises(st.CprocCudaError):
        ctx.batch(st.PDM_V2, 8, order=5)
    with pytest.raises(st.CprocCudaError):
        ctx.batch(st.PDM_V2, 8, order=2, out_shift=16)
    b = ctx.batch(st.PDM_V2, 8, order=2, bank_size=3, ctl_div_log=4)
    with pytest.raises(st.CprocCudaError):     # not enough setpoint rows for the boundaries crossed
        b.run(64, ctl=np.zeros((1, 8), np.uint32), out=np.zeros(8 * 64, np.uint8))
    with pytest.raises(st.CprocCudaError):     # TILED needs F % 16 == 0
        b.run(24, out=np.zeros(8 * 24, np.uint8), layout=st.TILED)
    with pytest.raises(st.CprocCudaError):
        b.run(16, out=None)
    b.run(0, out=np.zeros(1, np.uint8))        # empty run is a no-op
    b.free()


# --------------------------------------------------------------------------- v1
@pytest.mark.parametrize("bank,tpb,persist,N", [(1, 1, 2, 301), (2, 1, 2, 301), (2, 1, 0, 301), (2, 0, 0, 301), (3, 1, 1, 301),
                                               (4, 1, 0, 301), (9, 1, 2, 301), (2, 1, 2, 65536), (1, 1, 2, 32 * 700 + 3)])
@pytest.mark.parametrize("layout", ["PLANAR", "INTERLEAVED", "TILED"])
@pytest.mark.parametrize("chains", [1, 2])
def test_pdm_v1(st, ctx, oracle, bank, tpb, persist, N, layout, chains):
    ctx.set_option("pdm_v1_chains", chains)
    F = 512 if N != 65536 or layout == "TILED" else 480          # 480: not whole 128-tick groups -- the word-at-a-time path of PLANAR / INTERLEAVED
    nb = (N + bank - 1) // bank
    ch0 = rng.integers(0, 2**32, (N, 2), dtype=np.uint32)
    prng0 = rng.integers(1, 2**32, nb, dtype=np.uint32)
    ca, pa = ch0.copy(), prng0.copy()
    bits = oracle.pdm_v1_run(ca, N, bank, pa, None, 0x0FFFFFFF, F)
    want = pack_bits(bits)
    ctx.set_option("pdm_tpb", tpb)
    ctx.set_option("pdm_persist", persist)
    b = ctx.batch(st.PDM_V1, N, bank_size=bank, dither_mask=0x0FFFFFFF, layout=getattr(st, layout))
    b.upload_state(ch0); b.upload_bank(prng0)
    out = np.zeros(N * F // 32, np.uint32)
    b.run(F, out=out)
    if layout == "PLANAR":
        got = out.reshape(N, F // 32)
    elif layout == "INTERLEAVED":
        got = out.reshape(F // 32, N).T
    else:
        got = out.reshape(F // 128, N, 4).transpose(1, 0, 2).reshape(N, F // 32)
    assert np.array_equal(got, want)
    assert np.array_equal(b.download_state(), ca)
    assert np.array_equal(b.download_bank()[0], pa)
    b.free()
    ctx.set_option("pdm_tpb", 2)
    ctx.set_option("pdm_persist", 1)
    ctx.set_option("pdm_v1_chains", 2)


@pytest.mark.parametrize("N,bank,layout", [(1 << 20, 7, "TILED"), (1 << 20, 4096, "INTERLEAVED"), ((1 << 20) + 3, 1 << 20, "PLANAR"), (1 << 20, 3, "INTERLEAVED")])
def test_pdm_v1_banks_wider_than_a_block(st, ctx, oracle, N, bank, layout):
    """Thread-per-channel v1 kernel with a bank replayed by many blocks (>= 1 Mi channels: more than one resident wave):
    the generator state is double buffered, no block may see another's write-back."""
    F = 128
    nb = (N + bank - 1) // bank
    ch0 = rng.integers(0, 2**32, (N, 2), dtype=np.uint32)
    prng0 = rng.integers(1, 2**32, nb, dtype=np.uint32)
    ca, pa = ch0.copy(), prng0.copy()
    want = pack_bits(oracle.pdm_v1_run(ca, N, bank, pa, None, 0x0FFFFFFF, F))
    ctx.set_option("pdm_tpb", 0 if bank <= 4 else 1)
    b = ctx.batch(st.PDM_V1, N, bank_size=bank, dither_mask=0x0FFFFFFF, layout=getattr(st, layout))
    b.upload_state(ch0); b.upload_bank(prng0)
    out = np.zeros(N * F // 32, np.uint32)
    for _ in range(1):
        b.run(F, out=out)
    ctx.set_option("pdm_tpb", 2)
    got = out.reshape(N, F // 32) if layout == "PLANAR" else out.reshape(F // 32, N).T if layout == "INTERLEAVED" else \
        out.reshape(F // 128, N, 4).transpose(1, 0, 2).reshape(N, F // 32)
    assert np.array_equal(got, want)
    assert np.array_equal(b.download_state(), ca) and np.array_equal(b.download_bank()[0], pa)
    b.free()


def test_pdm_v1_external_dither_and_density(st, ctx, oracle):
    N, F, bank = 64, 1024, 2
    ch0 = np.zeros((N, 2), np.uint32)
    ch0[:, 0] = np.linspace(0x40000000, 0xC0000000, N).astype(np.uint32)
    dext = rng.integers(0, 2**32, (N // bank, F), dtype=np.uint32)
    ca = ch0.copy()
    want = pack_bits(oracle.pdm_v1_run(ca, N, bank, None, dext, 0x0FFFFFFF, F))
    b = ctx.batch(st.PDM_V1, N, bank_size=bank, dither_mask=0x0FFFFFFF)
    b.upload_state(ch0)
    out = np.zeros((N, F // 32), np.uint32)
    b.run(F, in2=dext, out=out)
    assert np.array_equal(out, want) and np.array_equal(b.download_state(), ca)
    # pulse density tracks setpoint / 2^32 (dither mean 2^27 adds 1/32)
    dens = np.unpackbits(out.view(np.uint8), axis=1).mean(axis=1)
    assert np.allclose(dens, ch0[:, 0] / 2.0**32 + 1 / 32, atol=0.02)
    with pytest.raises(st.CprocCudaError):
        b.run(48, out=out)
    b.free()


# --------------------------------------------------------------------- pdm raw, pwm
@pytest.mark.parametrize("order", [1, 2, 3, 4])
@pytest.mark.parametrize("layout,N,F", [("PLANAR", 130, 300), ("INTERLEAVED", 130, 300), ("INTERLEAVED", 132, 301), ("INTERLEAVED", 4 * 700, 64)])
def test_pdm_raw(st, ctx, oracle, order, layout, N, F):
    """PLANAR through the staging template; INTERLEAVED four instances per thread when the count allows (n % 4 == 0), else a thread each."""
    sh = 24
    s0 = rng.integers(0, 2**32, (N, order), dtype=np.uint32)
    inp = rng.integers(0, 2**32, (N, F), dtype=np.uint32)
    dith = rng.integers(0, 1024, F, dtype=np.uint32)
    cst = rng.integers(0x40000000, 0xC0000000, (N, 1), dtype=np.uint32)
    sa = s0.copy()
    want1 = oracle.pdm_run(order, sa, N, F, inp, None, sh, dith)
    want2 = oracle.pdm_run(order, sa, N, F, None, cst[:, 0].copy(), sh, None)
    b = ctx.batch(st.PDM, N, order=order, out_shift=sh, layout=getattr(st, layout))
    b.upload_state(s0); b.upload_param(cst)
    il = layout == "INTERLEAVED"
    out = np.zeros((F, N) if il else (N, F), np.uint32)
    b.run(F, inp=np.ascontiguousarray(inp.T) if il else inp, in2=dith, out=out)
    assert np.array_equal(out.T if il else out, want1)
    b.run(F, out=out)
    assert np.array_equal(out.T if il else out, want2)
    assert np.array_equal(b.download_state(), sa)
    b.free()


@pytest.mark.parametrize("N,F,layout", [(77, 512, "PLANAR"), (1000, 4096, "PLANAR"), (33, 48, "PLANAR"), (300, 1024, "TILED"),
                                        (65, 16, "TILED"), (50, 200, "INTERLEAVED")])
def test_pwm_layouts(st, ctx, oracle, N, F, layout):
    """pwm_update through the bulk-staged PLANAR kernel (four ticks per staged word), the TILED
    kernel and the scalar one; a second block continues from the device state."""
    ph0 = rng.integers(0, 1 << 24, (N, 1), dtype=np.uint32)
    sp = rng.integers(0, 1 << 16, (N, 1), dtype=np.uint32)
    pa = ph0[:, 0].copy()
    b = ctx.batch(st.PWM, N, layout=getattr(st, layout))
    b.upload_state(ph0); b.upload_param(sp)
    for _ in range(2):
        want = oracle.pwm_run(pa, sp[:, 0].copy(), N, F)
        out = np.zeros(N * F, np.uint8)
        b.run(F, out=out)
        got = tiled16_to_planar(out, N, F) if layout == "TILED" else (out.reshape(F, N).T if layout == "INTERLEAVED" else out.reshape(N, F))
        assert np.array_equal(got, want) and np.array_equal(b.download_state()[:, 0], pa)
    b.free()


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("N,F", [(130, 320), (33, 64), (1000, 1024), (70, 100), (5, 36)])
def test_planar_template_modes(st, ctx, oracle, mode, N, F):
    """pdm raw (with and without an input stream), one-pole and pwm through the scalar kernels (0), the
    per-lane bulk-copy template (1) and its tensor-TMA form (2): ragged instance counts and tiles."""
    ctx.set_option("planar_bulk", mode)
    try:
        for order in (1, 3):
            s0 = rng.integers(0, 2**32, (N, order), dtype=np.uint32)
            inp = rng.integers(0, 2**32, (N, F), dtype=np.uint32)
            dith = rng.integers(0, 1024, F, dtype=np.uint32)
            cst = rng.integers(0x40000000, 0xC0000000, (N, 1), dtype=np.uint32)
            for use_in in (True, False):
                sa = s0.copy()
                want = oracle.pdm_run(order, sa, N, F, inp if use_in else None, cst[:, 0].copy(), 24, dith)
                b = ctx.batch(st.PDM, N, order=order, out_shift=24)
                b.upload_state(s0); b.upload_param(cst)
                out = np.zeros((N, F), np.uint32)
                b.run(F, inp=inp if use_in else None, in2=dith, out=out)
                assert np.array_equal(out, want) and np.array_equal(b.download_state(), sa), (order, use_in)
                b.free()
        x = rng.uniform(-1, 1, (N, F)).astype(np.float32)
        a = rng.uniform(0.001, 0.9, (N, 1)).astype(np.float32); y0 = rng.uniform(-1, 1, (N, 1)).astype(np.float32)
        ya = y0[:, 0].copy()
        want = oracle.onepole_run(ya, a[:, 0].copy(), N, F, x)
        b = ctx.batch(st.ONEPOLE, N); b.upload_state(y0); b.upload_param(a)
        out = np.zeros((N, F), np.float32)
        b.run(F, inp=x, out=out)
        assert np.array_equal(out.view(np.uint32), want.view(np.uint32))
        b.free()
        if F % 16 == 0:
            ph0 = rng.integers(0, 1 << 24, (N, 1), dtype=np.uint32); sp = rng.integers(0, 1 << 16, (N, 1), dtype=np.uint32)
            pa = ph0[:, 0].copy()
            want = oracle.pwm_run(pa, sp[:, 0].copy(), N, F)
            b = ctx.batch(st.PWM, N); b.upload_state(ph0); b.upload_param(sp)
            out = np.zeros((N, F), np.uint8)
            b.run(F, out=out)
            assert np.array_equal(out, want) and np.array_equal(b.download_state()[:, 0], pa)
            b.free()
    finally:
        ctx.set_option("planar_bulk", 2)


def test_pwm(st, ctx, oracle):
    N, F = 77, 500
    ph0 = rng.integers(0, 1 << 24, (N, 1), dtype=np.uint32)
    sp = rng.integers(0, 1 << 16, (N, 1), dtype=np.uint32)
    sp[0] = 256 * 13                                   # mod_pdm.c:161
    pa = ph0[:, 0].copy()
    want = oracle.pwm_run(pa, sp[:, 0].copy(), N, F)
    b = ctx.batch(st.PWM, N)
    b.upload_state(ph0); b.upload_param(sp)
    out = np.zeros((N, F), np.uint8)
    b.run(F, out=out)
    assert np.array_equal(out, want) and np.array_equal(b.download_state()[:, 0], pa)
    b.free()


# ------------------------------------------------------------------------- graphs
def _graph_case(st, ctx, oracle, rows, layout, masked, N=150, F=64, out_node=None, jit=1):
    n_in = max(1, max(max(-r[1], -r[3] if len(r) > 3 else 0) for r in rows))
    out_node = len(rows) - 1 if out_node is None else out_node
    inp = rng.integers(0, 2, (N, n_in, F), dtype=np.uint32)
    inp[::7] = rng.integers(0, 2**32, inp[::7].shape, dtype=np.uint32)
    changed = rng.integers(0, 8, (N, F), dtype=np.uint32) if masked else None
    sw = sum(po.node_words(r[0]) for r in rows)
    s0 = rng.integers(0, 2**32, (N, sw), dtype=np.uint32)
    o = 0
    for r in rows:                                         # glide: the divider count lives below 2^L
        t = r[0]
        if t & 0xFF == po.NODE_GLIDE:
            s0[:, o + 4] &= (1 << (t >> 8)) - 1
        o += po.node_words(t)
    sa = s0.copy()
    want = oracle.graph_run(rows, n_in, out_node, sa, N, F, inp, changed)
    ctx.set_option("graph_jit", jit)
    try:
        b = ctx.batch(st.GRAPH, N, nodes=rows, n_inputs=n_in, out_node=out_node, layout=getattr(st, layout))
        assert b.state_bytes == 4 * sw
        b.upload_state(s0)
        il = layout == "INTERLEAVED"
        out = np.zeros((F, N) if il else (N, F), np.uint32)
        b.run(F, inp=np.ascontiguousarray(inp.transpose(2, 1, 0)) if il else inp,
              in2=None if changed is None else (np.ascontiguousarray(changed.T) if il else changed), out=out)
        if jit:
            assert "not found" not in b.jit_log and "failed" not in b.jit_log, b.jit_log    # the generated kernel ran
        assert np.array_equal(out.T if il else out, want)
        assert np.array_equal(b.download_state(), sa)
        # a second block continues from the device state
        inp2 = rng.integers(0, 3, (N, n_in, F), dtype=np.uint32)
        want2 = oracle.graph_run(rows, n_in, out_node, sa, N, F, inp2, changed)
        b.run(F, inp=np.ascontiguousarray(inp2.transpose(2, 1, 0)) if il else inp2,
              in2=None if changed is None else (np.ascontiguousarray(changed.T) if il else changed), out=out)
        assert np.array_equal(out.T if il else out, want2)
        assert np.array_equal(b.download_state(), sa)
        b.free()
    finally:
        ctx.set_option("graph_jit", 1)


@pytest.mark.parametrize("rows", [po.GRAPH_TEST_CPROC, po.GRAPH_BP5,
                                  [(po.NODE_ACC, -1, 1), (po.NODE_ACC, -2, 2), (po.NODE_EDGE, 1, 4), (po.NODE_ACC, 2, 3)],
                                  [(po.NODE_ACC, -1, 0xFFFFFFFF)]])
@pytest.mark.parametrize("layout", ["PLANAR", "INTERLEAVED"])
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("jit", [0, 1])
def test_graph(st, ctx, oracle, rows, layout, masked, jit):
    _graph_case(st, ctx, oracle, rows, layout, masked, jit=jit)


def _random_graph(n_nodes, n_in, seed, glide=False, pdm=False):
    r = np.random.default_rng(seed)
    rows = []
    for k in range(n_nodes):
        src = int(r.integers(-n_in, k)) if k else -int(r.integers(1, n_in + 1))
        t = int(r.integers(0, 4 if pdm else (3 if glide else 2)))
        mask = int(r.choice([1, 2, 3, 4, 6, 0xFFFFFFFF]))
        if t == po.NODE_GLIDE:
            rows.append((po.node_glide(int(r.integers(1, 7))), src, mask))
        elif t == po.NODE_PDM:
            src2 = int(r.integers(-n_in, k)) if k else -int(r.integers(1, n_in + 1))
            rows.append((po.node_pdm(int(r.integers(1, 5)), int(r.choice([0, 8, 24, 31]))), src, mask, src2))
        else:
            rows.append((t, src, mask))
    return rows


@pytest.mark.parametrize("n_nodes,n_in,N,F", [(16, 2, 300, 256), (40, 3, 97, 100), (64, 1, 70, 33), (7, 4, 1000, 192), (3, 1, 5000, 1024)])
@pytest.mark.parametrize("layout", ["PLANAR", "INTERLEAVED"])
@pytest.mark.parametrize("masked", [False, True])
def test_graph_generated_kernels(st, ctx, oracle, n_nodes, n_in, N, F, layout, masked):
    """NVRTC-generated kernels for random ANF graphs up to the 64-node limit: several input
    streams, every mask, an inner node as the output, frame counts that are not multiples of
    the staging tile (and F = 33: the unaligned planar path)."""
    rows = _random_graph(n_nodes, n_in, seed=n_nodes * 131 + n_in)
    _graph_case(st, ctx, oracle, rows, layout, masked, N=N, F=F, out_node=n_nodes // 2)


@pytest.mark.parametrize("n_nodes,n_in,N,F,jit", [(12, 2, 300, 256, 1), (9, 2, 100, 96, 0), (40, 3, 97, 100, 1), (5, 1, 2000, 512, 1)])
@pytest.mark.parametrize("layout", ["PLANAR", "INTERLEAVED"])
@pytest.mark.parametrize("masked", [False, True])
def test_graph_with_glide_nodes(st, ctx, oracle, n_nodes, n_in, N, F, jit, layout, masked):
    """Graphs that contain glide nodes (control-rate -> audio-rate line interpolation,
    mod_pdm_pwm.c:97-143 / mod_controlrate.c:28-40) with dividers 2..64, JIT and table kernels."""
    rows = _random_graph(n_nodes, n_in, seed=n_nodes * 17 + n_in, glide=True)
    assert any(r[0] & 0xFF == po.NODE_GLIDE for r in rows)
    _graph_case(st, ctx, oracle, rows, layout, masked, N=N, F=F, out_node=n_nodes - 1, jit=jit)


@pytest.mark.parametrize("n_nodes,n_in,N,F,jit", [(10, 2, 300, 256, 1), (8, 3, 100, 96, 0), (30, 3, 97, 100, 1)])
@pytest.mark.parametrize("layout", ["PLANAR", "INTERLEAVED"])
@pytest.mark.parametrize("masked", [False, True])
def test_graph_with_pdm_nodes(st, ctx, oracle, n_nodes, n_in, N, F, jit, layout, masked):
    """Graphs with pdmK nodes (two inputs, orders 1..4, several shifts) mixed with acc / edge / glide."""
    rows = _random_graph(n_nodes, n_in, seed=n_nodes * 29 + n_in, pdm=True)
    assert any(r[0] & 0xFF == po.NODE_PDM for r in rows)
    _graph_case(st, ctx, oracle, rows, layout, masked, N=N, F=F, out_node=n_nodes - 1, jit=jit)


@pytest.mark.parametrize("layout", ["PLANAR", "INTERLEAVED"])
def test_v2_channel_as_a_generated_graph(st, ctx, oracle, layout):
    """The firmware's whole v2 channel (mod_pdm_pwm.c:97-116) written as generated graph text --
    glide(setpoint) -> pdm2(in, dither) -- and compiled by the JIT: its output stream is the duty
    stream of the hand-written PDM v2 kernel and of the v2 channel oracle, byte for byte."""
    N, F, L = 500, 2048, 6
    rows, n_in, out_node, _ = st.graph_parse("""
        #define CPROC_NB_INPUTS 2
        void cproc_update(w *input, w g) {
            PROC(line, glide, &(glide_config){ .div_log = 6 }, NULL, .in = input[0]);
            PROC(mod, pdm2, &(pdm_config){ .out_shift = 24 }, NULL, .in = line.out, .dither = input[1]);
            cproc_output(0, mod.out);
        }""")
    sp = po.pdm_setpoints(N, (F >> L) + 1)
    dext = rng.integers(0, 2**32, (N, F), dtype=np.uint32)
    chan = np.zeros((N, 7), np.uint32)
    want, _ = oracle.pdm_v2_run(chan, 2, N, 1, np.ones(N, np.uint32), dext, 0x3FF, 0, L, 24, sp, F)
    inp = np.zeros((N, 2, F), np.uint32)
    inp[:, 0, :] = np.repeat(sp.T, 1 << L, axis=1)[:, :F]
    inp[:, 1, :] = dext & 0x3FF
    il = layout == "INTERLEAVED"
    b = ctx.batch(st.GRAPH, N, nodes=rows, n_inputs=n_in, out_node=out_node, layout=getattr(st, layout))
    out = np.zeros((F, N) if il else (N, F), np.uint32)
    b.run(F, inp=np.ascontiguousarray(inp.transpose(2, 1, 0)) if il else inp, out=out)
    got = out.T if il else out
    assert got.max() < 256 and np.array_equal(got.astype(np.uint8), want)
    gs = b.download_state()
    assert np.array_equal(gs[:, 0:4], chan[:, 1:5]) and np.array_equal(gs[:, 6:8], chan[:, 5:7])
    # and the hand-written v2 kernel with the same external dither
    bv = ctx.batch(st.PDM_V2, N, order=2, bank_size=1, ctl_div_log=L, layout=st.PLANAR)
    duty = np.zeros((N, F), np.uint8)
    bv.run(F, in2=dext, ctl=sp, out=duty)
    assert np.array_equal(duty, got.astype(np.uint8))
    b.free(); bv.free()


def test_glide_node_is_the_pdm_v2_line(st, ctx, oracle):
    """A glide node fed with the setpoint rows reproduces line[0].position of the PDM v2
    channels tick for tick: glide -> (raw) pdm2 by hand equals the v2 duty stream."""
    N, F, L = 64, 1024, 6
    sp = po.pdm_setpoints(N, F >> L)                                     # [rows][N]
    # the v2 oracle on zero state, one bank per channel, external dither 0
    chan = np.zeros((N, 7), np.uint32); prng = np.ones(N, np.uint32)
    dext = np.zeros((N, F), np.uint32)
    want_duty, _ = oracle.pdm_v2_run(chan, 2, N, 1, prng, dext, 0x3FF, 0, L, 24, sp, F)
    # glide node over the same setpoints held for 2^L ticks each
    inp = np.repeat(sp.T[:, None, :], 1 << L, axis=2).astype(np.uint32)  # [N][1][F]
    inp = np.ascontiguousarray(inp)
    b = ctx.batch(st.GRAPH, N, nodes=[(st.node_glide(L), -1, 0xFFFFFFFF)])
    pos = np.zeros((N, F), np.uint32)
    b.run(F, inp=inp, out=pos)
    gl = b.download_state()
    assert np.array_equal(gl[:, 0:4], chan[:, 1:5])                      # line[0], line[1] after F ticks
    # pdm2_update on the glide output (CPROC_CUDA_PDM takes an input stream)
    bp = ctx.batch(st.PDM, N, order=2, out_shift=24)
    q = np.zeros((N, F), np.uint32)
    bp.run(F, inp=pos, out=q)
    assert np.array_equal(q.astype(np.uint8), want_duty)
    b.free(); bp.free()


@pytest.mark.parametrize("rows", [po.GRAPH_TEST_CPROC, po.GRAPH_BP5,
                                  [(po.NODE_ACC, -1, 1), (po.NODE_EDGE, -2, 2), (po.NODE_EDGE, 1, 4), (po.NODE_ACC, 2, 3), (po.NODE_ACC, 0, 6), (po.NODE_EDGE, 3, 0xFFFFFFFF)],
                                  [(po.NODE_EDGE, -1, 0)]])
@pytest.mark.parametrize("layout", ["PLANAR", "INTERLEAVED"])
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("N,F,chunk", [(1, 50000, 0), (3, 4099, 64), (70, 1000, 7), (2, 65, 1)])
def test_graph_scan(st, ctx, oracle, rows, layout, masked, N, F, chunk):
    """Time-parallel acc / edge graphs: bit-exact against the sequential oracle, output stream and
    every state word, for ragged chunkings, sparse masks (long runs without an executed tick), an
    interior output node and a never-executed node."""
    n_in = max(1, max(-r[1] for r in rows))
    out_node = min(2, len(rows) - 1)
    inp = rng.integers(0, 2, (N, n_in, F), dtype=np.uint32)
    inp[:, :, ::17] = rng.integers(0, 2**32, inp[:, :, ::17].shape, dtype=np.uint32)
    changed = None
    if masked:
        changed = rng.integers(0, 8, (N, F), dtype=np.uint32)
        changed[:, F // 3: F // 3 + min(F // 3, 300)] = 0                 # a stretch where nothing executes
    sw = sum(po.node_words(r[0]) for r in rows)
    s0 = rng.integers(0, 2**32, (N, sw), dtype=np.uint32)
    sa = s0.copy()
    want = oracle.graph_run(rows, n_in, out_node, sa, N, F, inp, changed)
    ctx.set_option("xvoice_chunk", chunk)
    try:
        b = ctx.batch(st.GRAPH, N, nodes=rows, n_inputs=n_in, out_node=out_node, layout=getattr(st, layout), mode=1)
        b.upload_state(s0)
        il = layout == "INTERLEAVED"
        out = np.zeros((F, N) if il else (N, F), np.uint32)
        l0 = ctx.launches
        b.run(F, inp=np.ascontiguousarray(inp.transpose(2, 1, 0)) if il else inp,
              in2=None if changed is None else (np.ascontiguousarray(changed.T) if il else changed), out=out)
        assert ctx.launches - l0 >= 3 * len(rows)          # reduce, scan, apply per node
        assert np.array_equal(out.T if il else out, want)
        assert np.array_equal(b.download_state(), sa)
        b.free()
    finally:
        ctx.set_option("xvoice_chunk", 0)
    with pytest.raises(st.CprocCudaError):                 # glide / pdm are not scannable
        bb = ctx.batch(st.GRAPH, 2, nodes=[(st.node_glide(4), -1, 1)], mode=1)
        bb.run(128, inp=np.zeros((2, 1, 128), np.uint32), out=np.zeros((2, 128), np.uint32))


@pytest.mark.parametrize("n_nodes,n_in,outs,N,F", [(6, 1, [5, 2], 200, 256), (20, 2, [19, 0, 7, 7, 12], 97, 100), (9, 3, [8, 1, 2, 3, 4, 5, 6, 7], 64, 33),
                                                 (12, 2, [3] * 16, 40, 64)])
@pytest.mark.parametrize("layout", ["PLANAR", "INTERLEAVED"])
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("path", ["jit", "table", "scan"])
def test_graph_several_outputs(st, ctx, oracle, n_nodes, n_in, outs, N, F, layout, masked, path):
    """Graphs with several cproc_output statements (more outputs than inputs included): output
    stream q is the .out of node outs[q]; generated kernels, table kernel and the time-parallel scan."""
    rows = _random_graph(n_nodes, n_in, seed=n_nodes * 7 + len(outs), glide=path != "scan", pdm=path == "jit")
    if path == "table" and (len(rows) > 16 or sum(po.node_words(r[0]) for r in rows) > 48):
        pytest.skip("the table kernel holds 16 nodes / 48 state words")
    n_in = max(1, max(max(-r[1], -r[3] if len(r) > 3 else 0) for r in rows))
    inp = rng.integers(0, 3, (N, n_in, F), dtype=np.uint32)
    changed = rng.integers(0, 8, (N, F), dtype=np.uint32) if masked else None
    sw = sum(po.node_words(r[0]) for r in rows)
    s0 = rng.integers(0, 2**32, (N, sw), dtype=np.uint32)
    o = 0
    for r in rows:
        if r[0] & 0xFF == po.NODE_GLIDE:
            s0[:, o + 4] &= (1 << (r[0] >> 8)) - 1
        o += po.node_words(r[0])
    sa = s0.copy()
    want = oracle.graph_run_multi(rows, n_in, outs, sa, N, F, inp, changed)       # [N][n_out][F]
    ctx.set_option("graph_jit", 0 if path == "table" else 1)
    try:
        b = ctx.batch(st.GRAPH, N, nodes=rows, n_inputs=n_in, out_node=outs, layout=getattr(st, layout), mode=1 if path == "scan" else 0)
        b.upload_state(s0)
        il = layout == "INTERLEAVED"
        out = np.zeros((F, len(outs), N) if il else (N, len(outs), F), np.uint32)
        b.run(F, inp=np.ascontiguousarray(inp.transpose(2, 1, 0)) if il else inp,
              in2=None if changed is None else (np.ascontiguousarray(changed.T) if il else changed), out=out)
        assert np.array_equal(out.transpose(2, 1, 0) if il else out, want)
        assert np.array_equal(b.download_state(), sa)
        b.free()
    finally:
        ctx.set_option("graph_jit", 1)


@pytest.mark.parametrize("vec4", [0, 1])
@pytest.mark.parametrize("N,F", [(1024, 200), (300, 64), (4, 1000), (1001, 50)])
@pytest.mark.parametrize("masked", [False, True])
def test_graph_interleaved_vec4(st, ctx, oracle, vec4, N, F, masked):
    """INTERLEAVED generated kernels with one and with four instances per thread (the latter only
    when n % 4 == 0: N = 1001 must take the scalar kernel either way), two inputs, three outputs."""
    rows = _random_graph(9, 2, seed=123, glide=True, pdm=True)
    ctx.set_option("graph_vec4", vec4)
    try:
        n_in = max(1, max(max(-r[1], -r[3] if len(r) > 3 else 0) for r in rows))
        outs = [8, 2, 5]
        inp = rng.integers(0, 3, (N, n_in, F), dtype=np.uint32)
        changed = rng.integers(0, 8, (N, F), dtype=np.uint32) if masked else None
        sw = sum(po.node_words(r[0]) for r in rows)
        s0 = rng.integers(0, 2**32, (N, sw), dtype=np.uint32)
        o = 0
        for r in rows:
            if r[0] & 0xFF == po.NODE_GLIDE:
                s0[:, o + 4] &= (1 << (r[0] >> 8)) - 1
            o += po.node_words(r[0])
        sa = s0.copy()
        want = oracle.graph_run_multi(rows, n_in, outs, sa, N, F, inp, changed)
        b = ctx.batch(st.GRAPH, N, nodes=rows, n_inputs=n_in, out_node=outs, layout=st.INTERLEAVED)
        b.upload_state(s0)
        out = np.zeros((F, len(outs), N), np.uint32)
        b.run(F, inp=np.ascontiguousarray(inp.transpose(2, 1, 0)), in2=None if changed is None else np.ascontiguousarray(changed.T), out=out)
        assert np.array_equal(out.transpose(2, 1, 0), want)
        assert np.array_equal(b.download_state(), sa)
        b.free()
    finally:
        ctx.set_option("graph_vec4", 1)


def test_graph_from_generated_text(st, ctx, oracle):
    """The wire format end to end: the generated C text of the reference's two graphs
    (linux/test_cproc.c:11-17, stm32f103/bp5_plugin.c:1-9) -> parser -> batch -> render."""
    for text, want_rows in ((GEN_TEST_CPROC, po.GRAPH_TEST_CPROC), (GEN_BP5, po.GRAPH_BP5)):
        rows, n_in, out_node, _ = st.abi.graph_parse(text)
        assert rows == want_rows
        _graph_case(st, ctx, oracle, rows, "PLANAR", True, N=200, F=128, out_node=out_node)


# the statements epid_cproc.erl generated for the reference's two shipped graphs
GEN_TEST_CPROC = """
#define CPROC_NB_INPUTS 1
void cproc_update(w *input, w g) {
    PROC_COND(g&0b1, n1, edge, NULL, NULL, .in = input[0]);
    PROC_COND(g&0b1, n2, acc,  NULL, NULL, .in = n1.out);
    cproc_output(2, n2.out);
}
"""
GEN_BP5 = """
#define CPROC_NB_INPUTS 1
void cproc_update(w *input, w g) {
    PROC_COND(g&0b1, n1, edge, NULL, NULL, .in = input[0]);
    PROC_COND(g&0b1, n2, acc, NULL, NULL, .in = n1.out);
    PROC_COND(g&0b1, n3, acc, NULL, NULL, .in = n2.out);
    cproc_output(3, n3.out);
}
"""


def test_graph_test_cproc_anchor(st, ctx):
    """SURVEY 8c anchor through the CUDA path: zero-initialised edge->acc graph,
    one instance, tick by tick (F=1 per call, like cproc_update)."""
    b = ctx.batch(st.GRAPH, 1, nodes=po.GRAPH_TEST_CPROC)
    got = []
    for x in [0, 1, 1, 0, 0, 1, 0, 1, 1, 1, 0]:
        out = np.zeros((1, 1), np.uint32)
        b.run(1, inp=np.array([[[x]]], np.uint32), out=out)
        got.append(int(out[0, 0]))
    assert got == [0, 1, 1, 2, 2, 3, 4, 5, 5, 5, 6]
    b.free()
    with pytest.raises(st.CprocCudaError):     # ANF: forward reference
        ctx.batch(st.GRAPH, 1, nodes=[(po.NODE_ACC, 1, 1), (po.NODE_ACC, -1, 1)])


# --------------------------------------------------------------------- voice bank
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("N,G,F", [(64, 64, 64), (64 * 37, 64, 64), (5000, 0, 512), (20000, 0, 700), (1000, 300, 129)])
def test_voice_bank(st, ctx, oracle, mode, N, G, F):
    v0 = np.zeros((N, 2), np.uint32)
    v0[:, 1] = rng.integers(0, 2**32, N, dtype=np.uint32)
    tab = np.array([oracle.note_to_inc(n) for n in range(128)], np.uint32)
    v0[:, 0] = np.where(rng.random(N) < 0.8, tab[rng.integers(0, 128, N)], 0)
    v0[: N // 8, 0] = 0x7FFFFFF1                     # loud voices: integer sum wraps
    va = v0.copy()
    Gq = G if G else N
    want_i, want_f = oracle.voice_bank_run(va, N, Gq, mode, F)
    b = ctx.batch(st.VOICE_BANK, N, mode=mode, voices_per_bus=G)
    b.upload_state(v0)
    n_bus = (N + Gq - 1) // Gq
    out = np.zeros((n_bus, F), np.float32)
    mix = np.zeros((n_bus, F), np.int32)
    b.run(F, out=out, mix=mix)
    assert np.array_equal(mix, want_i)
    assert np.array_equal(out.view(np.uint32), want_f.view(np.uint32))
    assert np.array_equal(b.download_state(), va)
    # float only, continuing from the advanced state
    want_i2, want_f2 = oracle.voice_bank_run(va, N, Gq, mode, F)
    b.run(F, out=out)
    assert np.array_equal(out.view(np.uint32), want_f2.view(np.uint32))
    b.free()


def test_voice_bank_synth_anchor(st, ctx):
    # SURVEY 8c: notes 69,60,127,0 on -> first 8 saw-mix samples of synth_run
    v = np.zeros((64, 2), np.uint32)
    v[:4, 0] = [39370533, 23409859, 1122405051, 731558]
    b = ctx.batch(st.VOICE_BANK, 64, voices_per_bus=64)
    b.upload_state(v)
    out = np.zeros((1, 8), np.float32)
    b.run(8, out=out)
    want = [0.0, float.fromhex("0x1.1abeap-6"), float.fromhex("-0x1.ca82bep-6"), float.fromhex("-0x1.5f883ap-7"),
            float.fromhex("0x1.abea1p-8"), float.fromhex("0x1.85b924p-6"), float.fromhex("-0x1.5f883ap-6"),
            float.fromhex("-0x1.132662p-8")]
    assert out[0].tolist() == want
    b.free()


@pytest.mark.parametrize("run_graph", [0, 1, 2, 3])
def test_run_period_state_rides_along(st, ctx, oracle, run_graph):
    """cproc_cuda_run_period == upload_state; run; download_state (the JACK / synth_run period: the host's structs hold the
    state, note_on / note_off write them between periods) on every period path of cproc_cuda_run -- staged copies, the
    captured CUDA graph, zero copy, direct launches on pinned staging -- and with a record stride (struct voice in a larger struct)."""
    ctx.set_option("run_graph", run_graph)
    try:
        V, F = 128, 64
        rec = np.zeros((V, 4), np.uint32)                          # stride 16: {inc, phase, unrelated, unrelated}
        rec[::3, 0] = [oracle.note_to_inc(int(n)) for n in rng.integers(30, 90, len(rec[::3]))]
        rec[:, 2:] = rng.integers(0, 2**32, (V, 2), dtype=np.uint32)
        tail = rec[:, 2:].copy()
        vb = ctx.batch(st.VOICE_BANK, V, voices_per_bus=64)
        syncs = []
        for k in range(6):
            if k == 3:
                rec[1, 0] = oracle.note_to_inc(69)                 # note on between periods
            voices = np.ascontiguousarray(rec[:, :2])
            _, want = oracle.voice_bank_run(voices, V, 64, po.MIX_SAW, F)   # advances `voices`
            out = np.zeros((2, F), np.float32)
            vb.run_period(F, rec, stride=16, out=out)
            assert np.array_equal(out.view(np.uint32), want.view(np.uint32)), k
            assert np.array_equal(rec[:, :2], voices) and np.array_equal(rec[:, 2:], tail), k
        assert np.array_equal(vb.download_state(), rec[:, :2])
        vb.free()
        # a graph batch (edge -> acc of test_cproc.c) with input stream and packed records
        N = 3
        stt = np.zeros((N, 3), np.uint32); sa = stt.copy()
        b = ctx.batch(st.GRAPH, N, nodes=po.GRAPH_TEST_CPROC, n_inputs=1)
        for k in range(4):
            x = rng.integers(0, 2, (N, 1, F), dtype=np.uint32)
            want = oracle.graph_run(po.GRAPH_TEST_CPROC, 1, 1, sa, N, F, x)
            out = np.zeros((N, F), np.uint32)
            b.run_period(F, stt, inp=x, out=out)
            assert np.array_equal(out, want) and np.array_equal(stt, sa), k
        b.free()
        with pytest.raises(st.CprocCudaError):
            vb2 = ctx.batch(st.VOICE_BANK, 8, voices_per_bus=8)
            try:
                vb2.run_period(8, np.zeros((8, 1), np.uint32), stride=4, out=np.zeros((1, 8), np.float32))   # stride smaller than the record
            finally:
                vb2.free()
    finally:
        ctx.set_option("run_graph", 2)


# -------------------------------------------------------------------- square_grain
def _square_grain_case(st, ctx, oracle, N, F, layout, neg_th=False, odd_state=False):
    inp = rng.uniform(-1, 1, (N, F)).astype(np.float32)
    th = rng.uniform(0.05, 0.5, (N, 1)).astype(np.float32)
    th[0] = 0.0
    if neg_th:
        th[3::5] = -th[3::5]
    s0 = rng.choice(np.array([0.0, 0.5, -0.5], np.float32), (N, 1))
    if odd_state:
        s0[1::4] = rng.choice(np.array([0.25, -0.125, 2.0], np.float32), s0[1::4].shape)   # output = state until the first flip
    sa = s0[:, 0].copy()
    want = oracle.square_grain_run(sa, th[:, 0].copy(), N, F, inp)
    b = ctx.batch(st.SQUARE_GRAIN, N, layout=getattr(st, layout))
    b.upload_state(s0); b.upload_param(th)
    il = layout == "INTERLEAVED"
    out = np.zeros((F, N) if il else (N, F), np.float32)
    b.run(F, inp=np.ascontiguousarray(inp.T) if il else inp, out=out)
    got = out.T if il else out
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert np.array_equal(b.download_state().view(np.float32)[:, 0], sa)
    # in place (Pd hands the same vector as in and out)
    b.upload_state(s0)
    io = np.ascontiguousarray(inp.T) if il else inp.copy()
    b.run(F, inp=io, out=io)
    assert np.array_equal((io.T if il else io).view(np.uint32), want.view(np.uint32))
    # a second block continues from the device state
    inp2 = rng.uniform(-1, 1, (N, F)).astype(np.float32)
    want2 = oracle.square_grain_run(sa, th[:, 0].copy(), N, F, inp2)
    b.run(F, inp=np.ascontiguousarray(inp2.T) if il else inp2, out=out)
    assert np.array_equal((out.T if il else out).view(np.uint32), want2.view(np.uint32))
    assert np.array_equal(b.download_state().view(np.float32)[:, 0], sa)
    b.free()


@pytest.mark.parametrize("N,F", [(1, 64), (33, 257), (1000, 256), (129, 31)])
@pytest.mark.parametrize("layout", ["PLANAR", "INTERLEAVED"])
def test_square_grain(st, ctx, oracle, N, F, layout):
    _square_grain_case(st, ctx, oracle, N, F, layout)


@pytest.mark.parametrize("vec4", [0, 1])
@pytest.mark.parametrize("N,F", [(1000, 256), (64, 7), (4100, 40), (1001, 33)])
def test_square_grain_interleaved_variants(st, ctx, oracle, vec4, N, F):
    ctx.set_option("grain_vec4", vec4)
    try:
        _square_grain_case(st, ctx, oracle, N, F, "INTERLEAVED", True, True)
    finally:
        ctx.set_option("grain_vec4", 1)


@pytest.mark.parametrize("bulk", [0, 1, 2, 3, 4, 5])
@pytest.mark.parametrize("N,F,neg_th,odd", [(1000, 256, False, False), (77, 100, False, False), (300, 1024, True, False),
                                            (64, 4, False, True), (4097, 64, True, True), (31, 392, False, False)])
def test_square_grain_bulk_variants(st, ctx, oracle, bulk, N, F, neg_th, odd):
    """k_grain_bulk tile/stage shapes against the register-transpose kernel's cases: ragged
    last tiles, ragged last warp, negative thresholds and non-reference state values
    (both take the literal two-branch form)."""
    ctx.set_option("grain_bulk", bulk)
    try:
        _square_grain_case(st, ctx, oracle, N, F, "PLANAR", neg_th, odd)
    finally:
        ctx.set_option("grain_bulk", 5)


@pytest.mark.parametrize("gen", [0, 1, 2])
@pytest.mark.parametrize("N,F,neg_th", [(3000, 256, False), (70000, 200, False), (517, 37, False), (3000, 128, True)])
def test_square_grain_mix(st, ctx, oracle, gen, N, F, neg_th):
    state = rng.choice(np.array([0.0, 0.5, -0.5], np.float32), N)
    th = rng.uniform(0.05, 0.5, N).astype(np.float32)
    th[0] = 0.0
    if neg_th:
        th[5::7] = -th[5::7]          # both flip conditions can hold: the literal two-branch kernels must take over
    phase = rng.integers(0, 2**32, N, dtype=np.uint32)
    inc = np.array([oracle.note_to_inc(n) for n in rng.integers(36, 97, N)], np.uint32)
    gl = rng.integers(0, 65, N).astype(np.uint8); gr = (64 - gl).astype(np.uint8)
    sa, pa = state.copy(), phase.copy()
    want_i, want_f = oracle.square_grain_mix_run(sa, th, pa, inc, gl, gr, N, F)
    ctx.set_option("grain_mix2", gen)
    try:
        b = ctx.batch(st.SQUARE_GRAIN_MIX, N)
        s_rec = np.zeros((N, 2), np.uint32); s_rec[:, 0] = state.view(np.uint32); s_rec[:, 1] = phase
        p_rec = np.zeros((N, 4), np.uint32); p_rec[:, 0] = th.view(np.uint32); p_rec[:, 1] = inc; p_rec[:, 2] = gl; p_rec[:, 3] = gr
        b.upload_state(s_rec); b.upload_param(p_rec)
        out = np.zeros((2, F), np.float32); mix = np.zeros((2, F), np.int32)
        b.run(F, out=out, mix=mix)
        assert np.array_equal(mix, want_i)
        assert np.array_equal(out.view(np.uint32), want_f.view(np.uint32))
        s1 = b.download_state()
        assert np.array_equal(s1[:, 0].view(np.float32), sa) and np.array_equal(s1[:, 1], pa)
        # a second block continues from the device state (split run == one run)
        want_i2, _ = oracle.square_grain_mix_run(sa, th, pa, inc, gl, gr, N, F)
        b.run(F, out=out, mix=mix)
        assert np.array_equal(mix, want_i2)
        s1 = b.download_state()
        assert np.array_equal(s1[:, 0].view(np.float32), sa) and np.array_equal(s1[:, 1], pa)
        b.free()
    finally:
        ctx.set_option("grain_mix2", 2)


# ------------------------------------------------------------- extension processors
def _xvoice_inputs(oracle, N):
    prm = np.zeros(N, po.xvoice_param_dtype)
    prm["inc"] = [oracle.note_to_inc(n) for n in rng.integers(24, 109, N)]
    prm["f"] = rng.uniform(0.01, 0.3, N); prm["q"] = rng.uniform(0.5, 2.0, N)
    prm["env_attack"] = rng.uniform(1e-3, 1e-1, N); prm["env_release"] = rng.uniform(1e-3, 1e-2, N)
    prm["gate_frames"] = rng.integers(0, 400, N)
    prm["gl"] = rng.uniform(0, 1, N); prm["gr"] = 1.0 - prm["gl"]
    stt = np.zeros(N, po.xvoice_state_dtype)
    stt["phase"] = rng.integers(0, 2**32, N, dtype=np.uint32)
    return stt, prm


@pytest.mark.parametrize("layout", ["PLANAR", "TILED"])
def test_xvoice_raw_bit_exact_and_mix(st, ctx, oracle, layout):
    N, F = 1000, 512
    s0, prm = _xvoice_inputs(oracle, N)
    sa = s0.copy()
    want_raw, want_mix = oracle.xvoice_run(sa, prm, N, F)
    b = ctx.batch(st.XVOICE, N, layout=getattr(st, layout))
    b.upload_state(s0.view(np.uint32).reshape(N, 5)); b.upload_param(prm.view(np.uint32).reshape(N, 8))
    raw = np.zeros(N * F * 2, np.float32); mix = np.zeros((2, F), np.float32)
    b.run(F, out=raw, mix=mix)
    got = raw.reshape(F // 2, N, 2, 2).transpose(1, 0, 2, 3).reshape(N, F, 2) if layout == "TILED" else raw.reshape(N, F, 2)
    assert np.array_equal(got.view(np.uint32), want_raw.view(np.uint32))       # bit-exact per voice
    assert np.array_equal(b.download_state(), sa.view(np.uint32).reshape(N, 5))
    # mix: float sum over voices, order differs from the oracle's double accumulation.
    # Tolerance (BASELINE.json north_star): <= 1e-5 relative to the mix peak, SNR >= 120 dB.
    err = np.abs(mix.astype(np.float64) - want_mix.astype(np.float64)).max()
    peak = np.abs(want_mix).max()
    assert err <= 1e-5 * peak
    snr = 10 * np.log10((want_mix.astype(np.float64) ** 2).sum() / max(((mix.astype(np.float64) - want_mix) ** 2).sum(), 1e-300))
    assert snr >= 120.0
    # deterministic run to run
    b.upload_state(s0.view(np.uint32).reshape(N, 5))
    mix2 = np.zeros((2, F), np.float32)
    b.run(F, out=raw, mix=mix2)
    assert np.array_equal(mix.view(np.uint32), mix2.view(np.uint32))
    b.free()


def _mix_close(mix, want_mix):
    err = np.abs(mix.astype(np.float64) - want_mix.astype(np.float64)).max()
    peak = np.abs(want_mix).max()
    assert err <= 1e-5 * peak
    snr = 10 * np.log10((want_mix.astype(np.float64) ** 2).sum() / max(((mix.astype(np.float64) - want_mix) ** 2).sum(), 1e-300))
    assert snr >= 120.0


@pytest.fixture(params=[1, 0], ids=["mix2", "mix1"])
def mixgen(request, ctx):
    """Both generations of the mix-only XVOICE kernel: k_xvoice_mix2 (voice pairs on the packed fp32 pipe, state tiles in
    shared memory; the default) and k_xvoice_mix."""
    ctx.set_option("xvoice_mix2", request.param)
    yield request.param
    ctx.set_option("xvoice_mix2", 1)


@pytest.mark.parametrize("N,F", [(1000, 512), (77, 45), (148 * 4 * 128 + 333, 96), (1, 32), (148 * 3 * 256 * 12 + 257, 64), (255, 33), (256, 32), (257, 70)])
def test_xvoice_mix_only(st, ctx, oracle, N, F, mixgen):
    """Mix-only render (register accumulators per thread, voices walked per 32-frame
    chunk): mix within the stated tolerance of the oracle's double-accumulated mix
    (<= 1e-5 of the peak, >= 120 dB SNR), voice state bit-exact, deterministic."""
    s0, prm = _xvoice_inputs(oracle, N)
    sa = s0.copy()
    _, want_mix = oracle.xvoice_run(sa, prm, N, F)
    b = ctx.batch(st.XVOICE, N)
    b.upload_state(s0.view(np.uint32).reshape(N, 5)); b.upload_param(prm.view(np.uint32).reshape(N, 8))
    mix = np.zeros((2, F), np.float32)
    b.run(F, mix=mix)
    _mix_close(mix, want_mix)
    assert np.array_equal(b.download_state(), sa.view(np.uint32).reshape(N, 5))
    b.upload_state(s0.view(np.uint32).reshape(N, 5))
    mix2 = np.zeros((2, F), np.float32)
    b.run(F, mix=mix2)
    assert np.array_equal(mix.view(np.uint32), mix2.view(np.uint32))
    # the same render in two calls continues seamlessly
    if F >= 64:
        b.upload_state(s0.view(np.uint32).reshape(N, 5))
        ma = np.zeros((2, 32), np.float32); mb = np.zeros((2, F - 32), np.float32)
        b.run(32, mix=ma); b.run(F - 32, mix=mb)
        assert np.array_equal(np.concatenate([ma, mb], axis=1).view(np.uint32), mix.view(np.uint32))
    b.free()


@pytest.mark.parametrize("closed", [1, 0])
@pytest.mark.parametrize("layout,groups", [("TILED", 4), ("PLANAR", 1), ("PLANAR", 3)])
def test_xvoice_scan_zero_state_forms(st, ctx, oracle, closed, layout, groups):
    """The closed-form zero-state pass (per phase wrap) and the ticked fp64 pass give chunk start states
    inside the same tolerance of the sequential oracle (1e-5 of the peak, benign filters), for every kind of
    increment: none, one wrap per 2^32 ticks, powers of two, increments past 2^31 (a wrap nearly every tick),
    gaps of exactly k and of k+1 ticks.  The same set at the slow filter f = 1e-3, voice by voice against the
    fp64 filter: tests/test_gpu_float_ref.py::test_xvoice_scan_slow_filter_increments."""
    special = np.array([0, 1, 2, 3, 1 << 20, 1 << 24, (1 << 24) + 1, (1 << 24) - 1, 3 << 28, 1 << 31, (1 << 31) + 5, (1 << 31) - 1,
                        0xFFFFFFFF, 0xFFFFFFFE, 0x12345678, 0x9ABCDEF0, 0x55555555, 0x55555556, 0x00F00F00, 715827883], np.uint32)
    N, F = 512, 1536
    s0, prm = _xvoice_inputs(oracle, N)
    prm["inc"][:len(special)] = special
    prm["inc"][len(special):2 * len(special)] = special
    prm["gate_frames"] = rng.integers(0, F, N)
    s0["lp"] = rng.uniform(-0.5, 0.5, N); s0["bp"] = rng.uniform(-0.5, 0.5, N)
    sa = s0.copy()
    want_raw, _ = oracle.xvoice_run(sa, prm, N, F)
    ctx.set_option("xvoice_chunk", 96); ctx.set_option("xvoice_groups", groups); ctx.set_option("xvoice_closed", closed)
    b = ctx.batch(st.XVOICE, N, layout=getattr(st, layout), mode=st.XVOICE_SCAN)
    try:
        b.upload_state(s0.view(np.uint32).reshape(N, 5)); b.upload_param(prm.view(np.uint32).reshape(N, 8))
        raw = np.zeros(N * F * 2, np.float32)
        b.run(F, out=raw)
        got = raw.reshape(F // 2, N, 2, 2).transpose(1, 0, 2, 3).reshape(N, F, 2) if layout == "TILED" else raw.reshape(N, F, 2)
        w64, g64 = want_raw.astype(np.float64), got.astype(np.float64)
        err = np.abs(g64 - w64).reshape(N, -1).max(axis=1)
        assert err.max() <= 1e-5 * np.abs(w64).max(), (int(err.argmax()), int(prm["inc"][err.argmax()]), float(err.max()))
        assert 10 * np.log10((w64 ** 2).sum() / max(((g64 - w64) ** 2).sum(), 1e-300)) >= 120.0
        got_state = b.download_state().view(po.xvoice_state_dtype).reshape(N)
        assert np.array_equal(got_state["phase"], sa["phase"])
    finally:
        b.free()
        ctx.set_option("xvoice_chunk", 0); ctx.set_option("xvoice_groups", 0); ctx.set_option("xvoice_closed", 1)


@pytest.mark.parametrize("N,F,chunk,groups,mode", [(70, 1001, 32, 0, 2), (200, 3000, 96, 0, 1), (700, 2048, 32, 3, 1), (40, 2050, 64, 0, 2), (500, 998, 32, 4, 2)])
def test_xvoice_scan_planar_store_paths(st, ctx, oracle, N, F, chunk, groups, mode):
    """PLANAR render: tensor-TMA stores (planar_bulk 2, even F) and the staged-row kernel it falls back to
    (odd F, planar_bulk 1) agree with the sequential oracle to 1e-5 of the peak at benign filters (the
    per-voice contract against the fp64 filter: tests/test_gpu_float_ref.py)."""
    s0, prm = _xvoice_inputs(oracle, N)
    prm["gate_frames"] = rng.integers(0, F, N)
    sa = s0.copy()
    want_raw, _ = oracle.xvoice_run(sa, prm, N, F)
    ctx.set_option("xvoice_chunk", chunk); ctx.set_option("xvoice_groups", groups); ctx.set_option("planar_bulk", mode)
    b = ctx.batch(st.XVOICE, N, layout=st.PLANAR, mode=st.XVOICE_SCAN)
    try:
        b.upload_state(s0.view(np.uint32).reshape(N, 5)); b.upload_param(prm.view(np.uint32).reshape(N, 8))
        raw = np.full(N * F * 2 + 64, 7.0, np.float32)
        b.run(F, out=raw[:N * F * 2])
        assert np.all(raw[N * F * 2:] == 7.0)
        w64, g64 = want_raw.astype(np.float64), raw[:N * F * 2].reshape(N, F, 2).astype(np.float64)
        assert np.abs(g64 - w64).max() <= 1e-5 * np.abs(w64).max()
        assert 10 * np.log10((w64 ** 2).sum() / max(((g64 - w64) ** 2).sum(), 1e-300)) >= 120.0
        got_state = b.download_state().view(po.xvoice_state_dtype).reshape(N)
        assert np.array_equal(got_state["phase"], sa["phase"]) and np.array_equal(got_state["t"], sa["t"])
    finally:
        b.free()
        ctx.set_option("xvoice_chunk", 0); ctx.set_option("xvoice_groups", 0); ctx.set_option("planar_bulk", 2)


@pytest.mark.parametrize("layout", ["PLANAR", "TILED"])
@pytest.mark.parametrize("N,F,chunk,groups", [(64, 4096, 256, 0), (200, 3000, 96, 0), (33, 8192, 0, 0), (5, 1000, 32, 0),
                                              (700, 2048, 64, 0), (700, 2048, 32, 3), (300, 1024, 512, 1), (129, 640, 64, 8), (1100, 1056, 96, 0), (1100, 1056, 96, 5)])
def test_xvoice_scan(st, ctx, oracle, layout, N, F, chunk, groups):
    """Time-parallel raw render: chunk start states from the fp64 scan of the SVF's affine
    recurrence.  phase / t / env bit-exact; at these benign filters (f 0.01..0.3, q 0.5..2), where the
    sequential render is itself within ~1e-6 of the exact filter, lp, bp and the output stay within
    <= 1e-5 of the peak and >= 120 dB SNR of the sequential oracle, for every chunking and grouping.
    The accuracy contract itself -- per voice against the fp64 filter, slow and resonant filters
    included -- is tests/test_gpu_float_ref.py."""
    s0, prm = _xvoice_inputs(oracle, N)
    prm["gate_frames"] = rng.integers(0, F, N)
    prm["env_release"] = rng.uniform(2e-4, 1e-2, N)
    s0["lp"] = rng.uniform(-0.5, 0.5, N); s0["bp"] = rng.uniform(-0.5, 0.5, N)
    s0["env"] = rng.uniform(0, 1, N); s0["t"] = rng.integers(0, 100, N)
    sa = s0.copy()
    want_raw, _ = oracle.xvoice_run(sa, prm, N, F)
    ctx.set_option("xvoice_chunk", chunk)
    ctx.set_option("xvoice_groups", groups)
    b = ctx.batch(st.XVOICE, N, layout=getattr(st, layout), mode=st.XVOICE_SCAN)
    try:
        b.upload_state(s0.view(np.uint32).reshape(N, 5)); b.upload_param(prm.view(np.uint32).reshape(N, 8))
        raw = np.zeros(N * F * 2, np.float32)
        l0 = ctx.launches
        b.run(F, out=raw)
        g_req = min(groups or 1, -(-N // 128))
        per = -(-(-(-N // g_req)) // 128) * 128              # variants per group, multiple of 128
        g_eff = -(-N // per)
        piped = False                                        # closed-form zero-state pass: always a kernel of its own
        # env; zsr (TILED pipeline: first two groups only, the rest is fused into the renders); scan + render per group
        # (+ the table kernel of the closed-form zero-state pass)
        assert ctx.launches - l0 == 2 + (2 if piped else g_eff) + 2 * g_eff
        got = raw.reshape(F // 2, N, 2, 2).transpose(1, 0, 2, 3).reshape(N, F, 2) if layout == "TILED" else raw.reshape(N, F, 2)
        w64, g64 = want_raw.astype(np.float64), got.astype(np.float64)
        peak = np.abs(w64).max()
        assert np.abs(g64 - w64).max() <= 1e-5 * peak
        snr = 10 * np.log10((w64 ** 2).sum() / max(((g64 - w64) ** 2).sum(), 1e-300))
        assert snr >= 120.0, snr
        got_state = b.download_state().view(po.xvoice_state_dtype).reshape(N)
        for k in ("phase", "t"):
            assert np.array_equal(got_state[k], sa[k])
        assert np.array_equal(got_state["env"].view(np.uint32), sa["env"].view(np.uint32))
        for k in ("lp", "bp"):
            assert np.abs(got_state[k].astype(np.float64) - sa[k]).max() <= 1e-5 * max(1.0, np.abs(sa[k]).max())
    finally:
        b.free()
        ctx.set_option("xvoice_chunk", 0)
        ctx.set_option("xvoice_groups", 0)


@pytest.mark.parametrize("layout,N,F", [("PLANAR", 300, 200), ("INTERLEAVED", 300, 201), ("INTERLEAVED", 301, 200), ("INTERLEAVED", 4 * 513, 37)])
def test_onepole(st, ctx, oracle, layout, N, F):
    inp = rng.uniform(-1, 1, (N, F)).astype(np.float32)
    a = rng.uniform(0.001, 0.9, (N, 1)).astype(np.float32)
    y0 = rng.uniform(-1, 1, (N, 1)).astype(np.float32)
    ya = y0[:, 0].copy()
    want = oracle.onepole_run(ya, a[:, 0].copy(), N, F, inp)
    b = ctx.batch(st.ONEPOLE, N, layout=getattr(st, layout))
    b.upload_state(y0); b.upload_param(a)
    il = layout == "INTERLEAVED"
    out = np.zeros((F, N) if il else (N, F), np.float32)
    b.run(F, inp=np.ascontiguousarray(inp.T) if il else inp, out=out)
    assert np.array_equal((out.T if il else out).view(np.uint32), want.view(np.uint32))
    assert np.array_equal(b.download_state().view(np.float32)[:, 0], ya)
    b.free()


@pytest.mark.parametrize("layout", ["PLANAR", "INTERLEAVED"])
@pytest.mark.parametrize("N,F,chunk", [(1, 100000, 0), (3, 65536, 0), (40, 5000, 96), (130, 777, 50), (2, 64, 0)])
def test_onepole_scan(st, ctx, oracle, layout, N, F, chunk):
    """Time-parallel one-pole (block scan of the affine recurrence over the time axis): at these
    coefficients (a 5e-4..0.5 on noise plus a slow sine), where the sequential render does not stall and
    is itself within ~1e-6 of the exact recurrence, within 1e-5 of the peak / 120 dB SNR of the
    sequential oracle, final state included.  At small coefficients the sequential float render drifts
    from the exact result and the scan is the more accurate of the two: the contract against the fp64
    recurrence, instance by instance, is tests/test_gpu_float_ref.py."""
    inp = rng.uniform(-1, 1, (N, F)).astype(np.float32)
    inp += np.sin(np.arange(F) * 0.001).astype(np.float32)            # slow component: the filter output is not just noise
    a = rng.uniform(0.0005, 0.5, (N, 1)).astype(np.float32)
    y0 = rng.uniform(-1, 1, (N, 1)).astype(np.float32)
    ya = y0[:, 0].copy()
    want = oracle.onepole_run(ya, a[:, 0].copy(), N, F, inp)
    ctx.set_option("xvoice_chunk", chunk)
    try:
        b = ctx.batch(st.ONEPOLE, N, layout=getattr(st, layout), mode=1)
        b.upload_state(y0); b.upload_param(a)
        il = layout == "INTERLEAVED"
        out = np.zeros((F, N) if il else (N, F), np.float32)
        l0 = ctx.launches
        b.run(F, inp=np.ascontiguousarray(inp.T) if il else inp, out=out)
        if F > 64:
            assert ctx.launches - l0 == 3                  # zero-state pass, scan, render
        got = (out.T if il else out).astype(np.float64)
        w64 = want.astype(np.float64)
        assert np.abs(got - w64).max() <= 1e-5 * np.abs(w64).max()
        assert 10 * np.log10((w64 ** 2).sum() / max(((got - w64) ** 2).sum(), 1e-300)) >= 120.0
        assert np.abs(b.download_state().view(np.float32)[:, 0].astype(np.float64) - ya).max() <= 1e-5 * max(1.0, np.abs(ya).max())
        b.free()
    finally:
        ctx.set_option("xvoice_chunk", 0)


def test_xvoice_mix_uniform_phase_chunks(st, ctx, oracle, mixgen):
    """Mix-only render where whole warps sit in one envelope phase (sustain at 1, released at 0,
    long attacks / releases) -- the three-instruction envelope path -- next to warps with gate
    crossings, negative and -0.0 rates and out-of-range envelopes, which must take the general path:
    final state of every voice bit-exact, mix within the stated tolerance."""
    N, F = 148 * 4 * 128 * 2 + 77, 96
    s0, prm = _xvoice_inputs(oracle, N)
    third = N // 3
    prm["gate_frames"][:third] = 10**6                       # attack for the whole render
    prm["gate_frames"][third:2 * third] = 0                  # release from the first tick
    s0["env"][:third:2] = 1.0                                # sustained
    s0["env"][third:2 * third] = rng.uniform(0, 1, third).astype(np.float32)
    s0["env"][third + 1:2 * third:5] = 0.0                   # already silent
    s0["t"][third:2 * third] = rng.integers(0, 1000, third)
    odd = slice(2 * third, N)                                 # general-path voices
    prm["env_attack"][2 * third + 1:N:7] = -0.01
    prm["env_release"][2 * third + 2:N:7] = np.float32(-0.0)
    s0["env"][2 * third + 3:N:7] = 1.5
    s0["env"][2 * third + 4:N:7] = np.float32(-0.0)
    sa = s0.copy()
    _, want_mix = oracle.xvoice_run(sa, prm, N, F, want_raw=False)
    b = ctx.batch(st.XVOICE, N)
    b.upload_state(s0.view(np.uint32).reshape(N, 5)); b.upload_param(prm.view(np.uint32).reshape(N, 8))
    mix = np.zeros((2, F), np.float32)
    b.run(F, mix=mix)
    got = b.download_state().view(po.xvoice_state_dtype).reshape(N)
    assert np.array_equal(got.view(np.uint32), sa.view(np.uint32))
    w64, g64 = np.asarray(want_mix, np.float64).reshape(2, F), mix.astype(np.float64)
    assert np.abs(g64 - w64).max() <= 1e-5 * np.abs(w64).max()
    b.free()


# ------------------------------------------------------------ device-resident path
def test_run_dev_and_stream(st, ctx, oracle):
    """Device-pointer API and the chunked host stream give the same bytes as run()."""
    N, F, ctl, order, bank = 300, 2048, 8, 2, 3
    nb = (N + bank - 1) // bank
    chan0 = rng.integers(0, 2**32, (N, 5 + order), dtype=np.uint32)
    prng0 = rng.integers(1, 2**32, nb, dtype=np.uint32)
    sp = po.pdm_setpoints(N, F // (1 << ctl))
    ca, pa = chan0.copy(), prng0.copy()
    want, _ = oracle.pdm_v2_run(ca, order, N, bank, pa, None, 0x3FF, 0, ctl, 24, sp, F)
    b = ctx.batch(st.PDM_V2, N, order=order, bank_size=bank, ctl_div_log=ctl, layout=st.TILED)
    # (1) device pointers
    b.upload_state(chan0); b.upload_bank(prng0, 0)
    d_out = ctx.dev_alloc(N * F); d_sp = ctx.dev_alloc(sp.nbytes)
    ctx.h2d(d_sp, sp)
    l0 = ctx.launches
    b.run_dev(F, ctl=d_sp, n_ctl=sp.shape[0], out=d_out)
    assert ctx.launches == l0 + 1
    got = np.zeros(N * F, np.uint8)
    ctx.d2h(got, d_out)
    assert np.array_equal(tiled16_to_planar(got, N, F), want)
    ctx.dev_free(d_out); ctx.dev_free(d_sp)
    # (2) chunked stream into pinned host memory, ring of 2 slabs + callback
    b.upload_state(chan0); b.upload_bank(prng0, 0)
    Fc = 512
    ring, ring_ptr = ctx.host_alloc(2 * N * Fc)
    seen = []

    def on_chunk(user, k, slab, nbytes):
        a = np.ctypeslib.as_array((__import__("ctypes").c_uint8 * nbytes).from_address(slab)).copy()
        seen.append((k, tiled16_to_planar(a, N, Fc)))

    b.run_stream(F, Fc, out=ring_ptr, ctl=sp, ring_chunks=2, on_chunk=on_chunk)
    assert [k for k, _ in seen] == list(range(F // Fc))
    assert np.array_equal(np.concatenate([a for _, a in seen], axis=1), want)
    assert np.array_equal(b.download_state(), ca)
    ctx.host_free(ring_ptr)
    b.free()


@pytest.mark.parametrize("layout", ["PLANAR", "INTERLEAVED"])
@pytest.mark.parametrize("N,F", [(300, 1000), (3, 64), (40, 1023), (1, 4096)])
def test_word_clock(st, ctx, oracle, layout, N, F):
    """linux/clock.c:109-120 as a batch: integer-divisor square waves, bit-exact against the restated loop
    over two consecutive blocks (state carried), including half periods of 0, 1, negative and huge values."""
    hp = rng.integers(1, 200, N).astype(np.int32)
    special = np.array([0, 1, -5, 2**31 - 1, 2, 500, 62, 8], np.int32)
    hp[:min(N, len(special))] = special[:min(N, len(special))]
    s0 = np.zeros((N, 2), np.int32); s0[:, 0] = rng.integers(0, 300, N); s0[:, 1] = rng.integers(0, 2, N)
    if N > 8:
        s0[8] = (2**31 - 3, 7)                                 # the phase counter wraps; pol is any integer
    sa = s0.copy()
    b = ctx.batch(st.WORD_CLOCK, N, layout=getattr(st, layout))
    b.upload_state(s0.view(np.uint32)); b.upload_param(hp.view(np.uint32).reshape(N, 1))
    for blk in range(2):
        want = oracle.word_clock_run(sa, hp, N, F)
        out = np.zeros((N, F) if layout == "PLANAR" else (F, N), np.float32)
        b.run(F, out=out)
        got = out if layout == "PLANAR" else out.T
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), blk
        assert np.array_equal(b.download_state().view(np.int32), sa)
    b.free()


@pytest.mark.parametrize("use_graph", [1, 0, 2, 3])
def test_small_blocks_replay_as_cuda_graph(st, ctx, oracle, use_graph):
    """cproc_cuda_run with host buffers: from the third call with one shape on, a period is two memcpys around one
    cudaGraphLaunch (captured at the second call: 1 = H2D, kernels, D2H; 2 = the kernels alone, working on the pinned
    staging; 3 = no graph, direct launches on the pinned staging; 0 = staged copies).  Eight consecutive periods of five processors,
    a shape change in the middle, state uploads between periods: bit-exact against the oracle either way, and the
    launch counter keeps counting the kernels of the replays."""
    ctx.set_option("run_graph", use_graph)
    try:
        F = 64
        # test_cproc chain, 3 voices
        b = ctx.batch(st.GRAPH, 3, nodes=po.GRAPH_TEST_CPROC)
        s = np.zeros((3, 3), np.uint32); sa = s.copy(); b.upload_state(s)
        per = []
        for k in range(8):
            f = F if k != 4 else 96                          # one period of another size
            x = rng.integers(0, 2, (3, f), dtype=np.uint32)
            want = oracle.graph_run(po.GRAPH_TEST_CPROC, 1, 1, sa, 3, f, x)
            out = np.zeros((3, f), np.uint32)
            l0 = ctx.launches
            b.run(f, inp=x, out=out)
            per.append(ctx.launches - l0)
            assert np.array_equal(out, want), k
        assert np.array_equal(b.download_state(), sa) and len(set(per)) == 1 and per[0] >= 1
        b.free()
        # voice bank with a note change between periods (state upload), word clock, square_grain in place, one-pole
        V = 128
        voices = np.zeros((V, 2), np.uint32); voices[::3, 0] = [oracle.note_to_inc(int(n)) for n in rng.integers(30, 90, len(voices[::3]))]
        vb = ctx.batch(st.VOICE_BANK, V, voices_per_bus=64)
        hp = np.array([62, 500, 8], np.int32); cs = np.zeros((3, 2), np.int32); cs[:, 1] = 1; csa = cs.copy()
        cb = ctx.batch(st.WORD_CLOCK, 3); cb.upload_state(cs.view(np.uint32)); cb.upload_param(hp.view(np.uint32).reshape(3, 1))
        G = 5
        gth = rng.uniform(0.05, 0.5, (G, 1)).astype(np.float32); gst = np.zeros(G, np.float32)
        gb = ctx.batch(st.SQUARE_GRAIN, G); gb.upload_param(gth)
        a = rng.uniform(0.01, 0.5, (G, 1)).astype(np.float32); y = np.zeros(G, np.float32)
        ob = ctx.batch(st.ONEPOLE, G); ob.upload_param(a)
        for k in range(8):
            if k == 5:
                voices[1, 0] = oracle.note_to_inc(69)
            vb.upload_state(voices)
            _, want = oracle.voice_bank_run(voices, V, 64, po.MIX_SAW, F)
            out = np.zeros((2, F), np.float32)
            vb.run(F, out=out)
            voices = vb.download_state()
            assert np.array_equal(out.view(np.uint32), want.view(np.uint32)), k
            wantc = oracle.word_clock_run(csa, hp, 3, F)
            outc = np.zeros((3, F), np.float32)
            cb.run(F, out=outc)
            assert np.array_equal(outc, wantc), k
            x = rng.uniform(-1, 1, (G, F)).astype(np.float32)
            wantg = oracle.square_grain_run(gst, gth[:, 0].copy(), G, F, x)
            io = x.copy()
            gb.run(F, inp=io, out=io)                        # in place, as Pd does
            assert np.array_equal(io.view(np.uint32), wantg.view(np.uint32)), k
            wanto = oracle.onepole_run(y, a[:, 0].copy(), G, F, x)
            outo = np.zeros((G, F), np.float32)
            ob.run(F, inp=x, out=outo)
            assert np.array_equal(outo.view(np.uint32), wanto.view(np.uint32)), k
        assert np.array_equal(cb.download_state().view(np.int32), csa)
        for q in (vb, cb, gb, ob):
            q.free()
    finally:
        ctx.set_option("run_graph", 2)
