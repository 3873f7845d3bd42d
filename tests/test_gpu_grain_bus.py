"""GPU: the square_grain mix (SQUARE_GRAIN_MIX) with a mix bus attached (cproc_cuda_bus_attach), world = 1.

The render launch exchanges its own mix: the render blocks accumulate into a batch-owned accumulator that every
launch leaves zero, the last block to finish pushes it to the bus, and the bus writes io.mix (int32) and io.out
((float)x * 2^-7).  Mode 1 completes the exchange in the same launch; mode 2 completes it in block 0 of the next
launch (or in bus_flush).  All three kernel generations carry that tail; everything is compared bit for bit with
the oracle, block after block."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
rng = np.random.default_rng(20261021)


@pytest.fixture(scope="module")
def st():
    import synth_tools_b200 as st_
    return st_


@pytest.fixture(scope="module")
def ctx(st):
    c = st.Context(0)
    yield c
    c.close()


def _grains(oracle, N, th_kind="pos"):
    """state, threshold, phase, inc, gl, gr.  th_kind "neg": some negative thresholds (both flip conditions can hold:
    the two-branch kernels k_grain_mix2 / k_grain_mix take over); "unrep": some below -1 as well (no integer
    threshold exists: k_grain_mix whatever grain_mix2 says)."""
    state = rng.choice(np.array([0.0, 0.5, -0.5], np.float32), N)
    th = rng.uniform(0.05, 0.5, N).astype(np.float32)
    th[0] = 0.0
    _set_th(th, th_kind)
    phase = rng.integers(0, 2**32, N, dtype=np.uint32)
    inc = np.array([oracle.note_to_inc(int(n)) for n in rng.integers(36, 97, N)], np.uint32)
    gl = rng.integers(0, 65, N).astype(np.uint8)
    gr = (64 - gl).astype(np.uint8)
    return state, th, phase, inc, gl, gr


def _set_th(th, kind):
    if kind in ("neg", "unrep"):
        th[1::7] = -np.abs(th[1::7])
    if kind == "unrep":
        th[3::11] = -1.5


def _batch(st, ctx, g):
    state, th, phase, inc, gl, gr = g
    N = state.size
    b = ctx.batch(st.SQUARE_GRAIN_MIX, N)
    s_rec = np.zeros((N, 2), np.uint32); s_rec[:, 0] = state.view(np.uint32); s_rec[:, 1] = phase
    b.upload_state(s_rec)
    _upload_param(b, g)
    return b


def _upload_param(b, g):
    _, th, _, inc, gl, gr = g
    p_rec = np.zeros((th.size, 4), np.uint32)
    p_rec[:, 0] = th.view(np.uint32); p_rec[:, 1] = inc; p_rec[:, 2] = gl; p_rec[:, 3] = gr
    b.upload_param(p_rec)


def _oracle_block(oracle, g, F):
    """The next block of the oracle; advances the state and phase of `g` in place."""
    state, th, phase, inc, gl, gr = g
    return oracle.square_grain_mix_run(state, th, phase, inc, gl, gr, state.size, F)


def _assert_state(b, g):
    s = b.download_state()
    assert np.array_equal(s[:, 0], g[0].view(np.uint32)) and np.array_equal(s[:, 1], g[2])


def _bufs(ctx, K, F):
    return [ctx.dev_alloc(8 * F) for _ in range(K)], [ctx.dev_alloc(8 * F) for _ in range(K)]


def _check_blocks(ctx, d_mix, d_out, wants, F, used):
    mix = np.zeros((2, F), np.int32); out = np.zeros((2, F), np.float32)
    for k, (w_i, w_f) in enumerate(wants):
        want_mix, want_out = used[k]
        if want_mix:
            ctx.d2h(mix, d_mix[k])
            assert np.array_equal(mix, w_i), "block %d: mix" % k
        if want_out:
            ctx.d2h(out, d_out[k])
            assert np.array_equal(out.view(np.uint32), w_f.view(np.uint32)), "block %d: out" % k


def _run_blocks(st, ctx, oracle, b, g, F, K, d_mix, d_out, before=None):
    """K consecutive blocks; block k % 3 == 1 passes out=None, k % 3 == 2 mix=None."""
    wants, used = [], []
    for k in range(K):
        if before:
            before(k)
        use_mix, use_out = k % 3 != 2, k % 3 != 1
        wants.append(_oracle_block(oracle, g, F))
        used.append((use_mix, use_out))
        b.run_dev(F, mix=d_mix[k] if use_mix else None, out=d_out[k] if use_out else None)
    return wants, used


@pytest.mark.parametrize("bus_mode", [1, 2])
@pytest.mark.parametrize("gen", [0, 1, 2])
@pytest.mark.parametrize("N,F,th_kind", [(3000, 256, "pos"), (70000, 200, "pos"), (517, 37, "pos"), (5, 64, "pos"),
                                         (3000, 128, "neg"), (3000, 128, "unrep")])
def test_grain_mix_bus(st, ctx, oracle, bus_mode, gen, N, F, th_kind):
    """Six consecutive blocks with the bus attached equal the oracle continued block by block, for every kernel
    generation (grain_mix2 0..2; "neg" / "unrep" thresholds force the fallback kernels); ragged chunks, fewer grains
    than a warp, blocks without io.mix or io.out.  Detached again, the launch writes its own mix."""
    g = _grains(oracle, N, th_kind)
    ctx.set_option("grain_mix2", gen)
    try:
        b = _batch(st, ctx, g)
        bus = st.Bus(ctx, 2 * F, 1, 0)
        bus.attach(b, bus_mode)
        K = 6
        d_mix, d_out = _bufs(ctx, K, F)
        wants, used = _run_blocks(st, ctx, oracle, b, g, F, K, d_mix, d_out)
        bus.flush()
        ctx.sync()
        assert bus.status() == 0
        _check_blocks(ctx, d_mix, d_out, wants, F, used)
        _assert_state(b, g)
        bus.detach(b)
        w = _oracle_block(oracle, g, F)
        b.run_dev(F, mix=d_mix[0], out=d_out[0])
        ctx.sync()
        _check_blocks(ctx, d_mix, d_out, [w], F, [(True, True)])
        _assert_state(b, g)
        bus.destroy(); b.free()
        for p in d_mix + d_out:
            ctx.dev_free(p)
    finally:
        ctx.set_option("grain_mix2", 2)


@pytest.mark.parametrize("gen", [1, 2])
def test_grain_mix_bus_reserved_slot(st, ctx, oracle, gen):
    """Pipelined, one render block per SM: the render grid is capped one block short of the chip so that the
    exchange block (block 0) has its own slot; the grid-stride walk over the grains uses the render blocks only."""
    N, F = 200000, 256
    g = _grains(oracle, N)
    ctx.set_option("grain_mix2", gen)
    ctx.set_option("grain_blocks_per_sm", 1)
    try:
        b = _batch(st, ctx, g)
        bus = st.Bus(ctx, 2 * F, 1, 0)
        bus.attach(b, 2)
        K = 4
        d_mix, d_out = _bufs(ctx, K, F)
        wants, used = _run_blocks(st, ctx, oracle, b, g, F, K, d_mix, d_out)
        bus.flush()
        ctx.sync()
        assert bus.status() == 0
        _check_blocks(ctx, d_mix, d_out, wants, F, used)
        _assert_state(b, g)
        bus.destroy(); b.free()
        for p in d_mix + d_out:
            ctx.dev_free(p)
    finally:
        ctx.set_option("grain_blocks_per_sm", 2)
        ctx.set_option("grain_mix2", 2)


@pytest.mark.parametrize("bus_mode", [1, 2])
def test_grain_mix_bus_four_blocks_per_launch(st, ctx, oracle, bus_mode):
    """One launch of 4 x 256 frames (one exchange of [2][1024]) equals four launches of 256 frames, per channel."""
    N, F = 70000, 256
    g = _grains(oracle, N)
    g4 = tuple(x.copy() for x in g)
    b1, b4 = _batch(st, ctx, g), _batch(st, ctx, g4)
    bus1, bus4 = st.Bus(ctx, 2 * F, 1, 0), st.Bus(ctx, 8 * F, 1, 0)
    bus1.attach(b1, bus_mode); bus4.attach(b4, bus_mode)
    d_mix, d_out = _bufs(ctx, 4, F)
    d_mix4, d_out4 = ctx.dev_alloc(32 * F), ctx.dev_alloc(32 * F)
    for k in range(4):
        b1.run_dev(F, mix=d_mix[k], out=d_out[k])
    b4.run_dev(4 * F, mix=d_mix4, out=d_out4)
    bus1.flush(); bus4.flush()
    ctx.sync()
    assert bus1.status() == 0 and bus4.status() == 0
    mix4 = np.zeros((2, 4 * F), np.int32); out4 = np.zeros((2, 4 * F), np.float32)
    ctx.d2h(mix4, d_mix4); ctx.d2h(out4, d_out4)
    w_i, w_f = _oracle_block(oracle, g4, 4 * F)
    assert np.array_equal(mix4, w_i) and np.array_equal(out4.view(np.uint32), w_f.view(np.uint32))
    mix = np.zeros((2, F), np.int32); out = np.zeros((2, F), np.float32)
    for k in range(4):
        ctx.d2h(mix, d_mix[k]); ctx.d2h(out, d_out[k])
        for c in range(2):
            assert np.array_equal(mix[c], mix4[c, k * F:(k + 1) * F]), (k, c)
            assert np.array_equal(out[c].view(np.uint32), out4[c, k * F:(k + 1) * F].view(np.uint32)), (k, c)
    assert np.array_equal(b1.download_state(), b4.download_state())
    _assert_state(b4, g4)
    for x in (bus1, bus4):
        x.destroy()
    b1.free(); b4.free()
    for p in d_mix + d_out + [d_mix4, d_out4]:
        ctx.dev_free(p)


def test_grain_mix_bus_generation_change_mid_pipeline(st, ctx, oracle):
    """Pipelined: parameter uploads between blocks switch the kernel generation (k_grain_mix3 -> k_grain_mix2 ->
    k_grain_mix) while the previous block's exchange is pending; whichever generation launches completes it."""
    N, F = 20000, 256
    g = _grains(oracle, N)
    b = _batch(st, ctx, g)
    bus = st.Bus(ctx, 2 * F, 1, 0)
    bus.attach(b, 2)
    K = 6
    d_mix, d_out = _bufs(ctx, K, F)
    base = g[1].copy()

    def before(k):
        kind = {3: "neg", 5: "unrep"}.get(k)
        if kind:
            g[1][:] = base
            _set_th(g[1], kind)
            _upload_param(b, g)

    wants, used = _run_blocks(st, ctx, oracle, b, g, F, K, d_mix, d_out, before=before)
    bus.flush()
    ctx.sync()
    assert bus.status() == 0
    _check_blocks(ctx, d_mix, d_out, wants, F, used)
    _assert_state(b, g)
    bus.destroy(); b.free()
    for p in d_mix + d_out:
        ctx.dev_free(p)


def test_grain_mix_bus_errors(st, ctx, oracle):
    N, F = 1000, 64
    bus = st.Bus(ctx, 2 * F, 1, 0)
    raw = ctx.batch(st.SQUARE_GRAIN, N)                    # no mix: nothing to exchange
    with pytest.raises(st.CprocCudaError) as e:
        bus.attach(raw, 1)
    assert e.value.code == st.abi.EINVAL
    raw.free()
    g = _grains(oracle, N)
    b = _batch(st, ctx, g)
    d_mix, d_out = _bufs(ctx, 2, F)
    small = st.Bus(ctx, 100, 1, 0)                         # 2 x 64 words do not fit in 100
    small.attach(b, 1)
    with pytest.raises(st.CprocCudaError) as e:
        b.run_dev(F, mix=d_mix[0], out=d_out[0])
    assert e.value.code == st.abi.EINVAL
    small.detach(b); small.destroy()
    bus.attach(b, 1)
    with pytest.raises(st.CprocCudaError) as e:            # out and mix both NULL
        b.run_dev(F)
    assert e.value.code == st.abi.EINVAL
    # none of the refused calls rendered: the state is still that of the upload
    wants = [_oracle_block(oracle, g, F)]
    bus.attach(b, 2)
    b.run_dev(F, mix=d_mix[0], out=d_out[0])
    bus.attach(b, 1)
    with pytest.raises(st.CprocCudaError) as e:            # mode 1 while a pipelined exchange is pending
        b.run_dev(F, mix=d_mix[1], out=d_out[1])
    assert e.value.code == st.abi.ESTATE
    bus.flush()
    wants.append(_oracle_block(oracle, g, F))
    b.run_dev(F, mix=d_mix[1], out=d_out[1])
    ctx.sync()
    assert bus.status() == 0
    _check_blocks(ctx, d_mix, d_out, wants, F, [(True, True)] * 2)
    _assert_state(b, g)
    bus.destroy(); b.free()
    for p in d_mix + d_out:
        ctx.dev_free(p)
