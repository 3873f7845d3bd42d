"""A reduced pass over every kernel family for compute-sanitizer (tools/sanitize.sh): small shapes, each checked against the oracle.
    compute-sanitizer --tool {memcheck|racecheck|synccheck|initcheck} python tools/sanitize_subset.py"""
import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import __graft_entry__ as ge
import synth_tools_b200 as st
from oracle import pyoracle as po

ge.smoke()                       # k_pdm_v2_ws4 (static + dynamic schedule), k_voice_mix, k_planar_tma<GrainOp>, graph_planar_tma (int and float graphs)
orc = po.Oracle()
ctx = st.Context(0)
rng = np.random.default_rng(1)

# PDM v2 PLANAR rows through tensor-TMA boxes, orders 1..4, ragged bank
for order, bank in ((1, 3), (2, 5), (3, 3), (4, 2)):
    N, F = 1000 + order, 512
    chan = rng.integers(0, 2**32, (N, 5 + order), dtype=np.uint32)
    nb = (N + bank - 1) // bank
    prng = rng.integers(1, 2**32, nb, dtype=np.uint32)
    sp = po.pdm_setpoints(N, F // 64 + 1)
    ca, pa = chan.copy(), prng.copy()
    want, _ = orc.pdm_v2_run(ca, order, N, bank, pa, None, 0x3FF, 0, 6, 24, sp, F)
    b = ctx.batch(st.PDM_V2, N, order=order, bank_size=bank, ctl_div_log=6, layout=st.PLANAR)
    b.upload_state(chan); b.upload_bank(prng, 0)
    out = np.zeros((N, F), np.uint8)
    b.run(F, ctl=sp, out=out)
    assert np.array_equal(out, want) and np.array_equal(b.download_state(), ca), "pdm_v2 planar order %d" % order
    b.free()
# PDM v1 (TILED + PLANAR), pdm raw planar (k_planar_tma), pwm, word clock, one-pole
N, F = 2048, 256
ch = np.zeros((N, 2), np.uint32); ch[:, 0] = rng.integers(0x40000000, 0xC0000000, N, dtype=np.uint32)
pr = (np.arange(N // 2) + 1).astype(np.uint32)
cha, pra = ch.copy(), pr.copy()
bits = orc.pdm_v1_run(cha, N, 2, pra, None, 0x0FFFFFFF, F)
for layout in (st.PLANAR, st.INTERLEAVED):
    b = ctx.batch(st.PDM_V1, N, bank_size=2, dither_mask=0x0FFFFFFF, layout=layout)
    b.upload_state(ch); b.upload_bank(pr)
    out = np.zeros((N, F // 32) if layout == st.PLANAR else (F // 32, N), np.uint32)
    b.run(F, out=out)
    got = out if layout == st.PLANAR else out.T
    assert np.array_equal(np.ascontiguousarray(got).view(np.uint8), np.packbits(bits, axis=1, bitorder="little")), "pdm v1"
    b.free()
inp = rng.integers(0, 2**32, (N, F), dtype=np.uint32); s2 = np.zeros((N, 2), np.uint32); sa = s2.copy()
want = orc.pdm_run(2, sa, N, F, inp, None, 24, None)
b = ctx.batch(st.PDM, N, order=2, out_shift=24); o = np.zeros((N, F), np.uint32); b.run(F, inp=inp, out=o)
assert np.array_equal(o, want), "pdm raw"
b.free()
# extension voice: raw (k_xvoice), mix (k_xvoice_mix2 and k_xvoice_mix), time-parallel scan
Nx, Fx = 3000, 96
xs = np.zeros(Nx, po.xvoice_state_dtype); xs["phase"] = rng.integers(0, 2**32, Nx, dtype=np.uint32)
xp = np.zeros(Nx, po.xvoice_param_dtype)
xp["inc"] = rng.integers(1 << 20, 1 << 28, Nx); xp["f"] = rng.uniform(0.01, 0.3, Nx); xp["q"] = rng.uniform(0.5, 2, Nx)
xp["env_attack"] = 0.01; xp["env_release"] = 0.002; xp["gate_frames"] = rng.integers(0, 90, Nx); xp["gl"] = 0.5; xp["gr"] = 0.5
xa = xs.copy()
raw, mix = orc.xvoice_run(xa, xp, Nx, Fx)
for gen in (1, 0):
    ctx.set_option("xvoice_mix2", gen)
    b = ctx.batch(st.XVOICE, Nx)
    b.upload_state(xs.view(np.uint32).reshape(Nx, 5)); b.upload_param(xp.view(np.uint32).reshape(Nx, 8))
    m = np.zeros((2, Fx), np.float32)
    b.run(Fx, mix=m)
    assert np.abs(m - mix).max() <= 1e-5 * np.abs(mix).max() and np.array_equal(b.download_state(), xa.view(np.uint32).reshape(Nx, 5)), "xvoice mix %d" % gen
    b.free()
b = ctx.batch(st.XVOICE, Nx)
b.upload_state(xs.view(np.uint32).reshape(Nx, 5)); b.upload_param(xp.view(np.uint32).reshape(Nx, 8))
r = np.zeros((Nx, Fx, 2), np.float32)
b.run(Fx, out=r)
assert np.array_equal(r.view(np.uint32), raw.reshape(Nx, Fx, 2).view(np.uint32)), "xvoice raw"
b.free()
# square_grain mix (k_grain_mix3), interleaved square_grain (k_interleaved4<GrainOp>), graph interleaved4, graph scan, patcher
Ng, Fg = 4096, 64
gs = np.zeros((Ng, 2), np.uint32); gs[:, 1] = rng.integers(0, 2**32, Ng, dtype=np.uint32)
gp = np.zeros((Ng, 4), np.uint32); gp[:, 0] = rng.uniform(0.05, 0.5, Ng).astype(np.float32).view(np.uint32); gp[:, 1] = rng.integers(1 << 20, 1 << 26, Ng)
gl = rng.integers(0, 65, Ng); gp[:, 2] = gl; gp[:, 3] = 64 - gl
b = ctx.batch(st.SQUARE_GRAIN_MIX, Ng); b.upload_state(gs); b.upload_param(gp)
im = np.zeros((2, Fg), np.int32); b.run(Fg, mix=im)
sta = np.zeros(Ng, np.float32); pha = gs[:, 1].copy()
wim, _ = orc.square_grain_mix_run(sta, gp[:, 0].copy().view(np.float32), pha, gp[:, 1].copy(), gl.astype(np.uint8), (64 - gl).astype(np.uint8), Ng, Fg)
assert np.array_equal(im, wim.reshape(2, Fg)), "grain mix"
b.free()
gi = rng.uniform(-1, 1, (Fg, Ng)).astype(np.float32)
b = ctx.batch(st.SQUARE_GRAIN, Ng, layout=st.INTERLEAVED); b.upload_param(gp[:, :1].copy())
go = np.zeros((Fg, Ng), np.float32); b.run(Fg, inp=gi, out=go)
s0 = np.zeros(Ng, np.float32)
assert np.array_equal(np.ascontiguousarray(go.T).view(np.uint32), orc.square_grain_run(s0, gp[:, 0].copy().view(np.float32), Ng, Fg, np.ascontiguousarray(gi.T)).view(np.uint32)), "grain interleaved"
b.free()
rows = po.GRAPH_BP5
gin = rng.integers(0, 2, (Fg, 1, Ng), dtype=np.uint32)
b = ctx.batch(st.GRAPH, Ng, nodes=rows, layout=st.INTERLEAVED)
gout = np.zeros((Fg, Ng), np.uint32); b.run(Fg, inp=gin, out=gout)
gst = np.zeros((Ng, 4), np.uint32)
assert np.array_equal(gout.T, orc.graph_run(rows, 1, 2, gst, Ng, Fg, np.ascontiguousarray(gin.transpose(2, 1, 0)))), "graph interleaved4"
b.free()
Fs = 4096
gin = rng.integers(0, 2, (2, 1, Fs), dtype=np.uint32)
b = ctx.batch(st.GRAPH, 2, nodes=po.GRAPH_TEST_CPROC, mode=1)
gout = np.zeros((2, Fs), np.uint32); b.run(Fs, inp=gin, out=gout)
gst = np.zeros((2, 3), np.uint32)
assert np.array_equal(gout, orc.graph_run(po.GRAPH_TEST_CPROC, 1, 1, gst, 2, Fs, gin)), "graph scan"
b.free()
# the mix bus kernels on one rank (k_bus_allreduce; fused exchange inside k_voice_mix)
bus = st.Bus(ctx, 1024, 1, 0)
bus.connect([bus.handle()])
Nv, Fv = 64 * 64, 128
v = np.zeros((Nv, 2), np.uint32); v[:, 0] = rng.integers(1 << 20, 1 << 28, Nv); v[:, 1] = rng.integers(0, 2**32, Nv, dtype=np.uint32)
va = v.copy()
isum, vec = orc.voice_bank_run(va, Nv, Nv, 0, Fv)
b = ctx.batch(st.VOICE_BANK, Nv, voices_per_bus=0); b.upload_state(v)
bus.attach(b, 1)
d_mix = ctx.dev_alloc(4 * Fv); d_out = ctx.dev_alloc(4 * Fv)
b.run_dev(Fv, out=d_out, mix=d_mix); ctx.sync()
hm = np.zeros(Fv, np.int32); ctx.d2h(hm, d_mix)
assert np.array_equal(hm, isum.reshape(-1)) and bus.status() == 0, "fused bus"
bus.detach(b); b.free(); bus.destroy()
print("sanitize subset ok: %d launches" % ctx.launches)
ctx.close()
