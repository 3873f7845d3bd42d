"""Run ONE configuration a few times (for ncu launch lists / --set full captures).
usage: python tools/prof_one.py {grain|grain_il|gmix|xvoice|sweep|sweep_planar|voice} [reps]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import synth_tools_b200 as st

which = sys.argv[1]
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 2
ctx = st.Context(0)
rng = np.random.default_rng(0)
for kv in sys.argv[3:]:
    k, v = kv.split("=")
    ctx.set_option(k, int(v))

def note_incs(n, lo=24, hi=109):
    tab12 = np.array([594573364, 629928536, 667386036, 707070875, 749115497, 793660223, 840853716, 890853479,
                      943826384, 999949221, 1059409296, 1122405051], np.uint32)
    notes = rng.integers(lo, hi, n)
    octave = np.where(notes < 8, 10, 9 - (notes - 8) // 12)
    idx = np.where(notes < 8, notes + 4, (notes - 8) % 12)
    return (tab12[idx] >> octave.astype(np.uint32)).astype(np.uint32)

def xvoice_records(N):
    prm = np.zeros((N, 8), np.uint32)
    prm[:, 0] = note_incs(N)
    prm[:, 1] = rng.uniform(0.01, 0.3, N).astype(np.float32).view(np.uint32)
    prm[:, 2] = rng.uniform(0.5, 2.0, N).astype(np.float32).view(np.uint32)
    prm[:, 3] = rng.uniform(1e-3, 1e-1, N).astype(np.float32).view(np.uint32)
    prm[:, 4] = rng.uniform(1e-3, 1e-2, N).astype(np.float32).view(np.uint32)
    prm[:, 5] = rng.integers(0, 400, N)
    g = rng.uniform(0, 1, N).astype(np.float32)
    prm[:, 6] = g.view(np.uint32); prm[:, 7] = (1 - g).astype(np.float32).view(np.uint32)
    stt = np.zeros((N, 5), np.uint32); stt[:, 0] = rng.integers(0, 2**32, N, dtype=np.uint32)
    return stt, prm

def timed(fn):
    fn(); ctx.sync()
    best = 1e9
    for _ in range(reps):
        ctx.timer_start(); fn(); best = min(best, ctx.timer_stop())
    return best

if which in ("grain", "grain_il"):
    N, F = int(os.environ.get("GRAIN_N", 1024 * 1024)), 256
    d_in = ctx.dev_alloc(4 * N * F); d_out = ctx.dev_alloc(4 * N * F)
    chunk = rng.uniform(-1, 1, (65536, F)).astype(np.float32)
    for k in range(N // 65536):
        ctx.h2d(d_in + k * chunk.nbytes, chunk)
    b = ctx.batch(st.SQUARE_GRAIN, N, layout=st.INTERLEAVED if which == "grain_il" else st.PLANAR)
    b.upload_param(rng.uniform(0.05, 0.5, (N, 1)).astype(np.float32))
    ms = timed(lambda: b.run_dev(F, inp=d_in, out=d_out))
    print("%s: %.3f ms  %.0f GB/s" % (which, ms, 8 * N * F / ms / 1e6))
elif which == "gmix":
    N, F = 1024 * 1024, 256
    s_rec = np.zeros((N, 2), np.uint32); s_rec[:, 1] = rng.integers(0, 2**32, N, dtype=np.uint32)
    p_rec = np.zeros((N, 4), np.uint32)
    p_rec[:, 0] = rng.uniform(0.05, 0.5, N).astype(np.float32).view(np.uint32); p_rec[:, 1] = note_incs(N, 36, 97)
    gl = rng.integers(0, 65, N); p_rec[:, 2] = gl; p_rec[:, 3] = 64 - gl
    b = ctx.batch(st.SQUARE_GRAIN_MIX, N); b.upload_state(s_rec); b.upload_param(p_rec)
    d_out = ctx.dev_alloc(8 * F); d_mix = ctx.dev_alloc(8 * F)
    ms = timed(lambda: b.run_dev(F, out=d_out, mix=d_mix))
    print("gmix: %.3f ms  %.1f G grain-samples/s" % (ms, N * F / ms / 1e6))
elif which == "xvoice":
    N, F = int(os.environ.get("XV_N", 4 * 1024 * 1024)), 512
    stt, prm = xvoice_records(N)
    if os.environ.get("XV_GATE"):                     # every voice in one envelope phase: the uniform-chunk path
        prm[:, 5] = int(os.environ["XV_GATE"])
    b = ctx.batch(st.XVOICE, N); b.upload_state(stt); b.upload_param(prm)
    d_mix = ctx.dev_alloc(8 * F)
    if os.environ.get("XV_STEADY"):                 # launches after the first: every voice is past its gate (released)
        ms = timed(lambda: b.run_dev(F, mix=d_mix))
    else:                                           # the block after note-on, gates crossed inside it: state back to t = 0 before every launch
        best = 1e9
        for _ in range(reps + 1):
            b.upload_state(stt); ctx.sync()
            ctx.timer_start(); b.run_dev(F, mix=d_mix); best = min(best, ctx.timer_stop())
        ms = best
    print("xvoice mix: %.3f ms  %.1f G voice-samples/s" % (ms, N * F / ms / 1e6))
elif which in ("sweep", "sweep_planar"):
    N, F = 2048, 480000
    stt, prm = xvoice_records(N)
    d_out = ctx.dev_alloc(8 * N * F)
    b = ctx.batch(st.XVOICE, N, layout=st.PLANAR if which == "sweep_planar" else st.TILED, mode=st.XVOICE_SCAN)
    b.upload_state(stt); b.upload_param(prm)
    ms = timed(lambda: b.run_dev(F, out=d_out))
    print("%s: %.3f ms  %.0f GB/s" % (which, ms, 8 * N * F / ms / 1e6))
elif which == "voice":
    N, F = 4 * 1024 * 1024, 512
    v = np.zeros((N, 2), np.uint32); v[:, 0] = note_incs(N); v[:, 1] = rng.integers(0, 2**32, N, dtype=np.uint32)
    b = ctx.batch(st.VOICE_BANK, N, voices_per_bus=0); b.upload_state(v)
    d_out = ctx.dev_alloc(4 * F); d_mix = ctx.dev_alloc(4 * F)
    ms = timed(lambda: b.run_dev(F, out=d_out, mix=d_mix))
    print("voice: %.3f ms  %.1f G voice-samples/s" % (ms, N * F / ms / 1e6))
elif which in ("graph", "graph_il"):
    # the reference's bp5 graph (edge -> acc -> acc), 4 Mi instances x 256 ticks: 4 B in + 4 B out per tick
    N, F = 4 * 1024 * 1024, 256
    rows = [(st.NODE_EDGE, -1, 1), (st.NODE_ACC, 0, 1), (st.NODE_ACC, 1, 1)]
    d_in = ctx.dev_alloc(4 * N * F); d_out = ctx.dev_alloc(4 * N * F)
    chunk = rng.integers(0, 2, (65536, F), dtype=np.uint32)
    for k in range(N // 65536):
        ctx.h2d(d_in + k * chunk.nbytes, chunk)
    b = ctx.batch(st.GRAPH, N, nodes=rows, layout=st.INTERLEAVED if which == "graph_il" else st.PLANAR)
    ms = timed(lambda: b.run_dev(F, inp=d_in, out=d_out))
    print("%s: %.3f ms  %.0f GB/s  %.1f G ticks/s  [%s]" % (which, ms, 8 * N * F / ms / 1e6, N * F / ms / 1e6, b.jit_log.strip()))
elif which in ("gvoice", "gvoice_il"):
    # the C4 voice as a generated graph of extension processors: no input stream, two float output streams
    from tools.bench_configs import VOICE_GRAPH_TEXT
    g = st.graph_parse_ex(VOICE_GRAPH_TEXT)
    F = int(os.environ.get("GV_F", 512))            # frames per launch: the row length of the PLANAR output
    N = 2 * 1024 * 1024 * 512 // F
    stt, prm = xvoice_records(N)
    gst = np.zeros((N, 9), np.uint32); gst[:, 1] = stt[:, 0]
    d_out = ctx.dev_alloc(8 * N * F)
    b = ctx.batch(st.GRAPH, N, nodes=g["rows"], n_inputs=0, out_node=g["out_nodes"], layout=st.INTERLEAVED if which == "gvoice_il" else st.PLANAR)
    b.upload_state(gst); b.upload_param(prm)
    ms = timed(lambda: b.run_dev(F, out=d_out))
    print("%s: %.3f ms  %.0f GB/s  %.1f G ticks/s  [%s]" % (which, ms, 8 * N * F / ms / 1e6, N * F / ms / 1e6, b.jit_log.strip()))
elif which == "onepole_long":
    # 4 instances x 16 Mi frames: sequential kernel vs time-parallel scan
    N, F = 4, 16 * 1024 * 1024
    d_in = ctx.dev_alloc(4 * N * F); d_out = ctx.dev_alloc(4 * N * F)
    x = rng.uniform(-1, 1, (N, F)).astype(np.float32)
    ctx.h2d(d_in, x)
    for mode, label in ((0, "sequential"), (1, "time-parallel scan")):
        b = ctx.batch(st.ONEPOLE, N, mode=mode)
        b.upload_param(np.full((N, 1), 0.01, np.float32))
        ms = timed(lambda: b.run_dev(F, inp=d_in, out=d_out))
        print("onepole %d x %d (%s): %.3f ms  %.2f G samples/s  %.0f GB/s" % (N, F, label, ms, N * F / ms / 1e6, 8 * N * F / ms / 1e6))
        b.free()
elif which == "graph_long":
    # the reference's own shape: ONE voice of the test_cproc chain, 16 Mi ticks
    N, F = 1, 16 * 1024 * 1024
    rows = [(st.NODE_EDGE, -1, 1), (st.NODE_ACC, 0, 1)]
    d_in = ctx.dev_alloc(4 * N * F); d_out = ctx.dev_alloc(4 * N * F)
    ctx.h2d(d_in, rng.integers(0, 2, (N, F), dtype=np.uint32))
    for mode, label in ((0, "sequential (generated kernel)"), (1, "time-parallel scan")):
        b = ctx.batch(st.GRAPH, N, nodes=rows, mode=mode)
        ms = timed(lambda: b.run_dev(F, inp=d_in, out=d_out))
        print("test_cproc graph %d x %d (%s): %.3f ms  %.2f G ticks/s" % (N, F, label, ms, N * F / ms / 1e6))
        b.free()
elif which == "pdmraw":
    # pdm2_update on an input stream, 1 Mi channels x 1024 ticks, PLANAR uint32 in/out (8 B per sample)
    N, F = 1024 * 1024, 1024
    d_in = ctx.dev_alloc(4 * N * F); d_out = ctx.dev_alloc(4 * N * F)
    chunk = rng.integers(0, 2**32, (16384, F), dtype=np.uint32)
    for k in range(N // 16384):
        ctx.h2d(d_in + k * chunk.nbytes, chunk)
    for mode in (0, 2):
        ctx.set_option("planar_bulk", mode)
        b = ctx.batch(st.PDM, N, order=2, out_shift=24)
        ms = timed(lambda: b.run_dev(F, inp=d_in, out=d_out))
        print("pdm raw planar_bulk=%d: %.3f ms  %.0f GB/s" % (mode, ms, 8 * N * F / ms / 1e6))
        b.free()
