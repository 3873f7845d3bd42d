"""Time the bus mix of a generated cproc graph (io.mix of a CPROC_CUDA_GRAPH batch) against the ways a host gets the same
bus without it, at the C4 shape: 4 Mi voices x 512 frames of the voice graph (bench_configs.VOICE_GRAPH_TEXT: phasor_f ->
svf -> env -> 2 x gain), buses of 4096 voices.

    python tools/time_graph_mix.py [--reps 10] [--json OUT]

Rows (CUDA events on the stream the library and torch share, best of --reps after a warm-up launch):
  graph mix-only            the steady block (every voice released) and the note-on block (state back to t = 0 before
                            every timed launch, untimed, as bench.py does for XVOICE)
  raw render                PLANAR and INTERLEAVED, 16 GiB of per-voice stereo out
  raw render + torch.sum    the PLANAR render and a torch sum over each bus's voices
  input-stream voice        the same voice with a pitch-modulation input (ext_voice.cproc): mix-only with PLANAR and
                            INTERLEAVED input, and the raw PLANAR render, for the mix kernel's lane-by-lane PLANAR reads
  k_xvoice_mix2             the hand-fused XVOICE mix of the same voices (one bus), note-on and steady
  JACK period               16 parts x 64 voices x 64 frames through cproc_cuda_run (host buffers), us per period
The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    import torch
    import synth_tools_b200 as st
    from tools import bench_configs

    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream(dev)                  # not the legacy default stream (handle 0): the library would make its own
    torch.cuda.set_stream(stream)
    ctx = st.Context(0, stream=stream.cuda_stream)

    def timed(fn, before=None):
        if before:
            before()
        fn()
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(a.reps):
            if before:
                before()
                torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            e1.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return best

    rows = {"card (name, power limit, max SM clock)": card()}
    print("card:", rows["card (name, power limit, max SM clock)"], flush=True)
    g = st.graph_parse_ex(bench_configs.VOICE_GRAPH_TEXT)
    N, F, vpb = 4 * 1024 * 1024, 512, 4096
    stt, prm = bench_configs.xvoice_records(np.random.default_rng(5), N)
    gst = np.zeros((N, 9), np.uint32)
    gst[:, 1] = stt[:, 0]
    samples = N * F

    def row(name, ms, note=""):
        rows[name] = {"ms": round(ms, 4), "voice_samples_per_s": float("%.4g" % (samples / (ms * 1e-3))), "note": note}
        print("%-44s %9.3f ms  %.3e voice-samples/s  %s" % (name, ms, samples / (ms * 1e-3), note), flush=True)

    b = ctx.batch(st.GRAPH, N, nodes=g["rows"], n_inputs=0, out_node=g["out_nodes"], voices_per_bus=vpb)
    b.upload_state(gst); b.upload_param(prm)
    mix = torch.empty((N // vpb, 2, F), dtype=torch.float32, device=dev)
    row("graph mix-only, note-on block", timed(lambda: b.run_dev(F, mix=mix.data_ptr()), before=lambda: b.upload_state(gst)))
    row("graph mix-only, steady block", timed(lambda: b.run_dev(F, mix=mix.data_ptr())))
    mix_ref = mix.clone()
    b.free()

    out = torch.empty((N, 2, F), dtype=torch.float32, device=dev)        # 16 GiB
    for name, layout in (("PLANAR", st.PLANAR), ("INTERLEAVED", st.INTERLEAVED)):
        b = ctx.batch(st.GRAPH, N, nodes=g["rows"], n_inputs=0, out_node=g["out_nodes"], layout=layout)
        b.upload_state(gst); b.upload_param(prm)
        row("graph raw render %s, steady" % name, timed(lambda: b.run_dev(F, out=out.data_ptr())), "16 GiB out")
        if layout == st.PLANAR:
            row("graph raw render PLANAR + torch.sum, steady",
                timed(lambda: (b.run_dev(F, out=out.data_ptr()), torch.sum(out.view(N // vpb, vpb, 2, F), dim=1, out=mix))),
                "sum over each bus's voices")
        b.free()
    # the same voice with a pitch-modulation input stream (tests/golden/ext_voice.cproc, same records): the mix kernel reads
    # PLANAR input rows lane by lane and INTERLEAVED ones coalesced; the raw PLANAR render stages them (tensor TMA)
    gv = st.graph_parse_ex(open(os.path.join(ROOT, "tests", "golden", "ext_voice.cproc")).read())
    inp = torch.randint(0, 1 << 20, (N * F,), dtype=torch.int32, device=dev)     # 8 GiB
    for name, layout in (("PLANAR", st.PLANAR), ("INTERLEAVED", st.INTERLEAVED)):
        b = ctx.batch(st.GRAPH, N, nodes=gv["rows"], n_inputs=1, out_node=gv["out_nodes"], layout=layout, voices_per_bus=vpb)
        b.upload_state(gst); b.upload_param(prm)
        row("input-stream voice mix-only, %s in, steady" % name, timed(lambda: b.run_dev(F, inp=inp.data_ptr(), mix=mix.data_ptr())), "8 GiB in")
        if layout == st.PLANAR:
            row("input-stream voice raw render PLANAR, steady", timed(lambda: b.run_dev(F, inp=inp.data_ptr(), out=out.data_ptr())), "8 GiB in, 16 GiB out")
        b.free()
    del out, inp
    torch.cuda.empty_cache()

    b = ctx.batch(st.XVOICE, N)
    b.upload_state(stt); b.upload_param(prm)
    xm = torch.empty((2, F), dtype=torch.float32, device=dev)
    row("k_xvoice_mix2, note-on block", timed(lambda: b.run_dev(F, mix=xm.data_ptr()), before=lambda: b.upload_state(stt)), "one bus")
    row("k_xvoice_mix2, steady block", timed(lambda: b.run_dev(F, mix=xm.data_ptr())), "one bus")
    b.free()

    # JACK period: 16 parts x 64 voices, 64 frames, host buffers (cproc_cuda_run, run_graph default)
    Np, Fp, vp = 16 * 64, 64, 64
    b = ctx.batch(st.GRAPH, Np, nodes=g["rows"], n_inputs=0, out_node=g["out_nodes"], voices_per_bus=vp)
    b.upload_state(gst[:Np]); b.upload_param(np.ascontiguousarray(prm[:Np]))
    hm = np.zeros((Np // vp, 2, Fp), np.float32)
    for _ in range(50):
        b.run(Fp, mix=hm)
    best = 1e9
    for _ in range(5):
        t0 = time.perf_counter()
        for _ in range(1000):
            b.run(Fp, mix=hm)
        best = min(best, (time.perf_counter() - t0) / 1000)
    b.free()
    rows["JACK period 16 x 64 voices x 64 frames, cproc_cuda_run"] = {"us_per_period": round(best * 1e6, 2)}
    print("%-44s %9.2f us per period (best of 5 x 1000)" % ("JACK period 16 x 64 x 64, cproc_cuda_run", best * 1e6), flush=True)
    rows["mix checksum"] = float(mix_ref.double().abs().sum())
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as f:
            json.dump(rows, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
