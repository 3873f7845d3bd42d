#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 cproc renderer.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes what the last timed step computed (rank 0's shard) to
DIR/<name>.npy, so that two builds can be compared output for output.  On the
native path the inputs depend only on the arguments.  The reference arm sizes
its sample by the host's core count, so its dumps compare only between runs on
hosts with the same number of cores.

Workload (BASELINE.json configs[1], SURVEY.md section 8d "C2"): the PDM
sigma-delta modulator, 65,536 independent channels x 16 Mi samples, integer,
bit-exact.  The modulator is the one the reference firmware builds
(stm32f103/mod_synth.c:37 includes mod_pdm_pwm.c): glide + pdm2_update with the
control-rate line generator, banks of 3 channels sharing one dither word per
tick, a fresh setpoint row every 4096 ticks; output one 8-bit duty per
channel-sample.

A "step" is one pass over the whole workload (2^40 channel-samples per GPU),
rendered as 128 launches of 131,072 ticks into two alternating 8 GiB output
slabs in HBM.  Multi-GPU is weak scaling: every rank renders its own 65,536
channels (independent shards, no data-path collective).

One JSON line on stdout (rank 0).
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_CH = 65536
F_TOTAL = 16 * 1024 * 1024
F_CHUNK = 131072                     # ticks per launch: 8 GiB duty slab (two alternate); 36.9 rounds of work items per launch
BANK = 3
CTL_LOG = 12
ALGO_BYTES_PER_SAMPLE = 1.0          # SURVEY 8d C2 v2: one uint8 duty per channel-sample
ALGO_INSTR_PER_SAMPLE = 10.0         # SURVEY 8d C2 v2: ~10 integer instructions per channel-sample
E2E_TICKS = 1024 * 1024              # e2e step: 65,536 ch x 1 Mi samples through host buffers
# 256 MiB slabs, ring of 4 in pinned memory.  Small on purpose: with 1 GiB slabs (4 GiB of pinned ring per rank) the
# device-to-host stream of a rank drops from 57 to 46 GB/s as soon as a second rank streams too, and to 11 GB/s per rank
# at eight (measured; plain concurrent copies into 1 GiB buffers do not show it) -- the DMA working set, not the fabric.
E2E_CHUNK = int(os.environ.get("E2E_CHUNK_TICKS", "4096"))
DUMP_CHANNELS = 256                  # --dump-outputs: seeded sample of channels whose duty is written tick by tick
DUMP_TICKS = 8192                    # ... over the last ticks of each launch written
DUMP_MAX_BYTES = 64 << 20


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons during the timed region (NVML)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = False
        self.sm = []
        self.reasons = set()
        self.sm_max = None
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        if not self.ok or not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons)}
        s = sorted(self.sm)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.sm_max, "reasons": sorted(self.reasons)}


def physical_gpu_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


# --------------------------------------------------------------------------- reference arm
def run_reference(args, rank, world):
    """The reference's own CPU implementation of the path: oracle/_ref (pdm2_update
    from the unmodified stm32f103/pdm.h inside the restated v2 ISR), OpenMP over
    all host cores, on a bounded sample of the same workload per step."""
    if rank != 0:
        return
    # torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host core
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
    import numpy as np
    from oracle import pyoracle as po
    kind = "reference"
    try:
        lib = po.Ref()
    except Exception:
        lib = po.Oracle()
        kind = "port"
    cores = os.cpu_count() or 1
    po.set_threads(cores)
    n_ch = 3 * 2048 * max(1, cores // 8)           # multiple of the bank size
    ticks = 256 * 1024
    chan = np.zeros((n_ch, 7), np.uint32)
    prng = (np.arange(n_ch // 3) + 1).astype(np.uint32)
    sp = po.pdm_setpoints(n_ch, ticks // 4096)
    duty = np.zeros((n_ch, ticks), np.uint8)       # allocated and touched once: the timed loop renders, it does not page-fault
    count = 0
    _, count = lib.pdm_v2_run(chan, 2, n_ch, 3, prng, None, 0x3FF, count, CTL_LOG, 24, sp, ticks, out=duty)
    for _ in range(args.warmup):
        _, count = lib.pdm_v2_run(chan, 2, n_ch, 3, prng, None, 0x3FF, count, CTL_LOG, 24, sp, ticks, out=duty)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        _, count = lib.pdm_v2_run(chan, 2, n_ch, 3, prng, None, 0x3FF, count, CTL_LOG, 24, sp, ticks, out=duty)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        idx = dump_channels(n_ch)
        write_outputs(args.dump_outputs, {"duty_channels": idx, "duty": duty[idx, -DUMP_TICKS:], "duty_sum": duty.sum(axis=1),
                                          "channel_state": chan, "bank_prng": prng, "bank_count": np.array([count], np.uint32)})
    value = n_ch * ticks * args.steps / dt
    sample = "%d ch x %d samples per step (same modulator, setpoints and dither as the native arm), gcc -O2, output buffer preallocated" % (n_ch, ticks)
    line = {
        "impl": "reference", "metric": "voice-samples/sec", "value": value, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": workload_config(),
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def workload_config():
    return {"workload": "C2 PDM v2 (mod_pdm_pwm.c glide + pdm2_update, banks of 3 share dither, setpoint row every "
                        "4096 ticks): 65,536 channels x 16 Mi samples per GPU, uint8 duty out",
            "channels_per_gpu": N_CH, "samples_per_channel": F_TOTAL, "launch_ticks": F_CHUNK,
            "out_layout": "TILED [t/16][ch][16]", "l2": "inputs+outputs larger than L2 (8 GiB output slab per launch)"}


# --------------------------------------------------------------------------- --dump-outputs
def dump_channels(n_ch):
    """The channels whose duty --dump-outputs writes tick by tick: a fixed, seeded, sorted sample."""
    import numpy as np
    return np.sort(np.random.default_rng(20261020).choice(n_ch, size=min(DUMP_CHANNELS, n_ch), replace=False))


def write_outputs(path, arrays):
    """DIR/<name>.npy per array: 8- and 16-bit integers as float32, wider integers as float64 (both exact)."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    out = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        out[name] = a.astype(np.float32 if a.dtype.kind == "f" or a.dtype.itemsize <= 2 else np.float64)
    total = sum(a.nbytes for a in out.values())
    assert total <= DUMP_MAX_BYTES, "dump of %d bytes exceeds %d" % (total, DUMP_MAX_BYTES)
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)
    print("bench: wrote %d arrays (%.1f MB) to %s" % (len(out), total / 1e6, path), file=sys.stderr)


def dump_native(path, torch, batch, slabs, n_chunks):
    """What the last timed step leaves its caller: the duty of its last two launches (the two slabs alternate, so these are
    the two still in HBM) -- tick by tick for the sampled channels over each launch's last DUMP_TICKS ticks, and summed
    over all ticks for every channel -- and the channel and dither-bank state the step ends with."""
    import numpy as np
    idx = dump_channels(N_CH)
    sel = torch.from_numpy(idx).to(slabs[0].device)
    arrays = {"duty_channels": idx}
    for name, k in (("prev_launch", n_chunks - 2), ("last_launch", n_chunks - 1)):
        tiles = slabs[k & 1].view(F_CHUNK // 16, N_CH, 16)                      # TILED: [t/16][ch][16]
        win = tiles[-(DUMP_TICKS // 16):].index_select(1, sel)
        arrays[name + "_duty"] = win.permute(1, 0, 2).reshape(len(idx), DUMP_TICKS).cpu().numpy()
        total = torch.zeros(N_CH, dtype=torch.int64, device=slabs[0].device)
        for r in range(0, F_CHUNK // 16, 512):                                  # int32 partial sums of 512 x 16 bytes
            total += tiles[r:r + 512].sum(dim=(0, 2), dtype=torch.int32)
        arrays[name + "_duty_sum"] = total.cpu().numpy()
    prng, count = batch.download_bank()
    arrays["channel_state"] = batch.download_state()
    arrays["bank_prng"] = prng
    arrays["bank_count"] = np.array([count], np.uint32)
    write_outputs(path, arrays)


# --------------------------------------------------------------------------- native arm
def cpu_baseline_sample():
    """The reference's pdm2_update inside the v2 ISR (oracle/_ref) on the host cores: all cores at -O2 (the value), plus one
    core, and the -O3 -march=x86-64-v3 build on all cores and on one (BASELINE.md 3).  The duty buffer is preallocated."""
    import numpy as np
    from oracle import pyoracle as po
    cores = os.cpu_count() or 1
    kind = "reference"
    try:
        lib = po.Ref()
    except Exception:
        lib = po.Oracle()
        kind = "port"
    lib_o3 = None
    try:
        if kind == "reference" and os.path.exists(po.REF_O3_SO):
            lib_o3 = po.Ref(po.REF_O3_SO)
    except Exception:
        lib_o3 = None
    n_ch = 3 * 2048 * max(1, cores // 8)
    ticks = 64 * 1024
    sp = po.pdm_setpoints(n_ch, 16)
    duty = np.zeros((n_ch, ticks), np.uint8)

    def rate(l, threads, n, seconds):
        po.set_threads(threads)
        chan = np.zeros((n, 7), np.uint32)
        prng = (np.arange(n // 3) + 1).astype(np.uint32)
        spn = np.ascontiguousarray(sp[:, :n])
        d = duty[:n]
        count = 0
        _, count = l.pdm_v2_run(chan, 2, n, 3, prng, None, 0x3FF, count, CTL_LOG, 24, spn, ticks, out=d)   # warm, first touch
        t0 = time.perf_counter()
        _, count = l.pdm_v2_run(chan, 2, n, 3, prng, None, 0x3FF, count, CTL_LOG, 24, spn, ticks, out=d)
        r = n * ticks / (time.perf_counter() - t0)
        reps = max(1, min(48, int(seconds * r / (n * ticks))))
        t0 = time.perf_counter()
        for _ in range(reps):
            _, count = l.pdm_v2_run(chan, 2, n, 3, prng, None, 0x3FF, count, CTL_LOG, 24, spn, ticks, out=d)
        return n * ticks * reps / (time.perf_counter() - t0), reps

    v, reps = rate(lib, cores, n_ch, 10.0)                       # about 10 s of CPU work
    one, _ = rate(lib, 1, 3 * 256, 2.0)
    res = {"value": v, "unit": "samples/s", "cores": cores, "kind": kind,
           "sample": "%d ch x %d samples, all host threads (OpenMP), gcc -O2, output buffer preallocated" % (n_ch, ticks * reps),
           "one_core": {"value": one, "sample": "768 ch x %d samples, one thread, gcc -O2" % ticks}}
    if lib_o3 is not None:
        v3, _ = rate(lib_o3, cores, n_ch, 3.0)
        one3, _ = rate(lib_o3, 1, 3 * 256, 2.0)
        res["o3"] = {"value": v3, "one_core": one3,
                     "flags": "-O3 -march=x86-64-v3 (not -march=native: the library is built where the reference sources are, not on this box)"}
    po.set_threads(cores)
    return res


def run_native(args, rank, local_rank, world):
    import numpy as np
    import torch
    import torch.distributed as dist
    import synth_tools_b200 as st
    from oracle import pyoracle as po           # input generator + cpu_baseline only

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = "unset"
    try:
        # run (and first-touch the pinned host ring) on the CPUs next to this GPU: the e2e leg is a
        # PCIe / host-memory stream, and 8 ranks on the wrong socket share one inter-socket link
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(physical_gpu_index(local_rank)))
        numa = "gpu-local cpus (%d)" % len(os.sched_getaffinity(0))
    except Exception as e:
        numa = "not set (%s)" % type(e).__name__
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    # a non-default torch stream: the library launches on it and torch's events time it
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    ctx = st.Context(local_rank, stream.cuda_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    n_rows = F_TOTAL // (1 << CTL_LOG)
    rows_per_chunk = F_CHUNK >> CTL_LOG
    # inputs resident in HBM before the timed region: 4096 setpoint rows (1 GiB)
    seed = 1 + rank * N_CH
    sp_host = po.pdm_setpoints(N_CH, 64, seed_base=seed)
    sp_dev = torch.empty((n_rows, N_CH), dtype=torch.int32, device=dev)
    sp64 = torch.from_numpy(sp_host.view(np.int32)).to(dev)
    for r in range(0, n_rows, 64):                        # 64 distinct rows, rolled per block of rows
        sp_dev[r:r + 64] = torch.roll(sp64, shifts=r // 64, dims=1)
    slabs = [torch.empty(N_CH * F_CHUNK, dtype=torch.uint8, device=dev) for _ in range(2)]
    batch = ctx.batch(st.PDM_V2, N_CH, order=2, bank_size=BANK, ctl_div_log=CTL_LOG, out_shift=24, dither_mask=0x3FF,
                      layout=st.TILED)
    batch.upload_bank((np.arange(batch.n_banks) + seed).astype(np.uint32), 0)
    n_chunks = F_TOTAL // F_CHUNK

    def step():
        for k in range(n_chunks):
            batch.run_dev(F_CHUNK, ctl=sp_dev.data_ptr() + 4 * N_CH * rows_per_chunk * k, n_ctl=rows_per_chunk,
                          out=slabs[k & 1].data_ptr())

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(physical_gpu_index(local_rank))
    sampler.start()
    l0 = ctx.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    barrier()
    sampler.stop_flag = True
    ms = e0.elapsed_time(e1)
    launches = ctx.launches - l0
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    ms_per_step = ms_max / args.steps
    value = world * N_CH * F_TOTAL / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_native(args.dump_outputs, torch, batch, slabs, n_chunks)    # before the e2e leg runs the batch on

    # ---- end to end through the C-ABI with HOST buffers: setpoints H2D, duty D2H
    e2e_rows = E2E_TICKS >> CTL_LOG
    slab_bytes = N_CH * E2E_CHUNK
    ring, ring_ptr = ctx.host_alloc(4 * slab_bytes)
    sp_pin, sp_pin_ptr = ctx.host_alloc(e2e_rows * N_CH * 4, np.uint32)
    sp_pin[:] = np.tile(sp_host, (e2e_rows // 64, 1)).reshape(-1)
    checks = []

    def on_chunk(user, k, slab, nbytes):
        if k == 0:
            checks.append(nbytes)

    def e2e_step():
        batch.run_stream(E2E_TICKS, E2E_CHUNK, out=ring_ptr, ctl=sp_pin_ptr, n_ctl=e2e_rows, ring_chunks=4, on_chunk=on_chunk)

    for _ in range(min(args.warmup, 3)):
        e2e_step()
    barrier()
    # the ceiling of this leg: plain device -> pinned-host copies of the same ring, all ranks at once (the ranks of one box share
    # the host's PCIe uplinks; tools/d2h_probe.py, profiles/r2_d2h_probe_8gpu.json).  Untimed for the metric.
    tp0 = time.perf_counter()
    for _ in range(8):
        ctx.d2h(ring, slabs[0].data_ptr())
    probe_gbs = 8 * ring.nbytes / (time.perf_counter() - tp0) / 1e9
    tpr = torch.tensor([probe_gbs], device=dev, dtype=torch.float64)
    probe_ranks = [probe_gbs]
    if world > 1:
        allp = [torch.zeros_like(tpr) for _ in range(world)]
        dist.all_gather(allp, tpr)
        probe_ranks = [float(x.item()) for x in allp]
    barrier()
    e2e_steps = max(1, min(args.steps, 5))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], device=dev, dtype=torch.float64)
    e2e_ranks = [dt]
    if world > 1:
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        e2e_ranks = [float(x.item()) for x in allt]
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * N_CH * E2E_TICKS * e2e_steps / float(t.item())
    ctx.host_free(ring_ptr)
    ctx.host_free(sp_pin_ptr)

    if rank == 0:
        peak, peak_src = measured_peaks()
        launch_ms = ms / launches
        algo_bytes = ALGO_BYTES_PER_SAMPLE * N_CH * F_CHUNK + 4.0 * N_CH * rows_per_chunk
        achieved = algo_bytes / (launch_ms * 1e-3) / 1e9
        clocks = sampler.summary()
        sm_hz = (clocks["sm_mhz"] or 1965) * 1e6
        issue_peak = 128.0 * 148 * sm_hz
        issue_ach = ALGO_INSTR_PER_SAMPLE * N_CH * F_CHUNK / (launch_ms * 1e-3)
        traffic, traffic_src, executed = None, None, None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            try:
                tj = json.load(open(tp))
                traffic = tj.get("k_pdm_v2_bytes_per_launch")
                traffic_src = tj.get("source")
                executed = tj.get("k_pdm_v2_thread_instr_per_sample")
            except Exception:
                traffic = None
        line = {
            "metric": "voice-samples/sec", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u32", "data": "synthetic", "config": workload_config(),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "samples/s",
                    "h2d_bytes_per_step": e2e_rows * N_CH * 4, "d2h_bytes_per_step": N_CH * E2E_TICKS,
                    "sample": "65,536 ch x 1 Mi samples per step per GPU via cproc_cuda_run_stream (pinned ring of 4 x %d MiB)" % (N_CH * E2E_CHUNK >> 20),
                    "cpu_affinity": numa,
                    "steps": e2e_steps, "seconds_per_rank": [round(x, 4) for x in e2e_ranks],
                    "d2h_gbs_per_rank": [round(N_CH * E2E_TICKS * e2e_steps / x / 1e9, 2) for x in e2e_ranks],
                    "d2h_copy_ceiling_gbs_per_rank": [round(x, 2) for x in probe_ranks],
                    "fraction_of_copy_ceiling_per_rank": [round(N_CH * E2E_TICKS * e2e_steps / x / 1e9 / max(pr, 1e-9), 3) for x, pr in zip(e2e_ranks, probe_ranks)],
                    "ceiling_note": "plain device -> pinned host copies of the same ring, all ranks at once, measured in this run before the e2e leg"},
            "gpu_launches": launches,
            # The kernel is bound by integer instruction issue (two half-rate pipes shared by ~4 warps per scheduler), not by
            # HBM: the roofline is stated against the issue peak at the observed SM clock, the HBM figure rides along.
            "roofline": {"bound": "issue", "achieved": issue_ach / 1e12, "peak": issue_peak / 1e12, "unit": "T thread-instr/s",
                         "frac": issue_ach / issue_peak, "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "k_pdm_v2_ws4<K=2,CW=3,TLOG=7,PL=0>", "launch_ms": launch_ms,
                         "algorithmic_instr_per_sample": ALGO_INSTR_PER_SAMPLE,
                         "executed_thread_instr_per_sample": executed,
                         "note": "SURVEY 8d: C2 is INT-issue bound; 10 algorithmic int instr per sample against 128 thread-instr/clk/SM "
                                 "(measured, tools/ubench_int.cu) at the observed SM clock; traffic = ncu dram bytes per launch of the same kernel",
                         "hbm": {"achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                                 "algorithmic_bytes_per_launch": algo_bytes}},
        }
        if world == 1:
            line["cpu_baseline"] = cpu_baseline_sample()
    batch.free()
    scaling = None
    if not args.no_other_configs:
        # the configurations that shard over the GPUs of a box (C4', C4, C3b with the mix bus exchange, C5 without), at this N,
        # strong scaling, outside every timed region above; all ranks take part
        try:
            from tools import bench_configs
            scaling = bench_configs.scaling_rows(st, ctx, torch, stream, dev, rank, world, dist if world > 1 else None)
        except Exception as e:
            scaling = [{"error": "%s: %s" % (type(e).__name__, e)}]
    if rank == 0:
        if scaling is not None:
            line["scaling_configs"] = scaling
        if world == 1 and not args.no_other_configs:
            # the other BASELINE.json configurations at full size (parity-test cases; reported for the
            # raw-output >= 70 % HBM / mixed-down >= 60 % issue targets), outside every timed region above
            from tools import bench_configs
            line["other_configs"] = bench_configs.run_all(st, ctx, peak)
        emit(line)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--no-other-configs", action="store_true", help="skip the secondary configuration rows (N=1)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (float32/float64, <= 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    # stdout carries the ONE JSON line and nothing else: libraries that write to fd 1 (NCCL prints its version
    # banner there) are sent to stderr, the line goes to the saved descriptor.  The re-exec below inherits fd 1.
    global _JSON_OUT
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under torch.distributed.run
        import subprocess
        port = os.environ.get("MASTER_PORT", "29531")
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", port, os.path.abspath(__file__),
               "--gpus", str(args.gpus), "--steps", str(args.steps), "--warmup", str(args.warmup)]
        cmd += ["--no-other-configs"] if args.no_other_configs else []
        cmd += ["--dump-outputs", args.dump_outputs] if args.dump_outputs else []
        sys.exit(subprocess.call(cmd))
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    run_native(args, rank, local_rank, world)


_JSON_OUT = None


def emit(line):
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    print(json.dumps(line), file=out, flush=True)


if __name__ == "__main__":
    main()
