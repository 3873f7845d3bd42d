"""Multi-GPU mix bus check + timing (BASELINE.json config 4: 4 Mi voices x 512-frame blocks, the
mix bus reduced across the GPUs of one box).  Run under torchrun, one rank per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 tools/multi_gpu_mix.py

Voices are sharded in contiguous ranges; each rank renders the INTEGER mix of its shard
(k_voice_mix).  The bus is then formed four ways: (A) NCCL all-reduce of the int32 mix + the
conversion kernel, (B) cproc_cuda_bus_allreduce -- one kernel per rank over NVLink peer
memory, reduce and float scale fused, (C) the exchange fused into the render launch
(cproc_cuda_bus_attach mode 1: reduce at the end of the same launch), (D) the same, pipelined
(mode 2: the reduce of block k beside the render of block k+1).  All must equal the
single-device oracle bit for bit.  Prints one JSON line per measurement (rank 0).
The C4 extension voices (float bus) and the C3b square_grain mix (1 Mi grains x 256-frame
blocks, integer bus in units of 2^-7) get the same treatment in their own sections.
--check-only: parity checks at reduced sizes, no timing (tests/test_gpu_multi.py)."""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

import synth_tools_b200 as st
from synth_tools_b200 import shard
from oracle import pyoracle as po

rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
stream = torch.cuda.Stream(device=dev)
torch.cuda.set_stream(stream)
ctx = st.Context(local, stream.cuda_stream)
orc = po.Oracle()
tab = np.array([orc.note_to_inc(k) for k in range(128)], np.uint32)


def voices(N, seed):
    r = np.random.default_rng(seed)
    v = np.zeros((N, 2), np.uint32)
    v[:, 0] = tab[r.integers(0, 128, N)]
    v[::53, 0] = 0
    v[:, 1] = r.integers(0, 2**32, N, dtype=np.uint32)
    return v


def check(N, F, mode):
    v = voices(N, 1234)                                   # same on every rank
    lo, hi = shard.shard_range(N, rank, world)
    full = v.copy()
    want_i, want_f = orc.voice_bank_run(full, N, N, mode, F)
    b = ctx.batch(st.VOICE_BANK, hi - lo, voices_per_bus=0, mode=mode)
    b.upload_state(np.ascontiguousarray(v[lo:hi]))
    imix = torch.zeros(F, dtype=torch.int32, device=dev)
    out = torch.zeros(F, dtype=torch.float32, device=dev)
    b.run_dev(F, mix=imix.data_ptr())
    keep = imix.clone()
    # (A) NCCL + conversion kernel
    shard.allreduce_mix(imix, mode)
    b.mix_to_float(imix.data_ptr(), out.data_ptr(), F)
    torch.cuda.synchronize()
    ok_a = np.array_equal(imix.cpu().numpy().view(np.uint32), want_i[0].view(np.uint32)) and \
        np.array_equal(out.cpu().numpy().view(np.uint32), want_f[0].view(np.uint32))
    # (B) one kernel over peer memory
    bus = shard.connect_bus(st.Bus(ctx, 4096, world, rank))
    imix.copy_(keep); out.zero_()
    for _ in range(3):                                    # consecutive epochs reuse the double-buffered slots
        imix.copy_(keep)
        bus.allreduce(imix.data_ptr(), F, out_dev=out.data_ptr(), op=st.Bus.OR if mode == 1 else st.Bus.SUM,
                      scale=st.Bus.SCALE_SQUARE if mode == 1 else st.Bus.SCALE_SAW)
    torch.cuda.synchronize()
    ok_b = bus.status() == 0 and np.array_equal(imix.cpu().numpy().view(np.uint32), want_i[0].view(np.uint32)) and \
        np.array_equal(out.cpu().numpy().view(np.uint32), want_f[0].view(np.uint32))
    # overlapped form: four blocks in flight over the two slots, every block continues the phases
    outs = [torch.zeros(F, dtype=torch.float32, device=dev) for _ in range(2)]
    mixes = [torch.zeros(F, dtype=torch.int32, device=dev) for _ in range(2)]
    b.upload_state(np.ascontiguousarray(v[lo:hi]))
    full2 = v.copy()
    wants = []
    for k in range(4):
        s = k & 1
        bus.wait(s)
        if k >= 2:
            ok_b = ok_b and np.array_equal(outs[s].cpu().numpy().view(np.uint32), wants[k - 2].view(np.uint32))
        wants.append(orc.voice_bank_run(full2, N, N, mode, F)[1][0].copy())
        b.run_dev(F, mix=mixes[s].data_ptr())
        bus.begin(s, mixes[s].data_ptr(), F, out_dev=outs[s].data_ptr(), op=st.Bus.OR if mode == 1 else st.Bus.SUM,
                  scale=st.Bus.SCALE_SQUARE if mode == 1 else st.Bus.SCALE_SAW)
    bus.wait(0); bus.wait(1)
    torch.cuda.synchronize()
    ok_b = ok_b and bus.status() == 0 and np.array_equal(outs[0].cpu().numpy().view(np.uint32), wants[2].view(np.uint32)) and \
        np.array_equal(outs[1].cpu().numpy().view(np.uint32), wants[3].view(np.uint32))
    # (C) / (D): the exchange as the tail of the render launch; six blocks continue the phases
    ok_f = []
    for bus_mode in (1, 2):
        okm = True
        b.upload_state(np.ascontiguousarray(v[lo:hi]))
        full3 = v.copy()
        bus.attach(b, bus_mode)
        outs6 = [torch.zeros(F, dtype=torch.float32, device=dev) for _ in range(6)]
        mixes6 = [torch.zeros(F, dtype=torch.int32, device=dev) for _ in range(6)]
        wants6 = []
        for k in range(6):
            wants6.append(orc.voice_bank_run(full3, N, N, mode, F))
            b.run_dev(F, mix=mixes6[k].data_ptr(), out=outs6[k].data_ptr())
        bus.flush()
        torch.cuda.synchronize()
        for k in range(6):
            okm = okm and np.array_equal(outs6[k].cpu().numpy().view(np.uint32), wants6[k][1][0].view(np.uint32)) and \
                np.array_equal(mixes6[k].cpu().numpy().view(np.uint32), wants6[k][0][0].view(np.uint32))
        bus.detach(b)
        ok_f.append(okm and bus.status() == 0)
    bus.destroy(); b.free()
    t = torch.tensor([int(ok_a), int(ok_b), int(ok_f[0]), int(ok_f[1])], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return [bool(x.item()) for x in t]


def timing(N, F, reps=50):
    v = voices(N, 99)
    lo, hi = shard.shard_range(N, rank, world)
    b = ctx.batch(st.VOICE_BANK, hi - lo, voices_per_bus=0)
    b.upload_state(np.ascontiguousarray(v[lo:hi]))
    imix = torch.zeros(F, dtype=torch.int32, device=dev)
    out = torch.zeros(F, dtype=torch.float32, device=dev)
    bus = shard.connect_bus(st.Bus(ctx, 4096, world, rank))
    res = {}

    def block_nccl():
        b.run_dev(F, mix=imix.data_ptr())
        dist.all_reduce(imix)
        b.mix_to_float(imix.data_ptr(), out.data_ptr(), F)

    def block_bus():
        b.run_dev(F, mix=imix.data_ptr())
        bus.allreduce(imix.data_ptr(), F, out_dev=out.data_ptr(), scale=st.Bus.SCALE_SAW)

    def block_render_only():
        b.run_dev(F, mix=imix.data_ptr())

    imix2 = [torch.zeros(F, dtype=torch.int32, device=dev) for _ in range(2)]
    out2 = [torch.zeros(F, dtype=torch.float32, device=dev) for _ in range(2)]
    kblk = [0]

    def block_bus_overlapped():
        s = kblk[0] & 1
        kblk[0] += 1
        bus.wait(s)                                        # the exchange that last used this buffer pair
        b.run_dev(F, mix=imix2[s].data_ptr())
        bus.begin(s, imix2[s].data_ptr(), F, out_dev=out2[s].data_ptr(), scale=st.Bus.SCALE_SAW)

    def block_fused():
        s = kblk[0] & 1
        kblk[0] += 1
        b.run_dev(F, mix=imix2[s].data_ptr(), out=out2[s].data_ptr())

    def block_fused_k4():                                  # four frame blocks per launch, one exchange of 4 x 512 words
        b.run_dev(4 * F, mix=imix4.data_ptr(), out=out4.data_ptr())

    imix4 = torch.zeros(4 * F, dtype=torch.int32, device=dev)
    out4 = torch.zeros(4 * F, dtype=torch.float32, device=dev)
    for name, fn in (("render_only", block_render_only), ("nccl_allreduce_plus_convert", block_nccl), ("peer_memory_bus_kernel", block_bus),
                     ("peer_memory_bus_overlapped", block_bus_overlapped), ("fused_in_launch", block_fused), ("fused_pipelined", block_fused),
                     ("fused_pipelined_4_blocks_per_launch", block_fused_k4), ("render_only_4_blocks_per_launch", block_fused_k4)):
        if name == "fused_in_launch":
            bus.attach(b, 1)
        elif name.startswith("fused_pipelined"):
            bus.attach(b, 2)
        else:
            bus.detach(b)
        for _ in range(5):
            fn()
        dist.barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            fn()
        bus.wait(0); bus.wait(1); bus.flush()
        e1.record(stream)
        dist.barrier(); torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / reps], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        res[name] = float(t.item()) / (4 if name.endswith("4_blocks_per_launch") else 1)
    ok = bus.status() == 0
    bus.detach(b)
    bus.destroy(); b.free()
    return res, ok


def xvoice_records(N, seed):
    r = np.random.default_rng(seed)
    prm = np.zeros(N, po.xvoice_param_dtype)
    prm["inc"] = tab[r.integers(24, 109, N)]
    prm["f"] = r.uniform(0.01, 0.3, N); prm["q"] = r.uniform(0.5, 2.0, N)
    prm["env_attack"] = r.uniform(1e-3, 1e-1, N); prm["env_release"] = r.uniform(1e-3, 1e-2, N)
    prm["gate_frames"] = r.integers(0, 400, N)
    prm["gl"] = r.uniform(0, 1, N); prm["gr"] = 1.0 - prm["gl"]
    s0 = np.zeros(N, po.xvoice_state_dtype)
    s0["phase"] = r.integers(0, 2**32, N, dtype=np.uint32)
    return s0, prm


def xvoice_check_and_timing(N_check, N, F, reps=20):
    """C4: float stereo mix of the extension voices; the bus is a float sum in rank order."""
    s0, prm = xvoice_records(N_check, 5)
    lo, hi = shard.shard_range(N_check, rank, world)
    sa = s0.copy()
    _, want = orc.xvoice_run(sa, prm, N_check, F, want_raw=False)
    b = ctx.batch(st.XVOICE, hi - lo)
    b.upload_state(np.ascontiguousarray(s0[lo:hi]).view(np.uint32).reshape(hi - lo, 5))
    b.upload_param(np.ascontiguousarray(prm[lo:hi]).view(np.uint32).reshape(hi - lo, 8))
    mix = torch.zeros(2 * F, dtype=torch.float32, device=dev)
    bus = shard.connect_bus(st.Bus(ctx, 4096, world, rank))
    b.run_dev(F, mix=mix.data_ptr())
    bus.allreduce(mix.data_ptr(), 2 * F, op=st.Bus.FSUM)
    torch.cuda.synchronize()
    g64, w64 = mix.cpu().numpy().astype(np.float64), np.asarray(want, np.float64).reshape(-1)
    detail = {}
    ok = bus.status() == 0 and np.abs(g64 - w64).max() <= 1e-5 * np.abs(w64).max() and \
        10 * np.log10((w64 ** 2).sum() / max(((g64 - w64) ** 2).sum(), 1e-300)) >= 120.0
    detail["separate_bus_within_tolerance"] = bool(ok)
    allmix = [torch.empty_like(mix) for _ in range(world)]
    dist.all_gather(allmix, mix)
    detail["identical_on_all_ranks"] = all(torch.equal(allmix[0], m) for m in allmix)
    ok = ok and detail["identical_on_all_ranks"]          # every rank holds the same bits
    # the exchange fused into the render launch: the same bits as the separate bus kernel, in both modes, over 3 blocks
    for bus_mode in (1, 2):
        b.upload_state(np.ascontiguousarray(s0[lo:hi]).view(np.uint32).reshape(hi - lo, 5))
        bus.attach(b, bus_mode)
        m3 = [torch.zeros(2 * F, dtype=torch.float32, device=dev) for _ in range(3)]
        for k in range(3):
            b.run_dev(F, mix=m3[k].data_ptr())
        bus.flush()
        torch.cuda.synchronize()
        bus.detach(b)
        detail["fused_mode%d_block0_equals_separate" % bus_mode] = bool(torch.equal(m3[0], mix)) and bus.status() == 0
        detail["fused_mode%d_block0_max_abs_diff" % bus_mode] = float((m3[0] - mix).abs().max().item())
        ok = ok and detail["fused_mode%d_block0_equals_separate" % bus_mode]
        # blocks 2 and 3 against the separate form
        b.upload_state(np.ascontiguousarray(s0[lo:hi]).view(np.uint32).reshape(hi - lo, 5))
        for k in range(3):
            mk = torch.zeros(2 * F, dtype=torch.float32, device=dev)
            b.run_dev(F, mix=mk.data_ptr())
            bus.allreduce(mk.data_ptr(), 2 * F, op=st.Bus.FSUM)
            torch.cuda.synchronize()
            detail["fused_mode%d_block%d_equals_separate" % (bus_mode, k)] = bool(torch.equal(m3[k], mk))
            ok = ok and torch.equal(m3[k], mk)
    b.free()
    if N == 0:
        bus.destroy()
        return ok, detail
    # timing at the full size
    s0, prm = xvoice_records(N, 6)
    lo, hi = shard.shard_range(N, rank, world)
    b = ctx.batch(st.XVOICE, hi - lo)
    b.upload_state(np.ascontiguousarray(s0[lo:hi]).view(np.uint32).reshape(hi - lo, 5))
    b.upload_param(np.ascontiguousarray(prm[lo:hi]).view(np.uint32).reshape(hi - lo, 8))
    mixes = [torch.zeros(2 * F, dtype=torch.float32, device=dev) for _ in range(2)]
    k = [0]

    def render_only():
        b.run_dev(F, mix=mixes[0].data_ptr())

    def nccl():
        b.run_dev(F, mix=mixes[0].data_ptr())
        dist.all_reduce(mixes[0])

    def overlapped():
        s = k[0] & 1
        k[0] += 1
        bus.wait(s)
        b.run_dev(F, mix=mixes[s].data_ptr())
        bus.begin(s, mixes[s].data_ptr(), 2 * F, op=st.Bus.FSUM)

    def fused():
        s = k[0] & 1
        k[0] += 1
        b.run_dev(F, mix=mixes[s].data_ptr())

    res = {}
    for name, fn in (("render_only", render_only), ("nccl_allreduce", nccl), ("peer_memory_bus_overlapped", overlapped), ("fused_in_launch", fused),
                     ("fused_pipelined", fused)):
        if name == "fused_in_launch":
            bus.attach(b, 1)
        elif name == "fused_pipelined":
            bus.attach(b, 2)
        else:
            bus.detach(b)
        for _ in range(3):
            fn()
        dist.barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            fn()
        bus.wait(0); bus.wait(1); bus.flush()
        e1.record(stream)
        dist.barrier(); torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / reps], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        res[name] = float(t.item())
    ok = ok and bus.status() == 0
    bus.detach(b)
    bus.destroy(); b.free()
    return ok, res


def grain_records(N, seed):
    """state, threshold, phase, inc, gl, gr of N grains (the same on every rank)"""
    r = np.random.default_rng(seed)
    state = r.choice(np.array([0.0, 0.5, -0.5], np.float32), N)
    th = r.uniform(0.05, 0.5, N).astype(np.float32)
    phase = r.integers(0, 2**32, N, dtype=np.uint32)
    inc = tab[r.integers(36, 97, N)]
    gl = r.integers(0, 65, N).astype(np.uint8)
    return state, th, phase, inc, gl, (64 - gl).astype(np.uint8)


def grain_batch(g, lo, hi):
    state, th, phase, inc, gl, gr = (x[lo:hi] for x in g)
    b = ctx.batch(st.SQUARE_GRAIN_MIX, hi - lo)
    s_rec = np.zeros((hi - lo, 2), np.uint32); s_rec[:, 0] = state.view(np.uint32); s_rec[:, 1] = phase
    p_rec = np.zeros((hi - lo, 4), np.uint32); p_rec[:, 0] = th.view(np.uint32); p_rec[:, 1] = inc; p_rec[:, 2] = gl; p_rec[:, 3] = gr
    b.upload_state(s_rec); b.upload_param(p_rec)
    return b


def grain_check(N, F, K=6):
    """C3b: K consecutive blocks of the sharded grain mix, the bus formed by the separate bus kernel and by the exchange fused
    into the render launch (modes 1 and 2), each compared on every rank with the single-device oracle."""
    g = grain_records(N, 77)
    lo, hi = shard.shard_range(N, rank, world)
    ga = tuple(x.copy() for x in g)
    wants = [orc.square_grain_mix_run(*ga, N, F) for _ in range(K)]

    def same(imix, out, k):
        return np.array_equal(imix.cpu().numpy().reshape(2, F), wants[k][0]) and \
            np.array_equal(out.cpu().numpy().reshape(2, F).view(np.uint32), wants[k][1].view(np.uint32))

    bus = shard.connect_bus(st.Bus(ctx, 4096, world, rank))
    mixes = [torch.zeros(2 * F, dtype=torch.int32, device=dev) for _ in range(K)]
    outs = [torch.zeros(2 * F, dtype=torch.float32, device=dev) for _ in range(K)]
    b = grain_batch(g, lo, hi)
    for k in range(K):                                    # the separate bus kernel after each render
        b.run_dev(F, mix=mixes[k].data_ptr())
        bus.allreduce(mixes[k].data_ptr(), 2 * F, out_dev=outs[k].data_ptr(), scale=st.Bus.SCALE_GRAIN)
    torch.cuda.synchronize()
    ok_sep = bus.status() == 0 and all(same(mixes[k], outs[k], k) for k in range(K))
    b.free()
    ok_f = []
    for bus_mode in (1, 2):
        b = grain_batch(g, lo, hi)
        bus.attach(b, bus_mode)
        for m, o in zip(mixes, outs):
            m.zero_(); o.zero_()
        for k in range(K):
            b.run_dev(F, mix=mixes[k].data_ptr(), out=outs[k].data_ptr())
        bus.flush()
        torch.cuda.synchronize()
        ok_f.append(bus.status() == 0 and all(same(mixes[k], outs[k], k) for k in range(K)))
        bus.detach(b)
        b.free()
    bus.destroy()
    t = torch.tensor([int(ok_sep), int(ok_f[0]), int(ok_f[1])], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return [bool(x.item()) for x in t]


def grain_timing(N, F, reps=400, rounds=3):
    """C3b at full size: ms per 256-frame block, CUDA events, max over ranks; each form timed `rounds` times, in turn."""
    g = grain_records(N, 78)
    lo, hi = shard.shard_range(N, rank, world)
    b = grain_batch(g, lo, hi)
    bus = shard.connect_bus(st.Bus(ctx, 4096, world, rank))
    mixes = [torch.zeros(2 * F, dtype=torch.int32, device=dev) for _ in range(2)]
    outs = [torch.zeros(2 * F, dtype=torch.float32, device=dev) for _ in range(2)]
    mix4 = torch.zeros(8 * F, dtype=torch.int32, device=dev)
    out4 = torch.zeros(8 * F, dtype=torch.float32, device=dev)
    k = [0]

    def render_only():
        b.run_dev(F, mix=mixes[0].data_ptr(), out=outs[0].data_ptr())

    def separate_bus():                                   # today's form: the bus kernel on the bus's stream, overlapped
        s = k[0] & 1
        k[0] += 1
        bus.wait(s)
        b.run_dev(F, mix=mixes[s].data_ptr(), out=outs[s].data_ptr())
        bus.begin(s, mixes[s].data_ptr(), 2 * F, out_dev=outs[s].data_ptr(), scale=st.Bus.SCALE_GRAIN)

    def fused():
        s = k[0] & 1
        k[0] += 1
        b.run_dev(F, mix=mixes[s].data_ptr(), out=outs[s].data_ptr())

    def fused_k4():                                       # four frame blocks per launch, one exchange of [2][4 x 256]
        b.run_dev(4 * F, mix=mix4.data_ptr(), out=out4.data_ptr())

    forms = (("render_only", 0, render_only, 1), ("separate_bus_kernel_overlapped", 0, separate_bus, 1), ("fused_in_launch", 1, fused, 1),
             ("fused_pipelined", 2, fused, 1), ("fused_pipelined_4_blocks_per_launch", 2, fused_k4, 4))
    res = {name: [] for name, _, _, _ in forms}
    for _ in range(rounds):
        for name, mode, fn, per in forms:
            if mode:
                bus.attach(b, mode)
            else:
                bus.detach(b)
            for _ in range(10):
                fn()
            bus.wait(0); bus.wait(1); bus.flush()
            dist.barrier(); torch.cuda.synchronize()
            n = max(1, reps // per)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(n):
                fn()
            bus.wait(0); bus.wait(1); bus.flush()
            e1.record(stream)
            dist.barrier(); torch.cuda.synchronize()
            t = torch.tensor([e0.elapsed_time(e1) / (n * per)], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            res[name].append(float(t.item()))
    ok = bus.status() == 0
    bus.detach(b)
    bus.destroy(); b.free()
    return res, ok


def card():
    """name and power limit of this rank's GPU, read in the same run as the measurement"""
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        limit = r.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        limit = None
    return {"name": torch.cuda.get_device_name(dev), "power_limit_and_max_sm_clock": limit}


CHECK_ONLY = "--check-only" in sys.argv
for mode in (0, 1):
    a, bb, c1, c2 = check(256 * 1024 + 77, 512, mode)
    if rank == 0:
        print(json.dumps({"check": "voice bank mix bus, mode %d" % mode, "n_gpus": world, "nccl_bit_exact": a, "peer_bus_bit_exact": bb,
                          "fused_in_launch_bit_exact": c1, "fused_pipelined_bit_exact": c2}), flush=True)
sep, f1, f2 = grain_check(256 * 1024 + 77, 256)
if rank == 0:
    print(json.dumps({"check": "square_grain mix bus", "n_gpus": world, "peer_bus_bit_exact": sep, "fused_in_launch_bit_exact": f1,
                      "fused_pipelined_bit_exact": f2}), flush=True)
if CHECK_ONLY:
    okx, detail = xvoice_check_and_timing(64 * 1024 + 5, 0, 512)
    if rank == 0:
        print(json.dumps({"check": "xvoice float bus", "n_gpus": world, "float_bus_within_tolerance_and_identical_on_all_ranks_ok": bool(okx), "detail": detail}), flush=True)
    ctx.close()
    dist.destroy_process_group()
    sys.exit(0)
res, ok = timing(4 * 1024 * 1024, 512)
if rank == 0:
    N, F = 4 * 1024 * 1024, 512
    print(json.dumps({"config": "C4' voice bank 4 Mi voices x 512 frames sharded over %d GPUs, int32 mix bus" % world, "n_gpus": world, "bus_ok": ok,
                      "ms_per_block": res, "voice_samples_per_s": {k: N * F / (v * 1e-3) for k, v in res.items()},
                      "exchange_cost_us": {"nccl": 1e3 * (res["nccl_allreduce_plus_convert"] - res["render_only"]),
                                           "peer_bus": 1e3 * (res["peer_memory_bus_kernel"] - res["render_only"]),
                                           "peer_bus_overlapped": 1e3 * (res["peer_memory_bus_overlapped"] - res["render_only"])}}), flush=True)
okx, resx = xvoice_check_and_timing(64 * 1024 + 5, 4 * 1024 * 1024, 512)
if rank == 0:
    N, F = 4 * 1024 * 1024, 512
    print(json.dumps({"config": "C4 poly voice 4 Mi voices x 512 frames sharded over %d GPUs, float stereo mix bus" % world, "n_gpus": world,
                      "float_bus_within_tolerance_and_identical_on_all_ranks": bool(okx), "ms_per_block": resx,
                      "voice_samples_per_s": {k: N * F / (v * 1e-3) for k, v in resx.items()}}), flush=True)
resg, okg = grain_timing(1024 * 1024, 256)
if rank == 0:
    N, F = 1024 * 1024, 256
    med = {k: float(np.median(v)) for k, v in resg.items()}
    print(json.dumps({"config": "C3b square_grain mix 1 Mi grains x 256-frame blocks sharded over %d GPUs, int32 mix bus" % world, "n_gpus": world, "bus_ok": okg,
                      "card": card(), "ms_per_block": med, "ms_per_block_rounds": resg,
                      "grain_samples_per_s": {k: N * F / (v * 1e-3) for k, v in med.items()}}), flush=True)
ctx.close()
dist.destroy_process_group()
