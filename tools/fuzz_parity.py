"""Randomised parity sweep (development tool): PDM v2 (all kernel generations are picked by shape),
square_grain, graphs (JIT) with random shapes / counters / layouts against the oracle.  Prints one line
per case and a summary; exits 1 on the first mismatch."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import synth_tools_b200 as st
from oracle import pyoracle as po

seed = int(sys.argv[1]) if len(sys.argv) > 1 else 1
n_cases = int(sys.argv[2]) if len(sys.argv) > 2 else 40
rng = np.random.default_rng(seed)
orc = po.Oracle()
ctx = st.Context(0)
bad = 0

def tiled16(a, N, F):
    return a.reshape(F // 16, N, 16).transpose(1, 0, 2).reshape(N, F)

for case in range(n_cases):
    kind = rng.choice(["pdm", "pdm_big", "grain", "graph", "voice", "gmix", "pdm_v1", "xmix", "planar", "sweep"])
    if kind in ("pdm", "pdm_big"):
        order = int(rng.integers(1, 5)) if kind == "pdm" else 2
        bank = int(rng.choice([1, 2, 3, 4, 7])) if kind == "pdm" else 3
        N = int(rng.integers(1, 4000)) if kind == "pdm" else int(rng.integers(96 * 149, 96 * 160))
        ctl = int(rng.integers(4, 10)) if kind == "pdm" else int(rng.integers(6, 10))
        unit = int(rng.choice([1, 16, 64]))
        F = int(rng.integers(1, 40)) * unit
        count0 = int(rng.integers(0, (1 << ctl) // unit + 1)) * unit % (1 << ctl)
        layout = st.TILED if (F % 16 == 0 and rng.random() < 0.6) else st.PLANAR
        opts = {}
        if kind == "pdm_big":
            opts = {"pdm_ctas_per_sm": 1, "pdm_slice_batches": int(rng.choice([2, 4, 8]))}
        for k, v in opts.items():
            ctx.set_option(k, v)
        nb = (N + bank - 1) // bank
        chan0 = rng.integers(0, 2**32, (N, 5 + order), dtype=np.uint32)
        prng0 = rng.integers(1, 2**32, nb, dtype=np.uint32)
        sp = po.pdm_setpoints(N, F // (1 << ctl) + 2)
        ca, pa = chan0.copy(), prng0.copy()
        want, wcnt = orc.pdm_v2_run(ca, order, N, bank, pa, None, 0x3FF, count0, ctl, 24, sp, F)
        b = ctx.batch(st.PDM_V2, N, order=order, bank_size=bank, ctl_div_log=ctl, layout=layout)
        b.upload_state(chan0); b.upload_bank(prng0, count0)
        out = np.zeros(N * F, np.uint8)
        b.run(F, ctl=sp, out=out)
        got = tiled16(out, N, F) if layout == st.TILED else out.reshape(N, F)
        p1, c1 = b.download_bank()
        ok = np.array_equal(got, want) and np.array_equal(b.download_state(), ca) and np.array_equal(p1, pa) and c1 == wcnt
        desc = "order=%d bank=%d N=%d F=%d ctl=%d count0=%d layout=%d %s" % (order, bank, N, F, ctl, count0, layout, opts)
        b.free()
        ctx.set_option("pdm_ctas_per_sm", 4); ctx.set_option("pdm_slice_batches", 64)
    elif kind == "grain":
        N, F = int(rng.integers(1, 3000)), int(rng.integers(1, 600))
        layout = st.PLANAR if rng.random() < 0.6 else st.INTERLEAVED
        inp = rng.uniform(-1, 1, (N, F)).astype(np.float32)
        th = rng.uniform(-0.1, 0.5, (N, 1)).astype(np.float32)
        s0 = rng.choice(np.array([0.0, 0.5, -0.5, 0.25], np.float32), (N, 1))
        sa = s0[:, 0].copy()
        want = orc.square_grain_run(sa, th[:, 0].copy(), N, F, inp)
        b = ctx.batch(st.SQUARE_GRAIN, N, layout=layout)
        b.upload_state(s0); b.upload_param(th)
        il = layout == st.INTERLEAVED
        io = np.ascontiguousarray(inp.T) if il else inp.copy()
        inplace = rng.random() < 0.5
        out = io if inplace else np.zeros_like(io)
        b.run(F, inp=io, out=out)
        ok = np.array_equal((out.T if il else out).view(np.uint32), want.view(np.uint32)) and np.array_equal(b.download_state().view(np.float32)[:, 0], sa)
        desc = "N=%d F=%d layout=%d inplace=%d" % (N, F, layout, inplace)
        b.free()
    elif kind == "voice":
        N, F, mode = int(rng.integers(1, 30000)), int(rng.integers(1, 1200)), int(rng.integers(0, 2))
        G = int(rng.choice([0, 64, 100, 4096, 5000]))
        v = np.zeros((N, 2), np.uint32)
        v[:, 0] = rng.integers(0, 2**32, N, dtype=np.uint32) * (rng.random(N) < 0.8)
        v[:, 1] = rng.integers(0, 2**32, N, dtype=np.uint32)
        va = v.copy()
        gg = G if 0 < G <= N else N
        want_i, want_f = orc.voice_bank_run(va, N, gg, mode, F)
        b = ctx.batch(st.VOICE_BANK, N, voices_per_bus=G, mode=mode)
        b.upload_state(v)
        nbus = (N + gg - 1) // gg
        vec = np.zeros((nbus, F), np.float32); mix = np.zeros((nbus, F), np.int32)
        b.run(F, out=vec, mix=mix)
        ok = np.array_equal(mix.view(np.uint32), want_i.view(np.uint32)) and np.array_equal(vec.view(np.uint32), want_f.view(np.uint32)) and np.array_equal(b.download_state(), va)
        desc = "N=%d F=%d G=%d mode=%d" % (N, F, G, mode)
        b.free()
    elif kind == "gmix":
        N, F = int(rng.integers(1, 90000)), int(rng.integers(1, 400))
        state = rng.choice(np.array([0.0, 0.5, -0.5], np.float32), N)
        th = rng.uniform(0.0, 0.5, N).astype(np.float32)
        if rng.random() < 0.3: th[::11] = -th[::11]
        phase = rng.integers(0, 2**32, N, dtype=np.uint32)
        inc = rng.integers(0, 2**30, N, dtype=np.uint32)
        gl = rng.integers(0, 65, N).astype(np.uint8); gr = (64 - gl).astype(np.uint8)
        sa, pa = state.copy(), phase.copy()
        want_i, want_f = orc.square_grain_mix_run(sa, th, pa, inc, gl, gr, N, F)
        gen = int(rng.integers(0, 3))
        ctx.set_option("grain_mix2", gen)
        b = ctx.batch(st.SQUARE_GRAIN_MIX, N)
        s_rec = np.zeros((N, 2), np.uint32); s_rec[:, 0] = state.view(np.uint32); s_rec[:, 1] = phase
        p_rec = np.zeros((N, 4), np.uint32); p_rec[:, 0] = th.view(np.uint32); p_rec[:, 1] = inc; p_rec[:, 2] = gl; p_rec[:, 3] = gr
        b.upload_state(s_rec); b.upload_param(p_rec)
        out = np.zeros((2, F), np.float32); mix = np.zeros((2, F), np.int32)
        b.run(F, out=out, mix=mix)
        s1 = b.download_state()
        ok = np.array_equal(mix, want_i) and np.array_equal(out.view(np.uint32), want_f.view(np.uint32)) and np.array_equal(s1[:, 0].view(np.float32), sa) and np.array_equal(s1[:, 1], pa)
        desc = "N=%d F=%d gen=%d" % (N, F, gen)
        b.free(); ctx.set_option("grain_mix2", 2)
    elif kind == "pdm_v1":
        bank = int(rng.choice([1, 2, 3, 4, 9]))
        N, F = int(rng.integers(1, 70000)), int(rng.integers(1, 12)) * 128
        layout = int(rng.choice([st.PLANAR, st.INTERLEAVED, st.TILED]))
        nb = (N + bank - 1) // bank
        ch0 = rng.integers(0, 2**32, (N, 2), dtype=np.uint32); prng0 = rng.integers(1, 2**32, nb, dtype=np.uint32)
        ca, pa = ch0.copy(), prng0.copy()
        bits = orc.pdm_v1_run(ca, N, bank, pa, None, 0x0FFFFFFF, F)
        want = np.packbits(bits.reshape(N, F // 32, 32), axis=2, bitorder="little").view("<u4").reshape(N, F // 32)
        b = ctx.batch(st.PDM_V1, N, bank_size=bank, dither_mask=0x0FFFFFFF, layout=layout)
        b.upload_state(ch0); b.upload_bank(prng0)
        out = np.zeros(N * F // 32, np.uint32)
        b.run(F, out=out)
        got = out.reshape(N, F // 32) if layout == st.PLANAR else (out.reshape(F // 32, N).T if layout == st.INTERLEAVED else out.reshape(F // 128, N, 4).transpose(1, 0, 2).reshape(N, F // 32))
        ok = np.array_equal(got, want) and np.array_equal(b.download_state(), ca) and np.array_equal(b.download_bank()[0], pa)
        desc = "bank=%d N=%d F=%d layout=%d" % (bank, N, F, layout)
        b.free()
    elif kind == "planar":
        # the PLANAR staging template (tensor TMA / scalar by planar_bulk) under four processors
        N, F = int(rng.integers(1, 3000)), int(rng.integers(1, 150)) * int(rng.choice([1, 4, 16]))
        mode = int(rng.choice([0, 2])); which = str(rng.choice(["pdm", "onepole", "pwm", "clock"]))
        ctx.set_option("planar_bulk", mode)
        if which == "pdm":
            order = int(rng.integers(1, 5)); use_in = bool(rng.random() < 0.6); sh = int(rng.choice([8, 24, 31]))
            s0 = rng.integers(0, 2**32, (N, order), dtype=np.uint32); inp = rng.integers(0, 2**32, (N, F), dtype=np.uint32)
            dith = rng.integers(0, 1 << min(sh, 12), F, dtype=np.uint32); cst = rng.integers(0, 2**32, (N, 1), dtype=np.uint32)
            sa = s0.copy()
            want = orc.pdm_run(order, sa, N, F, inp if use_in else None, cst[:, 0].copy(), sh, dith)
            b = ctx.batch(st.PDM, N, order=order, out_shift=sh); b.upload_state(s0); b.upload_param(cst)
            out = np.zeros((N, F), np.uint32)
            b.run(F, inp=inp if use_in else None, in2=dith, out=out)
            ok = np.array_equal(out, want) and np.array_equal(b.download_state(), sa)
        elif which == "onepole":
            x = rng.uniform(-1, 1, (N, F)).astype(np.float32); a = rng.uniform(0.001, 0.9, (N, 1)).astype(np.float32); y0 = rng.uniform(-1, 1, (N, 1)).astype(np.float32)
            ya = y0[:, 0].copy()
            want = orc.onepole_run(ya, a[:, 0].copy(), N, F, x)
            b = ctx.batch(st.ONEPOLE, N); b.upload_state(y0); b.upload_param(a)
            out = np.zeros((N, F), np.float32)
            b.run(F, inp=x, out=out)
            ok = np.array_equal(out.view(np.uint32), want.view(np.uint32)) and np.array_equal(b.download_state()[:, 0].view(np.uint32), ya.view(np.uint32))
        elif which == "pwm":
            F = (F + 15) // 16 * 16
            ph0 = rng.integers(0, 1 << 24, (N, 1), dtype=np.uint32); sp = rng.integers(0, 1 << 16, (N, 1), dtype=np.uint32)
            pa = ph0[:, 0].copy()
            want = orc.pwm_run(pa, sp[:, 0].copy(), N, F)
            b = ctx.batch(st.PWM, N); b.upload_state(ph0); b.upload_param(sp)
            out = np.zeros((N, F), np.uint8)
            b.run(F, out=out)
            ok = np.array_equal(out, want) and np.array_equal(b.download_state()[:, 0], pa)
        else:
            hp = rng.integers(-2, 300, N).astype(np.int32)
            s0 = np.zeros((N, 2), np.int32); s0[:, 0] = rng.integers(0, 400, N); s0[:, 1] = rng.integers(0, 2, N)
            sa = s0.copy()
            want = orc.word_clock_run(sa, hp, N, F)
            b = ctx.batch(st.WORD_CLOCK, N); b.upload_state(s0.view(np.uint32)); b.upload_param(hp.view(np.uint32).reshape(N, 1))
            out = np.zeros((N, F), np.float32)
            b.run(F, out=out)
            ok = np.array_equal(out.view(np.uint32), want.view(np.uint32)) and np.array_equal(b.download_state().view(np.int32), sa)
        desc = "%s N=%d F=%d planar_bulk=%d" % (which, N, F, mode)
        b.free()
        ctx.set_option("planar_bulk", 2)
    elif kind == "sweep":
        # time-parallel raw render: closed-form / ticked zero-state pass, any increment
        N, F = int(rng.integers(1, 700)), int(rng.integers(33, 3000)) * 2
        layout = st.TILED if rng.random() < 0.5 else st.PLANAR
        closed = int(rng.random() < 0.7); groups = int(rng.choice([0, 1, 2, 4, 8])); chunk = int(rng.choice([0, 32, 64, 96, 256, 1024]))
        prm = np.zeros(N, po.xvoice_param_dtype)
        prm["inc"] = np.where(rng.random(N) < 0.7, rng.integers(0, 2**29, N), rng.integers(0, 2**32, N)).astype(np.uint32)
        prm["f"] = rng.uniform(0.01, 0.3, N); prm["q"] = rng.uniform(0.5, 2.0, N)
        prm["env_attack"] = rng.uniform(1e-3, 1e-1, N); prm["env_release"] = rng.uniform(2e-4, 1e-2, N)
        prm["gate_frames"] = rng.integers(0, F, N)
        prm["gl"] = rng.uniform(0, 1, N); prm["gr"] = 1.0 - prm["gl"]
        s0 = np.zeros(N, po.xvoice_state_dtype)
        s0["phase"] = rng.integers(0, 2**32, N, dtype=np.uint32); s0["env"] = rng.uniform(0, 1, N); s0["t"] = rng.integers(0, 100, N)
        s0["lp"] = rng.uniform(-0.5, 0.5, N); s0["bp"] = rng.uniform(-0.5, 0.5, N)
        sa = s0.copy()
        want_raw, _ = orc.xvoice_run(sa, prm, N, F, want_mix=False)
        ctx.set_option("xvoice_closed", closed); ctx.set_option("xvoice_groups", groups); ctx.set_option("xvoice_chunk", chunk)
        b = ctx.batch(st.XVOICE, N, layout=layout, mode=st.XVOICE_SCAN)
        b.upload_state(s0.view(np.uint32).reshape(N, 5)); b.upload_param(prm.view(np.uint32).reshape(N, 8))
        raw = np.zeros(N * F * 2, np.float32)
        b.run(F, out=raw)
        got = raw.reshape(F // 2, N, 2, 2).transpose(1, 0, 2, 3).reshape(N, F, 2) if layout == st.TILED else raw.reshape(N, F, 2)
        w64, g64 = want_raw.astype(np.float64), got.astype(np.float64)
        gs = b.download_state().view(po.xvoice_state_dtype).reshape(N)
        snr = 10 * np.log10((w64 ** 2).sum() / max(((g64 - w64) ** 2).sum(), 1e-300))
        ok = np.abs(g64 - w64).max() <= 1e-5 * max(np.abs(w64).max(), 1e-30) and snr >= 120.0 and np.array_equal(gs["phase"], sa["phase"]) \
            and np.array_equal(gs["t"], sa["t"]) and np.array_equal(gs["env"].view(np.uint32), sa["env"].view(np.uint32))
        desc = "N=%d F=%d layout=%d closed=%d groups=%d chunk=%d snr=%.1f" % (N, F, layout, closed, groups, chunk, snr)
        b.free()
        ctx.set_option("xvoice_closed", 1); ctx.set_option("xvoice_groups", 0); ctx.set_option("xvoice_chunk", 0)
    elif kind == "xmix":
        N, F = int(rng.integers(1, 200000)), int(rng.integers(1, 200))
        prm = np.zeros(N, po.xvoice_param_dtype)
        prm["inc"] = rng.integers(0, 2**28, N, dtype=np.uint32)
        prm["f"] = rng.uniform(0.01, 0.3, N); prm["q"] = rng.uniform(0.5, 2.0, N)
        prm["env_attack"] = rng.uniform(1e-3, 1e-1, N); prm["env_release"] = rng.uniform(1e-3, 1e-2, N)
        prm["gate_frames"] = rng.integers(0, 2 * F + 2, N)
        prm["gl"] = rng.uniform(0, 1, N); prm["gr"] = 1.0 - prm["gl"]
        s0 = np.zeros(N, po.xvoice_state_dtype)
        s0["phase"] = rng.integers(0, 2**32, N, dtype=np.uint32); s0["env"] = rng.uniform(0, 1, N); s0["t"] = rng.integers(0, F + 1, N)
        sa = s0.copy()
        _, want_mix = orc.xvoice_run(sa, prm, N, F, want_raw=False)
        b = ctx.batch(st.XVOICE, N)
        b.upload_state(s0.view(np.uint32).reshape(N, 5)); b.upload_param(prm.view(np.uint32).reshape(N, 8))
        mix = np.zeros((2, F), np.float32)
        b.run(F, mix=mix)
        got = b.download_state().view(po.xvoice_state_dtype).reshape(N)
        w64, g64 = np.asarray(want_mix, np.float64).reshape(2, F), mix.astype(np.float64)
        ok = np.array_equal(got.view(np.uint32), sa.view(np.uint32)) and np.abs(g64 - w64).max() <= 1e-5 * max(np.abs(w64).max(), 1e-30)
        desc = "N=%d F=%d" % (N, F)
        b.free()
    else:
        nn, n_in = int(rng.integers(1, 30)), int(rng.integers(1, 4))
        rows = []
        for k in range(nn):
            src = int(rng.integers(-n_in, k)) if k else -int(rng.integers(1, n_in + 1))
            t = int(rng.integers(0, 4)); mask = int(rng.choice([1, 2, 3, 6, 0xFFFFFFFF]))
            if t == 2: rows.append((po.node_glide(int(rng.integers(1, 7))), src, mask))
            elif t == 3: rows.append((po.node_pdm(int(rng.integers(1, 5)), int(rng.choice([0, 8, 24, 31]))), src, mask, int(rng.integers(-n_in, k)) if k else -1))
            else: rows.append((t, src, mask))
        n_in = max(1, max(max(-r[1], -r[3] if len(r) > 3 else 0) for r in rows))
        outs = [int(x) for x in rng.integers(0, nn, int(rng.integers(1, 6)))]
        N, F = int(rng.integers(1, 1500)), int(rng.integers(1, 300))
        layout = st.PLANAR if rng.random() < 0.5 else st.INTERLEAVED
        masked = rng.random() < 0.5
        inp = rng.integers(0, 4, (N, n_in, F), dtype=np.uint32)
        changed = rng.integers(0, 8, (N, F), dtype=np.uint32) if masked else None
        sw = sum(po.node_words(r[0]) for r in rows)
        s0 = rng.integers(0, 2**32, (N, sw), dtype=np.uint32)
        o = 0
        for r in rows:
            if r[0] & 0xFF == po.NODE_GLIDE: s0[:, o + 4] &= (1 << (r[0] >> 8)) - 1
            o += po.node_words(r[0])
        sa = s0.copy()
        want = orc.graph_run_multi(rows, n_in, outs, sa, N, F, inp, changed)
        pmode = int(rng.choice([0, 2]))                        # generated planar kernel: scalar graph_planar_simple / tensor TMA
        ctx.set_option("planar_bulk", pmode)
        b = ctx.batch(st.GRAPH, N, nodes=rows, n_inputs=n_in, out_node=outs, layout=layout)
        b.upload_state(s0)
        il = layout == st.INTERLEAVED
        out = np.zeros((F, len(outs), N) if il else (N, len(outs), F), np.uint32)
        b.run(F, inp=np.ascontiguousarray(inp.transpose(2, 1, 0)) if il else inp, in2=None if changed is None else (np.ascontiguousarray(changed.T) if il else changed), out=out)
        ok = np.array_equal(out.transpose(2, 1, 0) if il else out, want) and np.array_equal(b.download_state(), sa)
        desc = "nodes=%d n_in=%d outs=%d N=%d F=%d layout=%d masked=%d planar_bulk=%d [%s]" % (nn, n_in, len(outs), N, F, layout, masked, pmode, b.jit_log.strip()[:60])
        b.free()
        ctx.set_option("planar_bulk", 2)
    print("%s %-8s %s" % ("ok  " if ok else "FAIL", kind, desc), flush=True)
    if not ok:
        bad += 1
        break
print("cases run: %d, failures: %d" % (case + 1, bad))
sys.exit(1 if bad else 0)
