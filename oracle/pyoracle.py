"""ctypes bindings for oracle/liboracle.so and oracle/_ref/libref.so.

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs.  The product package
(synth_tools_b200) never imports this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(HERE, "liboracle.so")
REF_SO = os.path.join(HERE, "_ref", "libref.so")
REF_O3_SO = os.path.join(HERE, "_ref", "libref_o3.so")     # the same sources, -O3 -march=x86-64-v3 (build_ref.sh)

u32p = np.ctypeslib.ndpointer(np.uint32, flags="C_CONTIGUOUS")
i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
u8p = np.ctypeslib.ndpointer(np.uint8, flags="C_CONTIGUOUS")
f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
VP = C.c_void_p

NODE_ACC, NODE_EDGE, NODE_GLIDE, NODE_PDM = 0, 1, 2, 3
NODE_PHASOR_F, NODE_SVF, NODE_ENV, NODE_ONEPOLE, NODE_GAIN, NODE_ASFLOAT, NODE_GLIDE_F, NODE_MUL = 4, 5, 6, 7, 8, 9, 10, 11   # include/cproc_ext.h
SRC_ZERO = -0x80000000


def node_glide(div_log):
    """glide node type word: kind | (control divider log2 << 8)."""
    return NODE_GLIDE | (div_log << 8)


def node_glide_f(div_log):
    """glide_f node type word (include/cproc_ext.h): kind | (control divider log2 << 8)."""
    return NODE_GLIDE_F | (div_log << 8)


def node_pdm(order, out_shift):
    """pdm node type word: kind | (order | out_shift << 3) << 8."""
    return NODE_PDM | ((order | (out_shift << 3)) << 8)


def node_words(t):
    if t & 0xFF == NODE_PDM:
        return 1 + ((t >> 8) & 7)
    return {NODE_EDGE: 2, NODE_GLIDE: 5, NODE_PHASOR_F: 2, NODE_SVF: 2, NODE_ENV: 3, NODE_GLIDE_F: 3}.get(t & 0xFF, 1)


def node_param_words(t):
    return {NODE_PHASOR_F: 1, NODE_SVF: 2, NODE_ENV: 3, NODE_ONEPOLE: 1, NODE_GAIN: 1}.get(t & 0xFF, 0)

MIX_SAW, MIX_SQUARE = 0, 1

node_dtype = np.dtype([("type", np.uint32), ("src", np.int32), ("cond_mask", np.uint32), ("src2", np.int32)])
xvoice_param_dtype = np.dtype([("inc", np.uint32), ("f", np.float32), ("q", np.float32),
                               ("env_attack", np.float32), ("env_release", np.float32),
                               ("gate_frames", np.uint32), ("gl", np.float32), ("gr", np.float32)])
xvoice_state_dtype = np.dtype([("phase", np.uint32), ("lp", np.float32), ("bp", np.float32),
                               ("env", np.float32), ("t", np.uint32)])


def set_threads(n):
    """OpenMP thread count of the oracle / reference libraries (torchrun exports
    OMP_NUM_THREADS=1; the CPU baseline is meant to use every host core)."""
    try:
        C.CDLL("libgomp.so.1").omp_set_num_threads(int(n))
    except OSError:
        pass


def build(force=False):
    """Compile the oracle (always possible) and oracle/_ref (only where the
    reference tree is present; elsewhere the prebuilt .so is used)."""
    if force or not os.path.exists(ORACLE_SO) or \
            os.path.getmtime(ORACLE_SO) < max(os.path.getmtime(os.path.join(HERE, f)) for f in ("cproc_oracle.c", "arm_v1_model.c", "build_oracle.sh")):
        subprocess.check_call(["bash", os.path.join(HERE, "build_oracle.sh")])
    if os.path.isdir(os.environ.get("REF", "/root/reference")):
        recipe = [os.path.join(HERE, "build_ref.sh")] + [os.path.join(d, f) for d in (os.path.join(HERE, "ref"), os.path.join(HERE, "shim"), os.path.join(HERE, "shim", "stm32"))
                                                         for f in os.listdir(d) if os.path.isfile(os.path.join(d, f))]
        root = os.path.dirname(HERE)                       # the extension processors and the graph texts are compiled into libref too
        recipe += [os.path.join(root, "include", "cproc_ext.h")] + [os.path.join(root, "tests", "golden", f) for f in os.listdir(os.path.join(root, "tests", "golden")) if f.endswith(".cproc")]
        if force or not os.path.exists(REF_SO) or not os.path.exists(REF_O3_SO) or os.path.getmtime(REF_O3_SO) < max(os.path.getmtime(f) for f in recipe):
            subprocess.check_call(["bash", os.path.join(HERE, "build_ref.sh")])


def _ptr(a):
    return None if a is None else a.ctypes.data_as(VP)


def make_nodes(rows):
    """rows: [(type, src, cond_mask)] -> structured array for *_graph_run."""
    a = np.zeros(len(rows), node_dtype)
    for i, r in enumerate(rows):                 # (type, src, cond_mask[, src2])
        a[i] = (r[0], r[1], r[2], r[3] if len(r) > 3 else 0)
    return a


GRAPH_TEST_CPROC = [(NODE_EDGE, -1, 1), (NODE_ACC, 0, 1)]            # linux/test_cproc.c:13-17
GRAPH_BP5 = [(NODE_EDGE, -1, 1), (NODE_ACC, 0, 1), (NODE_ACC, 1, 1)]  # stm32f103/bp5_plugin.c:4-9


class _Lib:
    prefix = ""

    def __init__(self, path):
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        self.path = path
        self.lib = C.CDLL(path)

    def _fn(self, name, restype, argtypes):
        f = getattr(self.lib, self.prefix + name)
        f.restype = restype
        f.argtypes = argtypes
        return f

    # ---- shared signatures (orc_* and ref_* agree where both exist) ----
    def graph_run(self, rows, n_inputs, out_node, state, N, F, inp, changed=None):
        nodes = make_nodes(rows)
        out = np.zeros((N, F), np.uint32)
        f = self._fn("graph_run", None, [VP, C.c_uint32, C.c_uint32, C.c_uint32, VP, C.c_uint64,
                                         C.c_uint64, VP, VP, VP])
        f(_ptr(nodes), len(rows), n_inputs, out_node, _ptr(state), N, F, _ptr(inp), _ptr(changed), _ptr(out))
        return out

    def graph_run_ext(self, rows, n_inputs, out_nodes, state, param, N, F, inp=None, changed=None):
        """Graphs with extension processors: param uint32 [N][param_words] (floats as bits) or None; returns out
        uint32 [N][len(out_nodes)][F].  liboracle: the restatement; libref: the DEF_PROC bodies of include/cproc_ext.h
        compiled against the reference's cproc.h (acc / edge / extension kinds only)."""
        nodes = make_nodes(rows)
        outs = np.asarray(out_nodes, np.uint32)
        out = np.zeros((N, len(outs), F), np.uint32)
        f = self._fn("graph_run_ext", None, [VP, C.c_uint32, C.c_uint32, VP, C.c_uint32, VP, VP, C.c_uint64, C.c_uint64, VP, VP, VP])
        f(_ptr(nodes), len(rows), n_inputs, _ptr(outs), len(outs), _ptr(state), _ptr(param), N, F, _ptr(inp), _ptr(changed), _ptr(out))
        return out

    def graph_run_multi(self, rows, n_inputs, out_nodes, state, N, F, inp, changed=None):
        """Several cproc_output statements: returns out [N][len(out_nodes)][F]."""
        nodes = make_nodes(rows)
        outs = np.asarray(out_nodes, np.uint32)
        out = np.zeros((N, len(outs), F), np.uint32)
        f = self._fn("graph_run_multi", None, [VP, C.c_uint32, C.c_uint32, VP, C.c_uint32, VP, C.c_uint64, C.c_uint64, VP, VP, VP])
        f(_ptr(nodes), len(rows), n_inputs, _ptr(outs), len(outs), _ptr(state), N, F, _ptr(inp), _ptr(changed), _ptr(out))
        return out

    def pdm_run(self, order, state, N, F, inp, in_const, out_shift, dither):
        out = np.zeros((N, F), np.uint32)
        f = self._fn("pdm_run", None, [C.c_uint32, VP, C.c_uint64, C.c_uint64, VP, VP, C.c_uint32, VP, VP])
        f(order, _ptr(state), N, F, _ptr(inp), _ptr(in_const), out_shift, _ptr(dither), _ptr(out))
        return out

    def pdm_v2_run(self, chan, order, N, bank_size, prng, dither_ext, dither_mask, count,
                   ctl_div_log, out_shift, setpoints, F, out=None):
        """chan [N][5+order] u32 (updated in place); prng [n_banks] u32 in place;
        returns (duty [N][F] u8, new_count).  out: a preallocated (and touched) duty buffer -- timed loops pass one, so
        that neither arm of a comparison pays for allocating and first-touching its output."""
        duty = np.zeros((N, F), np.uint8) if out is None else out
        assert duty.dtype == np.uint8 and duty.size >= N * F and duty.flags["C_CONTIGUOUS"]
        cnt = C.c_uint32(count)
        f = self._fn("pdm_v2_run", None, [VP, C.c_uint32, C.c_uint64, C.c_uint32, VP, VP, C.c_uint32,
                                          C.POINTER(C.c_uint32), C.c_uint32, C.c_uint32, VP, C.c_uint64, VP])
        f(_ptr(chan), order, N, bank_size, _ptr(prng), _ptr(dither_ext), dither_mask, C.byref(cnt),
          ctl_div_log, out_shift, _ptr(setpoints), F, _ptr(duty))
        return duty, cnt.value

    def pwm_run(self, phase, speed, N, F):
        duty = np.zeros((N, F), np.uint8)
        f = self._fn("pwm_run", None, [VP, VP, C.c_uint64, C.c_uint64, VP])
        f(_ptr(phase), _ptr(speed), N, F, _ptr(duty))
        return duty

    def square_grain_run(self, state, threshold, N, F, inp, out=None):
        if out is None:
            out = np.zeros((N, F), np.float32)
        f = self._fn("square_grain_run", None, [VP, VP, C.c_uint64, C.c_uint64, VP, VP])
        f(_ptr(state), _ptr(threshold), N, F, _ptr(inp), _ptr(out))
        return out


class Oracle(_Lib):
    prefix = "orc_"

    def __init__(self):
        build()
        super().__init__(ORACLE_SO)

    def xorshift32(self, state):
        s = C.c_uint32(state)
        f = self._fn("xorshift32", C.c_uint32, [C.POINTER(C.c_uint32)])
        r = f(C.byref(s))
        return r, s.value

    def pdm_v1_run(self, ch, N, bank_size, prng, dither_ext, dither_mask, F):
        """ch [N][2] u32 {setpoint, accu} in place; returns bits [N][F] u8."""
        bits = np.zeros((N, F), np.uint8)
        f = self._fn("pdm_v1_run", None, [VP, C.c_uint64, C.c_uint32, VP, VP, C.c_uint32, C.c_uint64, VP])
        f(_ptr(ch), N, bank_size, _ptr(prng), _ptr(dither_ext), dither_mask, F, _ptr(bits))
        return bits

    def arm_v1_mcu_run(self, chan, pin_chan0, rng, dmask, F):
        """oracle/arm_v1_model.c: the reference's adds / rrx sequence (mod_pdm.c:214-275) on a model of the ARM flags, ONE MCU of
        chan.shape[0] channels.  chan uint32 [n][2] in/out; returns (gpio set_bits uint32 [F], rng')."""
        gpio = np.zeros(F, np.uint32)
        r = C.c_uint32(int(rng))
        f = getattr(self.lib, "arm_v1_mcu_run")
        f.restype = None
        f.argtypes = [VP, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32), C.c_uint32, C.c_uint64, VP]
        f(_ptr(chan), chan.shape[0], pin_chan0, C.byref(r), dmask, F, _ptr(gpio))
        return gpio, r.value

    def note_to_inc(self, note):
        return self._fn("note_to_inc", C.c_uint32, [C.c_int])(note)

    def voice_bank_run(self, voices, N, voices_per_bus, mode, F, want_isum=True, want_vec=True):
        """voices [N][2] u32 {inc, state} in place; returns (isum [n_bus][F] i32, vec [n_bus][F] f32)."""
        n_bus = (N + voices_per_bus - 1) // voices_per_bus
        isum = np.zeros((n_bus, F), np.int32) if want_isum else None
        vec = np.zeros((n_bus, F), np.float32) if want_vec else None
        f = self._fn("voice_bank_run", None, [VP, C.c_uint64, C.c_uint64, C.c_int, C.c_uint64, VP, VP])
        f(_ptr(voices), N, voices_per_bus, mode, F, _ptr(isum), _ptr(vec))
        return isum, vec

    def square_grain_mix_run(self, state, threshold, phase, inc, gl, gr, N, F):
        imix = np.zeros((2, F), np.int32)
        mix = np.zeros((2, F), np.float32)
        f = self._fn("square_grain_mix_run", None, [VP, VP, VP, VP, VP, VP, C.c_uint64, C.c_uint64, VP, VP])
        f(_ptr(state), _ptr(threshold), _ptr(phase), _ptr(inc), _ptr(gl), _ptr(gr), N, F, _ptr(imix), _ptr(mix))
        return imix, mix

    def xvoice_run(self, state, param, N, F, want_raw=True, want_mix=True):
        raw = np.zeros((N, F, 2), np.float32) if want_raw else None
        mix = np.zeros((2, F), np.float32) if want_mix else None
        f = self._fn("xvoice_run", None, [VP, VP, C.c_uint64, C.c_uint64, VP, VP])
        f(_ptr(state), _ptr(param), N, F, _ptr(raw), _ptr(mix))
        return raw, mix

    def word_clock_run(self, state, hperiod, N, F):
        """state int32 [N][2] = {phase, pol} (advanced in place); returns float [N][F]"""
        out = np.zeros((N, F), np.float32)
        f = self._fn("word_clock_run", None, [VP, VP, C.c_uint64, C.c_uint64, VP])
        f(_ptr(state), _ptr(hperiod), N, F, _ptr(out))
        return out

    def onepole_run(self, y, a, N, F, inp):
        out = np.zeros((N, F), np.float32)
        f = self._fn("onepole_run", None, [VP, VP, C.c_uint64, C.c_uint64, VP, VP])
        f(_ptr(y), _ptr(a), N, F, _ptr(inp), _ptr(out))
        return out


class Ref(_Lib):
    """The reference's own code, compiled from /root/reference (oracle/_ref)."""
    prefix = "ref_"

    def __init__(self, path=None):
        if path is None:
            build()
            path = REF_SO
        super().__init__(path)

    def sizeof(self, what):
        return self._fn("sizeof", C.c_uint32, [C.c_int])(what)

    def pdm_sizeof(self, order):
        return self._fn("pdm_sizeof", C.c_uint32, [C.c_uint32])(order)

    def test_cproc_tick(self, inp, g):
        idx = C.c_uint32(0)
        v = self._fn("test_cproc_tick", C.c_uint32, [C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32)])(inp, g, C.byref(idx))
        return idx.value, v

    def synth_sizeof(self, what):
        return self._fn("synth_sizeof", C.c_uint32, [C.c_int])(what)

    def v2_isr_config(self):
        """(channels per MCU, sizeof(struct channel), CONTROL_DIV_LOG) of the compiled mod_pdm_pwm.c"""
        return tuple(self._fn("v2_isr_" + k, C.c_uint32, [])() for k in ("nb_channels", "sizeof_channel", "control_div_log"))

    def v2_isr_run(self, chan, prng, count, setpoints, F):
        """The real TIM3 ISR of mod_pdm_pwm.c (+ mod_controlrate.c) called F times for ONE MCU.
        chan uint32 [nb][7] in/out; returns (duty uint8 [nb][F], prng', count')."""
        nb = chan.shape[0]
        duty = np.zeros((nb, F), np.uint8)
        pr, cn = C.c_uint32(int(prng)), C.c_uint32(int(count))
        f = self._fn("v2_isr_run", None, [VP, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), VP, C.c_uint64, C.c_uint64, VP])
        f(_ptr(chan), C.byref(pr), C.byref(cn), _ptr(setpoints), 0 if setpoints is None else setpoints.shape[0], F, _ptr(duty))
        return duty, pr.value, cn.value

    def word_clock_run(self, state, hperiod, N, F, ev_clock=0, ev_cap=4096):
        """linux/clock.c:108-120 itself.  Returns (out float [N][F], sample times of the MIDI clock bytes of clock ev_clock)."""
        out = np.zeros((N, F), np.float32)
        ev = np.zeros(ev_cap, np.uint32)
        f = self._fn("word_clock_run", C.c_uint32, [VP, VP, C.c_uint64, C.c_uint64, VP, C.c_uint64, VP, C.c_uint32])
        n_ev = f(_ptr(state), _ptr(hperiod), N, F, _ptr(out), ev_clock, _ptr(ev), ev_cap)
        return out, ev[:min(n_ev, ev_cap)].copy()

    def note_table(self):
        t = np.zeros(128, np.uint32)
        self._fn("note_table", None, [VP])(_ptr(t))
        return t

    def note_tab12(self):
        t = np.zeros(12, np.uint32)
        self._fn("note_tab12", None, [VP])(_ptr(t))
        return t

    def voice_bank_run(self, voices, n_synth, mode, F):
        vec = np.zeros((n_synth, F), np.float32)
        self._fn("voice_bank_run", None, [VP, C.c_uint64, C.c_int, C.c_uint64, VP])(_ptr(voices), n_synth, mode, F, _ptr(vec))
        return vec

    def synth_play(self, notes, F):
        notes = np.asarray(notes, np.int32)
        vec = np.zeros(F, np.float32)
        voices = np.zeros((64, 2), np.uint32)
        self._fn("synth_play", None, [VP, C.c_int, C.c_uint64, VP, VP])(_ptr(notes), len(notes), F, _ptr(vec), _ptr(voices))
        return vec, voices

    def ext_sizeof(self, what):
        """sizeof of the DEF_PROC_STRUCTS-generated structs of include/cproc_ext.h: 3 * kind + {0 state, 1 param, 2 input}."""
        return self._fn("ext_sizeof", C.c_uint32, [C.c_int])(what)

    def ext_text_run(self, which, inp, changed, F, n_out):
        """tests/golden/ext_voice.cproc (0) / ext_chain.cproc (1) compiled as C against the reference's cproc.h: F ticks of
        the ONE instance of this loaded library copy.  inp uint32 [n_in][F]; returns uint32 [n_out][F]."""
        out = np.zeros((n_out, F), np.uint32)
        self._fn("ext_text_run", None, [C.c_int, VP, VP, C.c_uint64, VP])(which, _ptr(inp), _ptr(changed), F, _ptr(out))
        return out

    def pixi_lfo_run(self, dac, adc0, ticks):
        """stm32f103/pixi.c:279,282-285 itself: `ticks` timer interrupts of the demo LFO bank.  dac uint16 [12] in/out;
        returns the DAC values after each tick, uint16 [ticks][12]."""
        trace = np.zeros((ticks, 12), np.uint16)
        self._fn("pixi_lfo_run", None, [VP, C.c_uint16, C.c_uint64, VP])(_ptr(dac), adc0, ticks, _ptr(trace))
        return trace

    def grain_sizeof(self):
        return self._fn("grain_sizeof", C.c_uint32, [])()


def have_ref():
    return os.path.exists(REF_SO) or os.path.isdir(os.environ.get("REF", "/root/reference"))


# ---- shared synthetic-input generators (SURVEY.md section 8d) -------------
def xorshift32_np(x):
    x = x.astype(np.uint32).copy()
    x ^= (x << np.uint32(13))
    x ^= (x >> np.uint32(17))
    x ^= (x << np.uint32(5))
    return x


def pdm_setpoints(n_ch, n_rows, seed_base=1):
    """setpoint ~ U[0x40000000, 0xC0000000] (mod_pdm.c:99-100) from
    xorshift32(seed = ch + seed_base), one row per control period."""
    s = (np.arange(n_ch, dtype=np.uint64) + seed_base).astype(np.uint32)
    s[s == 0] = 0x9E3779B9
    rows = np.zeros((n_rows, n_ch), np.uint32)
    for r in range(n_rows):
        s = xorshift32_np(s)
        rows[r] = np.uint32(0x40000000) + (s >> np.uint32(1))
    return rows
