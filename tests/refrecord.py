"""The reference's side of the oracle-vs-reference tests, recorded (tests/golden/ref_calls.json).

The tests that take the `ref` fixture compare the oracle with the reference's own code, compiled from the upstream
sources into oracle/_ref/libref.so (oracle/build_ref.sh).  Those sources are not part of this repository, so every call
such a test makes on `ref` is recorded: per test, in call order, a digest of the inputs and, for every output (the
return values and every array argument after the call, which is how state written in place comes back), its SHA-256,
shape, dtype and a sample of its values.

* libref.so present: the tests run against it, and each call is also checked against the record.
* libref.so absent: the calls are answered by `StandIn`, the same entry points on the oracle, and each answer must
  match the record -- so the oracle is still compared, bit for bit, with what the reference computed.
* tests/golden/gen_golden_ref.py writes the record (CPROC_REF_RECORD=<path> makes the fixture record there).

The module-level generator of test_oracle_vs_ref.py is consumed in test order; its state at the start of each test is
recorded too and restored before the test, so the inputs do not depend on which tests a run selects.
"""
import hashlib
import json
import os
import shutil
import tempfile

import numpy as np

from oracle import pyoracle as po

HERE = os.path.dirname(os.path.abspath(__file__))
RECORD = os.path.join(HERE, "golden", "ref_calls.json")
SAMPLE = 16                    # values kept per output, evenly spaced over the flattened array


def _digest_inputs(name, args, kw):
    h = hashlib.sha256(name.encode())
    for a in list(args) + [kw[k] for k in sorted(kw)]:
        if isinstance(a, np.ndarray):
            h.update(("%s%s" % (a.dtype.str, a.shape)).encode())
            h.update(np.ascontiguousarray(a).tobytes())
        else:
            h.update(repr(a if not isinstance(a, (np.integer, np.floating)) else a.item()).encode())
    return h.hexdigest()


def _outputs(ret, args, kw):
    """Return values (tuples flattened) and the array arguments after the call."""
    outs = list(ret) if isinstance(ret, tuple) else [ret]
    outs += [a for a in list(args) + [kw[k] for k in sorted(kw)] if isinstance(a, np.ndarray)]
    return outs


def _describe(x):
    a = np.ascontiguousarray(np.asarray(x))
    bits = a.view(np.uint32) if a.dtype.itemsize == 4 and a.dtype.kind == "f" else a
    flat = bits.reshape(-1)
    idx = np.linspace(0, flat.size - 1, min(SAMPLE, flat.size)).astype(np.int64) if flat.size else np.zeros(0, np.int64)
    return {"sha256": hashlib.sha256(a.tobytes()).hexdigest(), "shape": list(a.shape), "dtype": a.dtype.str,
            "sample": [int(v) for v in flat[idx]]}


class Recorded:
    """Wraps a reference (libref.so or StandIn): every call is recorded into, or checked against, `calls`."""

    def __init__(self, source, calls, mode):
        self._source, self._calls, self._mode = source, calls, mode
        self._pos = [0]                                  # shared with private copies: one call sequence per test

    def private_copy(self):
        """A fresh copy of the library (the reference keeps some state in function statics)."""
        r = Recorded(self._source.private_copy(), self._calls, self._mode)
        r._pos = self._pos
        return r

    def __getattr__(self, name):
        fn = getattr(self._source, name)
        if not callable(fn):
            return fn

        def call(*args, **kw):
            key = _digest_inputs(name, args, kw)
            ret = fn(*args, **kw)
            got = [_describe(o) for o in _outputs(ret, args, kw)]
            i = self._pos[0]
            self._pos[0] += 1
            if self._mode == "record":
                self._calls.append({"fn": name, "inputs": key, "outputs": got})
                return ret
            assert i < len(self._calls), "call %d (%s) is not in %s: regenerate it with tests/golden/gen_golden_ref.py" % (i, name, RECORD)
            want = self._calls[i]
            assert (want["fn"], want["inputs"]) == (name, key), \
                "call %d: %s on other inputs than the recorded %s: regenerate %s" % (i, name, want["fn"], RECORD)
            for k, (g, w) in enumerate(zip(got, want["outputs"])):
                assert g["sha256"] == w["sha256"], "call %d (%s), output %d differs from the reference's: %s vs %s" % (
                    i, name, k, {x: g[x] for x in ("shape", "dtype", "sample")}, {x: w[x] for x in ("shape", "dtype", "sample")})
            assert len(got) == len(want["outputs"])
            return ret
        return call


class Ref(po.Ref):
    """libref.so, with private copies."""

    def private_copy(self):
        d = tempfile.mkdtemp()
        p = os.path.join(d, "libref_private.so")
        shutil.copy(self.path, p)
        return Ref(p)


class StandIn:
    """The entry points of libref.so that the tests call, on the oracle (and on the project's own state layouts for the
    struct sizes).  Stateful entry points keep their state per copy, like the function statics of the reference."""

    def __init__(self, oracle):
        self.o = oracle
        self._tick_state = np.zeros((1, 3), np.uint32)
        self._text_state = {}

    def private_copy(self):
        return StandIn(self.o)

    # struct sizes, from the word counts of the project's state / param / input records
    def sizeof(self, what):
        acc, edge = po.NODE_ACC, po.NODE_EDGE
        return [po.node_words(acc) * 4, 4, 0, po.node_param_words(acc) * 4, po.node_words(edge) * 4, 4, 4][what]

    def pdm_sizeof(self, order):
        return (po.node_words(po.node_pdm(order, 24)) - 1) * 4            # the pdm node's words: order accumulators + out

    def synth_sizeof(self, what):
        return [2 * 4, 1024][what]                                        # voice {inc, state}; struct synth as the reference has it

    def ext_sizeof(self, what):
        if what == 24:
            return 4                                                      # glide_f_config {w div_log}
        kind, part = po.NODE_PHASOR_F + what // 3, what % 3
        return [po.node_words(kind) * 4, po.node_param_words(kind) * 4, 8 if kind == po.NODE_MUL else 4][part]

    def v2_isr_config(self):
        return (3, 28, 12)                                                # PDM_FOR_CHANNELS c(0) c(1) c(2); 7 words; CONTROL_DIV_LOG

    # processors
    def graph_run(self, *a, **kw):
        return self.o.graph_run(*a, **kw)

    def graph_run_ext(self, *a, **kw):
        return self.o.graph_run_ext(*a, **kw)

    def pdm_run(self, *a, **kw):
        return self.o.pdm_run(*a, **kw)

    def pdm_v2_run(self, *a, **kw):
        return self.o.pdm_v2_run(*a, **kw)

    def pwm_run(self, *a, **kw):
        return self.o.pwm_run(*a, **kw)

    def square_grain_run(self, *a, **kw):
        return self.o.square_grain_run(*a, **kw)

    def test_cproc_tick(self, inp, g):
        out = self.o.graph_run(po.GRAPH_TEST_CPROC, 1, 1, self._tick_state, 1, 1, np.array([[[inp]]], np.uint32),
                               np.array([[g]], np.uint32))
        return 2, int(out[0, 0])

    def v2_isr_run(self, chan, prng, count, setpoints, F):
        p = np.array([prng], np.uint32)
        duty, cnt = self.o.pdm_v2_run(chan, 2, chan.shape[0], 3, p, None, 0x3FF, count, 12, 24, setpoints, F)
        return duty, int(p[0]), cnt

    def word_clock_run(self, state, hperiod, N, F, ev_clock=0, ev_cap=4096):
        prev = int(state[ev_clock, 1])
        out = self.o.word_clock_run(state, hperiod, N, F)
        pol = np.concatenate([[prev], out[ev_clock].astype(np.int64)])
        ev = np.flatnonzero((pol[1:] == 1) & (pol[:-1] != 1)).astype(np.uint32)      # a MIDI clock byte where the polarity turns 1
        return out, ev[:ev_cap]

    def note_table(self):
        return np.array([self.o.note_to_inc(n) for n in range(128)], np.uint32)

    def note_tab12(self):
        # synth.c's 12-entry table as the reference has it (SURVEY a-9); the oracle has no counterpart to compute it from
        return np.array([594573364, 629928536, 667386036, 707070875, 749115497, 793660223,
                         840853716, 890853479, 943826384, 999949221, 1059409296, 1122405051], np.uint32)

    def voice_bank_run(self, voices, n_synth, mode, F):
        return self.o.voice_bank_run(voices, n_synth * 64, 64, mode, F)[1]

    def synth_play(self, notes, F):
        v = np.zeros((64, 2), np.uint32)
        v[:len(notes), 0] = [self.o.note_to_inc(int(n)) for n in notes]
        vec = self.o.voice_bank_run(v, 64, 64, po.MIX_SAW, F)[1]
        return vec[0].copy(), v

    def pixi_lfo_run(self, dac, adc0, ticks):
        st = dac.astype(np.uint32).reshape(-1, 1).copy()
        inp = np.full((len(dac), 1, ticks), int(adc0) >> 5, np.uint32)
        out = self.o.graph_run([(po.NODE_ACC, -1, 0xFFFFFFFF)], 1, 0, st, len(dac), ticks, inp)
        dac[:] = st[:, 0] & 0xFFF
        return (out & 0xFFF).T.astype(np.uint16)

    def ext_text_run(self, which, inp, changed, F, n_out):
        from synth_tools_b200 import abi
        name = ["voice", "chain", "gain"][which]
        g = abi.graph_parse_ex(open(os.path.join(HERE, "golden", "ext_%s.cproc" % name)).read())
        st = self._text_state.setdefault(which, np.zeros((1, sum(po.node_words(r[0]) for r in g["rows"])), np.uint32))
        n_in = g["n_inputs"]
        out = self.o.graph_run_ext(g["rows"], n_in, g["out_nodes"], st, g["param_init"].reshape(1, -1).copy(), 1, F,
                                   np.ascontiguousarray(inp).reshape(1, n_in, F), None if changed is None else changed.reshape(1, F))
        return out[0]


def load():
    if os.path.exists(RECORD):
        with open(RECORD) as f:
            return json.load(f)
    return {}


def save(path, record):
    with open(path, "w") as f:
        json.dump(record, f, indent=0, sort_keys=True)
        f.write("\n")
