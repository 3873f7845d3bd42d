"""ctypes binding of include/cproc_cuda.h (libcproc_cuda.so).

This is plumbing for tests, bench.py and Python hosts; the product is the
shared library.  There is no CPU fallback anywhere: if the library is missing
the import fails, and without a CUDA device `Context()` raises.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libcproc_cuda.so")

# enum cproc_cuda_proc
GRAPH, PDM, PDM_V1, PDM_V2, PWM, VOICE_BANK, SQUARE_GRAIN, SQUARE_GRAIN_MIX, XVOICE, ONEPOLE, WORD_CLOCK = range(1, 12)
NODE_ACC, NODE_EDGE, NODE_GLIDE, NODE_PDM = 0, 1, 2, 3
# extension processors (include/cproc_ext.h)
NODE_PHASOR_F, NODE_SVF, NODE_ENV, NODE_ONEPOLE, NODE_GAIN, NODE_ASFLOAT, NODE_GLIDE_F, NODE_MUL = 4, 5, 6, 7, 8, 9, 10, 11
SRC_ZERO = -0x80000000          # CPROC_CUDA_SRC_ZERO: an input the PROC statement does not name


def node_glide(div_log):
    """CPROC_CUDA_NODE_GLIDE_L(L)"""
    return NODE_GLIDE | (div_log << 8)


def node_glide_f(div_log):
    """CPROC_CUDA_NODE_GLIDE_F_L(L)"""
    return NODE_GLIDE_F | (div_log << 8)


def node_pdm(order, out_shift):
    """CPROC_CUDA_NODE_PDM_K(K, SH)"""
    return NODE_PDM | ((order | (out_shift << 3)) << 8)


def _node(r):
    return Node(r[0], r[1], r[2], r[3] if len(r) > 3 else 0)


def _row(n):
    """Node -> (type, src, cond_mask) for one-input kinds, (type, src, cond_mask, src2) for pdm."""
    return (n.type, n.src, n.cond_mask, n.src2) if n.type & 0xFF in (NODE_PDM, NODE_MUL) else (n.type, n.src, n.cond_mask)

MIX_SAW, MIX_SQUARE = 0, 1
XVOICE_SEQ, XVOICE_SCAN = 0, 1
PLANAR, INTERLEAVED, TILED = 0, 1, 2
OK, EINVAL, ENODEV, ENOMEM, ECUDA, ESTATE = 0, -1, -2, -3, -4, -5


class Node(C.Structure):
    _fields_ = [("type", C.c_uint32), ("src", C.c_int32), ("cond_mask", C.c_uint32), ("src2", C.c_int32)]


class Config(C.Structure):
    _fields_ = [("proc", C.c_uint32), ("layout", C.c_uint32), ("order", C.c_uint32), ("out_shift", C.c_uint32),
                ("bank_size", C.c_uint32), ("dither_mask", C.c_uint32), ("ctl_div_log", C.c_uint32),
                ("mode", C.c_uint32), ("voices_per_bus", C.c_uint64), ("nodes", C.POINTER(Node)),
                ("n_nodes", C.c_uint32), ("n_inputs", C.c_uint32), ("out_node", C.c_uint32), ("n_outputs", C.c_uint32),
                ("out_nodes", C.POINTER(C.c_uint32))]


class GraphInfo(C.Structure):
    _fields_ = [("n_nodes", C.c_uint32), ("n_inputs", C.c_uint32), ("out_node", C.c_uint32), ("out_index", C.c_uint32),
                ("n_outputs", C.c_uint32), ("out_nodes", C.c_uint32 * 16), ("out_indices", C.c_uint32 * 16),
                ("out_is_float", C.c_uint32), ("n_param_words", C.c_uint32), ("param_init", C.c_uint32 * 192)]


GRAPH_MAX_NODES = 64


class IO(C.Structure):
    _fields_ = [("in_", C.c_void_p), ("in2", C.c_void_p), ("ctl", C.c_void_p), ("out", C.c_void_p),
                ("mix", C.c_void_p), ("layout", C.c_uint32), ("n_ctl", C.c_uint32)]


CHUNK_FN = C.CFUNCTYPE(None, C.c_void_p, C.c_uint64, C.c_void_p, C.c_size_t)

# name -> (restype, argtypes): every symbol include/cproc_cuda.h declares
SYMBOLS = {
    "cproc_cuda_open": (C.c_int, [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]),
    "cproc_cuda_close": (C.c_int, [C.c_void_p]),
    "cproc_cuda_sync": (C.c_int, [C.c_void_p]),
    "cproc_cuda_last_error": (C.c_char_p, [C.c_void_p]),
    "cproc_cuda_abi_version": (C.c_int, []),
    "cproc_cuda_device_count": (C.c_int, []),
    "cproc_cuda_launch_count": (C.c_uint64, [C.c_void_p]),
    "cproc_cuda_alloc": (C.c_int, [C.c_void_p, C.POINTER(Config), C.c_uint64, C.POINTER(C.c_void_p)]),
    "cproc_cuda_free": (C.c_int, [C.c_void_p]),
    "cproc_cuda_state_bytes": (C.c_size_t, [C.c_void_p]),
    "cproc_cuda_param_bytes": (C.c_size_t, [C.c_void_p]),
    "cproc_cuda_upload_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "cproc_cuda_download_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "cproc_cuda_upload_param": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "cproc_cuda_upload_bank": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32]),
    "cproc_cuda_download_bank": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_uint32)]),
    "cproc_cuda_run": (C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(IO)]),
    "cproc_cuda_run_dev": (C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(IO)]),
    "cproc_cuda_run_period": (C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(IO), C.c_void_p, C.c_size_t]),
    "cproc_cuda_run_stream": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.POINTER(IO), C.c_uint32, CHUNK_FN, C.c_void_p]),
    "cproc_cuda_mix_to_float": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]),
    "cproc_cuda_dev_alloc": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "cproc_cuda_dev_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "cproc_cuda_host_alloc": (C.c_int, [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]),
    "cproc_cuda_host_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "cproc_cuda_memcpy_h2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "cproc_cuda_memcpy_d2h": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "cproc_cuda_memset": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_size_t]),
    "cproc_cuda_timer_start": (C.c_int, [C.c_void_p]),
    "cproc_cuda_timer_stop": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "cproc_cuda_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    "cproc_cuda_patch_class_count": (C.c_int, []),
    "cproc_cuda_patch_class_name": (C.c_char_p, [C.c_uint32]),
    "cproc_cuda_patch_class_field": (C.c_int, [C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(C.c_char_p)]),
    "cproc_cuda_patch_open": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p)]),
    "cproc_cuda_patch_close": (C.c_int, [C.c_void_p]),
    "cproc_cuda_patch_reset": (C.c_int, [C.c_void_p]),
    "cproc_cuda_patch_node_count": (C.c_int, [C.c_void_p]),
    "cproc_cuda_patch_apply": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32), C.c_uint32, C.c_uint32]),
    "cproc_cuda_patch_output": (C.c_int, [C.c_void_p, C.c_uint32]),
    "cproc_cuda_patch_tick": (C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(IO), C.c_int]),
    "cproc_cuda_patch_get": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, C.POINTER(C.c_uint32)]),
    "cproc_cuda_patch_set": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint32]),
    "cproc_cuda_patch_batch": (C.c_void_p, [C.c_void_p]),
    "cproc_cuda_bus_create": (C.c_int, [C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "cproc_cuda_bus_handle_bytes": (C.c_size_t, []),
    "cproc_cuda_bus_handle": (C.c_int, [C.c_void_p, C.c_void_p]),
    "cproc_cuda_bus_connect": (C.c_int, [C.c_void_p, C.c_void_p]),
    "cproc_cuda_bus_allreduce": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32]),
    "cproc_cuda_bus_allreduce_begin": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32]),
    "cproc_cuda_bus_wait": (C.c_int, [C.c_void_p, C.c_uint32]),
    "cproc_cuda_bus_attach": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32]),
    "cproc_cuda_bus_flush": (C.c_int, [C.c_void_p]),
    "cproc_cuda_bus_status": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint32)]),
    "cproc_cuda_bus_destroy": (C.c_int, [C.c_void_p]),
    "cproc_cuda_graph_parse": (C.c_int, [C.c_char_p, C.POINTER(Node), C.c_uint32, C.POINTER(GraphInfo)]),
    "cproc_cuda_graph_jit_log": (C.c_char_p, [C.c_void_p]),
    "cproc_cuda_graph_set_input": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32]),
    "cproc_cuda_graph_tick": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p]),
    "cproc_cuda_graph_event": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p]),
    "cproc_cuda_graph_jit_source": (C.c_int, [C.POINTER(Node), C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32), C.c_uint32, C.c_int, C.c_char_p, C.c_size_t]),
}


class CprocCudaError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("cproc_cuda error %d: %s" % (code, msg))
        self.code = code


def load(path=LIB_PATH):
    if not os.path.exists(path):
        raise ImportError("%s is missing: build it with `python synth_tools_b200/build.py` "
                          "(there is no CPU fallback)" % path)
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        f = getattr(lib, name)          # AttributeError if the ABI symbol is missing
        f.restype = res
        f.argtypes = args
    return lib


lib = load()


def graph_parse(text):
    """Generated cproc graph text (epid_cproc.erl output, linux/test_cproc.c:11-17) ->
    ([(type, src, cond_mask)], n_inputs, out_node, out_index).  Needs no device."""
    nodes = (Node * GRAPH_MAX_NODES)()
    info = GraphInfo()
    rc = lib.cproc_cuda_graph_parse(text.encode(), nodes, GRAPH_MAX_NODES, C.byref(info))
    if rc:
        raise CprocCudaError(rc, (lib.cproc_cuda_last_error(None) or b"").decode())
    rows = [_row(nodes[k]) for k in range(info.n_nodes)]
    return rows, info.n_inputs, info.out_node, info.out_index


def graph_parse_outputs(text):
    """Like graph_parse, for graphs with several cproc_output statements:
    (rows, n_inputs, [out_node...], [out_index...])."""
    nodes = (Node * GRAPH_MAX_NODES)()
    info = GraphInfo()
    rc = lib.cproc_cuda_graph_parse(text.encode(), nodes, GRAPH_MAX_NODES, C.byref(info))
    if rc:
        raise CprocCudaError(rc, (lib.cproc_cuda_last_error(None) or b"").decode())
    rows = [_row(nodes[k]) for k in range(info.n_nodes)]
    return rows, info.n_inputs, list(info.out_nodes[:info.n_outputs]), list(info.out_indices[:info.n_outputs])


def graph_parse_ex(text):
    """Everything cproc_cuda_graph_parse reports: {rows, n_inputs, out_nodes, out_indices, out_is_float: [bool],
    param_init: uint32 [n_param_words] (the param record's initial value from the text's compound literals)}."""
    nodes = (Node * GRAPH_MAX_NODES)()
    info = GraphInfo()
    rc = lib.cproc_cuda_graph_parse(text.encode(), nodes, GRAPH_MAX_NODES, C.byref(info))
    if rc:
        raise CprocCudaError(rc, (lib.cproc_cuda_last_error(None) or b"").decode())
    return {"rows": [_row(nodes[k]) for k in range(info.n_nodes)], "n_inputs": info.n_inputs,
            "out_nodes": list(info.out_nodes[:info.n_outputs]), "out_indices": list(info.out_indices[:info.n_outputs]),
            "out_is_float": [bool((info.out_is_float >> q) & 1) for q in range(info.n_outputs)],
            "param_init": np.array(info.param_init[:info.n_param_words], np.uint32)}


def graph_jit_source(rows, n_inputs, out_node, has_changed=False):
    """The CUDA source the library generates (and NVRTC-compiles) for a node table."""
    arr = (Node * len(rows))(*[_node(r) for r in rows])
    outs = [out_node] if isinstance(out_node, int) else list(out_node)
    oarr = (C.c_uint32 * len(outs))(*outs)
    n = lib.cproc_cuda_graph_jit_source(arr, len(rows), n_inputs, oarr, len(outs), int(has_changed), None, 0)
    if n < 0:
        raise CprocCudaError(n, (lib.cproc_cuda_last_error(None) or b"").decode())
    buf = C.create_string_buffer(n + 1)
    lib.cproc_cuda_graph_jit_source(arr, len(rows), n_inputs, oarr, len(outs), int(has_changed), buf, n + 1)
    return buf.value.decode()


def patch_classes():
    """The class map of the patcher: [{name, state: [...], input: [...], param: [...], config: [...]}]."""
    out = []
    for c in range(lib.cproc_cuda_patch_class_count()):
        d = {"name": lib.cproc_cuda_patch_class_name(c).decode()}
        for kind, key in ((0, "param"), (1, "state"), (2, "input"), (3, "config")):
            n = lib.cproc_cuda_patch_class_field(c, kind, 0, None)
            names = []
            for k in range(n):
                s = C.c_char_p()
                lib.cproc_cuda_patch_class_field(c, kind, k, C.byref(s))
                names.append(s.value.decode())
            d[key] = names
        out.append(d)
    return out


def _vp(a):
    """numpy array / int device pointer / None -> c_void_p value."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        assert a.flags["C_CONTIGUOUS"]
        return a.ctypes.data
    return int(a)


class Context:
    """cproc_cuda_ctx: one device + stream."""

    def __init__(self, device=0, stream=None):
        h = C.c_void_p()
        rc = lib.cproc_cuda_open(device, stream, C.byref(h))
        if rc:
            raise CprocCudaError(rc, (lib.cproc_cuda_last_error(None) or b"").decode())
        self.h = h
        self.device = device

    def _ck(self, rc):
        if rc:
            raise CprocCudaError(rc, (lib.cproc_cuda_last_error(self.h) or b"").decode())

    def close(self):
        if self.h:
            lib.cproc_cuda_close(self.h)
            self.h = None

    def sync(self):
        self._ck(lib.cproc_cuda_sync(self.h))

    def set_option(self, name, value):
        self._ck(lib.cproc_cuda_set_option(self.h, name.encode(), int(value)))

    @property
    def launches(self):
        return lib.cproc_cuda_launch_count(self.h)

    def dev_alloc(self, nbytes):
        p = C.c_void_p()
        self._ck(lib.cproc_cuda_dev_alloc(self.h, nbytes, C.byref(p)))
        return p.value

    def dev_free(self, p):
        self._ck(lib.cproc_cuda_dev_free(self.h, p))

    def host_alloc(self, nbytes, dtype=np.uint8):
        """Pinned host buffer as a numpy array (keeps the raw pointer in .base_ptr)."""
        p = C.c_void_p()
        self._ck(lib.cproc_cuda_host_alloc(self.h, nbytes, C.byref(p)))
        buf = (C.c_uint8 * nbytes).from_address(p.value)
        a = np.frombuffer(buf, dtype=np.uint8).view(dtype)
        return a, p.value

    def host_free(self, p):
        self._ck(lib.cproc_cuda_host_free(self.h, p))

    def h2d(self, dev, arr):
        self._ck(lib.cproc_cuda_memcpy_h2d(self.h, dev, _vp(arr), arr.nbytes))

    def d2h(self, arr, dev):
        self._ck(lib.cproc_cuda_memcpy_d2h(self.h, _vp(arr), dev, arr.nbytes))

    def memset(self, dev, value, nbytes):
        self._ck(lib.cproc_cuda_memset(self.h, dev, value, nbytes))

    def timer_start(self):
        self._ck(lib.cproc_cuda_timer_start(self.h))

    def timer_stop(self):
        ms = C.c_float()
        self._ck(lib.cproc_cuda_timer_stop(self.h, C.byref(ms)))
        return ms.value

    def batch(self, proc, n, **kw):
        return Batch(self, proc, n, **kw)


class Batch:
    """cproc_cuda_batch: N instances of one reference processor."""

    def __init__(self, ctx, proc, n, layout=PLANAR, order=2, out_shift=24, bank_size=1, dither_mask=0x3FF,
                 ctl_div_log=12, mode=MIX_SAW, voices_per_bus=0, nodes=None, n_inputs=1, out_node=None):
        self.ctx = ctx
        cfg = Config()
        cfg.proc, cfg.layout, cfg.order, cfg.out_shift = proc, layout, order, out_shift
        cfg.bank_size, cfg.dither_mask, cfg.ctl_div_log = bank_size, dither_mask, ctl_div_log
        cfg.mode, cfg.voices_per_bus = mode, voices_per_bus
        self._nodes = None
        if nodes is not None:
            arr = (Node * len(nodes))(*[_node(r) for r in nodes])
            self._nodes = arr
            cfg.nodes = arr
            cfg.n_nodes = len(nodes)
            cfg.n_inputs = n_inputs
            if isinstance(out_node, (list, tuple)):               # several cproc_output statements
                self._outs = (C.c_uint32 * len(out_node))(*out_node)
                cfg.out_nodes = self._outs
                cfg.n_outputs = len(out_node)
                cfg.out_node = out_node[0]
            else:
                cfg.out_node = len(nodes) - 1 if out_node is None else out_node
        h = C.c_void_p()
        ctx._ck(lib.cproc_cuda_alloc(ctx.h, C.byref(cfg), n, C.byref(h)))
        self.h = h
        self.n = n
        self.proc = proc
        self.layout = layout
        self.state_bytes = lib.cproc_cuda_state_bytes(h)
        self.param_bytes = lib.cproc_cuda_param_bytes(h)
        self.bank_size = min(bank_size, n)
        self.n_banks = (n + self.bank_size - 1) // self.bank_size

    def free(self):
        if self.h:
            lib.cproc_cuda_free(self.h)
            self.h = None

    def upload_state(self, aos, stride=0):
        self.ctx._ck(lib.cproc_cuda_upload_state(self.h, _vp(aos), stride))

    def download_state(self, aos=None, stride=0):
        if aos is None:
            aos = np.zeros((self.n, self.state_bytes // 4), np.uint32)
        self.ctx._ck(lib.cproc_cuda_download_state(self.h, _vp(aos), stride))
        return aos

    def upload_param(self, aos, stride=0):
        self.ctx._ck(lib.cproc_cuda_upload_param(self.h, _vp(aos), stride))

    def upload_bank(self, prng=None, count=0):
        self.ctx._ck(lib.cproc_cuda_upload_bank(self.h, _vp(prng), count))

    def download_bank(self):
        prng = np.zeros(self.n_banks, np.uint32)
        cnt = C.c_uint32()
        self.ctx._ck(lib.cproc_cuda_download_bank(self.h, _vp(prng), C.byref(cnt)))
        return prng, cnt.value

    def _io(self, inp, in2, ctl, out, mix, layout, n_ctl):
        io = IO()
        io.in_, io.in2, io.ctl, io.out, io.mix = _vp(inp), _vp(in2), _vp(ctl), _vp(out), _vp(mix)
        io.layout = self.layout if layout is None else layout
        if n_ctl is None:
            n_ctl = ctl.shape[0] if isinstance(ctl, np.ndarray) else 0
        io.n_ctl = n_ctl
        return io

    # evented graph driver (handle_tag_u32 of stm32f103/mod_cproc_plugin.c:24-38)
    def set_input(self, i, v, instance=None):
        """cproc_input[i] = v for one instance (None: every instance)."""
        self.ctx._ck(lib.cproc_cuda_graph_set_input(self.h, 0xFFFFFFFFFFFFFFFF if instance is None else instance, i, v))

    def tick(self, changed=0xFFFFFFFF, n_outputs=1):
        """cproc_update(cproc_input, changed) once per instance -> uint32 [inst][n_outputs]."""
        out = np.zeros((self.n, n_outputs), np.uint32)
        self.ctx._ck(lib.cproc_cuda_graph_tick(self.h, changed, _vp(out)))
        return out

    def event(self, instance, i, v, n_outputs=1):
        """One TAG_U32 message [i, v] to one graph instance -> its cproc_output values."""
        out = np.zeros(n_outputs, np.uint32)
        self.ctx._ck(lib.cproc_cuda_graph_event(self.h, instance, i, v, _vp(out)))
        return out

    def run(self, F, inp=None, in2=None, ctl=None, out=None, mix=None, layout=None, n_ctl=None):
        """Host buffers (numpy), synchronous."""
        io = self._io(inp, in2, ctl, out, mix, layout, n_ctl)
        self.ctx._ck(lib.cproc_cuda_run(self.h, F, C.byref(io)))

    def run_period(self, F, state, stride=0, inp=None, in2=None, ctl=None, out=None, mix=None, layout=None, n_ctl=None):
        """One real-time period with the state in the host's records: records in, render, records out, one synchronisation
        (`state` is updated in place)."""
        io = self._io(inp, in2, ctl, out, mix, layout, n_ctl)
        self.ctx._ck(lib.cproc_cuda_run_period(self.h, F, C.byref(io), _vp(state), stride))

    def run_dev(self, F, inp=None, in2=None, ctl=None, out=None, mix=None, layout=None, n_ctl=0):
        """Device pointers (ints), asynchronous on the context stream."""
        io = self._io(inp, in2, ctl, out, mix, layout, n_ctl)
        self.ctx._ck(lib.cproc_cuda_run_dev(self.h, F, C.byref(io)))

    def run_stream(self, F_total, F_chunk, out, ctl=None, layout=None, n_ctl=None, ring_chunks=0, on_chunk=None):
        io = self._io(None, None, ctl, out, None, layout, n_ctl)
        cb = CHUNK_FN(on_chunk) if on_chunk is not None else C.cast(None, CHUNK_FN)
        self.ctx._ck(lib.cproc_cuda_run_stream(self.h, F_total, F_chunk, C.byref(io), ring_chunks, cb, None))

    @property
    def jit_log(self):
        return (lib.cproc_cuda_graph_jit_log(self.h) or b"").decode()

    def mix_to_float(self, imix_dev, out_dev, count):
        self.ctx._ck(lib.cproc_cuda_mix_to_float(self.h, imix_dev, out_dev, count))


class Patch:
    """cproc_cuda_patch: the dynamic patcher (mod_bpmodular.c RPC tree) on device state."""
    PARAM, STATE = 0, 1

    def __init__(self, ctx, n, n_inputs=1, layout=PLANAR):
        self.ctx = ctx
        h = C.c_void_p()
        ctx._ck(lib.cproc_cuda_patch_open(ctx.h, n, n_inputs, layout, C.byref(h)))
        self.h = h
        self.n = n
        self.layout = layout
        self.classes = {d["name"]: i for i, d in enumerate(patch_classes())}

    def close(self):
        if self.h:
            lib.cproc_cuda_patch_close(self.h)
            self.h = None

    def apply(self, cls, *in_nodes, config=0):
        c = self.classes[cls] if isinstance(cls, str) else cls
        arr = (C.c_uint32 * max(1, len(in_nodes)))(*in_nodes)
        rc = lib.cproc_cuda_patch_apply(self.h, c, arr, len(in_nodes), config)
        if rc < 0:
            self.ctx._ck(rc)
        return rc

    def output(self, node):
        self.ctx._ck(lib.cproc_cuda_patch_output(self.h, node))

    def reset(self):
        self.ctx._ck(lib.cproc_cuda_patch_reset(self.h))

    def tick(self, F, inp, out, device=False):
        io = IO()
        io.in_, io.out, io.layout = _vp(inp), _vp(out), self.layout
        self.ctx._ck(lib.cproc_cuda_patch_tick(self.h, F, C.byref(io), int(device)))

    def get(self, node, field, instance=0, kind=1):
        v = C.c_uint32()
        self.ctx._ck(lib.cproc_cuda_patch_get(self.h, node, kind, field, instance, C.byref(v)))
        return v.value

    def set(self, node, field, value, instance=0, kind=1):
        self.ctx._ck(lib.cproc_cuda_patch_set(self.h, node, kind, field, instance, value))

    @property
    def node_count(self):
        return lib.cproc_cuda_patch_node_count(self.h)


class Bus:
    """cproc_cuda_bus: the shared mix bus of the ranks of one box over NVLink peer memory."""
    SUM, OR, FSUM = 0, 1, 2
    SCALE_NONE, SCALE_SAW, SCALE_SQUARE, SCALE_GRAIN = 0, 1, 2, 3

    def __init__(self, ctx, max_words, world, rank):
        self.ctx = ctx
        h = C.c_void_p()
        ctx._ck(lib.cproc_cuda_bus_create(ctx.h, max_words, world, rank, C.byref(h)))
        self.h = h
        self.world, self.rank = world, rank

    def handle(self):
        buf = np.zeros(lib.cproc_cuda_bus_handle_bytes(), np.uint8)
        self.ctx._ck(lib.cproc_cuda_bus_handle(self.h, _vp(buf)))
        return buf

    def connect(self, handles):
        handles = np.ascontiguousarray(handles, np.uint8)
        assert handles.size == self.world * lib.cproc_cuda_bus_handle_bytes()
        self.ctx._ck(lib.cproc_cuda_bus_connect(self.h, _vp(handles)))

    def allreduce(self, imix_dev, count, out_dev=None, op=0, scale=0):
        self.ctx._ck(lib.cproc_cuda_bus_allreduce(self.h, imix_dev, out_dev, count, op, scale))

    def begin(self, slot, imix_dev, count, out_dev=None, op=0, scale=0):
        self.ctx._ck(lib.cproc_cuda_bus_allreduce_begin(self.h, slot, imix_dev, out_dev, count, op, scale))

    def wait(self, slot):
        self.ctx._ck(lib.cproc_cuda_bus_wait(self.h, slot))

    IN_LAUNCH, PIPELINED = 1, 2

    def attach(self, batch, mode=1):
        """The batch's render launch exchanges its mix itself (mode 1: reduce in the same launch, 2: beside the next one).
        VOICE_BANK, XVOICE (mix only) and SQUARE_GRAIN_MIX batches."""
        self.ctx._ck(lib.cproc_cuda_bus_attach(self.h, batch.h, mode))

    def detach(self, batch):
        self.ctx._ck(lib.cproc_cuda_bus_attach(None, batch.h, 0))

    def flush(self):
        self.ctx._ck(lib.cproc_cuda_bus_flush(self.h))

    def status(self):
        v = C.c_uint32()
        self.ctx._ck(lib.cproc_cuda_bus_status(self.h, C.byref(v)))
        return v.value

    def destroy(self):
        if self.h:
            lib.cproc_cuda_bus_destroy(self.h)
            self.h = None
