"""ctypes binding of libb200serve.so (include/b200serve.h).

There is NO fallback: if the shared library is missing or a CUDA device is absent every compute
entry point raises.  Importing this module only dlopens the library (works on a CPU-only box so
the symbol-export test can run); `init()` needs a GPU.
"""
import ctypes
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200serve.so")

B2S_OK = 0
B2S_ERR_INVALID = -1
B2S_ERR_CUDA = -2
B2S_ERR_OOM = -3
B2S_ERR_NOT_INITIALISED = -4
B2S_ERR_BUSY = -5
B2S_ERR_NOT_READY = 1

MODEL_FOREST, MODEL_LINEAR, MODEL_GRAPH = 1, 2, 3

DTYPES = {  # b2s_dtype <-> numpy
    0: np.float32, 1: np.float64, 2: np.int32, 3: np.int64, 4: np.uint8, 5: np.int8,
    6: np.bool_, 7: np.uint64, 8: np.float16, 9: np.uint32,
}
DTYPE_CODES = {np.dtype(v): k for k, v in DTYPES.items()}
MAX_DIMS = 8


class Tensor(ctypes.Structure):
    _fields_ = [("data", ctypes.c_void_p), ("dtype", ctypes.c_int32), ("ndim", ctypes.c_int32),
                ("shape", ctypes.c_int64 * MAX_DIMS)]


class ModelInfo(ctypes.Structure):
    _fields_ = [("kind", ctypes.c_int32), ("n_inputs", ctypes.c_int32), ("n_outputs", ctypes.c_int32),
                ("in_dtype", ctypes.c_int32 * 4), ("out_dtype", ctypes.c_int32 * 4),
                ("in_row_elems", ctypes.c_int64 * 4), ("out_row_elems", ctypes.c_int64 * 4),
                ("weight_bytes", ctypes.c_int64), ("algo_bytes_fixed", ctypes.c_int64),
                ("algo_bytes_per_row", ctypes.c_int64)]


class LlmConfig(ctypes.Structure):
    _fields_ = [("vocab", ctypes.c_int32), ("hidden", ctypes.c_int32), ("inter", ctypes.c_int32),
                ("n_layers", ctypes.c_int32), ("n_heads", ctypes.c_int32), ("n_kv_heads", ctypes.c_int32),
                ("head_dim", ctypes.c_int32), ("max_batch", ctypes.c_int32), ("max_ctx", ctypes.c_int32),
                ("max_tokens", ctypes.c_int32), ("tp_size", ctypes.c_int32), ("tp_rank", ctypes.c_int32),
                ("rope_theta", ctypes.c_float), ("rms_eps", ctypes.c_float), ("kv_pages", ctypes.c_int32)]


class B2SError(ValueError):
    """Raised for every non-zero status. A ValueError so the reference's REST layer maps it to 422
    (clearml_serving/serving/main.py:155-161) -- and a message containing "CUDA out of memory. "
    triggers its restart path (main.py:116-123)."""

    def __init__(self, code, message):
        super(B2SError, self).__init__(message)
        self.code = code


# (name, restype, argtypes): must list every prototype of include/b200serve.h
_vp, _i, _i32, _i64, _u64, _sz = (ctypes.c_void_p, ctypes.c_int, ctypes.c_int32, ctypes.c_int64,
                                  ctypes.c_uint64, ctypes.c_size_t)
_P = ctypes.POINTER
PROTOTYPES = [
    ("b2s_init", _i, [_i, _sz]),
    ("b2s_shutdown", _i, []),
    ("b2s_abi_version", _i, []),
    ("b2s_last_error", ctypes.c_char_p, []),
    ("b2s_launch_count", _u64, []),
    ("b2s_device_count", _i, []),
    ("b2s_model_load", _i, [_i, _i, _vp, _sz, ctypes.c_char_p, _P(_u64)]),
    ("b2s_model_free", _i, [_u64]),
    ("b2s_model_get_info", _i, [_u64, _P(ModelInfo)]),
    ("b2s_debug_read", _i, [_u64, _vp]),
    ("b2s_stream_create", _i, [_u64, _i64, _i64, _i, _P(_u64)]),
    ("b2s_stream_destroy", _i, [_u64]),
    ("b2s_stream_synchronize", _i, [_u64]),
    ("b2s_stream_cuda_handle", _vp, [_u64]),
    ("b2s_infer_batch", _i, [_u64, _u64, _i32, _P(Tensor), _P(Tensor), _P(_u64)]),
    ("b2s_slot_acquire", _i, [_u64, _P(_i32), _P(_vp), _P(_vp)]),
    ("b2s_slot_submit", _i, [_u64, _u64, _i32, _i64, _vp, _P(_u64)]),
    ("b2s_slot_collate", _i, [_u64, _u64, _i32, _i32, _vp, _vp, _vp, _P(_u64)]),
    ("b2s_slot_release", _i, [_u64, _i32]),
    ("b2s_event_wait", _i, [_u64]),
    ("b2s_event_query", _i, [_u64]),
    ("b2s_infer_device", _i, [_u64, _u64, _i64, _P(_vp), _P(_vp), _vp]),
    ("b2s_device_malloc", _i, [_i, _sz, _P(_vp)]),
    ("b2s_device_free", _i, [_i, _vp]),
    ("b2s_memcpy_h2d", _i, [_i, _vp, _vp, _sz]),
    ("b2s_memcpy_d2h", _i, [_i, _vp, _vp, _sz]),
    ("b2s_flush_l2", _i, [_i]),
    ("b2s_stream_flush_l2", _i, [_u64]),
    ("b2s_timer_create", _i, [_u64, _P(_u64)]),
    ("b2s_timer_start", _i, [_u64]),
    ("b2s_timer_stop", _i, [_u64]),
    ("b2s_timer_elapsed_ms", _i, [_u64, _P(ctypes.c_float)]),
    ("b2s_timer_destroy", _i, [_u64]),
    ("b2s_op_gemm", _i, [_i, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _i, _i, _i]),
    ("b2s_op_conv", _i, [_i, _vp, _vp, _i64, _i, _i, _i, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _i, _i]),
    ("b2s_op_conv_stem", _i, [_i, _vp, _vp, _i, _i64, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _i]),
    ("b2s_op_layernorm", _i, [_i, _vp, _vp, _i64, _i, _vp, _vp, ctypes.c_float, _vp, _vp]),
    ("b2s_op_embed_layernorm", _i, [_i, _vp, _vp, _vp, _vp, _i, _i64, _i, _vp, _vp, _vp, _i, _i, _i, _vp, _vp,
                                    ctypes.c_float, _vp, _vp]),
    ("b2s_op_attention", _i, [_i, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i64]),
    ("b2s_debug_attention_stamps", _i, [_vp]),
    ("b2s_llm_create", _i, [_i, _P(LlmConfig), _P(_vp)]),
    ("b2s_llm_free", _i, [_vp]),
    ("b2s_llm_init_random", _i, [_vp, _u64, ctypes.c_float]),
    ("b2s_llm_tensor", _i, [_vp, ctypes.c_char_p, _i, _P(_vp), _P(_i64), _P(_i64), _P(_i)]),
    ("b2s_llm_comm_export", _i, [_vp, _vp, _P(_u64)]),
    ("b2s_llm_comm_attach", _i, [_vp, _vp]),
    ("b2s_llm_prefill", _i, [_vp, _i, _vp, _vp]),
    ("b2s_llm_kv_info", _i, [_vp, _P(_i32), _P(_i32), _P(_i32)]),
    ("b2s_llm_set_pages", _i, [_vp, _i, _i, _i, _vp]),
    ("b2s_llm_prefill_slots", _i, [_vp, _i, _vp, _vp, _vp]),
    ("b2s_llm_set_rows", _i, [_vp, _i, _vp, _vp, _vp]),
    ("b2s_llm_decode", _i, [_vp, _i, _i]),
    ("b2s_llm_get_tokens", _i, [_vp, _vp, _i]),
    ("b2s_llm_keep_logits", _i, [_vp, _i]),
    ("b2s_llm_get_logits", _i, [_vp, _vp]),
    ("b2s_llm_synchronize", _i, [_vp]),
    ("b2s_llm_event_record", _i, [_vp, _i]),
    ("b2s_llm_elapsed_ms", _i, [_vp, _i, _i, _P(ctypes.c_float)]),
    ("b2s_llm_flush_l2", _i, [_vp]),
    ("b2s_op_skinny_gemm", _i, [_i, _vp, _vp, _vp, _vp, _i, _i, _i]),
    ("b2s_op_llm_attn_decode", _i, [_i, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _i, _vp, _vp, _i, _vp, _i, _i, _i, _i, _i,
                                    _vp, _vp]),
    ("b2s_op_llm_attn_prefill", _i, [_i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _i, _vp, _i, _i, _i, _i]),
    ("b2s_op_llm_argmax", _i, [_i, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
]

_lib = None
_lib_lock = threading.Lock()
_inited_devices = set()


def lib():
    """dlopen libb200serve.so (built in-tree by clearml_serving_b200.build). Fails loudly."""
    global _lib
    if _lib is None:
        with _lib_lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        "libb200serve.so is missing at {} -- build it with `python -m clearml_serving_b200.build` "
                        "(there is no CPU fallback for the b200 engine)".format(LIB_PATH))
                l = ctypes.CDLL(LIB_PATH)
                for name, restype, argtypes in PROTOTYPES:
                    fn = getattr(l, name)
                    fn.restype = restype
                    fn.argtypes = argtypes
                if l.b2s_abi_version() != 2:
                    raise RuntimeError("libb200serve.so ABI version mismatch")
                _lib = l
    return _lib


def last_error():
    msg = lib().b2s_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc):
    if rc != 0:
        raise B2SError(rc, "b200serve: {}".format(last_error() or "error {}".format(rc)))


def device_count():
    return int(lib().b2s_device_count())


def init(device=0, pinned_arena_bytes=0):
    check(lib().b2s_init(int(device), int(pinned_arena_bytes)))
    _inited_devices.add(int(device))


def ensure_init(device=0, pinned_arena_bytes=0):
    if int(device) not in _inited_devices:
        init(device, pinned_arena_bytes)


def shutdown():
    check(lib().b2s_shutdown())
    _inited_devices.clear()


def launch_count():
    return int(lib().b2s_launch_count())


def flush_l2(device=0):
    check(lib().b2s_flush_l2(int(device)))


class Model(object):
    def __init__(self, kind, blob, device=0):
        ensure_init(device)
        self.device = int(device)
        self.kind = int(kind)
        blob = bytes(blob)
        h = ctypes.c_uint64(0)
        check(lib().b2s_model_load(self.device, self.kind, blob, len(blob), None, ctypes.byref(h)))
        self.handle = h.value
        info = ModelInfo()
        check(lib().b2s_model_get_info(self.handle, ctypes.byref(info)))
        self.info = info
        self.n_inputs = info.n_inputs
        self.n_outputs = info.n_outputs
        self.in_dtypes = [np.dtype(DTYPES[info.in_dtype[i]]) for i in range(info.n_inputs)]
        self.out_dtypes = [np.dtype(DTYPES[info.out_dtype[i]]) for i in range(info.n_outputs)]
        self.in_row_elems = [int(info.in_row_elems[i]) for i in range(info.n_inputs)]
        self.out_row_elems = [int(info.out_row_elems[i]) for i in range(info.n_outputs)]

    def algo_bytes(self, n_rows):
        return int(self.info.algo_bytes_fixed) + int(n_rows) * int(self.info.algo_bytes_per_row)

    def free(self):
        if self.handle:
            try:
                check(lib().b2s_model_free(self.handle))
            finally:
                self.handle = 0

    def __del__(self):
        try:
            if getattr(self, "handle", 0) and _lib is not None:
                lib().b2s_model_free(self.handle)
        except Exception:  # noqa
            pass


def _view(ptr, nbytes, dtype):
    buf = (ctypes.c_char * nbytes).from_address(ptr)
    return np.frombuffer(buf, dtype=dtype)


class Slot(object):
    """A pinned staging slot exposed as numpy views (inputs: [max_rows, row_elems])."""
    __slots__ = ("index", "inputs", "outputs")

    def __init__(self, index, inputs, outputs):
        self.index, self.inputs, self.outputs = index, inputs, outputs


class Stream(object):
    """One CUDA stream + pinned staging slots: one per endpoint."""

    def __init__(self, model, max_rows, max_row_elems=0, n_slots=4):
        self.model = model
        self.max_rows = int(max_rows)
        self.max_row_elems = int(max_row_elems)
        self.n_slots = int(n_slots)
        h = ctypes.c_uint64(0)
        check(lib().b2s_stream_create(model.handle, self.max_rows, self.max_row_elems, self.n_slots, ctypes.byref(h)))
        self.handle = h.value
        self._slot_views = {}

    # ---- general C-ABI path: per-request host tensors, gather/scatter inside the library --------
    def infer_batch(self, requests, outputs=None):
        """requests: list (per request) of list (per model input) of C-contiguous numpy arrays.
        Returns (event, outs) where outs[r][o] are numpy arrays filled when wait(event) returns."""
        m = self.model
        n_req = len(requests)
        tin = (Tensor * (n_req * m.n_inputs))()
        tout = (Tensor * (n_req * m.n_outputs))()
        outs = []
        keep = []
        for r, req in enumerate(requests):
            rows = None
            for i in range(m.n_inputs):
                a = req[i]
                if not (isinstance(a, np.ndarray) and a.flags["C_CONTIGUOUS"]):
                    a = np.ascontiguousarray(a)
                keep.append(a)
                t = tin[r * m.n_inputs + i]
                t.data = a.ctypes.data
                code = DTYPE_CODES.get(a.dtype)
                if code is None:
                    raise B2SError(B2S_ERR_INVALID, "b200serve: unsupported input dtype {}".format(a.dtype))
                t.dtype = code
                t.ndim = a.ndim if a.ndim > 0 else 1
                if a.ndim == 0:
                    t.shape[0] = 1
                for d in range(a.ndim):
                    t.shape[d] = a.shape[d]
                if m.in_row_elems[i] > 0:
                    rows = a.size // m.in_row_elems[i]
                else:  # variable length: [rows, len] (or [len] = one row)
                    rows = a.shape[0] if a.ndim >= 2 else 1
            rows = rows or 0
            ro = []
            for o in range(m.n_outputs):
                if outputs is not None:
                    buf = outputs[r][o]
                else:
                    shape = (rows,) if m.out_row_elems[o] == 1 else (rows, m.out_row_elems[o])
                    buf = np.empty(shape, dtype=m.out_dtypes[o])
                ro.append(buf)
                tout[r * m.n_outputs + o].data = buf.ctypes.data
            outs.append(ro)
        ev = ctypes.c_uint64(0)
        check(lib().b2s_infer_batch(m.handle, self.handle, n_req, tin, tout, ctypes.byref(ev)))
        return ev.value, outs, keep

    # ---- staged path: collate straight into the pinned slot -------------------------------------
    def acquire(self):
        m = self.model
        idx = ctypes.c_int32(-1)
        ins = (ctypes.c_void_p * 4)()
        outs = (ctypes.c_void_p * 4)()
        check(lib().b2s_slot_acquire(self.handle, ctypes.byref(idx), ins, outs))
        slot = self._slot_views.get(idx.value)
        if slot is None:
            vin, vout = [], []
            for i in range(m.n_inputs):
                re = m.in_row_elems[i]
                if re > 0:
                    v = _view(ins[i], self.max_rows * re * m.in_dtypes[i].itemsize, m.in_dtypes[i]).reshape(self.max_rows, re)
                else:
                    v = _view(ins[i], self.max_rows * self.max_row_elems * m.in_dtypes[i].itemsize, m.in_dtypes[i])
                vin.append(v)
            for o in range(m.n_outputs):
                re = m.out_row_elems[o]
                v = _view(outs[o], self.max_rows * re * m.out_dtypes[o].itemsize, m.out_dtypes[o])
                vout.append(v if re == 1 else v.reshape(self.max_rows, re))
            slot = Slot(idx.value, vin, vout)
            self._slot_views[idx.value] = slot
        return slot

    def submit(self, slot, n_rows, row_offsets=None):
        ev = ctypes.c_uint64(0)
        ro = None
        if row_offsets is not None:
            row_offsets = np.ascontiguousarray(row_offsets, dtype=np.int64)
            ro = row_offsets.ctypes.data
        check(lib().b2s_slot_submit(self.model.handle, self.handle, slot.index, int(n_rows), ro, ctypes.byref(ev)))
        return ev.value

    def collate_submit(self, slot, requests):
        """Collate `requests` (objects with .ptrs = host addresses of their inputs, .rows, .row_len) into `slot` INSIDE
        the library (b2s_slot_collate: memcpy without the GIL, worker pool for large batches) and submit the batch.
        Returns (event, n_rows)."""
        n = len(requests)
        ni = self.model.n_inputs
        ptrs = np.fromiter((p for r in requests for p in r.ptrs), dtype=np.uint64, count=n * ni)
        rows = np.fromiter((r.rows for r in requests), dtype=np.int64, count=n)
        lens = None
        if any(e < 0 for e in self.model.in_row_elems):
            lens = np.fromiter((r.row_len for r in requests), dtype=np.int64, count=n)
        ev = ctypes.c_uint64(0)
        check(lib().b2s_slot_collate(self.model.handle, self.handle, slot.index, n, ptrs.ctypes.data, rows.ctypes.data,
                                     lens.ctypes.data if lens is not None else None, ctypes.byref(ev)))
        return ev.value, int(rows.sum())

    def release(self, slot):
        check(lib().b2s_slot_release(self.handle, slot.index))

    @staticmethod
    def wait(event):
        check(lib().b2s_event_wait(event))

    @staticmethod
    def query(event):
        rc = lib().b2s_event_query(event)
        if rc == B2S_ERR_NOT_READY:
            return False
        check(rc)
        return True

    def synchronize(self):
        check(lib().b2s_stream_synchronize(self.handle))

    def flush_l2(self):
        check(lib().b2s_stream_flush_l2(self.handle))

    def cuda_handle(self):
        return lib().b2s_stream_cuda_handle(self.handle)

    def infer_device(self, n_rows, d_in, d_out, d_row_offsets=None):
        ins = (ctypes.c_void_p * 4)(*[int(p) for p in d_in])
        outs = (ctypes.c_void_p * 4)(*[int(p) for p in d_out])
        check(lib().b2s_infer_device(self.model.handle, self.handle, int(n_rows), ins, outs,
                                     int(d_row_offsets) if d_row_offsets else None))

    def destroy(self):
        if self.handle:
            try:
                check(lib().b2s_stream_destroy(self.handle))
            finally:
                self.handle = 0
                self._slot_views = {}

    def __del__(self):
        try:
            if getattr(self, "handle", 0) and _lib is not None:
                lib().b2s_stream_destroy(self.handle)
        except Exception:  # noqa
            pass


class Timer(object):
    def __init__(self, stream):
        h = ctypes.c_uint64(0)
        check(lib().b2s_timer_create(stream.handle, ctypes.byref(h)))
        self.handle = h.value

    def start(self):
        check(lib().b2s_timer_start(self.handle))

    def stop(self):
        check(lib().b2s_timer_stop(self.handle))

    def elapsed_ms(self):
        ms = ctypes.c_float(0)
        check(lib().b2s_timer_elapsed_ms(self.handle, ctypes.byref(ms)))
        return float(ms.value)

    def destroy(self):
        if self.handle:
            lib().b2s_timer_destroy(self.handle)
            self.handle = 0


class DeviceBuffer(object):
    def __init__(self, nbytes, device=0):
        self.device = int(device)
        self.nbytes = int(nbytes)
        p = ctypes.c_void_p(0)
        check(lib().b2s_device_malloc(self.device, self.nbytes, ctypes.byref(p)))
        self.ptr = p.value

    def upload(self, arr):
        arr = np.ascontiguousarray(arr)
        assert arr.nbytes <= self.nbytes
        check(lib().b2s_memcpy_h2d(self.device, self.ptr, arr.ctypes.data, arr.nbytes))

    def download(self, dtype, count):
        out = np.empty(count, dtype=dtype)
        assert out.nbytes <= self.nbytes
        check(lib().b2s_memcpy_d2h(self.device, out.ctypes.data, self.ptr, out.nbytes))
        return out

    def free(self):
        if self.ptr:
            lib().b2s_device_free(self.device, self.ptr)
            self.ptr = 0


class Llm(object):
    """Decoder-only LLM executor (b2s_llm_* of include/b200serve.h).  One instance = one tensor-parallel rank."""

    def __init__(self, device=0, vocab=0, hidden=0, inter=0, n_layers=0, n_heads=0, n_kv_heads=0, head_dim=128,
                 max_batch=32, max_ctx=1024, max_tokens=None, tp_size=1, tp_rank=0, rope_theta=500000.0, rms_eps=1e-5,
                 kv_pages=0):
        ensure_init(device)
        self.device = int(device)
        if max_tokens is None:
            max_tokens = max_batch * max_ctx
        self.cfg = LlmConfig(vocab, hidden, inter, n_layers, n_heads, n_kv_heads, head_dim, max_batch, max_ctx,
                             int(max_tokens), tp_size, tp_rank, rope_theta, rms_eps, int(kv_pages))
        h = ctypes.c_void_p(0)
        check(lib().b2s_llm_create(self.device, ctypes.byref(self.cfg), ctypes.byref(h)))
        self.handle = h
        self.vocab_shard = vocab // tp_size
        self.n_seq = 0

    def init_random(self, seed=0, std=0.02):
        check(lib().b2s_llm_init_random(self.handle, int(seed), float(std)))

    def tensor(self, name, layer=0):
        """-> (device pointer, rows, cols, numpy dtype of the host image: uint16 for bf16 / float32)"""
        ptr, rows, cols, eb = ctypes.c_void_p(0), ctypes.c_int64(0), ctypes.c_int64(0), ctypes.c_int(0)
        check(lib().b2s_llm_tensor(self.handle, name.encode(), int(layer), ctypes.byref(ptr), ctypes.byref(rows),
                                   ctypes.byref(cols), ctypes.byref(eb)))
        return ptr.value, rows.value, cols.value, (np.uint16 if eb.value == 2 else np.float32)

    def load_tensor(self, name, layer, host):
        """host: uint16 (bf16 bit patterns) or float32 array of exactly this rank's shard shape"""
        ptr, rows, cols, dt = self.tensor(name, layer)
        a = np.ascontiguousarray(host, dtype=dt).reshape(-1)
        if a.size != rows * cols:
            raise B2SError(B2S_ERR_INVALID, "llm tensor {}[{}]: expected {} x {} elements, got {}".format(
                name, layer, rows, cols, a.size))
        check(lib().b2s_memcpy_h2d(self.device, ptr, a.ctypes.data, a.nbytes))

    def read_tensor(self, name, layer=0):
        ptr, rows, cols, dt = self.tensor(name, layer)
        out = np.empty((rows, cols), dtype=dt)
        check(lib().b2s_memcpy_d2h(self.device, out.ctypes.data, ptr, out.nbytes))
        return out

    def comm_export(self):
        buf = (ctypes.c_ubyte * 64)()
        n = ctypes.c_uint64(0)
        check(lib().b2s_llm_comm_export(self.handle, buf, ctypes.byref(n)))
        return bytes(buf)

    def comm_attach(self, peer_handle):
        buf = (ctypes.c_ubyte * 64).from_buffer_copy(bytes(peer_handle))
        check(lib().b2s_llm_comm_attach(self.handle, buf))

    def prefill(self, prompts):
        """prompts: list of int sequences (token ids); enqueues the prompt wave + the first sampled token"""
        offs = np.zeros(len(prompts) + 1, dtype=np.int32)
        offs[1:] = np.cumsum([len(p) for p in prompts])
        toks = np.ascontiguousarray(np.concatenate([np.asarray(p, dtype=np.int32).reshape(-1) for p in prompts]))
        check(lib().b2s_llm_prefill(self.handle, len(prompts), toks.ctypes.data, offs.ctypes.data))
        self.n_seq = len(prompts)

    # ---- continuous batching over the paged KV cache (the host scheduler owns slots and pages)
    def kv_info(self):
        """-> (pages in the pool, tokens per page, page-table entries per slot)"""
        a, b, c = ctypes.c_int32(0), ctypes.c_int32(0), ctypes.c_int32(0)
        check(lib().b2s_llm_kv_info(self.handle, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)))
        return a.value, b.value, c.value

    def set_pages(self, slot, first, pages):
        pg = np.ascontiguousarray(pages, dtype=np.int32)
        check(lib().b2s_llm_set_pages(self.handle, int(slot), int(first), int(pg.size), pg.ctypes.data))

    def prefill_slots(self, prompts, slots):
        """like prefill(), sequence i into KV slot slots[i]; other slots keep their sequences"""
        offs = np.zeros(len(prompts) + 1, dtype=np.int32)
        offs[1:] = np.cumsum([len(p) for p in prompts])
        toks = np.ascontiguousarray(np.concatenate([np.asarray(p, dtype=np.int32).reshape(-1) for p in prompts]))
        sl = np.ascontiguousarray(slots, dtype=np.int32)
        check(lib().b2s_llm_prefill_slots(self.handle, len(prompts), toks.ctypes.data, offs.ctypes.data, sl.ctypes.data))
        self.n_seq = len(prompts)

    def set_rows(self, slots, ctx_len, next_tok):
        sl, cl, nt = (np.ascontiguousarray(a, dtype=np.int32) for a in (slots, ctx_len, next_tok))
        check(lib().b2s_llm_set_rows(self.handle, int(sl.size), sl.ctypes.data, cl.ctypes.data, nt.ctypes.data))
        self.n_seq = int(sl.size)

    def decode(self, n_steps, use_graph=True):
        check(lib().b2s_llm_decode(self.handle, int(n_steps), int(use_graph)))   # 0 eager, 1 CUDA graph, 2 eager + per-kernel timing

    def tokens(self, n):
        out = np.empty((self.n_seq, int(n)), dtype=np.int32)
        check(lib().b2s_llm_get_tokens(self.handle, out.ctypes.data, int(n)))
        return out

    def keep_logits(self, on=True):
        check(lib().b2s_llm_keep_logits(self.handle, 1 if on else 0))

    def logits(self):
        out = np.empty((self.n_seq, self.vocab_shard), dtype=np.float32)
        check(lib().b2s_llm_get_logits(self.handle, out.ctypes.data))
        return out

    def synchronize(self):
        check(lib().b2s_llm_synchronize(self.handle))

    def record(self, which):
        check(lib().b2s_llm_event_record(self.handle, int(which)))

    def elapsed_ms(self, a, b):
        ms = ctypes.c_float(0)
        check(lib().b2s_llm_elapsed_ms(self.handle, int(a), int(b), ctypes.byref(ms)))
        return float(ms.value)

    def flush_l2(self):
        check(lib().b2s_llm_flush_l2(self.handle))

    def free(self):
        if self.handle:
            lib().b2s_llm_free(self.handle)
            self.handle = None

    def __del__(self):
        try:
            if getattr(self, "handle", None) and _lib is not None:
                lib().b2s_llm_free(self.handle)
        except Exception:  # noqa
            pass
