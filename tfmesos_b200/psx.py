"""ctypes binding of libpsx.so (include/psx.h) -- the stub a tfmesos maintainer
would add where tfmesos/server.py:51-66 hands the process to tf.train.Server.

There is no fallback: if the library has not been built this module raises on
first use, and without a CUDA device every compute call raises
``RuntimeError(psx_last_error())`` (the reference's error style,
tfmesos/scheduler.py:398).
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# TFMESOS_PSX_LIB selects another build of the same ABI (kernel A/B experiments)
LIB_PATH = os.environ.get("TFMESOS_PSX_LIB") or os.path.join(HERE, "lib", "libpsx.so")

ABI_VERSION = 11
OPT_SGD, OPT_ADAM, OPT_MOMENTUM, OPT_ADAGRAD, OPT_RMSPROP = 0, 1, 2, 3, 4
# f32 state arrays each optimizer keeps beside var: PSX_M [, PSX_V]
OPT_STATE_ARRAYS = {OPT_SGD: 0, OPT_ADAM: 2, OPT_MOMENTUM: 1, OPT_ADAGRAD: 1, OPT_RMSPROP: 2}
MODE_ASYNC_ORDERED, MODE_SUM, MODE_SYNC_MEAN = 0, 1, 2
F32, BF16 = 0, 1
VAR, M, V, SLOT0 = 0, 1, 2, 16
MAX_SLOTS = 16
HANDLE_BYTES = 128

_u64 = ctypes.c_uint64
_u32 = ctypes.c_uint32
_i32 = ctypes.c_int
_vp = ctypes.c_void_p
_fp = ctypes.POINTER(ctypes.c_float)

(OP_PUSH, OP_PULL, OP_APPLY, OP_ROUND, OP_SIGNAL, OP_WAIT_APPLIED, OP_WAIT_SLOTS,
 OP_SIGNAL_MANY, OP_WAIT_ARRIVALS, OP_WAIT_MAILBOX, OP_ROUND_COUNTED, OP_APPLY_COUNTED,
 OP_SIGNAL_COUNTED, OP_MAILBOX_WAIT, OP_MAILBOX_CONSUME) = range(1, 16)


class Op(ctypes.Structure):
    """struct psx_op (include/psx.h)."""
    _fields_ = [("op", ctypes.c_int32), ("a", ctypes.c_int32), ("b", ctypes.c_int32),
                ("c", ctypes.c_int32), ("id", _u64), ("off", _u64), ("n", _u64),
                ("ptr", _vp), ("stream", _vp), ("seq", _u32), ("reserved", _u32)]


# name -> (restype, argtypes); every symbol include/psx.h declares
SIGNATURES = {
    "psx_abi_version": (_i32, []),
    "psx_last_error": (ctypes.c_char_p, []),
    "psx_device_count": (_i32, [ctypes.POINTER(_i32)]),
    "psx_init": (_i32, [_i32]),
    "psx_enable_peer": (_i32, [_i32, _i32]),
    "psx_shard_create": (_i32, [_i32, _u64, _i32, _fp, _i32, _i32, ctypes.POINTER(_u64)]),
    "psx_shard_destroy": (_i32, [_u64]),
    "psx_shard_export": (_i32, [_u64, _vp]),
    "psx_shard_set_hyper": (_i32, [_u64, _fp]),
    "psx_set_values": (_i32, [_u64, _i32, _vp, _u64, _u64]),
    "psx_get_values": (_i32, [_u64, _i32, _vp, _u64, _u64]),
    "psx_get_state": (_i32, [_u64, _fp, _fp, ctypes.POINTER(ctypes.c_int64),
                             ctypes.POINTER(_u32)]),
    "psx_set_state": (_i32, [_u64, ctypes.c_float, ctypes.c_float, ctypes.c_int64]),
    "psx_apply": (_i32, [_u64, _i32, _i32, _i32, _u32, _vp]),
    "psx_apply_range": (_i32, [_u64, _i32, _i32, _i32, _u64, _u64, _i32, _u32, _vp]),
    "psx_wait_slots": (_i32, [_u64, _i32, _i32, _u32, _vp]),
    "psx_shard_open": (_i32, [_vp, _i32, _i32, ctypes.POINTER(_u64)]),
    "psx_shard_close": (_i32, [_u64]),
    "psx_client_export": (_i32, [_u64, _vp]),
    "psx_shard_register_client": (_i32, [_u64, _i32, _vp]),
    "psx_push": (_i32, [_u64, _vp, _u64, _u64, _i32, _u32, _vp]),
    "psx_pull": (_i32, [_u64, _vp, _u64, _u64, _i32, _u32, _vp]),
    "psx_list_create": (_i32, [_u64, ctypes.POINTER(_vp), ctypes.POINTER(_u64),
                               ctypes.POINTER(_u64), _i32, ctypes.POINTER(_u64)]),
    "psx_list_destroy": (_i32, [_u64]),
    "psx_push_list": (_i32, [_u64, _u32, _i32, _vp]),
    "psx_pull_list": (_i32, [_u64, _u32, _i32, _vp]),
    "psx_buffer_create": (_i32, [_i32, _u64, ctypes.POINTER(_u64), ctypes.POINTER(_vp)]),
    "psx_buffer_export": (_i32, [_u64, _vp]),
    "psx_buffer_destroy": (_i32, [_u64]),
    "psx_round_bind": (_i32, [_u64, _i32, _vp, _vp, _u64]),
    "psx_signal": (_i32, [_u64, _u32, _vp]),
    "psx_wait_applied": (_i32, [_u64, _u32, _vp]),
    "psx_round": (_i32, [_u64, _i32, _i32, _i32, _u32, _vp]),
    "psx_signal_many": (_i32, [ctypes.POINTER(_u64), _i32, _u32, _vp]),
    "psx_round_counted": (_i32, [_u64, _i32, _i32, _i32, _vp]),
    "psx_apply_counted": (_i32, [_u64, _i32, _i32, _i32, _vp]),
    "psx_signal_counted": (_i32, [ctypes.POINTER(_u64), _i32, _u32, _u64, _u32, _vp]),
    "psx_mailbox_consume": (_i32, [_u64, _u32, _vp]),
    "psx_mailbox_set": (_i32, [_u64, _u32]),
    "psx_wait_arrivals": (_i32, [_u64, _u32, _vp]),
    "psx_mailbox_create": (_i32, [_i32, ctypes.POINTER(_u64)]),
    "psx_mailbox_export": (_i32, [_u64, _vp]),
    "psx_mailbox_destroy": (_i32, [_u64]),
    "psx_shard_register_mailbox": (_i32, [_u64, _i32, _vp]),
    "psx_wait_mailbox": (_i32, [_u64, _u32, _vp]),
    "psx_nvls_supported": (_i32, [_i32, ctypes.POINTER(_i32)]),
    "psx_mc_create": (_i32, [ctypes.POINTER(_i32), _i32, _u64, ctypes.POINTER(_u64)]),
    "psx_mc_destroy": (_i32, [_u64]),
    "psx_mc_ptrs": (_i32, [_u64, _i32, ctypes.POINTER(_vp), ctypes.POINTER(_vp),
                           ctypes.POINTER(_u64)]),
    "psx_mc_broadcast": (_i32, [_u64, _i32, _vp, _u64, _u64, _vp]),
    "psx_mc_reduce": (_i32, [_u64, _i32, _vp, _u64, _u64, _vp]),
    "psx_shard_unregister_client": (_i32, [_u64, _i32]),
    "psx_mcx_create": (_i32, [_i32, _i32, _u64, ctypes.POINTER(_i32), ctypes.POINTER(_u64)]),
    "psx_mcx_import": (_i32, [_i32, _i32, _u64, _i32, ctypes.POINTER(_u64)]),
    "psx_mcx_add_device": (_i32, [_u64]),
    "psx_mcx_bind": (_i32, [_u64, ctypes.POINTER(_vp), ctypes.POINTER(_vp),
                            ctypes.POINTER(_u64)]),
    "psx_mcx_destroy": (_i32, [_u64]),
    "psx_round_bind_mc": (_i32, [_u64, _u64, _u64, _u64, _u64, _i32]),
    "psx_serve_start": (_i32, [_u64, _i32, _i32, _i32]),
    "psx_serve_stop": (_i32, [_u64]),
    "psx_serve_stats": (_i32, [_u64, ctypes.POINTER(_u64), ctypes.POINTER(_u32),
                               ctypes.POINTER(_u32), ctypes.POINTER(ctypes.c_int64)]),
    "psx_push_stamped": (_i32, [_u64, _vp, _u64, _u64, _i32, _u32, _u32, _vp]),
    "psx_wait_tokens": (_i32, [_u64, _u32, _vp]),
    "psx_read_step_async": (_i32, [_u64, _vp, _vp]),
    "psx_client_poll": (_i32, [_u64, ctypes.POINTER(_u32), ctypes.POINTER(_u32),
                               ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(_i32)]),
    "psx_push_rows": (_i32, [_u64, _vp, _vp, _u64, _u64, _i32, _u32, _vp]),
    "psx_apply_rows": (_i32, [_u64, _i32, _i32, _i32, _u64, _u32, _vp]),
    "psx_batch": (_i32, [ctypes.POINTER(Op), _i32, ctypes.POINTER(_i32)]),
    "psx_launch_count": (_u64, []),
    "psx_shard_ptr": (_i32, [_u64, _i32, ctypes.POINTER(_vp)]),
    "psx_copy": (_i32, [_i32, _vp, _vp, _u64, _vp]),
}

_lib = None


def lib():
    """The loaded library; raises if it was never built (no CPU fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libpsx.so is missing (%s): build it with "
                "`python -m tfmesos_b200.build`; there is no CPU fallback" % LIB_PATH)
        l = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        if l.psx_abi_version() != ABI_VERSION:
            raise RuntimeError("libpsx.so ABI %d, binding expects %d"
                               % (l.psx_abi_version(), ABI_VERSION))
        _lib = l
    return _lib


def last_error():
    return lib().psx_last_error().decode("utf-8", "replace")


def _check(rc):
    if rc != 0:
        raise RuntimeError("psx error %d: %s" % (rc, last_error()))


def _stream_ptr(stream):
    if stream is None:
        import torch
        return torch.cuda.current_stream().cuda_stream
    if isinstance(stream, int):
        return stream
    return stream.cuda_stream


def device_count():
    n = _i32(0)
    _check(lib().psx_device_count(ctypes.byref(n)))
    return n.value


def init(device):
    _check(lib().psx_init(int(device)))


def enable_peer(device, peer):
    _check(lib().psx_enable_peer(int(device), int(peer)))


def launch_count():
    return int(lib().psx_launch_count())


def _hyper(lr, beta1, beta2, epsilon):
    return (ctypes.c_float * 4)(lr, beta1, beta2, epsilon)


class Shard(object):
    """PS-side handle of one shard in HBM (psx_shard_create)."""

    def __init__(self, device, nelem, opt=OPT_SGD, lr=0.01, beta1=0.9, beta2=0.999,
                 epsilon=1e-8, n_slots=1, wire=F32):
        sid = _u64(0)
        _check(lib().psx_shard_create(int(device), int(nelem), int(opt),
                                      _hyper(lr, beta1, beta2, epsilon), int(n_slots),
                                      int(wire), ctypes.byref(sid)))
        self.id = sid.value
        self.device = int(device)
        self.nelem = int(nelem)
        self.opt = int(opt)
        self.n_slots = int(n_slots)
        self.wire = int(wire)

    def destroy(self):
        if self.id:
            _check(lib().psx_shard_destroy(self.id))
            self.id = 0

    def export(self):
        buf = ctypes.create_string_buffer(HANDLE_BYTES)
        _check(lib().psx_shard_export(self.id, buf))
        return buf.raw

    def set_hyper(self, lr, beta1=0.9, beta2=0.999, epsilon=1e-8):
        _check(lib().psx_shard_set_hyper(self.id, _hyper(lr, beta1, beta2, epsilon)))

    def set_values(self, which, host, off=0):
        import numpy as np
        a = np.ascontiguousarray(host, dtype=np.float32).ravel()
        _check(lib().psx_set_values(self.id, int(which), a.ctypes.data, int(off), a.size))

    def get_values(self, which, off=0, n=None):
        import numpy as np
        n = self.nelem - off if n is None else n
        out = np.empty(n, np.float32)
        _check(lib().psx_get_values(self.id, int(which), out.ctypes.data, int(off), int(n)))
        return out

    def state(self):
        b1p, b2p = ctypes.c_float(0), ctypes.c_float(0)
        step, seq = ctypes.c_int64(0), _u32(0)
        _check(lib().psx_get_state(self.id, ctypes.byref(b1p), ctypes.byref(b2p),
                                   ctypes.byref(step), ctypes.byref(seq)))
        return {"beta1_power": b1p.value, "beta2_power": b2p.value,
                "global_step": step.value, "apply_seq": seq.value}

    def set_state(self, beta1_power, beta2_power, global_step):
        _check(lib().psx_set_state(self.id, beta1_power, beta2_power, int(global_step)))

    def ptr(self, which):
        p = _vp(0)
        _check(lib().psx_shard_ptr(self.id, int(which), ctypes.byref(p)))
        return p.value

    def register_client(self, slot, client_handle):
        _check(lib().psx_shard_register_client(self.id, int(slot), client_handle))

    def apply_rows(self, mode, first_slot, count, row_len, wait_seq=0, stream=None):
        _check(lib().psx_apply_rows(self.id, int(mode), int(first_slot), int(count),
                                    int(row_len), int(wait_seq), _stream_ptr(stream)))

    def serve_start(self, mode, replicas_to_aggregate=1, idle_sleep_us=0):
        """Request-free serving loop on this shard (psx_serve_start)."""
        _check(lib().psx_serve_start(self.id, int(mode), int(replicas_to_aggregate),
                                     int(idle_sleep_us)))

    def serve_stop(self):
        _check(lib().psx_serve_stop(self.id))

    def serve_stats(self):
        it, served, dropped, step = _u64(0), _u32(0), _u32(0), ctypes.c_int64(0)
        _check(lib().psx_serve_stats(self.id, ctypes.byref(it), ctypes.byref(served),
                                     ctypes.byref(dropped), ctypes.byref(step)))
        return {"iterations": it.value, "served": served.value, "dropped": dropped.value,
                "global_step": step.value}

    def unregister_client(self, slot):
        _check(lib().psx_shard_unregister_client(self.id, int(slot)))

    def round_bind_mc(self, member, grad_off_bytes, param_off_bytes, elem_off, n_members):
        _check(lib().psx_round_bind_mc(self.id, member.id, int(grad_off_bytes),
                                       int(param_off_bytes), int(elem_off), int(n_members)))

    def register_mailbox(self, slot, mailbox_handle):
        _check(lib().psx_shard_register_mailbox(self.id, int(slot), mailbox_handle))

    def wait_arrivals(self, target, stream=None):
        _check(lib().psx_wait_arrivals(self.id, int(target) & 0xFFFFFFFF, _stream_ptr(stream)))

    def apply(self, mode, first_slot=0, count=1, wait_seq=0, stream=None):
        _check(lib().psx_apply(self.id, int(mode), int(first_slot), int(count),
                               int(wait_seq), _stream_ptr(stream)))

    def apply_range(self, mode, first_slot, count, elem_off, elem_n, finish=True, wait_seq=0,
                    stream=None):
        _check(lib().psx_apply_range(self.id, int(mode), int(first_slot), int(count),
                                     int(elem_off), int(elem_n), int(bool(finish)),
                                     int(wait_seq), _stream_ptr(stream)))

    def wait_slots(self, first_slot, count, wait_seq, stream=None):
        _check(lib().psx_wait_slots(self.id, int(first_slot), int(count), int(wait_seq),
                                    _stream_ptr(stream)))

    def round_bind(self, slot, grad_handle, param_handle, elem_off=0):
        _check(lib().psx_round_bind(self.id, int(slot), grad_handle, param_handle,
                                    int(elem_off)))

    def round(self, mode, first_slot=0, count=1, wait_seq=0, stream=None):
        _check(lib().psx_round(self.id, int(mode), int(first_slot), int(count),
                               int(wait_seq), _stream_ptr(stream)))

    def round_counted(self, mode, first_slot, count, stream=None):
        _check(lib().psx_round_counted(self.id, int(mode), int(first_slot), int(count),
                                       _stream_ptr(stream)))

    def apply_counted(self, mode, first_slot, count, stream=None):
        _check(lib().psx_apply_counted(self.id, int(mode), int(first_slot), int(count),
                                       _stream_ptr(stream)))


class Client(object):
    """Worker-side attachment to a shard (psx_shard_open)."""

    def __init__(self, handle, device, slot):
        cid = _u64(0)
        _check(lib().psx_shard_open(handle, int(device), int(slot), ctypes.byref(cid)))
        self.id = cid.value
        self.device = int(device)
        self.slot = int(slot)

    def close(self):
        if self.id:
            _check(lib().psx_shard_close(self.id))
            self.id = 0

    def export(self):
        buf = ctypes.create_string_buffer(HANDLE_BYTES)
        _check(lib().psx_client_export(self.id, buf))
        return buf.raw

    def push(self, grad_ptr, n, off=0, dtype=F32, seq=0, stream=None):
        _check(lib().psx_push(self.id, grad_ptr, int(off), int(n), int(dtype), int(seq),
                              _stream_ptr(stream)))

    def pull(self, param_ptr, n, off=0, dtype=F32, wait_seq=0, stream=None):
        _check(lib().psx_pull(self.id, param_ptr, int(off), int(n), int(dtype),
                              int(wait_seq), _stream_ptr(stream)))

    def push_rows(self, idx_ptr, rows_ptr, k, row_len, dtype=F32, seq=1, stream=None):
        """IndexedSlices push: k rows (k x row_len at rows_ptr) with strictly ascending
        int64 row indices at idx_ptr."""
        _check(lib().psx_push_rows(self.id, idx_ptr, rows_ptr, int(k), int(row_len), int(dtype),
                                   int(seq), _stream_ptr(stream)))

    def push_stamped(self, grad_ptr, n, off=0, dtype=F32, seq=1, stamp=0, stream=None):
        _check(lib().psx_push_stamped(self.id, grad_ptr, int(off), int(n), int(dtype), int(seq),
                                      int(stamp) & 0xFFFFFFFF, _stream_ptr(stream)))

    def wait_tokens(self, target, stream=None):
        _check(lib().psx_wait_tokens(self.id, int(target) & 0xFFFFFFFF, _stream_ptr(stream)))

    def poll(self):
        """Host-side read of the client block: {applied, tokens, global_step, in_process}."""
        a, t, st, ip = _u32(0), _u32(0), ctypes.c_int64(0), _i32(0)
        _check(lib().psx_client_poll(self.id, ctypes.byref(a), ctypes.byref(t), ctypes.byref(st),
                                     ctypes.byref(ip)))
        return {"applied": a.value, "tokens": t.value, "global_step": st.value,
                "in_process": bool(ip.value)}

    def wait_host(self, key, target, timeout=60.0):
        """Spin on poll() until block[key] >= target (in-process clients of a served
        shard; anything else stream-waits)."""
        import time
        t0 = time.time()
        while True:
            st = self.poll()
            if ((st[key] - int(target)) & 0xFFFFFFFF) < 0x80000000:
                return st
            if time.time() - t0 > timeout:
                raise RuntimeError("timed out waiting for %s >= %d (%r)" % (key, target, st))

    def read_step_async(self, host_ptr, stream=None):
        _check(lib().psx_read_step_async(self.id, host_ptr, _stream_ptr(stream)))

    def signal(self, seq, stream=None):
        _check(lib().psx_signal(self.id, int(seq), _stream_ptr(stream)))

    def wait_applied(self, seq, stream=None):
        _check(lib().psx_wait_applied(self.id, int(seq), _stream_ptr(stream)))


class Mailbox(object):
    """A worker's completion counter in its own HBM (psx_mailbox_create): every
    shard it is registered with bumps it when an apply / round completes."""

    def __init__(self, device):
        mid = _u64(0)
        _check(lib().psx_mailbox_create(int(device), ctypes.byref(mid)))
        self.id = mid.value
        self.device = int(device)

    def export(self):
        buf = ctypes.create_string_buffer(HANDLE_BYTES)
        _check(lib().psx_mailbox_export(self.id, buf))
        return buf.raw

    def wait(self, target, stream=None):
        _check(lib().psx_wait_mailbox(self.id, int(target) & 0xFFFFFFFF, _stream_ptr(stream)))

    def set(self, value):
        _check(lib().psx_mailbox_set(self.id, int(value)))

    def consume(self, n, stream=None):
        _check(lib().psx_mailbox_consume(self.id, int(n), _stream_ptr(stream)))

    def destroy(self):
        if self.id:
            _check(lib().psx_mailbox_destroy(self.id))
            self.id = 0


def signal_many(clients, seq, stream=None):
    ids = (_u64 * len(clients))(*[c.id for c in clients])
    _check(lib().psx_signal_many(ids, len(clients), int(seq), _stream_ptr(stream)))


def signal_counted(clients, seq, mailbox, consume, stream=None):
    ids = (_u64 * len(clients))(*[c.id for c in clients])
    _check(lib().psx_signal_counted(ids, len(clients), int(seq), mailbox.id, int(consume),
                                    _stream_ptr(stream)))


class TensorList(object):
    """A list of device tensors mapped onto shard offsets (psx_list_create):
    one launch pushes / pulls all of them."""

    def __init__(self, client, ptrs, offs, counts):
        k = len(ptrs)
        lid = _u64(0)
        _check(lib().psx_list_create(client.id, (_vp * k)(*ptrs), (_u64 * k)(*offs),
                                     (_u64 * k)(*counts), k, ctypes.byref(lid)))
        self.id = lid.value
        self.client = client

    def push(self, seq=0, tma=True, stream=None):
        _check(lib().psx_push_list(self.id, int(seq), int(bool(tma)), _stream_ptr(stream)))

    def pull(self, wait_seq=0, tma=True, stream=None):
        _check(lib().psx_pull_list(self.id, int(wait_seq), int(bool(tma)), _stream_ptr(stream)))

    def destroy(self):
        if self.id:
            _check(lib().psx_list_destroy(self.id))
            self.id = 0


class Buffer(object):
    """Exportable device buffer (psx_buffer_create); ``tensor()`` views it as a
    torch tensor without copying."""

    def __init__(self, device, nbytes):
        bid, p = _u64(0), _vp(0)
        _check(lib().psx_buffer_create(int(device), int(nbytes), ctypes.byref(bid),
                                       ctypes.byref(p)))
        self.id = bid.value
        self.ptr = p.value
        self.device = int(device)
        self.nbytes = int(nbytes)

    def export(self):
        buf = ctypes.create_string_buffer(HANDLE_BYTES)
        _check(lib().psx_buffer_export(self.id, buf))
        return buf.raw

    def destroy(self):
        if self.id:
            _check(lib().psx_buffer_destroy(self.id))
            self.id = 0

    @property
    def __cuda_array_interface__(self):
        return {"shape": (self.nbytes // 2,), "typestr": "<i2", "data": (self.ptr, False),
                "version": 2, "strides": None}

    def tensor(self, dtype=None):
        """Zero-copy torch view of the buffer (float32 unless ``dtype`` says bfloat16)."""
        import torch
        raw = torch.as_tensor(self, device="cuda:%d" % self.device)
        return raw.view(torch.float32 if dtype is None else dtype)


def nvls_supported(device):
    v = _i32(0)
    _check(lib().psx_nvls_supported(int(device), ctypes.byref(v)))
    return bool(v.value)


class MulticastBuffer(object):
    """One buffer per GPU bound to one NVSwitch multicast object (experimental)."""

    def __init__(self, devices, nbytes):
        arr = (_i32 * len(devices))(*devices)
        mid = _u64(0)
        _check(lib().psx_mc_create(arr, len(devices), int(nbytes), ctypes.byref(mid)))
        self.id = mid.value
        self.devices = list(devices)
        self.nbytes = int(nbytes)

    def ptrs(self, member):
        uc, mc, size = _vp(0), _vp(0), _u64(0)
        _check(lib().psx_mc_ptrs(self.id, int(member), ctypes.byref(uc), ctypes.byref(mc),
                                 ctypes.byref(size)))
        return uc.value, mc.value, size.value

    def tensor(self, member):
        """float32 torch view of this member's own (unicast) copy."""
        import torch
        uc, _, _ = self.ptrs(member)

        class _View(object):
            __cuda_array_interface__ = {"shape": (self.nbytes // 4,), "typestr": "<f4",
                                        "data": (uc, False), "version": 2, "strides": None}
        v = _View()
        v.owner = self
        return torch.as_tensor(v, device="cuda:%d" % self.devices[member])

    def broadcast(self, member, src_ptr, nbytes, off=0, stream=None):
        _check(lib().psx_mc_broadcast(self.id, int(member), src_ptr, int(off), int(nbytes),
                                      _stream_ptr(stream)))

    def reduce(self, member, dst_ptr, nbytes, off=0, stream=None):
        _check(lib().psx_mc_reduce(self.id, int(member), dst_ptr, int(off), int(nbytes),
                                   _stream_ptr(stream)))

    def destroy(self):
        if self.id:
            _check(lib().psx_mc_destroy(self.id))
            self.id = 0


def device_tensor(ptr, numel, dtype, device, owner=None):
    """Zero-copy torch view of raw device memory (kept alive by ``owner``)."""
    import torch
    esz = torch.empty(0, dtype=dtype).element_size()

    class _View(object):
        __cuda_array_interface__ = {"shape": (int(numel) * esz,), "typestr": "|u1",
                                    "data": (int(ptr), False), "version": 2, "strides": None}
    v = _View()
    v.owner = owner
    return torch.as_tensor(v, device="cuda:%d" % device).view(dtype)


class McMember(object):
    """This process's member of a multi-process NVSwitch multicast object
    (psx_mcx_*).  ``fd`` (creator only) is the descriptor to ship to the other
    members over an AF_UNIX socket."""

    def __init__(self, mid, device, fd=-1):
        self.id, self.device, self.fd = mid, int(device), fd

    @classmethod
    def create(cls, device, n_devices, nbytes):
        fd, mid = _i32(-1), _u64(0)
        _check(lib().psx_mcx_create(int(device), int(n_devices), int(nbytes),
                                    ctypes.byref(fd), ctypes.byref(mid)))
        return cls(mid.value, device, fd.value)

    @classmethod
    def import_fd(cls, device, n_devices, nbytes, fd):
        mid = _u64(0)
        _check(lib().psx_mcx_import(int(device), int(n_devices), int(nbytes), int(fd),
                                    ctypes.byref(mid)))
        return cls(mid.value, device)

    def add_device(self):
        _check(lib().psx_mcx_add_device(self.id))

    def bind(self):
        uc, mc, size = _vp(0), _vp(0), _u64(0)
        _check(lib().psx_mcx_bind(self.id, ctypes.byref(uc), ctypes.byref(mc),
                                  ctypes.byref(size)))
        return uc.value, mc.value, size.value

    def destroy(self):
        if self.id:
            _check(lib().psx_mcx_destroy(self.id))
            self.id = 0


class Batch(object):
    """A fixed sequence of ops replayed with fresh sequence numbers: one ABI
    crossing per PS round (psx_batch)."""

    def __init__(self, ops):
        """ops: list of dicts with the psx_op field names (stream: torch stream,
        raw pointer or None)."""
        self.array = (Op * len(ops))()
        self.seq_slots = []
        for i, spec in enumerate(ops):
            o = self.array[i]
            for k, v in spec.items():
                if k == "stream":
                    v = _stream_ptr(v)
                elif k == "uses_seq":
                    continue
                setattr(o, k, v)
            if spec.get("uses_seq", True):
                self.seq_slots.append(i)
        self.n = len(ops)
        self._failed = _i32(-1)

    def run(self, seq):
        for i in self.seq_slots:
            self.array[i].seq = seq
        rc = lib().psx_batch(self.array, self.n, ctypes.byref(self._failed))
        if rc != 0:
            raise RuntimeError("psx batch op %d failed (%d): %s"
                               % (self._failed.value, rc, last_error()))


def copy(device, dst_ptr, src_ptr, nbytes, stream=None):
    _check(lib().psx_copy(int(device), dst_ptr, src_ptr, int(nbytes), _stream_ptr(stream)))
