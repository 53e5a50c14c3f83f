"""ctypes binding of libalm_ocr.so (include/alm_ocr.h).

There is no fallback: if the shared library is missing or cannot be loaded this module raises, and
every adapter built on it fails loudly.  Build it with ``python -c "import __graft_entry__ as g; g.build()"``
or ``make`` at the repo root.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# ALM_OCR_LIB: developer knob for A/B runs of two builds of the same library on one GPU box (never a different backend)
LIB_PATH = os.environ.get('ALM_OCR_LIB') or os.path.join(_HERE, 'libalm_ocr.so')

ALM_OK = 0
MODEL_OMNI_SPOT, MODEL_OMNI_KIE, MODEL_MGPSTR = 1, 2, 3
DT_F32, DT_F16, DT_BF16, DT_I64 = 0, 1, 2, 3


class TensorDesc(C.Structure):
    _fields_ = [('name', C.c_char_p), ('data', C.c_void_p), ('dtype', C.c_int), ('ndim', C.c_int),
                ('shape', C.c_int64 * 4)]


class DecodeCfg(C.Structure):
    _fields_ = [(n, C.c_int) for n in (
        'num_bins', 'pt_eos', 'poly_eos', 'rec_eos', 'pt_sos', 'poly_sos', 'rec_sos', 'recog_pad',
        'pt_seq_length', 'rec_length', 'poly_length', 'vie_categories', 'max_instances')]


class AlmError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f'libalm_ocr error {code}: {msg}')
        self.code = code


_lib = None

# name -> (restype, argtypes); this table is also what tests/test_abi.py checks against include/alm_ocr.h
SIGNATURES = {
    'alm_init': (C.c_int, [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]),
    'alm_free': (None, [C.c_void_p]),
    'alm_last_error': (C.c_char_p, [C.c_void_p]),
    'alm_version': (C.c_char_p, []),
    'alm_set_option': (C.c_int, [C.c_void_p, C.c_char_p, C.c_long]),
    'alm_launch_count': (C.c_long, [C.c_void_p, C.c_int]),
    'alm_synchronize': (C.c_int, [C.c_void_p]),
    'alm_profile_read': (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_long)]),
    'alm_trace_read': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int)]),
    'alm_bench_graph_floor': (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    'alm_bench_gemm_ex': (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                    C.POINTER(C.c_float), C.c_void_p]),
    'alm_bench_gemm': (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    'alm_load_weights': (C.c_int, [C.c_void_p, C.c_int, C.POINTER(TensorDesc), C.c_int]),
    'alm_share_weights': (C.c_int, [C.c_void_p, C.c_void_p]),
    'alm_stream_wait': (C.c_int, [C.c_void_p, C.c_void_p]),
    'alm_stream_release': (C.c_int, [C.c_void_p, C.c_void_p]),
    'alm_comm_unique_id': (C.c_int, [C.c_void_p]),
    'alm_comm_init': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    'alm_comm_attach': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    'alm_broadcast_weights': (C.c_int, [C.c_void_p, C.c_int]),
    'alm_gather_sequences': (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    'alm_omni_encode': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]),
    'alm_omni_get_feature': (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]),
    'alm_omni_get_memory': (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]),
    'alm_omni_memory_shape': (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    'alm_omni_decode': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(DecodeCfg), C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_void_p]),
    'alm_omni_decode_kie': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(DecodeCfg), C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'alm_omni_decode_points': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(DecodeCfg), C.c_void_p, C.c_void_p,
                                         C.c_void_p]),
    'alm_omni_decode_prompted': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(DecodeCfg), C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'alm_omni_decode_points_prompted': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(DecodeCfg),
                                                  C.c_void_p, C.c_void_p, C.c_void_p]),
    'alm_omni_decode_logits': (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    'alm_omni_vocab': (C.c_int, [C.c_void_p]),
    'alm_omni_last_timing': (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    'alm_mgpstr_forward': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p]),
    'alm_mgpstr_info': (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int),
                                  C.POINTER(C.c_int), C.c_void_p]),
    'alm_op_linear': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                C.c_int, C.c_int]),
    'alm_op_attention': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]),
    'alm_op_layernorm': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_long,
                                   C.c_int]),
    'alm_op_window_attention': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                          C.c_int, C.c_int, C.c_int]),
    'alm_op_gemv': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_long, C.c_void_p, C.c_void_p, C.c_void_p,
                              C.c_long, C.c_void_p, C.c_long, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                              C.c_float, C.c_void_p, C.c_int]),
    'alm_op_self_attn_step': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                        C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    'alm_op_cross_attention': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                         C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    'alm_op_head_select': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(DecodeCfg),
                                     C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    # test-time image pipeline
    'alm_pre_omni_plan': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_int),
                                    C.POINTER(C.c_int)]),
    'alm_pre_coeffs': (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.c_void_p, C.c_void_p, C.c_size_t]),
    'alm_pre_omni_pages': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                     C.c_void_p]),
    'alm_pre_mgp_crops': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    # host-only post-processing (no context, no GPU)
    'alm_post_last_error': (C.c_char_p, []),
    'alm_post_omni_spotting': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.c_int, C.c_char_p, C.c_long, C.c_long, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_size_t]),
    'alm_post_omni_json': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                     C.c_int, C.c_char_p, C.c_long, C.c_long, C.c_char_p, C.c_void_p, C.c_size_t,
                                     C.POINTER(C.c_size_t)]),
    'alm_post_omni_kie_json': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                         C.c_int, C.c_int, C.c_int, C.c_char_p, C.POINTER(C.c_char_p), C.c_int, C.c_int,
                                         C.c_long, C.c_long, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]),
    'alm_post_mgp_fuse': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_char_p), C.c_int,
                                    C.POINTER(C.c_char_p), C.c_int, C.POINTER(C.c_char_p), C.c_int, C.c_void_p, C.c_void_p,
                                    C.c_size_t, C.c_void_p, C.c_void_p]),
}


def load():
    """dlopen libalm_ocr.so and bind every symbol of include/alm_ocr.h."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f'{LIB_PATH} not found: build it first (make / __graft_entry__.build()); '
                          'there is no CPU or PyTorch fallback')
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class Context:
    """One alm_ctx: one GPU, one stream, not thread-safe."""

    def __init__(self, device: int = 0, stream: int | None = None):
        self.lib = load()
        h = C.c_void_p()
        rc = self.lib.alm_init(int(device), C.c_void_p(stream) if stream else None, C.byref(h))
        if rc != ALM_OK:
            raise AlmError(rc, 'alm_init failed (no sm_100a CUDA device? this library has no fallback path)')
        self.h = h
        self.device = device
        self.comm_rank, self.comm_world = 0, 1
        # ALM_OCR_OPTIONS="name=value,...": developer knob, applied to every new context (A/B runs of kernel variants
        # through the unchanged tests / bench; the options are the documented alm_set_option ones)
        for kv in filter(None, os.environ.get('ALM_OCR_OPTIONS', '').split(',')):
            k, v = kv.split('=')
            self.set_option(k.strip(), int(v))

    def check(self, rc):
        if rc != ALM_OK:
            raise AlmError(rc, self.lib.alm_last_error(self.h).decode())

    def synchronize(self):
        self.check(self.lib.alm_synchronize(self.h))

    def set_option(self, key: str, value: int):
        self.check(self.lib.alm_set_option(self.h, key.encode(), int(value)))

    def profile_read(self):
        ms, fl, n = C.c_double(), C.c_double(), C.c_long()
        self.check(self.lib.alm_profile_read(self.h, C.byref(ms), C.byref(fl), C.byref(n)))
        return ms.value, fl.value, n.value

    def trace_read(self, max_records=200000):
        import numpy as np
        buf = np.zeros((max_records, 6), dtype=np.uint64)
        n = C.c_int()
        self.check(self.lib.alm_trace_read(self.h, buf.ctypes.data, max_records, C.byref(n)))
        return buf[:n.value]

    def omni_last_timing(self):
        e, p, r = C.c_float(), C.c_float(), C.c_float()
        self.check(self.lib.alm_omni_last_timing(self.h, C.byref(e), C.byref(p), C.byref(r)))
        return {'encode_ms': e.value, 'pt_loop_ms': p.value, 'poly_rec_loops_ms': r.value}

    def bench_gemm_ex(self, M, N, K, batch=1, split_out=0, act=0, iters=10, detail=False):
        import numpy as np
        ms = C.c_float()
        buf = np.zeros((64, 6), dtype=np.uint64)
        self.check(self.lib.alm_bench_gemm_ex(self.h, M, N, K, batch, split_out, act, iters, C.byref(ms),
                                              buf.ctypes.data if detail else None))
        return ms.value, buf

    def bench_gemm(self, M, N, K, iters=20) -> float:
        ms = C.c_float()
        self.check(self.lib.alm_bench_gemm(self.h, M, N, K, iters, C.byref(ms)))
        return ms.value

    def launch_count(self, reset=False) -> int:
        return int(self.lib.alm_launch_count(self.h, 1 if reset else 0))

    def load_state_dict(self, kind: int, state_dict):
        """state_dict: name -> torch.Tensor (any device) in the reference checkpoint layout."""
        import torch
        descs = (TensorDesc * len(state_dict))()
        keep = []
        for i, (k, v) in enumerate(state_dict.items()):
            t = v.detach().to('cpu').contiguous()
            if t.dtype == torch.float32:
                dt = DT_F32
            elif t.dtype == torch.float16:
                dt = DT_F16
            elif t.dtype == torch.bfloat16:
                dt = DT_BF16
            elif t.dtype == torch.int64:
                dt = DT_I64
            else:
                t = t.float()
                dt = DT_F32
            keep.append(t)
            assert t.dim() <= 4, k
            descs[i].name = k.encode()
            descs[i].data = t.data_ptr()
            descs[i].dtype = dt
            descs[i].ndim = t.dim()
            for j, s in enumerate(t.shape):
                descs[i].shape[j] = s
        self.check(self.lib.alm_load_weights(self.h, kind, descs, len(state_dict)))

    def load_placeholders(self, kind: int, meta):
        """Shape-only load (data == NULL) of [(name, shape, dtype_code), ...]: lays the weights out exactly like
        `load_state_dict` would; the values arrive through `broadcast_weights` (non-root ranks of a multi-GPU job)."""
        descs = (TensorDesc * len(meta))()
        for i, (k, shape, dt) in enumerate(meta):
            assert len(shape) <= 4, k
            descs[i].name = k.encode()
            descs[i].data = None
            descs[i].dtype = dt
            descs[i].ndim = len(shape)
            for j, s in enumerate(shape):
                descs[i].shape[j] = s
        self.check(self.lib.alm_load_weights(self.h, kind, descs, len(meta)))

    @staticmethod
    def state_dict_meta(state_dict):
        """[(name, shape, dtype_code)] of a reference state dict, as `load_placeholders` takes it."""
        import torch
        code = {torch.float32: DT_F32, torch.float16: DT_F16, torch.bfloat16: DT_BF16, torch.int64: DT_I64}
        return [(k, tuple(v.shape), code.get(v.dtype, DT_F32)) for k, v in state_dict.items()]

    def share_weights(self, owner: 'Context'):
        """Serve the weights resident in `owner` (same GPU) from this context too: no copy (alm_share_weights)."""
        self.check(self.lib.alm_share_weights(self.h, owner.h))
        self._weights_owner = owner  # keeps the Python object alive; the device slabs are ref-counted in the library

    def wait_stream(self, cuda_stream: int):
        """The context's stream waits for everything enqueued so far on `cuda_stream` (device inputs written there)."""
        self.check(self.lib.alm_stream_wait(self.h, C.c_void_p(cuda_stream)))

    def release_stream(self, cuda_stream: int):
        """`cuda_stream` waits for everything this context has enqueued so far (device outputs read there)."""
        self.check(self.lib.alm_stream_release(self.h, C.c_void_p(cuda_stream)))

    def wait_torch(self, *tensors):
        """Order the context's stream after torch's current stream when any argument is a CUDA tensor."""
        import torch
        for t in tensors:
            if t is not None and t.is_cuda:
                self.wait_stream(torch.cuda.current_stream(t.device).cuda_stream)
                return

    # ---- multi-GPU (alm_comm_*): one weight broadcast, one gather per batch
    def comm_unique_id(self) -> bytes:
        buf = C.create_string_buffer(128)
        rc = self.lib.alm_comm_unique_id(buf)
        if rc != ALM_OK:
            raise AlmError(rc, 'alm_comm_unique_id failed (NCCL not loadable?)')
        return buf.raw

    def comm_init(self, uid: bytes, rank: int, world: int):
        assert len(uid) == 128
        self.check(self.lib.alm_comm_init(self.h, C.create_string_buffer(uid, 128), int(rank), int(world)))
        self.comm_rank, self.comm_world = int(rank), int(world)

    def broadcast_weights(self, root: int = 0):
        self.check(self.lib.alm_broadcast_weights(self.h, int(root)))

    def gather(self, send, world: int):
        """All-gather of one equal-size buffer per rank (numpy array in, [world, ...] numpy array out)."""
        import numpy as np
        send = np.ascontiguousarray(send)
        recv = np.empty((world,) + send.shape, dtype=send.dtype)
        self.check(self.lib.alm_gather_sequences(self.h, send.ctypes.data, send.nbytes, recv.ctypes.data))
        return recv

    def close(self):
        if getattr(self, 'h', None):
            self.lib.alm_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
