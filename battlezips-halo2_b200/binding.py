"""ctypes binding of libbzhalo2.so (include/bzhalo2.h).  Plain pointers and sizes only."""
import ctypes, os, re, subprocess
import numpy as np

FIELD_FP, FIELD_FQ = 0, 1
CURVE_VESTA, CURVE_PALLAS = 0, 1

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
_lib = None


class BzError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"bzhalo2 error {code}: {msg}")
        self.code = code


def lib_path():
    return os.environ.get("BZ_LIB") or os.path.join(_HERE, "lib", "libbzhalo2.so")       # BZ_LIB: A/B builds only


def header_path():
    return os.path.join(_ROOT, "include", "bzhalo2.h")


def build_library(verbose=False):
    """Compile every CUDA source for sm_100a in-tree (nvcc cross-compiles without a GPU)."""
    subprocess.run(["make", "-C", os.path.join(_HERE, "csrc"), "-j8"], check=True,
                   stdout=None if verbose else subprocess.DEVNULL)
    return lib_path()


def _declared_exports():
    """Every function name include/bzhalo2.h declares."""
    src = open(header_path()).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(bz_[a-z0-9_]+)\s*\(", src)))


EXPORTS = _declared_exports()


ALLGATHER_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_size_t)


def load_library():
    """dlopen the CUDA library; fails loudly when it has not been built (no fallback path exists)."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise BzError(-1, f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(the product has no CPU fallback)")
    lib = ctypes.CDLL(path)
    vp, u64, u32, i32 = ctypes.c_void_p, ctypes.c_uint64, ctypes.c_uint32, ctypes.c_int
    sigs = {
        "bz_ctx_create": (i32, [i32, vp, ctypes.POINTER(vp)]),
        "bz_ctx_destroy": (None, [vp]),
        "bz_last_error": (ctypes.c_char_p, [vp]),
        "bz_sync": (i32, [vp]),
        "bz_kernel_launches": (u64, [vp]),
        "bz_version": (ctypes.c_char_p, []),
        "bz_profile_enable": (i32, [vp, i32]),
        "bz_profile_read": (i32, [vp, i32, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(u64)]),
        "bz_profile_counter": (i32, [vp, i32, ctypes.POINTER(u64), i32]),
        "bz_imad_peak": (i32, [vp, ctypes.POINTER(ctypes.c_double)]),
        "bz_imad_wide_peak": (i32, [vp, ctypes.POINTER(ctypes.c_double)]),
        "bz_dfma_peak": (i32, [vp, i32, ctypes.POINTER(ctypes.c_double)]),
        "bz_dev_alloc": (i32, [vp, ctypes.c_size_t, ctypes.POINTER(vp)]),
        "bz_dev_free": (i32, [vp, vp]),
        "bz_h2d": (i32, [vp, vp, vp, ctypes.c_size_t]),
        "bz_d2h": (i32, [vp, vp, vp, ctypes.c_size_t]),
        "bz_field_op": (i32, [vp, i32, i32, vp, vp, vp, u64]),
        "bz_curve_op": (i32, [vp, i32, i32, vp, vp, vp, u64]),
        "bz_best_multiexp": (i32, [vp, i32, vp, vp, u64, vp]),
        "bz_msm_dev": (i32, [vp, i32, vp, vp, u64, vp, i32]),
        "bz_batch_normalize_dev": (i32, [vp, i32, vp, vp, u64]),
        "bz_point_sum_dev": (i32, [vp, i32, vp, u32, vp]),
        "bz_best_fft": (i32, [vp, i32, vp, vp, u32]),
        "bz_ntt_dev": (i32, [vp, i32, vp, vp, u32, i32, i32]),
        "bz_lagrange_to_coeff_dev": (i32, [vp, i32, vp, vp, u32, i32]),
        "bz_coeff_to_extended_dev": (i32, [vp, i32, vp, vp, u32, u32, i32]),
        "bz_extended_to_coeff_dev": (i32, [vp, i32, vp, vp, u32, i32]),
        "bz_lagrange_to_coeff": (i32, [vp, i32, vp, u32]),
        "bz_coeff_to_extended": (i32, [vp, i32, vp, vp, u32, u32]),
        "bz_extended_to_coeff": (i32, [vp, i32, vp, u32]),
        "bz_params_new": (i32, [vp, u32, i32, vp, vp, vp, vp]),
        "bz_points_compress": (i32, [vp, i32, vp, u64, vp]),
        "bz_points_decompress": (i32, [vp, i32, vp, u64, vp, vp]),
        "bz_hash_to_curve": (i32, [vp, i32, ctypes.c_char_p, vp, u32, u64, vp]),
        "bz_batch_invert_assigned": (i32, [vp, i32, vp, vp, vp, u64]),
        "bz_batch_invert_assigned_dev": (i32, [vp, i32, vp, vp, vp, u64]),
        "bz_perm_product": (i32, [vp, i32, u32, u32, ctypes.POINTER(vp), ctypes.POINTER(vp), vp, vp, vp, vp, vp]),
        "bz_lookup_permute": (i32, [vp, i32, u32, u32, vp, vp, vp, vp]),
        "bz_lookup_product": (i32, [vp, i32, u32, vp, vp, vp, vp, vp, vp, vp]),
        "bz_divide_by_vanishing": (i32, [vp, i32, u32, u32, vp]),
        "bz_pk_quotient": (i32, [vp, vp, vp, vp, vp, vp, vp, vp]),
        "bz_pk_num_poly_slots": (u32, [vp]),
        "bz_eval_many": (i32, [vp, i32, u64, u32, ctypes.POINTER(vp), vp, vp]),
        "bz_kate_div": (i32, [vp, i32, u64, vp, vp, vp]),
        "bz_axpy": (i32, [vp, i32, u64, vp, vp, vp]),
        "bz_ipa_begin": (i32, [vp, vp, vp, vp, ctypes.POINTER(vp)]),
        "bz_ipa_round": (i32, [vp, vp, vp, vp, vp, vp, vp]),
        "bz_ipa_fold": (i32, [vp, vp, vp, vp]),
        "bz_ipa_finish": (i32, [vp, vp, vp]),
        "bz_ipa_destroy": (None, [vp]),
        "bz_quotient_program": (i32, [vp, u32, vp, u32, ctypes.POINTER(u32), vp, u32, ctypes.POINTER(u32), ctypes.POINTER(u64)]),
        "bz_pk_quotient_generated": (i32, [vp, u32]),
        "bz_ctx_set_sharding": (i32, [vp, u32, u32, vp, vp, ctypes.c_size_t, ALLGATHER_FN, vp]),
    }
    declared_elsewhere = {"bz_params_create", "bz_params_destroy", "bz_params_commit", "bz_pk_create", "bz_pk_destroy",
                          "bz_pk_num_random", "bz_pk_proof_size", "bz_pk_quotient_muls", "bz_create_proofs", "bz_pk_create_from_assembly", "bz_pk_vk_commitments", "bz_verify_proofs", "bz_params_commit_batch_dev",
                          "bz_vk_create", "bz_vk_destroy", "bz_vk_proof_size", "bz_verify_proofs_vk"}     # bound in plonk/prover.py
    missing = [n for n in EXPORTS if n not in sigs and n not in declared_elsewhere]
    assert not missing, f"unbound C-ABI symbols: {missing}"
    for name, (res, args) in sigs.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def _np_ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


class DeviceBuffer:
    def __init__(self, ctx, nbytes):
        self.ctx, self.nbytes = ctx, nbytes
        p = ctypes.c_void_p()
        ctx._check(ctx.lib.bz_dev_alloc(ctx.h, nbytes, ctypes.byref(p)))
        self.ptr = p

    def upload(self, arr):
        arr = np.ascontiguousarray(arr)
        assert arr.nbytes <= self.nbytes
        self.ctx._check(self.ctx.lib.bz_h2d(self.ctx.h, self.ptr, _np_ptr(arr), arr.nbytes))
        return self

    def download(self, shape, dtype=np.uint64):
        out = np.empty(shape, dtype=dtype)
        assert out.nbytes <= self.nbytes
        self.ctx._check(self.ctx.lib.bz_d2h(self.ctx.h, _np_ptr(out), self.ptr, out.nbytes))
        return out

    def free(self):
        if self.ptr:
            self.ctx.lib.bz_dev_free(self.ctx.h, self.ptr)
            self.ptr = None


class Context:
    """One GPU + one CUDA stream.  stream: an int cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream) or None."""

    def __init__(self, device=0, stream=None):
        self.lib = load_library()
        h = ctypes.c_void_p()
        rc = self.lib.bz_ctx_create(device, ctypes.c_void_p(stream) if stream else None, ctypes.byref(h))
        if rc != 0:
            raise BzError(rc, "bz_ctx_create failed (no CUDA device / driver?) -- the product has no CPU fallback")
        self.h = h
        self.device = device
        self.stream_handle = stream

    def _check(self, rc):
        if rc != 0:
            raise BzError(rc, self.lib.bz_last_error(self.h).decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.bz_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_sharding(self, rank, world, group=None, capacity=1 << 16):
        """One large proof across `world` GPUs (bz_ctx_set_sharding): the exchange buffers are torch CUDA tensors and the
        all-gather is torch.distributed's (NCCL), issued on the stream this context was created on (torch's current stream is
        thread-local, and bz_create_proofs may be called from a worker thread)."""
        if world <= 1:
            self._check(self.lib.bz_ctx_set_sharding(self.h, 0, 1, None, None, 0, ALLGATHER_FN(0), None))
            self._shard = None
            return
        import torch
        import torch.distributed as dist
        assert self.stream_handle, "sharding needs a context created on a caller-owned (torch) stream"
        send = torch.zeros(capacity, dtype=torch.uint8, device=f"cuda:{self.device}")
        recv = torch.zeros(capacity * world, dtype=torch.uint8, device=f"cuda:{self.device}")
        stream = torch.cuda.ExternalStream(self.stream_handle, device=f"cuda:{self.device}")

        def exchange(_user, nbytes):
            try:
                with torch.cuda.stream(stream):
                    dist.all_gather_into_tensor(recv[: world * nbytes], send[:nbytes], group=group)
                return 0
            except Exception:      # noqa: BLE001  (reported through the C status code)
                return -1
        cb = ALLGATHER_FN(exchange)
        self._shard = (send, recv, cb)          # keep the buffers and the callback alive
        self._check(self.lib.bz_ctx_set_sharding(self.h, rank, world, ctypes.c_void_p(send.data_ptr()), ctypes.c_void_p(recv.data_ptr()),
                                                 capacity, cb, None))

    def sync(self):
        self._check(self.lib.bz_sync(self.h))

    def kernel_launches(self):
        return int(self.lib.bz_kernel_launches(self.h))

    PROF_TAGS = ["ntt_pass", "msm_digits", "msm_sort", "msm_bucket", "msm_reduce", "msm_combine", "fixed_msm",
                 "quotient", "scan", "eval", "poly", "ipa", "other"]

    def profile_enable(self, on=True):
        self._check(self.lib.bz_profile_enable(self.h, 1 if on else 0))

    def profile_read(self):
        """{tag: (total_ms, launches)} measured with CUDA events on this context's stream."""
        out = {}
        for i, name in enumerate(self.PROF_TAGS):
            ms, cnt = ctypes.c_double(), ctypes.c_uint64()
            self._check(self.lib.bz_profile_read(self.h, i, ctypes.byref(ms), ctypes.byref(cnt)))
            if cnt.value:
                out[name] = (ms.value, cnt.value)
        return out

    def profile_counter(self, which=0, reset=True):
        v = ctypes.c_uint64()
        self._check(self.lib.bz_profile_counter(self.h, which, ctypes.byref(v), 1 if reset else 0))
        return v.value

    def imad_peak(self):
        v = ctypes.c_double()
        self._check(self.lib.bz_imad_peak(self.h, ctypes.byref(v)))
        return v.value

    def dfma_peak(self, mixed=False):
        v = ctypes.c_double()
        self._check(self.lib.bz_dfma_peak(self.h, 1 if mixed else 0, ctypes.byref(v)))
        return v.value

    def imad_wide_peak(self):
        v = ctypes.c_double()
        self._check(self.lib.bz_imad_wide_peak(self.h, ctypes.byref(v)))
        return v.value

    def alloc(self, nbytes):
        return DeviceBuffer(self, nbytes)

    def to_device(self, arr):
        arr = np.ascontiguousarray(arr)
        return DeviceBuffer(self, max(arr.nbytes, 32)).upload(arr)
