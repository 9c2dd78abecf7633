"""rife-ncnn-vulkan_b200 -- host-side mirror of the reference's `class RIFE` (/root/reference/src/rife.h:11-52)
over the C ABI of librife_b200.so (include/rife_b200.h).  Python is used here only as the test / bench host;
the drop-in host code for src/main.cpp is the C++ shim in host/ (same ABI).

The directory name is not an importable identifier; load it with `__graft_entry__.load_package()`.
There is no CPU fallback: constructing RIFE without the built CUDA library raises.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# RIFE_B200_LIB: an alternative build of the same library (A/B timing of compile-time switches); the default is the in-tree build
LIB_PATH = os.environ.get("RIFE_B200_LIB") or os.path.join(_HERE, "lib", "librife_b200.so")

ERRORS = {0: "ok", -1: "bad argument", -2: "CUDA device error", -3: "model error", -4: "process before load", -5: "internal error"}

_lib = None


def lib():
    """dlopen librife_b200.so once and declare the prototypes of include/rife_b200.h."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("librife_b200.so is not built (%s): run `python -c 'import __graft_entry__ as g; g.build()'`; "
                           "there is no CPU fallback" % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    vp, ci, cf = ctypes.c_void_p, ctypes.c_int, ctypes.c_float
    L.rife_b200_device_count.restype = ci
    L.rife_b200_create.argtypes = [ctypes.POINTER(vp), ci, ci, ci, ci, ci, ci, ci]
    L.rife_b200_load.argtypes = [vp, ctypes.c_char_p]
    L.rife_b200_load_w.argtypes = [vp, ctypes.c_wchar_p]
    L.rife_b200_forget_frames.argtypes = [vp]
    L.rife_b200_stage_report.argtypes = [vp, ctypes.c_char_p, ctypes.c_size_t]
    L.rife_b200_process.argtypes = [vp, vp, vp, ci, ci, cf, vp]
    L.rife_b200_process_device.argtypes = [vp, vp, vp, ci, ci, cf, vp]
    L.rife_b200_process_batch.argtypes = [vp, ci, ctypes.POINTER(vp), ctypes.POINTER(vp), ci, ci, ctypes.POINTER(cf), ctypes.POINTER(vp)]
    L.rife_b200_process_batch_device.argtypes = L.rife_b200_process_batch.argtypes
    L.rife_b200_get_option.argtypes = [vp, ctypes.c_char_p, ctypes.POINTER(ci)]
    L.rife_b200_set_option.argtypes = [vp, ctypes.c_char_p, ci]
    L.rife_b200_weights_size.argtypes = [vp, ctypes.POINTER(ctypes.c_size_t)]
    L.rife_b200_weights_export.argtypes = [vp, vp, ctypes.c_size_t]
    L.rife_b200_load_packed.argtypes = [vp, vp, ctypes.c_size_t]
    L.rife_b200_set_stream.argtypes = [vp, vp]
    L.rife_b200_bench_conv.argtypes = [ci, vp, ci, ci, ci, ci, ci, ci]
    L.rife_b200_bench_conv_batched.argtypes = [ci, vp, ci, ci, ci, ci, ci, ci, ci]
    L.rife_b200_selftest_conv.argtypes = [ci, ci, ci, ci, ci, ci, ci, ci, vp, vp, vp, vp, cf, vp, vp]
    L.rife_b200_debug_parse_model.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.POINTER(ci), ctypes.POINTER(ci), ctypes.POINTER(ctypes.c_ulonglong), ctypes.c_char_p, ci]
    L.rife_b200_debug_pack_weights.argtypes = [ci, ci, ci, ci, ci, ci, vp, vp, ctypes.c_size_t]
    L.rife_b200_debug_hbm.argtypes = [ci, vp, ci, ci, ci, ci, ci, vp, vp, vp]
    L.rife_b200_launch_count.restype = ctypes.c_ulonglong
    L.rife_b200_h2d_bytes.restype = ctypes.c_ulonglong
    L.rife_b200_d2h_bytes.restype = ctypes.c_ulonglong
    L.rife_b200_last_error.argtypes = [vp]
    L.rife_b200_last_error.restype = ctypes.c_char_p
    L.rife_b200_destroy.argtypes = [vp]
    L.rife_b200_destroy.restype = None
    _lib = L
    return L


EXPORTS = ["rife_b200_device_count", "rife_b200_create", "rife_b200_load", "rife_b200_load_w", "rife_b200_forget_frames", "rife_b200_stage_report", "rife_b200_process", "rife_b200_process_device",
           "rife_b200_process_batch", "rife_b200_process_batch_device", "rife_b200_set_option", "rife_b200_get_option", "rife_b200_weights_size", "rife_b200_weights_export",
           "rife_b200_load_packed", "rife_b200_selftest_conv", "rife_b200_set_stream", "rife_b200_bench_conv", "rife_b200_bench_conv_batched",
           "rife_b200_debug_conv_timeline", "rife_b200_debug_hbm", "rife_b200_debug_pack_weights", "rife_b200_debug_parse_model",
           "rife_b200_launch_count", "rife_b200_h2d_bytes", "rife_b200_d2h_bytes", "rife_b200_last_error", "rife_b200_destroy"]


def family_flags(model_name):
    """(rife_v2, rife_v4) from the model directory name, as src/main.cpp:658-683 sniffs them."""
    n = os.path.basename(os.path.normpath(model_name))
    if n.startswith("rife-v4"):
        return False, True
    if n.startswith("rife-v2") or n.startswith("rife-v3"):
        return True, False
    return False, False


class RifeError(RuntimeError):
    pass


class RIFE:
    """Same constructor arguments and methods as the reference class (rife.h:14-24)."""

    def __init__(self, gpuid, tta_mode=False, tta_temporal_mode=False, uhd_mode=False, num_threads=1, rife_v2=False, rife_v4=False):
        self._h = ctypes.c_void_p()
        self._lib = lib()
        r = self._lib.rife_b200_create(ctypes.byref(self._h), int(gpuid), int(tta_mode), int(tta_temporal_mode), int(uhd_mode),
                                       int(num_threads), int(rife_v2), int(rife_v4))
        if r != 0:
            self._h = ctypes.c_void_p()
            raise RifeError("rife_b200_create(gpuid=%d): %s" % (gpuid, ERRORS.get(r, r)))

    def _check(self, r, what):
        if r != 0:
            msg = self._lib.rife_b200_last_error(self._h)
            raise RifeError("%s: %s (%s)" % (what, ERRORS.get(r, r), msg.decode() if msg else ""))

    def load(self, modeldir):
        self._check(self._lib.rife_b200_load(self._h, os.fsencode(modeldir)), "load(%s)" % modeldir)
        return 0

    def load_w(self, modeldir):
        self._check(self._lib.rife_b200_load_w(self._h, str(modeldir)), "load_w(%s)" % modeldir)
        return 0

    def stage_report(self):
        """{lane: {"batches": n, "stages": [(name, us_per_batch, launches_per_batch), ...]}} (option "ktime" = 1)."""
        buf = ctypes.create_string_buffer(16384)
        self._check(self._lib.rife_b200_stage_report(self._h, buf, len(buf)), "stage_report")
        out, cur = {}, None
        for line in buf.value.decode().splitlines():
            f = line.split("\t")
            if f[0] == "lane":
                cur = out.setdefault(int(f[1]), {"batches": 0, "stages": []})
            elif f[0] == "batches" and cur is not None:
                cur["batches"] = int(f[1])
            elif cur is not None and len(f) == 3:
                cur["stages"].append((f[0], float(f[1]), int(f[2])))
        return out

    def forget_frames(self):
        self._check(self._lib.rife_b200_forget_frames(self._h), "forget_frames")

    def set_option(self, key, value):
        self._check(self._lib.rife_b200_set_option(self._h, key.encode(), int(value)), "set_option(%s)" % key)

    def get_option(self, key):
        v = ctypes.c_int()
        self._check(self._lib.rife_b200_get_option(self._h, key.encode(), ctypes.byref(v)), "get_option(%s)" % key)
        return v.value

    def process(self, in0image, in1image, timestep, outimage=None):
        """in0image/in1image: uint8 arrays (h, w, 3), C-contiguous host memory. Returns outimage."""
        a = np.ascontiguousarray(in0image, dtype=np.uint8)
        b = np.ascontiguousarray(in1image, dtype=np.uint8)
        if a.ndim != 3 or a.shape[2] != 3 or a.shape != b.shape:
            raise RifeError("process: frames must both be (h, w, 3) uint8")
        if outimage is None:
            outimage = np.empty_like(a)
        if outimage.shape != a.shape or outimage.dtype != np.uint8 or not outimage.flags.c_contiguous:
            raise RifeError("process: outimage must be a C-contiguous (h, w, 3) uint8 array")
        h, w = a.shape[:2]
        self._check(self._lib.rife_b200_process(self._h, a.ctypes.data, b.ctypes.data, w, h, float(timestep), outimage.ctypes.data), "process")
        return outimage

    def process_ptr(self, in0_ptr, in1_ptr, w, h, timestep, out_ptr, device=False):
        """Raw-pointer form (host pointers, or device pointers with device=True)."""
        fn = self._lib.rife_b200_process_device if device else self._lib.rife_b200_process
        self._check(fn(self._h, in0_ptr, in1_ptr, int(w), int(h), float(timestep), out_ptr), "process_ptr")

    def process_batch_ptr(self, in0_ptrs, in1_ptrs, w, h, timesteps, out_ptrs, device=False):
        n = len(in0_ptrs)
        VP = ctypes.c_void_p * n
        ts = (ctypes.c_float * n)(*[float(t) for t in timesteps])
        fn = self._lib.rife_b200_process_batch_device if device else self._lib.rife_b200_process_batch
        self._check(fn(self._h, n, VP(*in0_ptrs), VP(*in1_ptrs), int(w), int(h), ts, VP(*out_ptrs)), "process_batch")

    def set_stream(self, cuda_stream_ptr):
        self._check(self._lib.rife_b200_set_stream(self._h, ctypes.c_void_p(cuda_stream_ptr)), "set_stream")

    def export_weights(self):
        n = ctypes.c_size_t()
        self._check(self._lib.rife_b200_weights_size(self._h, ctypes.byref(n)), "weights_size")
        buf = np.empty(n.value, np.uint8)
        self._check(self._lib.rife_b200_weights_export(self._h, buf.ctypes.data, n.value), "weights_export")
        return buf

    def load_packed(self, blob):
        blob = np.ascontiguousarray(blob, dtype=np.uint8)
        self._check(self._lib.rife_b200_load_packed(self._h, blob.ctypes.data, blob.size), "load_packed")

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self._lib.rife_b200_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def bench_conv(cuda_stream_ptr, cin, cout, h, w, split, iters, gpuid=0, batch=1):
    rc = lib().rife_b200_bench_conv_batched(gpuid, ctypes.c_void_p(cuda_stream_ptr), cin, cout, h, w, int(split), int(batch), iters)
    if rc != 0:
        raise RifeError("bench_conv failed: %d" % rc)


def debug_conv_timeline(cin, cout, h, w, split=True, max_ctas=148, gpuid=0, batch=1, skip_tiles=0):
    buf = np.zeros((max_ctas, 64), np.uint64)
    L = lib()
    L.rife_b200_debug_conv_timeline.argtypes = [ctypes.c_int] * 6 + [ctypes.c_void_p, ctypes.c_int]
    rc = L.rife_b200_debug_conv_timeline(gpuid, cin, cout, h, w, int(bool(split)) | (int(batch) << 8) | (int(skip_tiles) << 16), buf.ctypes.data, max_ctas)
    if rc != 0:
        raise RifeError("debug_conv_timeline failed: %d" % rc)
    return buf


HBM_KERNELS = {"preproc": 0, "postproc": 1, "flow_tta_avg": 2, "warp": 3, "temporal_merge_v2": 4, "temporal_merge_v1": 5}


def debug_hbm(which, w, h, c, a=None, b=None, out=None, iters=0, cuda_stream_ptr=None, gpuid=0):
    """One of the HBM-side kernels on host arrays (iters = 0) or `iters` launches on synthetic device data (timing)."""
    rc = lib().rife_b200_debug_hbm(gpuid, ctypes.c_void_p(cuda_stream_ptr or 0), HBM_KERNELS[which], int(w), int(h), int(c), int(iters),
                                   None if a is None else a.ctypes.data, None if b is None else b.ctypes.data, None if out is None else out.ctypes.data)
    if rc != 0:
        raise RifeError("debug_hbm(%s) failed: %d" % (which, rc))
    return out


def launch_count():
    return int(lib().rife_b200_launch_count())


def copy_bytes():
    return int(lib().rife_b200_h2d_bytes()), int(lib().rife_b200_d2h_bytes())


def device_count():
    return int(lib().rife_b200_device_count())


def selftest_conv(mode, x, weight, bias, res=None, slope=0.2, split=True, ps=2, gpuid=0):
    """Runs one layer through the tcgen05 kernel and the fp32 CUDA-core kernel; returns (out_tc, out_ref)."""
    x = np.ascontiguousarray(x, np.float32)
    weight = np.ascontiguousarray(weight, np.float32)
    bias = np.ascontiguousarray(bias, np.float32)
    cin, h, w = x.shape
    cout = weight.shape[0]
    if mode == 3:
        assert ps == 2 and cout == 24
    if mode in (0, 4):
        oshape = (cout, h, w)
    elif mode == 2:
        oshape = (cout, h // 2, w // 2)
    else:
        oshape = (cout // (ps * ps), 2 * h * ps, 2 * w * ps)
    o1 = np.zeros(oshape, np.float32)
    o2 = np.zeros(oshape, np.float32)
    r = None if res is None else np.ascontiguousarray(res, np.float32)
    rc = lib().rife_b200_selftest_conv(gpuid, mode, cin, cout, h, w, int(split), ps, x.ctypes.data, weight.ctypes.data, bias.ctypes.data,
                                       None if r is None else r.ctypes.data, float(slope), o1.ctypes.data, o2.ctypes.data)
    if rc != 0:
        raise RifeError("selftest_conv failed: %d" % rc)
    return o1, o2
