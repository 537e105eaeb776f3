"""ctypes binding of libcnnacc.so (include/cnnacc.h).  Loading never falls back to a CPU path."""
import ctypes
import os
import subprocess

_DIR = os.path.dirname(os.path.abspath(__file__))
# CNNACC_LIB_PATH: load another build of the same library instead (the -DCNNACC_TRACE build of tools/trace_run.py)
LIB_PATH = os.environ.get("CNNACC_LIB_PATH") or os.path.join(_DIR, "libcnnacc.so")
CSRC = os.path.join(_DIR, "csrc")

OK, ERR_TIMEOUT, ERR_ARG, ERR_CUDA, ERR_STATE = 0, -1, -2, -3, -4
FLAG_DEVICE_PTRS, FLAG_DIRECT, FLAG_KEEP_MAPS, FLAG_CLS_GIVEN, FLAG_BBOX_UPSAMPLED, FLAG_LOGITS = 0x1, 0x2, 0x4, 0x8, 0x10, 0x20
FLAG_TWO_KERNELS = 0x40
FLAG_CLASS_AGNOSTIC = 0x80
FLAG_RECTS = 0x100
MERGE_MAX_DET, MERGE_MAX_PER_FRAME = 1024, 16384
PYRAMID_MAX_LEVELS = 16
MAX_PENDING = 8

# every symbol include/cnnacc.h declares: name -> (restype, argtypes)
_c = ctypes
_H = _c.c_void_p
SYMBOLS = {
    "cnnacc_create": (_c.c_int, [_c.c_int, _c.POINTER(_H)]),
    "cnnacc_destroy": (_c.c_int, [_H]),
    "cnnacc_set_stream": (_c.c_int, [_H, _c.c_void_p]),
    "cnnacc_last_error": (_c.c_char_p, [_H]),
    "cnnacc_launch_count": (_c.c_int64, [_H]),
    "cnnacc_load_weights": (_c.c_int, [_H, _c.c_void_p, _c.c_size_t]),
    "cnnacc_set_shifts": (_c.c_int, [_H, _c.c_int, _c.c_int, _c.c_int]),
    "cnnacc_get_shifts": (_c.c_int, [_H, _c.POINTER(_c.c_int)]),
    "cnnacc_set_accumulator_bits": (_c.c_int, [_H, _c.c_int]),
    "cnnacc_get_accumulator_bits": (_c.c_int, [_H]),
    "cnnacc_pack_weights_host": (_c.c_int, [_c.c_void_p, _c.c_size_t, _c.c_void_p, _c.c_void_p, _c.c_void_p]),
    "cnnacc_pdl_chain_host": (_c.c_int, [_c.c_int, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_int, _c.c_void_p]),
    "cnnacc_chunk_plan_host": (_c.c_int, [_c.c_int64, _c.c_int, _c.c_int, _c.c_int, _c.c_void_p, _c.c_int]),
    "cnnacc_tile_plan_host": (_c.c_int, [_c.c_int, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_int]),
    "cnnacc_run_batch": (_c.c_int, [_H, _c.c_void_p, _c.c_int64, _c.c_int, _c.c_int, _c.c_void_p, _c.c_uint32]),
    "cnnacc_run_batch_async": (_c.c_int, [_H, _c.c_void_p, _c.c_int64, _c.c_int, _c.c_int, _c.c_void_p, _c.c_uint32,
                                          _c.POINTER(_c.c_int64)]),
    "cnnacc_wait_batch": (_c.c_int, [_H, _c.c_int64]),
    "cnnacc_load_image": (_c.c_int, [_H, _c.c_void_p, _c.c_size_t]),
    "cnnacc_start": (_c.c_int, [_H]),
    "cnnacc_status": (_c.c_int, [_H]),
    "cnnacc_wait": (_c.c_int, [_H, _c.c_int]),
    "cnnacc_read_features": (_c.c_int, [_H, _c.c_void_p, _c.c_int, _c.c_int]),
    "cnnacc_read_feature_map": (_c.c_int, [_H, _c.c_int, _c.c_int, _c.c_void_p]),
    "cnnacc_infer_one": (_c.c_int, [_H, _c.c_void_p, _c.c_void_p, _c.POINTER(_c.c_float), _c.POINTER(_c.c_float)]),
    "cnnacc_load_classifier": (_c.c_int, [_H, _c.c_void_p, _c.c_void_p, _c.c_int]),
    "cnnacc_classify_batch": (_c.c_int, [_H, _c.c_void_p, _c.c_int64, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_uint32]),
    "cnnacc_infer_batch": (_c.c_int, [_H, _c.c_void_p, _c.c_int64, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_uint32]),
    "cnnacc_pool_features": (_c.c_int, [_H, _c.c_void_p, _c.c_int64, _c.c_void_p, _c.c_uint32]),
    "cnnacc_cam_bbox_batch": (_c.c_int, [_H, _c.c_void_p, _c.c_int64, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_uint32]),
    "cnnacc_preprocess_bgr": (_c.c_int, [_H, _c.c_void_p, _c.c_int64, _c.c_int, _c.c_int, _c.c_void_p, _c.c_uint32]),
    "cnnacc_detect_frames": (_c.c_int, [_H, _c.c_void_p, _c.c_int64, _c.c_int, _c.c_int, _c.c_void_p, _c.c_void_p, _c.c_void_p,
                                        _c.c_void_p, _c.c_uint32]),
    "cnnacc_preprocess_regions": (_c.c_int, [_H, _c.c_void_p, _c.c_int64, _c.c_int, _c.c_int, _c.c_void_p, _c.c_int64,
                                             _c.c_void_p, _c.c_uint32]),
    "cnnacc_detect_regions": (_c.c_int, [_H, _c.c_void_p, _c.c_int64, _c.c_int, _c.c_int, _c.c_void_p, _c.c_int64, _c.c_void_p,
                                         _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_uint32]),
    "cnnacc_detect_objects": (_c.c_int, [_H, _c.c_void_p, _c.c_int64, _c.c_int, _c.c_int, _c.c_void_p, _c.c_int64, _c.c_float,
                                         _c.c_float, _c.c_int] + [_c.c_void_p] * 5 + [_c.c_uint32]),
    "cnnacc_merge_regions": (_c.c_int, [_H, _c.c_void_p, _c.c_int64, _c.c_int64, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_float,
                                        _c.c_float, _c.c_int] + [_c.c_void_p] * 5 + [_c.c_uint32]),
    "cnnacc_merge_regions_host": (_c.c_int, [_c.c_void_p, _c.c_int64, _c.c_int64, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_float,
                                             _c.c_float, _c.c_int] + [_c.c_void_p] * 5 + [_c.c_uint32]),
    "cnnacc_scan_frames": (_c.c_int, [_H, _c.c_void_p, _c.c_int64, _c.c_int, _c.c_int, _c.c_int, _c.c_void_p, _c.c_void_p,
                                      _c.c_void_p, _c.c_uint32]),
    "cnnacc_scan_objects": (_c.c_int, [_H, _c.c_void_p, _c.c_int64, _c.c_int, _c.c_int, _c.c_int, _c.c_float, _c.c_float,
                                       _c.c_int] + [_c.c_void_p] * 5 + [_c.c_uint32]),
    "cnnacc_preprocess_pyramid": (_c.c_int, [_H, _c.c_void_p, _c.c_int64, _c.c_int, _c.c_int, _c.c_void_p, _c.c_int, _c.c_void_p,
                                             _c.c_uint32]),
    "cnnacc_scan_pyramid": (_c.c_int, [_H, _c.c_void_p, _c.c_int64, _c.c_int, _c.c_int, _c.c_void_p, _c.c_int, _c.c_int,
                                       _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_uint32]),
    "cnnacc_scan_pyramid_objects": (_c.c_int, [_H, _c.c_void_p, _c.c_int64, _c.c_int, _c.c_int, _c.c_void_p, _c.c_int, _c.c_int,
                                               _c.c_float, _c.c_float, _c.c_int] + [_c.c_void_p] * 5 + [_c.c_uint32]),
    "cnnacc_pyramid_windows_host": (_c.c_int, [_c.c_int, _c.c_int, _c.c_void_p, _c.c_int, _c.c_int, _c.c_void_p, _c.c_int64]),
    "cnnacc_region_plan_host": (_c.c_int, [_c.c_void_p, _c.c_int64, _c.c_int64, _c.c_int, _c.c_int, _c.c_void_p, _c.c_int]),
    "cnnacc_rect_plan_host": (_c.c_int, [_c.c_void_p, _c.c_int64, _c.c_int64, _c.c_int, _c.c_int, _c.c_void_p, _c.c_int]),
    "cnnacc_area_tab_host": (_c.c_int, [_c.c_int, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_int]),
    "cnnacc_image_to_gray128": (_c.c_int, [_H, _c.c_void_p, _c.c_int64, _c.c_int, _c.c_int, _c.c_int, _c.c_void_p, _c.c_uint32]),
    "cnnacc_run_batch_sharded": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_void_p, _c.c_int64, _c.c_int, _c.c_int, _c.c_void_p,
                                            _c.c_uint32, _c.POINTER(_c.c_int)]),
    "cnnacc_infer_batch_sharded": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_void_p, _c.c_int64, _c.c_void_p, _c.c_void_p,
                                              _c.c_void_p, _c.c_uint32, _c.POINTER(_c.c_int)]),
    "cnnacc_detect_frames_sharded": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_void_p, _c.c_int64, _c.c_int, _c.c_int, _c.c_void_p,
                                                _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_uint32, _c.POINTER(_c.c_int)]),
    "cnnacc_shard_plan_host": (_c.c_int, [_c.c_int64, _c.c_int, _c.c_int64, _c.c_void_p, _c.c_int]),
    "cnnacc_alloc_host": (_c.c_int, [_c.c_size_t, _c.POINTER(_c.c_void_p)]),
    "cnnacc_free_host": (_c.c_int, [_c.c_void_p]),
    "cnnacc_register_host": (_c.c_int, [_c.c_void_p, _c.c_size_t]),
    "cnnacc_unregister_host": (_c.c_int, [_c.c_void_p]),
    "cnnacc_probe_int8_peak": (_c.c_int, [_H, _c.c_double, _c.POINTER(_c.c_double), _c.POINTER(_c.c_double)]),
    "cnnacc_timer_start": (_c.c_int, [_H]),
    "cnnacc_timer_stop": (_c.c_int, [_H, _c.POINTER(_c.c_float)]),
    "cnnacc_synchronize": (_c.c_int, [_H]),
    # same symbol and ctypes convention as the reference (realtime_detect.py:389-391)
    "cnn_infer": (_c.c_int, [_c.c_void_p] * 4),
}

_lib = None


def build(force=False):
    """Compile libcnnacc.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", CSRC] + (["-B"] if force else [])
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"building libcnnacc.so failed:\n{r.stdout}\n{r.stderr}")
    return LIB_PATH


def load():
    """Load the C-ABI library; raise (never fall back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)            # AttributeError if the header and the library drift apart
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def check(rc, handle=None, prefix=""):
    """Map C status codes to the reference's Python exceptions (SURVEY.md 8b); `prefix` goes in front of the error text."""
    if rc == OK:
        return
    msg = load().cnnacc_last_error(handle)
    msg = prefix + (msg.decode() if msg else "")
    if rc == ERR_TIMEOUT:
        raise TimeoutError(msg or "timed out")
    if rc == ERR_ARG:
        raise ValueError(msg or "bad argument")
    raise RuntimeError(f"cnnacc error {rc}: {msg}")
