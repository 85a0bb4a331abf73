"""ctypes binding of libdct_b200.so (the C ABI declared in include/dct_b200.h).

There is no CPU fallback: if the shared library is missing it is built from
csrc/ with nvcc (sm_100a), and if that is impossible the import fails loudly.
"""
import ctypes as C
import os
import subprocess
import threading

_PKG = os.path.dirname(os.path.abspath(__file__))
# DCT_B200_LIB: developer override (A/B of two builds on the same box); the product always loads the in-tree library
_SO = os.environ.get("DCT_B200_LIB") or os.path.join(_PKG, "libdct_b200.so")
_CSRC = os.path.join(_PKG, "csrc")

OK = 0
ERR_UNSUPPORTED = -2
IN_PROBS, IN_LOGITS = 0, 1
COUNTS_ACCUMULATE, COUNTS_OVERWRITE = 0, 1
ABI_VERSION = 2
FLAG_SIMPLEX, FLAG_LABEL, FLAG_PRED, FLAG_ONEHOT, NUM_FLAGS = 0, 1, 2, 3, 4
MAX_VIEWS, MAX_CLASSES = 8, 64
MAX_PEERS, PUB_ROW_WORDS, PUB_MAX_VALUES, IPC_HANDLE_BYTES = 8, 16, 8, 64

_p, _i, _i64, _f = C.c_void_p, C.c_int, C.c_int64, C.c_float


class PeerPub(C.Structure):
    """``dct_peer_pub`` of include/dct_b200.h (host struct; device pointers inside)."""
    _fields_ = [("src", C.c_void_p), ("seq", C.c_void_p), ("mailbox_table", C.c_void_p), ("n", C.c_int32),
                ("rank", C.c_int32), ("world", C.c_int32), ("nslots", C.c_int32)]


# name -> argtypes (restype is int unless listed in _RESTYPES); must match include/dct_b200.h
_SIGNATURES = {
    "dct_abi_version": [],
    "dct_error_string": [_i],
    "dct_last_cuda_error": [],
    "dct_device_check": [_i],
    "dct_workspace_bytes": [],
    "dct_jsd_fwd_f32": [_p, _i, _i, _i64, _i64, _i, _p, _p, _p, _p, _p],
    "dct_jsd_bwd_f32": [_p, _i, _i, _i64, _i64, _i, _p, _p, _f, _p, _p],
    "dct_jsd_fwdbwd_f32": [_p, _i, _i, _i64, _i64, _i, _f, _p, _p, _p, _p, _p, _i, _p, _p, _p],
    "dct_jsd_fwdbwd_pub_f32": [_p, _i, _i, _i64, _i64, _i, _f, _p, _p, _p, _p, _p, _i, _p, _p, _p, _p],
    "dct_jsd_vat_kl_fwdbwd_f32": [_p, _i, _i, _i64, _i64, _f, _p, _p, _p, _p, _i, _p, _f, _p, _p, _p, _p, _p, _p],
    "dct_scale_if_not_one_f32": [_p, _i64, _p, _p],
    "dct_scale_if_not_one_bf16": [_p, _i64, _p, _p],
    "dct_kl_fwd_f32": [_p, _p, _i, _i64, _i64, _f, _p, _p, _p, _p, _p],
    "dct_kl_bwd_f32": [_p, _p, _i, _i64, _i64, _f, _p, _p, _f, _p, _p, _p],
    "dct_kl_logit_f32": [_p, _p, _i, _i64, _i64, _p, _p, _i, _p, _p, _f, _p, _p, _p, _p],
    "dct_kl_from_logits_fwdbwd_f32": [_p, _p, _i, _i64, _i64, _f, _f, _p, _p, _p, _p, _p, _p],
    "dct_kl_div_fwd_f32": [_p, _p, _i, _i64, _i64, _f, _p, _p, _p, _p, _p],
    "dct_kl_div_bwd_f32": [_p, _p, _i, _i64, _i64, _f, _p, _p, _f, _p, _p, _p],
    "dct_entropy_fwd_f32": [_p, _i, _i64, _i64, _p, _p, _p, _p, _p],
    "dct_entropy_bwd_f32": [_p, _i, _i64, _i64, _p, _p, _f, _p, _p],
    "dct_softmax_fwd_f32": [_p, _i, _i64, _i64, _p, _p],
    "dct_softmax_bwd_f32": [_p, _p, _i, _i64, _i64, _p, _p],
    "dct_l2_normalize_f32": [_p, _p, _i64, _i64, _i, _f, _p, _p, _p, _p],
    "dct_fgsm_f32": [_p, _p, _f, _p, _p, _i64, _p],
    "dct_dice_counts_f32": [_p, _p, _i, _i64, _i64, _p, _i, _p, _p],
    "dct_dice_from_counts_f32": [_p, _i64, _i, _i, _p, _p],
    "dct_confusion_f32": [_p, _p, _i, _i64, _i64, _p, _p],
    "dct_confusion_labels_i64": [_p, _p, _i64, _i, _p, _p, _p],
    "dct_label_hist_i64": [_p, _i64, _i, _i64, _p, _p],
    "dct_ce_fwd_f32": [_p, _p, _i, _i64, _i64, _p, _i64, _p, _p, _p, _p, _p],
    "dct_ce_bwd_f32": [_p, _p, _i, _i64, _i64, _p, _i64, _p, _p, _f, _p, _p, _p],
    "dct_ce_fwdbwd_f32": [_p, _p, _i, _i64, _i64, _p, _i64, _p, _f, _p, _p, _p, _p, _p, _p, _p],
    "dct_ce_fwdbwd_conf_f32": [_p, _p, _i, _i64, _i64, _p, _i64, _p, _f, _p, _p, _p, _p, _p, _p, _p],
    "dct_classmap_f32": [_p, _i, _i64, _i64, _i, _p, _p, _p, _p, _p],
    "dct_onehot_from_labels_i64": [_p, _i, _i64, _i64, _p, _p, _p],
    "dct_onehot_dice_counts_i32": [_p, _p, _i, _i64, _i64, _p, _p, _p],
    "dct_vote_f32": [_p, _i, _i, _i64, _i64, _i, _p, _p, _p, _p],
    "dct_hausdorff_scratch_bytes": [_i, _i64, _i64, _i64, _i],
    "dct_hausdorff_i64": [_p, _p, _i, _i64, _i64, _i64, _i, _p, _p, _p, _p, _p],
    "dct_surface_distance_scratch_bytes": [_i, _i64, _i64, _i64, _i],
    "dct_surface_distances_i64": [_p, _p, _i, _i64, _i64, _i64, _i, _p, _p, _p, _p, _p],
    "dct_surface_dice_scratch_bytes": [_i, _i64, _i64, _i64, _i],
    "dct_surface_dice_i64": [_p, _p, _i, _i64, _i64, _i64, _i, _p, _p, _p, _p, _p, _p, _p],
    "dct_distance_map_scratch_bytes": [_i, _i, _i64, _i64, _i64, _i, _i],
    "dct_distance_map_i64": [_p, _i, _i, _i64, _i64, _i64, _i, _p, _i, _p, _p, _p, _p],
    "dct_components_scratch_bytes": [_i, _i64, _i64, _i64, _i],
    "dct_components_i64": [_p, _i, _i64, _i64, _i64, _i, _i, _p, _p, _p, _p, _p, _p],
    "dct_boundary_iou_scratch_bytes": [_i, _i64, _i64, _i64],
    "dct_boundary_iou_i64": [_p, _p, _i, _i64, _i64, _i64, _i64, _i64, _p, _p, _p, _p, _p],
    "dct_jsd_fwdbwd_bf16": [_p, _i, _i, _i64, _i64, _f, _p, _p, _p, _p, _p, _i, _p, _p, _p],
    "dct_kl_logit_bf16": [_p, _p, _i, _i64, _i64, _p, _p, _i, _p, _p, _f, _p, _p, _p, _p],
    "dct_kl_from_logits_fwdbwd_bf16": [_p, _p, _i, _i64, _i64, _f, _f, _p, _p, _p, _p, _p, _p],
    "dct_ce_fwdbwd_bf16": [_p, _p, _i, _i64, _i64, _p, _i64, _p, _f, _p, _p, _p, _p, _p, _p, _p],
    "dct_dev_trace_begin": [_p, _i, _i],
    "dct_dev_trace_end": [],
    "dct_dev_tile_image": [_i, _i],
    "dct_peer_pub_bytes": [],
    "dct_mailbox_create": [C.c_size_t, _p, _p],
    "dct_mailbox_open": [_p, _p],
    "dct_mailbox_close": [_p, _i],
    "dct_exchange_publish": [_p, _p],
    "dct_kl_from_logits_fwdbwd_pub_f32": [_p, _p, _i, _i64, _i64, _f, _f, _p, _p, _p, _p, _p, _p, _p],
}
_RESTYPES = {"dct_error_string": C.c_char_p, "dct_last_cuda_error": C.c_char_p, "dct_workspace_bytes": C.c_size_t,
             "dct_peer_pub_bytes": C.c_size_t, "dct_hausdorff_scratch_bytes": C.c_size_t,
             "dct_surface_distance_scratch_bytes": C.c_size_t, "dct_components_scratch_bytes": C.c_size_t,
             "dct_surface_dice_scratch_bytes": C.c_size_t, "dct_distance_map_scratch_bytes": C.c_size_t,
             "dct_boundary_iou_scratch_bytes": C.c_size_t}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None
_lock = threading.Lock()


class DctError(RuntimeError):
    pass


def library_path() -> str:
    return _SO


def build(force: bool = False, jobs: int = 8) -> str:
    """Compile csrc/*.cu for sm_100a into libdct_b200.so (in-tree, next to this file)."""
    cmd = ["make", "-C", _CSRC, f"-j{jobs}"] + (["-B"] if force else [])
    subprocess.check_call(cmd, stdout=subprocess.DEVNULL)
    return _SO


def lib():
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(_SO):
                    try:
                        build()
                    except Exception as e:  # no nvcc / no make: nothing to run on
                        raise ImportError(
                            f"{_SO} is missing and could not be built ({e}); "
                            "run `python -c 'import __graft_entry__ as g; g.build()'` on a box with nvcc. "
                            "There is no CPU fallback.") from e
                h = C.CDLL(_SO)
                for name, argtypes in _SIGNATURES.items():
                    fn = getattr(h, name)  # AttributeError == ABI mismatch: fail loudly
                    fn.argtypes = argtypes
                    fn.restype = _RESTYPES.get(name, C.c_int)
                if h.dct_abi_version() != ABI_VERSION:
                    raise ImportError("libdct_b200.so ABI version mismatch; rebuild with build(force=True)")
                _lib = h
    return _lib


def check(rc: int, what: str) -> None:
    if rc != OK:
        h = lib()
        msg = h.dct_error_string(rc).decode()
        if rc == -4:
            msg += ": " + h.dct_last_cuda_error().decode()
        raise DctError(f"{what} failed: {msg} (code {rc})")


def ptr_array(tensors):
    """HOST array of device pointers (`const float* const*` in the ABI)."""
    return (C.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])
