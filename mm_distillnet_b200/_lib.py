"""ctypes binding of libmmd_b200.so (the C ABI declared in include/mmd.h).

There is no CPU fallback: if the shared library is missing or a call fails, this raises.
"""
import ctypes as C
import os
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(_HERE, "libmmd_b200.so")
SOURCES = ("api.cu", "mta.cu", "prep.cu", "bifpn_fwd.cu", "bifpn_fwd_tc.cu", "bifpn_fwd_v4.cu", "bifpn_proj_tma.cu", "bifpn_bwd.cu",
           "bifpn_bwd_tc.cu", "bifpn_bwd_v4.cu", "heads.cu", "focal.cu", "pseudo.cu", "adam.cu", "bifpn_run.cu")

MMD_F32, MMD_BF16 = 0, 1
MMD_NHWC, MMD_NCHW = 0, 1
MTA_MAX_LEVELS, MTA_MAX_TEACHERS = 8, 4
STATS_REPLICAS = 1   # MMD_STATS_REPLICAS

IN_SAME, IN_UP2, IN_POOL = 0, 1, 2
CONS_SAME, CONS_UP2, CONS_POOL = 0, 1, 2
OP_NODE_FWD, OP_PROJ_FWD, OP_BNAPPLY, OP_NODE_BWD, OP_PROJ_BWD, OP_PULL, OP_SLOT, OP_POOLFUSE = 1, 2, 3, 4, 5, 6, 7, 8
OP_ACT_FWD, OP_ACT_BWD, OP_HEAD_GATHER, OP_HEAD_SCATTER, OP_COPY = 9, 10, 11, 12, 13


class MtaArgs(C.Structure):
    _fields_ = [
        ("n_levels", C.c_int32), ("n_teachers", C.c_int32), ("B", C.c_int32), ("C", C.c_int32),
        ("dtype", C.c_int32), ("layout", C.c_int32), ("T", C.c_float), ("p", C.c_float),
        ("separate", C.c_int32), ("pad_", C.c_int32),
        ("H", C.c_int32 * MTA_MAX_LEVELS), ("W", C.c_int32 * MTA_MAX_LEVELS),
        ("fs", C.c_void_p * MTA_MAX_LEVELS),
        ("ft", (C.c_void_p * MTA_MAX_LEVELS) * MTA_MAX_TEACHERS),
        ("att_ws", C.c_void_p), ("ga_ws", C.c_void_p), ("loss_b", C.c_void_p), ("loss", C.c_void_p),
    ]


class FocalArgs(C.Structure):
    _fields_ = [("B", C.c_int32), ("N", C.c_int32), ("K", C.c_int32), ("M", C.c_int32), ("dtype", C.c_int32), ("pad_", C.c_int32),
                ("alpha", C.c_float), ("gamma", C.c_float), ("cls", C.c_void_p), ("reg", C.c_void_p), ("anchors", C.c_void_p),
                ("boxes", C.c_void_p), ("acc", C.c_void_p), ("assign", C.c_void_p), ("loss", C.c_void_p)]


FOCAL_MAX_BOXES = 2048
PL_MAX_TEACHERS, PL_MAX_CAP, PL_MAX_IGNORE = 8, 8192, 8


class PseudoArgs(C.Structure):
    _fields_ = [("B", C.c_int32), ("N", C.c_int32), ("K", C.c_int32), ("T", C.c_int32), ("dtype", C.c_int32), ("cap", C.c_int32),
                ("max_rows", C.c_int32), ("max_labels", C.c_int32), ("raw_rows", C.c_int32), ("n_ignore", C.c_int32),
                ("ignore", C.c_int32 * PL_MAX_IGNORE), ("merge01", C.c_int32), ("pad_", C.c_int32), ("conf_threshold", C.c_float), ("image_size", C.c_float),
                ("nms_threshold", C.c_double), ("merge_iou", C.c_double),
                ("cls", C.c_void_p * PL_MAX_TEACHERS), ("reg", C.c_void_p * PL_MAX_TEACHERS), ("anchors", C.c_void_p),
                ("label_of", C.c_void_p), ("workspace", C.c_void_p), ("teacher_rows", C.c_void_p),
                ("teacher_counts", C.c_void_p), ("labels", C.c_void_p), ("counts", C.c_void_p)]


class AdamArgs(C.Structure):
    _fields_ = [("n_chunks", C.c_int32), ("decoupled_weight_decay", C.c_int32), ("n_elements", C.c_int64),
                ("lr", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double), ("eps", C.c_double), ("weight_decay", C.c_double),
                ("chunks", C.c_void_p), ("offsets", C.c_void_p), ("params", C.c_void_p), ("grad", C.c_void_p),
                ("exp_avg", C.c_void_p), ("exp_avg_sq", C.c_void_p), ("step", C.c_void_p)]


class Ref(C.Structure):
    _fields_ = [("base", C.c_int32), ("pad_", C.c_int32), ("off", C.c_int64)]


class Tensor(C.Structure):
    _fields_ = [("data", Ref), ("bn", Ref), ("H", C.c_int32), ("W", C.c_int32), ("C", C.c_int32), ("pad_", C.c_int32)]


class Cons(C.Structure):
    _fields_ = [("du", Tensor), ("mode", C.c_int32), ("fw_k", C.c_int32), ("fw_n", C.c_int32), ("fw_eps", C.c_float),
                ("fw", C.c_void_p), ("slot", Ref), ("pidx", Ref)]


class Op(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("train", C.c_int32), ("n_in", C.c_int32), ("swish", C.c_int32),
        ("inp", Tensor * 3), ("mode", C.c_int32 * 3), ("fw_eps", C.c_float),
        ("fw", C.c_void_p),
        ("dw_w", C.c_void_p), ("pw_w", C.c_void_p), ("pw_b", C.c_void_p), ("bn_w", C.c_void_p), ("bn_b", C.c_void_p),
        ("bn_rm", C.c_void_p), ("bn_rv", C.c_void_p), ("bn_nbt", C.c_void_p),
        ("in_bn_w", C.c_void_p * 3), ("in_bn_b", C.c_void_p * 3),
        ("Cin", C.c_int32), ("accumulate_dx", C.c_int32), ("bn_eps", C.c_float), ("bn_momentum", C.c_float),
        ("out", Tensor),
        ("save_d", Ref), ("pidx", Ref * 3), ("packed", Ref), ("stats", Ref), ("counter", Ref),
        ("n_cons", C.c_int32), ("pad_", C.c_int32),
        ("cons", Cons * 3),
        ("du", Ref), ("dd", Ref), ("in_slot", Ref * 3), ("dx", Ref),
        ("g_dw", Ref), ("g_pw", Ref), ("g_pb", Ref), ("g_bn_w", Ref), ("g_bn_b", Ref), ("g_fw", Ref),
        ("fw_n", C.c_int32), ("fw_idx", C.c_int32 * 3),
        ("aux", Ref), ("praw", Ref),
        ("head_K", C.c_int32), ("head_tot", C.c_int32), ("head_off", C.c_int32), ("head_act", C.c_int32),
        ("copy_src", C.c_void_p), ("copy_dst", C.c_void_p), ("copy_n", C.c_int64),
        ("frozen_bn", C.c_int32), ("pad2_", C.c_int32),
    ]


NULL_REF = (-1, 0, 0)


NVCC_FLAGS = ("-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC")


def nvcc_command(out_path=LIB_PATH, extra=()):
    """The single-command equivalent of build() (documentation / manual builds)."""
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    return ["nvcc", *NVCC_FLAGS, "-shared", "-o", out_path, *extra, *srcs]


HASH_PATH = LIB_PATH + ".srchash"


def _deps():
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    deps = srcs + sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h")))
    deps.append(os.path.join(os.path.dirname(_HERE), "include", "mmd.h"))
    return deps


def source_hash():
    """SHA-256 over every source / header the library is built from (content, not mtimes: the snapshot that carries the
    tree to the GPU box does not have to preserve timestamps)."""
    import hashlib
    h = hashlib.sha256()
    for d in _deps():
        h.update(os.path.basename(d).encode())
        with open(d, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def is_stale():
    """True when libmmd_b200.so is missing or was built from other sources than the ones in the tree."""
    if not os.path.exists(LIB_PATH) or not os.path.exists(HASH_PATH):
        return True
    with open(HASH_PATH) as f:
        return f.read().strip() != source_hash()


def build(force=False, verbose=False):
    """Compile the CUDA sources into mm_distillnet_b200/libmmd_b200.so (in-tree, sm_100a only).  Skipped when the library
    on disk was built from exactly the current sources (content hash in libmmd_b200.so.srchash)."""
    if not force and not is_stale():
        return LIB_PATH
    digest = source_hash()
    # one nvcc process per translation unit (the v4 kernels are template-heavy), then one link
    import concurrent.futures
    import tempfile
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    tmp = tempfile.mkdtemp(prefix="mmd_build_")
    objs = [os.path.join(tmp, os.path.splitext(os.path.basename(s))[0] + ".o") for s in srcs]

    def cc(pair):
        src, obj = pair
        cmd = ["nvcc", *NVCC_FLAGS, "-c", "-o", obj, src]
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        return subprocess.run(cmd, capture_output=True, text=True)

    try:
        with concurrent.futures.ThreadPoolExecutor(max_workers=min(len(srcs), os.cpu_count() or 1)) as ex:
            results = list(ex.map(cc, zip(srcs, objs)))
        bad = [r for r in results if r.returncode != 0]
        if bad:
            raise RuntimeError("nvcc failed:\n" + "\n".join(r.stdout + r.stderr for r in bad))
        cmd = ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB_PATH, *objs]
        if verbose:
            print(" ".join(cmd), file=sys.stderr)
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc link failed:\n" + r.stdout + r.stderr)
    finally:
        import shutil
        shutil.rmtree(tmp, ignore_errors=True)
    with open(HASH_PATH, "w") as f:
        f.write(digest + "\n")
    return LIB_PATH


_lib = None


def lib():
    """Load the shared library, (re)building it first when it is missing or was built from other sources than the tree
    holds (content hash, see is_stale()).  Raises if unavailable: there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    build()
    L = C.CDLL(LIB_PATH)
    L.mmd_version.restype = C.c_int
    L.mmd_last_error.restype = C.c_char_p
    L.mmd_launch_count.restype = C.c_ulonglong
    L.mmd_sizeof_op.restype = C.c_size_t
    L.mmd_sizeof_mta_args.restype = C.c_size_t
    L.mmd_mta_fwd.restype = C.c_int
    L.mmd_mta_fwd.argtypes = [C.POINTER(MtaArgs), C.c_void_p]
    L.mmd_mta_bwd.restype = C.c_int
    L.mmd_mta_bwd.argtypes = [C.POINTER(MtaArgs), C.c_void_p, C.POINTER(C.c_void_p), C.c_void_p]
    L.mmd_focal_fwd.restype = C.c_int
    L.mmd_focal_fwd.argtypes = [C.POINTER(FocalArgs), C.c_void_p]
    L.mmd_focal_bwd.restype = C.c_int
    L.mmd_focal_bwd.argtypes = [C.POINTER(FocalArgs), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.mmd_sizeof_focal_args.restype = C.c_size_t
    L.mmd_pseudo_labels.restype = C.c_int
    L.mmd_pseudo_labels.argtypes = [C.POINTER(PseudoArgs), C.c_void_p]
    L.mmd_pseudo_workspace_bytes.restype = C.c_size_t
    L.mmd_pseudo_workspace_bytes.argtypes = [C.POINTER(PseudoArgs)]
    L.mmd_sizeof_pseudo_args.restype = C.c_size_t
    L.mmd_adam_step.restype = C.c_int
    L.mmd_adam_step.argtypes = [C.POINTER(AdamArgs), C.c_void_p]
    L.mmd_sizeof_adam_args.restype = C.c_size_t
    L.mmd_bifpn_run.restype = C.c_int
    L.mmd_bifpn_run.argtypes = [C.POINTER(Op), C.c_int32, C.POINTER(C.c_void_p), C.c_int32,
                                C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
    L.mmd_bifpn_run_multi.restype = C.c_int
    L.mmd_bifpn_run_multi.argtypes = [C.POINTER(C.POINTER(Op)), C.POINTER(C.c_int32), C.POINTER(C.POINTER(C.c_void_p)),
                                      C.POINTER(C.c_int32), C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
    L.mmd_bifpn_prep.restype = C.c_int
    L.mmd_bifpn_prep.argtypes = [C.POINTER(Op), C.c_int32, C.POINTER(C.c_void_p), C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
    L.mmd_packed_bytes.restype = C.c_size_t
    L.mmd_packed_bytes.argtypes = [C.c_int32, C.c_int32, C.c_int32]
    L.mmd_set_option.restype = C.c_int
    L.mmd_set_option.argtypes = [C.c_char_p, C.c_int32]
    L.mmd_prof_enable.argtypes = [C.c_int]
    L.mmd_prof_enable.restype = None
    L.mmd_prof_num_kinds.restype = C.c_int
    L.mmd_prof_kind_name.restype = C.c_char_p
    L.mmd_prof_kind_name.argtypes = [C.c_int]
    L.mmd_prof_collect.restype = C.c_int
    L.mmd_prof_collect.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_longlong), C.POINTER(C.c_double)]
    if L.mmd_sizeof_focal_args() != C.sizeof(FocalArgs):
        raise RuntimeError("libmmd_b200.so / _lib.py struct mismatch: MmdFocalArgs %d vs %d" % (L.mmd_sizeof_focal_args(), C.sizeof(FocalArgs)))
    if L.mmd_sizeof_adam_args() != C.sizeof(AdamArgs):
        raise RuntimeError("libmmd_b200.so / _lib.py struct mismatch: MmdAdamArgs %d vs %d" % (L.mmd_sizeof_adam_args(), C.sizeof(AdamArgs)))
    if L.mmd_sizeof_pseudo_args() != C.sizeof(PseudoArgs):
        raise RuntimeError("libmmd_b200.so / _lib.py struct mismatch: MmdPseudoArgs %d vs %d" % (L.mmd_sizeof_pseudo_args(), C.sizeof(PseudoArgs)))
    if L.mmd_sizeof_op() != C.sizeof(Op) or L.mmd_sizeof_mta_args() != C.sizeof(MtaArgs):
        raise RuntimeError("libmmd_b200.so struct layout mismatch: Op %d vs %d, MtaArgs %d vs %d" % (
            L.mmd_sizeof_op(), C.sizeof(Op), L.mmd_sizeof_mta_args(), C.sizeof(MtaArgs)))
    _lib = L
    return L


def check(rc, what):
    if rc != 0:
        msg = lib().mmd_last_error()
        raise RuntimeError("%s failed (code %d): %s" % (what, rc, msg.decode() if msg else "?"))


def set_option(name, value):
    """Runtime switch of the library (include/mmd.h: mmd_set_option), e.g. set_option("chain_fwd", 1)."""
    check(lib().mmd_set_option(name.encode(), int(value)), "mmd_set_option")


def launch_count():
    return int(lib().mmd_launch_count())


def prof_enable(on):
    lib().mmd_prof_enable(1 if on else 0)


def prof_collect():
    """{kernel kind: {"ms": total ms, "launches": n, "algo_bytes": total algorithmic bytes}} since the last collect."""
    L = lib()
    n = L.mmd_prof_num_kinds()
    ms, cnt, by = (C.c_double * n)(), (C.c_longlong * n)(), (C.c_double * n)()
    check(L.mmd_prof_collect(ms, cnt, by), "mmd_prof_collect")
    return {L.mmd_prof_kind_name(i).decode(): {"ms": ms[i], "launches": int(cnt[i]), "algo_bytes": by[i]}
            for i in range(n) if cnt[i] > 0}


EXPORTS = ("mmd_version", "mmd_last_error", "mmd_launch_count", "mmd_set_option", "mmd_mta_fwd", "mmd_mta_bwd", "mmd_focal_fwd",
           "mmd_focal_bwd", "mmd_sizeof_focal_args", "mmd_pseudo_labels", "mmd_pseudo_workspace_bytes", "mmd_sizeof_pseudo_args", "mmd_adam_step", "mmd_sizeof_adam_args", "mmd_bifpn_run", "mmd_bifpn_run_multi",
           "mmd_bifpn_prep", "mmd_packed_bytes",
           "mmd_sizeof_op", "mmd_sizeof_mta_args", "mmd_prof_enable", "mmd_prof_num_kinds", "mmd_prof_kind_name",
           "mmd_prof_collect")
