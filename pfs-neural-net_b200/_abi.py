"""ctypes binding of libpfs_b200.so (include/pfs_b200.h).

This is the whole Python<->CUDA boundary: plain pointers and sizes, one argument struct per
module, the caller's CUDA stream.  The library is built in-tree by `build_library()` (called from
`__graft_entry__.build()`); importing this module never compiles anything.  There is NO CPU
fallback: if the shared library is missing, or a tensor is not a contiguous fp32 CUDA tensor, the
call raises.
"""
import ctypes as ct
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(CSRC, "libpfs_b200.so")
HEADER = os.path.join(os.path.dirname(_HERE), "include", "pfs_b200.h")

PFS_LAYOUT_DENSE = 0
PFS_LAYOUT_CSR = 1
PFS_TILE_EDGES = 256
ABI_VERSION = 9

_P = ct.c_void_p


def _fields(spec):
    out = []
    for ctype, names in spec:
        for n in names.split():
            out.append((n, ctype))
    return out


class TopologyStruct(ct.Structure):
    _fields_ = _fields([
        (ct.c_int32, "layout G F S T E"),
        (_P, "csr_rowptr csr_eid csr_src csr_tgt tile_fibre"),
        (ct.c_int32, "ntiles"),
        (_P, "csc_colptr csc_q"),
        (_P, "tile_q tile_slot split_fibre split_ptr"),     # ABI 7: split tiles
        (ct.c_int32, "nsplit nslots"),
    ])


class EdgeArgs(ct.Structure):
    _fields_ = _fields([
        (TopologyStruct, "topo"),
        (_P, "x_s x_t x_e u w1 b1 w2 b2 gamma beta running_mean running_var num_batches_tracked"),
        (ct.c_int32, "training normed"),
        (ct.c_float, "eps momentum"),
        (_P, "x_e_out bn_save g_out g_x_s g_x_t g_x_e g_u g_w1 g_b1 g_w2 g_b2 g_gamma g_beta workspace"),
        (ct.c_size_t, "workspace_bytes"),
        (_P, "stream"),
        (ct.c_int32, "defer_affine reserved0"),
        (_P, "table_s table_t"),
    ])


class SourceArgs(ct.Structure):
    _fields_ = _fields([
        (TopologyStruct, "topo"),
        (_P, "x_s x_t x_e u w1 b1 w2 b2 w3 b3 w4 b4 gamma beta running_mean running_var num_batches_tracked"),
        (ct.c_int32, "training normed"),
        (ct.c_float, "eps momentum"),
        (_P, "x_s_out moments hidden y_pre bn_save g_out g_x_e_add g_x_s g_x_t g_x_e g_u "
             "g_w1 g_b1 g_w2 g_b2 g_w3 g_b3 g_w4 g_b4 g_gamma g_beta workspace"),
        (ct.c_size_t, "workspace_bytes"),
        (_P, "stream"),
        (_P, "x_e_affine x_e_norm_out"),
    ])


class TargetArgs(ct.Structure):
    _fields_ = _fields([
        (TopologyStruct, "topo"),
        (_P, "x_s x_t x_e u w1 b1 w2 b2 w3 b3 w4 b4 gamma beta running_mean running_var num_batches_tracked"),
        (ct.c_int32, "training normed"),
        (ct.c_float, "eps momentum"),
        (_P, "x_t_out act_sum y_pre bn_save g_out g_x_e_add g_x_s g_x_t g_x_e g_u "
             "g_w1 g_b1 g_w2 g_b2 g_w3 g_b3 g_w4 g_b4 g_gamma g_beta workspace"),
        (ct.c_size_t, "workspace_bytes"),
        (_P, "stream"),
        (_P, "table_s"),
    ])


class GlobalArgs(ct.Structure):
    _fields_ = _fields([
        (ct.c_int32, "G F S T"),
        (_P, "x_s x_t u w1 b1 w2 b2 rms_weight"),
        (ct.c_int32, "normed"),
        (ct.c_float, "rms_eps"),
        (_P, "u_out g_out g_x_s g_x_t g_u g_w1 g_b1 g_w2 g_b2 g_rms_weight workspace"),
        (ct.c_size_t, "workspace_bytes"),
        (_P, "stream"),
    ])


class HeadArgs(ct.Structure):
    _fields_ = _fields([
        (TopologyStruct, "topo"),
        (_P, "x_e w1 b1 w2 b2"),
        (ct.c_float, "scale"),
        (_P, "class_hours edge_tgt time visits time_int g_time g_x_e g_w1 g_b1 g_w2 g_b2 workspace"),
        (ct.c_size_t, "workspace_bytes"),
        (_P, "stream"),
    ])


class WideGemmArgs(ct.Structure):
    _fields_ = [
        ("A", _P), ("lda", ct.c_int64), ("B", _P), ("ldb", ct.c_int64),
        ("M", ct.c_int32), ("N", ct.c_int32), ("K", ct.c_int32),
        ("bias", _P), ("bias_rowscale", _P),
        ("tab0", _P), ("idx0", _P), ("div0", ct.c_int32),
        ("tab1", _P), ("idx1", _P), ("mod1", ct.c_int32),
        ("mask", _P), ("ldmask", ct.c_int64),
        ("act", ct.c_int32),
        ("out_bf16", _P), ("ldc", ct.c_int64),
        ("out_f32", _P), ("ldf", ct.c_int64),
        ("stream", _P),
        ("A2", _P), ("lda2", ct.c_int64), ("K2", ct.c_int32), ("a2_mod", ct.c_int32),
        ("bias_rows", _P), ("bias_rows_div", ct.c_int32),
    ]


class LossArgs(ct.Structure):
    _fields_ = [("S", ct.c_int32), ("T", ct.c_int32), ("time", _P), ("noise", _P), ("hours", _P), ("counts", _P)] + \
        [(n, ct.c_float) for n in "total_time wutils wvar pclass pfiber sharpness noiselevel".split()] + \
        [(n, _P) for n in "galaxies time2 fibre_time n_prime class_mean class_coef scalars g_loss g_time workspace".split()] + \
        [("workspace_bytes", ct.c_size_t), ("stream", _P), ("sharpness_dev", _P)] + \
        [("G", ct.c_int32), ("class_tables", ct.c_int32)] + \
        [("S_total", ct.c_int32), ("world", ct.c_int32), ("shard_record", _P), ("shard_records", _P)]
# ABI 8 appended the graph dimension (G, class_tables), ABI 9 the fibre-sharded graph (S_total ... shard_records)


class WideSegments(ct.Structure):
    _fields_ = [("mode", ct.c_int32), ("nseg", ct.c_int32), ("S", ct.c_int32), ("T", ct.c_int32),
                ("ptr", _P), ("list", _P)]


# every symbol include/pfs_b200.h declares: name -> (restype, argtypes)
_I64, _I32 = ct.c_int64, ct.c_int32
SYMBOLS = {
    "pfs_abi_version": (ct.c_int, []),
    "pfs_last_error": (ct.c_char_p, []),
    "pfs_supports_fdim": (ct.c_int, [_I32]),
    "pfs_sizeof_topology": (ct.c_size_t, []),
    "pfs_sizeof_edge_args": (ct.c_size_t, []),
    "pfs_sizeof_source_args": (ct.c_size_t, []),
    "pfs_sizeof_target_args": (ct.c_size_t, []),
    "pfs_sizeof_global_args": (ct.c_size_t, []),
    "pfs_sizeof_head_args": (ct.c_size_t, []),
    "pfs_launch_count": (ct.c_longlong, []),
    "pfs_profile_enable": (ct.c_int, [ct.c_int]),
    "pfs_profile_report": (ct.c_int, [ct.c_char_p, ct.c_size_t]),
    "pfs_workspace_bytes": (ct.c_size_t, [ct.POINTER(TopologyStruct)]),
    "pfs_detect_dense": (ct.c_int, [_P, _I64, _I32, _I32, _P, _P]),
    "pfs_build_topology_temp_bytes": (ct.c_size_t, [_I64, _I32, _I32]),
    "pfs_build_topology": (ct.c_int, [_P, _I64, _I32, _I32] + [_P] * 9 + [_P, ct.c_size_t, _P]),
    "pfs_build_split_tiles": (ct.c_int, [_P, _I32] + [_P] * 6 + [_P]),
    "pfs_edge_fwd": (ct.c_int, [ct.POINTER(EdgeArgs)]),
    "pfs_edge_bwd": (ct.c_int, [ct.POINTER(EdgeArgs)]),
    "pfs_source_fwd": (ct.c_int, [ct.POINTER(SourceArgs)]),
    "pfs_source_bwd": (ct.c_int, [ct.POINTER(SourceArgs)]),
    "pfs_target_fwd": (ct.c_int, [ct.POINTER(TargetArgs)]),
    "pfs_target_bwd": (ct.c_int, [ct.POINTER(TargetArgs)]),
    "pfs_global_fwd": (ct.c_int, [ct.POINTER(GlobalArgs)]),
    "pfs_global_bwd": (ct.c_int, [ct.POINTER(GlobalArgs)]),
    "pfs_time_head_fwd": (ct.c_int, [ct.POINTER(HeadArgs)]),
    "pfs_time_head_bwd": (ct.c_int, [ct.POINTER(HeadArgs)]),
    # wide-feature path (bf16, tcgen05 GEMMs + HBM-bound row kernels)
    "pfs_sizeof_wide_gemm_args": (ct.c_size_t, []),
    "pfs_sizeof_wide_segments": (ct.c_size_t, []),
    "pfs_wide_gemm_nt": (ct.c_int, [ct.POINTER(WideGemmArgs)]),
    "pfs_wide_gemm_tn_workspace": (ct.c_size_t, [_I64, _I32, _I32]),
    "pfs_wide_gemm_tn": (ct.c_int, [_P, _I64, _P, _I64, _I64, _I32, _I32, _P, _I64, _I32, _P, ct.c_size_t, _P]),
    "pfs_wide_colstats_workspace": (ct.c_size_t, [_I64, _I32]),
    "pfs_wide_colstats": (ct.c_int, [_I32, _P, _I32, _I64, _P, _I32, _I64, _P, _P, _P, _I64, _I32, _P, _P, ct.c_size_t, _P]),
    "pfs_wide_rowmap": (ct.c_int, [_I32, _P, _I32, _I64, _P, _I32, _I64, _P, _P, _P, _P, _P, _I64, _I32, _P, _I64, _P]),
    "pfs_wide_segsum_workspace": (ct.c_size_t, [ct.POINTER(WideSegments), _I32]),
    "pfs_wide_segsum": (ct.c_int, [ct.POINTER(WideSegments), _P, _I32, _I64, _I32, _P, _P, _P, ct.c_size_t, _P]),
    "pfs_wide_moments_fwd": (ct.c_int, [ct.POINTER(WideSegments), _P, _I32, _I32, _P, _P]),
    "pfs_wide_source_hcat": (ct.c_int, [_P, _P, _I32, _I32, _P, _I64, _I32, _P]),
    "pfs_wide_split": (ct.c_int, [_P, _I64, _I64, _I32, _P, _I64, _P]),
    "pfs_wide_source_coef": (ct.c_int, [ct.POINTER(WideSegments), _P, _P, _I32, _I32, _P, _P, _P]),
    "pfs_wide_source_dm": (ct.c_int, [_P, _I32, _P, _P, _P, _I32, _I64, _I32, _P, _P]),
    "pfs_wide_source_dm_seg": (ct.c_int, [ct.POINTER(WideSegments), _P, _I32, _P, _P, _I32, _P, _P]),
    "pfs_wide_gather_mask": (ct.c_int, [_P, _P, _I32, _P, _I64, _I32, _P, _P]),
    "pfs_wide_head_fwd": (ct.c_int, [_P, _P, _P, ct.c_float, _I64, _I32, _P, _P, _I32, _P, _P, _P, _P, _P]),
    "pfs_wide_head_bwd": (ct.c_int, [_P, _P, _P, _P, ct.c_float, _I64, _I32, _P, _P, _P]),
    "pfs_wide_cast": (ct.c_int, [_P, _I32, _P, _I32, _I64, _P]),
    # training loss (reference src/train.py:21-80)
    "pfs_sizeof_loss_args": (ct.c_size_t, []),
    "pfs_loss_workspace_bytes": (ct.c_size_t, [_I32, _I32]),
    "pfs_loss_fwd": (ct.c_int, [ct.POINTER(LossArgs)]),
    "pfs_loss_bwd": (ct.c_int, [ct.POINTER(LossArgs)]),
    "pfs_loss_shard_fwd": (ct.c_int, [ct.POINTER(LossArgs)]),
    "pfs_loss_shard_merge": (ct.c_int, [ct.POINTER(LossArgs)]),
    "pfs_wide_transpose": (ct.c_int, [_P, _I32, _I32, _I64, _P, _P]),
}
_SIZEOF_CHECKS = {
    "pfs_sizeof_topology": TopologyStruct, "pfs_sizeof_edge_args": EdgeArgs, "pfs_sizeof_source_args": SourceArgs,
    "pfs_sizeof_target_args": TargetArgs, "pfs_sizeof_global_args": GlobalArgs, "pfs_sizeof_head_args": HeadArgs,
    "pfs_sizeof_wide_gemm_args": WideGemmArgs, "pfs_sizeof_wide_segments": WideSegments,
    "pfs_sizeof_loss_args": LossArgs,
}


class PfsError(RuntimeError):
    pass


_lib = None


# translation units of the library: source -> headers it depends on (besides include/pfs_b200.h)
_WIDE_HEADERS = ("wide_gemm.cuh", "wide_ops.cuh", "tc_ptx.cuh")
_UNITS = {
    "api.cu": lambda f: f.endswith(".cuh") and not f.startswith("wide_"),
    "wide.cu": lambda f: f in _WIDE_HEADERS,
    "loss.cu": lambda f: False,
}


def nvcc_command(src, obj):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    return [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
            "-Xcompiler", "-fPIC", "-c", "-o", obj, src]


def link_command(objs, out_path=LIB_PATH):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    return [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-Xcompiler", "-fPIC", "-o", out_path] + objs


def build_library(force=False, verbose=False):
    """Compile csrc/*.cu for sm_100a (one object per translation unit, in parallel) and link them
    into csrc/libpfs_b200.so; nvcc cross-compiles without a GPU.  Only stale objects are rebuilt."""
    procs, objs = [], []
    for unit, dep in _UNITS.items():
        src = os.path.join(CSRC, unit)
        obj = os.path.join(CSRC, unit[:-3] + ".o")
        objs.append(obj)
        deps = [src, HEADER] + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if dep(f)]
        if not force and os.path.exists(obj) and os.path.getmtime(obj) >= max(os.path.getmtime(d) for d in deps):
            continue
        cmd = nvcc_command(src, obj)
        if verbose:
            print(" ".join(cmd))
        procs.append((cmd, subprocess.Popen(cmd, cwd=CSRC)))
    for cmd, p in procs:
        if p.wait() != 0:
            raise subprocess.CalledProcessError(p.returncode, cmd)
    if procs or force or not os.path.exists(LIB_PATH) or \
            os.path.getmtime(LIB_PATH) < max(os.path.getmtime(o) for o in objs):
        cmd = link_command(objs)
        if verbose:
            print(" ".join(cmd))
        subprocess.run(cmd, check=True, cwd=CSRC)
    return LIB_PATH


def load_library():
    """dlopen the in-tree library, declare every prototype and verify the struct layouts."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PfsError("libpfs_b200.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'`); "
                       "there is no CPU fallback for the message-passing layer")
    lib = ct.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SYMBOLS.items():
        fn = getattr(lib, name)      # AttributeError if the library lacks a declared symbol
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.pfs_abi_version() != ABI_VERSION:
        raise PfsError("libpfs_b200.so ABI version %d != binding %d" % (lib.pfs_abi_version(), ABI_VERSION))
    for fn, struct in _SIZEOF_CHECKS.items():
        if getattr(lib, fn)() != ct.sizeof(struct):
            raise PfsError("%s: C sizeof %d != ctypes %d" % (fn, getattr(lib, fn)(), ct.sizeof(struct)))
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load_library().pfs_last_error()
        raise PfsError("%s failed (%d): %s" % (what, rc, msg.decode() if msg else "?"))


def profile_report():
    """{kernel: (launches, total_ms)} recorded since pfs_profile_enable(1); synchronises."""
    lib = load_library()
    buf = ct.create_string_buffer(1 << 16)
    n = lib.pfs_profile_report(buf, len(buf))
    out = {}
    if n > 0:
        for line in buf.value.decode().splitlines():
            name, cnt, ms = line.rsplit(" ", 2)
            out[name] = (int(cnt), float(ms))
    return out


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()
