"""ctypes binding of libmlcg_b200.so (C ABI declared in include/mlcg.h) and the in-tree build recipe.

The library is the product: there is no torch / CPU fallback behind it.  If it is missing or no sm_100 device is
present the loaders raise."""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
LIB_PATH = os.path.join(_HERE, "libmlcg_b200.so")
SOURCES = [os.path.join(_HERE, "csrc", f) for f in ("mlcg_api.cu", "mlcg_tc.cuh", "mlcg_tc3.cuh", "mlcg_kernels.cuh", "mlcg_shape.cuh", "mlcg_ifm.cuh",
                                                     "mlcg_common.cuh")]
HEADER = os.path.join(_ROOT, "include", "mlcg.h")

EXPORTS = [
    "mlcg_version", "mlcg_create", "mlcg_destroy", "mlcg_last_error", "mlcg_load_egnn", "mlcg_load_seer",
    "mlcg_set_batch", "mlcg_egnn_forward", "mlcg_noise_init", "mlcg_step", "mlcg_reinject", "mlcg_forward_diffuse",
    "mlcg_decode", "mlcg_sample", "mlcg_seer_inputs", "mlcg_seer_forward", "mlcg_generate", "mlcg_num_edge_tiles",
    "mlcg_num_edges", "mlcg_kernel_launches", "mlcg_time_edge_kernel", "mlcg_edge_phase_profile", "mlcg_test_gemm",
    "mlcg_shape_moments", "mlcg_shape_tanimoto", "mlcg_gemm_phase_profile", "mlcg_plan_edge_tiles",
    "mlcg_egnn_forward_breakdown", "mlcg_ifm_context", "mlcg_ifm_merge_inputs", "mlcg_nonfinite", "mlcg_edge_block_order",
    "mlcg_generate_fragment", "mlcg_generate_fragment_jobs", "mlcg_graph_captures",
]


class WeightDesc(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("rows", C.c_int), ("cols", C.c_int)]


class Noise(C.Structure):
    _fields_ = [("raw", C.c_void_p), ("seed", C.c_uint64), ("draw", C.c_uint64), ("sample_offset", C.c_int64),
                ("sample_ids", C.c_void_p)]


class StepScalars(C.Structure):
    _fields_ = [("t", C.c_float), ("alpha_ts", C.c_float), ("c_eps", C.c_float), ("c_sigma", C.c_float),
                ("alpha_s", C.c_float), ("sigma_s", C.c_float), ("blend", C.c_float)]


class Fragment(C.Structure):
    _fields_ = [("mode", C.c_int), ("n_ff", C.c_int), ("ff_x_host", C.c_void_p), ("ff_h_host", C.c_void_p),
                ("diffusion_level", C.c_int), ("merge_alpha", C.c_float), ("merge_sigma", C.c_float),
                ("moi_gen_origin_host", C.c_void_p), ("ff_weighted_com_host", C.c_void_p), ("norm_mean_host", C.c_void_p),
                ("norm_mad_host", C.c_void_p)]


class FragmentJobs(C.Structure):
    _fields_ = [("mode", C.c_int), ("n_jobs", C.c_int), ("job_of_sample_host", C.c_void_p), ("n_ff_host", C.c_void_p),
                ("ff_x_host", C.c_void_p), ("ff_h_host", C.c_void_p), ("diffusion_level", C.c_int),
                ("merge_alpha", C.c_float), ("merge_sigma", C.c_float), ("moi_gen_origin_host", C.c_void_p),
                ("ff_weighted_com_host", C.c_void_p), ("norm_mean_host", C.c_void_p), ("norm_mad_host", C.c_void_p)]


STAMP_PATH = LIB_PATH + ".stamp"
BUILD_INFO = {"action": None, "sources_sha256": None}


def sources_digest() -> str:
    """sha256 over the CUDA sources + the C header: identifies the source state a binary was compiled from."""
    import hashlib
    h = hashlib.sha256()
    for p in SOURCES + [HEADER]:
        h.update(open(p, "rb").read())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile libmlcg_b200.so in-tree for sm_100a (nvcc cross-compiles without a GPU).  The binary carries a stamp with
    the digest of the sources it was compiled from; it is rebuilt whenever the stamp does not match the sources in the
    tree (file times do not survive a snapshot), so a stale or foreign binary is never used.  BUILD_INFO records whether
    this call compiled or found a binary of exactly these sources."""
    digest = sources_digest()
    BUILD_INFO["sources_sha256"] = digest
    if not force and os.path.exists(LIB_PATH) and os.path.exists(STAMP_PATH) and open(STAMP_PATH).read().strip() == digest:
        BUILD_INFO["action"] = "up to date (binary stamp == sha256 of the sources in the tree)"
        return LIB_PATH
    cmd = ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-shared",
           "-Xcompiler", "-fPIC", "-I" + os.path.join(_ROOT, "include"), "-o", LIB_PATH, SOURCES[0]]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    with open(STAMP_PATH, "w") as fh:
        fh.write(digest + "\n")
    BUILD_INFO["action"] = "compiled with nvcc"
    return LIB_PATH


_lib = None


def load() -> C.CDLL:
    """dlopen the library and declare the prototypes.  Raises if the library has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("libmlcg_b200.so is not built; run `python -c 'import __graft_entry__ as g; g.build()'`. "
                           "There is no fallback implementation.")
    lib = C.CDLL(LIB_PATH)
    vp, ci, cf = C.c_void_p, C.c_int, C.c_float
    lib.mlcg_version.restype = C.c_char_p
    lib.mlcg_create.argtypes = [C.POINTER(vp), ci, ci]
    lib.mlcg_destroy.argtypes = [vp]
    lib.mlcg_destroy.restype = None
    lib.mlcg_last_error.argtypes = [vp]
    lib.mlcg_last_error.restype = C.c_char_p
    lib.mlcg_load_egnn.argtypes = [vp, C.POINTER(WeightDesc), ci]
    lib.mlcg_load_seer.argtypes = [vp, C.POINTER(WeightDesc), ci]
    lib.mlcg_set_batch.argtypes = [vp, vp, ci, ci]
    lib.mlcg_egnn_forward.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.mlcg_egnn_forward_breakdown.argtypes = [vp, vp, vp, vp, vp, C.POINTER(C.c_double), vp]
    lib.mlcg_noise_init.argtypes = [vp, vp, C.POINTER(Noise), vp]
    lib.mlcg_step.argtypes = [vp, vp, vp, C.POINTER(StepScalars), C.POINTER(Noise), vp]
    lib.mlcg_reinject.argtypes = [vp, vp, vp, vp, C.POINTER(StepScalars), C.POINTER(Noise), vp]
    lib.mlcg_forward_diffuse.argtypes = [vp, vp, vp, cf, cf, C.POINTER(Noise), vp]
    lib.mlcg_decode.argtypes = [vp, vp, vp, cf, cf, cf, C.POINTER(Noise), vp, vp, vp]
    lib.mlcg_sample.argtypes = [vp, ci, ci, C.POINTER(StepScalars), ci, ci, cf, cf, cf, cf, cf, vp, vp, vp, vp,
                                C.c_uint64, C.c_int64, vp, vp, vp, vp, vp, vp, vp]
    lib.mlcg_seer_inputs.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    lib.mlcg_seer_forward.argtypes = [vp, vp, vp, vp, vp, vp, ci, vp]
    lib.mlcg_generate.argtypes = [vp, vp, ci, ci, vp, ci, C.POINTER(StepScalars), ci, cf, cf, cf, C.c_uint64,
                                  C.c_int64, vp, vp, vp, vp, vp]
    lib.mlcg_generate_fragment.argtypes = [vp, C.POINTER(Fragment), vp, ci, ci, vp, ci, C.POINTER(StepScalars), ci, cf, cf,
                                           cf, C.c_uint64, C.c_int64, vp, vp, vp, vp, vp]
    lib.mlcg_generate_fragment_jobs.argtypes = [vp, C.POINTER(FragmentJobs), vp, ci, ci, vp, ci, C.POINTER(StepScalars), ci,
                                                cf, cf, cf, C.c_uint64, C.c_int64, vp, vp, vp, vp, vp]
    lib.mlcg_nonfinite.argtypes = [vp, vp]
    lib.mlcg_num_edge_tiles.argtypes = [vp]
    lib.mlcg_num_edges.argtypes = [vp]
    lib.mlcg_num_edges.restype = C.c_int64
    lib.mlcg_kernel_launches.argtypes = [vp]
    lib.mlcg_kernel_launches.restype = C.c_int64
    lib.mlcg_graph_captures.argtypes = [vp]
    lib.mlcg_graph_captures.restype = C.c_int64
    lib.mlcg_time_edge_kernel.argtypes = [vp, ci, ci, vp]
    lib.mlcg_time_edge_kernel.restype = cf
    lib.mlcg_edge_phase_profile.argtypes = [vp, ci, C.POINTER(C.c_double), vp]
    lib.mlcg_test_gemm.argtypes = [vp, ci, ci, vp, vp, vp, vp, ci, ci, ci, vp]
    lib.mlcg_gemm_phase_profile.argtypes = [vp, ci, C.POINTER(C.c_double), vp]
    lib.mlcg_ifm_context.argtypes = [vp, vp, vp, ci, vp, vp, vp, ci, vp, vp, vp, vp, vp]
    lib.mlcg_ifm_merge_inputs.argtypes = [vp, vp, vp, vp, vp, vp, vp, ci, ci, ci, ci, vp, vp, vp]
    lib.mlcg_plan_edge_tiles.argtypes = [vp, ci, ci, ci, vp, vp, ci, vp]
    lib.mlcg_edge_block_order.argtypes = [ci, vp]
    lib.mlcg_shape_moments.argtypes = [vp, vp, vp, ci, ci, C.c_float, C.c_float, ci, vp, vp]
    lib.mlcg_shape_tanimoto.argtypes = [vp, vp, ci, vp, vp, ci, ci, vp, vp, ci, vp, ci, C.c_float, C.c_float, vp, vp, vp, vp]
    _lib = lib
    return lib
