"""ctypes binding of the C ABI in include/ecw_b200.h (one prototype per entry point)."""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libecw_b200.so")
_SRC = ["gemm.cu", "gemm_tma.cu", "ewise.cu", "ozaki.cu", "synth.cu", "ftao.cu", "maps.cu", "capi.cu", "plan.cpp", "ccsd_plan.cpp",
        "ccsd_plan_slab.cpp", "ccs_plan.cpp"]

ECW_HAS_ALPHA = 1
ECW_EQUATION = 2
ECW_ANTISYM = 4
ECW_SUBDIFF_SINGLES = 8


class EcwError(RuntimeError):
    pass


def build(force=False, verbose=False):
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU).
    One object per source under csrc/build/ (recompiled only when stale), then one link."""
    csrc = os.path.join(_HERE, "csrc")
    hdrs = [os.path.join(csrc, h) for h in ("plan.h", "kernels.h", "ccsd_plan.h", "ccsd_plan_detail.h")]
    hdrs.append(os.path.join(_HERE, "..", "include", "ecw_b200.h"))
    hdr_mt = max(os.path.getmtime(h) for h in hdrs)
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    flags = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
             "-Xcompiler", "-fPIC", "-diag-suppress", "550"]
    bdir = os.path.join(csrc, "build")
    os.makedirs(bdir, exist_ok=True)
    objs, jobs = [], []
    for s in _SRC:
        src, obj = os.path.join(csrc, s), os.path.join(bdir, s + ".o")
        objs.append(obj)
        if force or not os.path.exists(obj) or os.path.getmtime(obj) < max(os.path.getmtime(src), hdr_mt):
            cmd = [nvcc] + flags + ["-c", src, "-o", obj]
            if verbose:
                print(" ".join(cmd))
            jobs.append((cmd, subprocess.Popen(cmd)))
    for cmd, pr in jobs:
        if pr.wait() != 0:
            raise subprocess.CalledProcessError(pr.returncode, cmd)
    if jobs or not os.path.exists(LIB_PATH) or any(os.path.getmtime(o) > os.path.getmtime(LIB_PATH) for o in objs):
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a"] + objs + ["-ldl", "-o", LIB_PATH]
        if verbose:
            print(" ".join(cmd))
        subprocess.check_call(cmd)
    return LIB_PATH


class _Lib(object):
    """Lazy loader: importing the package must work before the library is built
    (`__graft_entry__.build()` imports it right after compiling)."""

    def __init__(self):
        self._dll = None

    def _load(self):
        if self._dll is not None:
            return self._dll
        if not os.path.exists(LIB_PATH):
            raise EcwError("libecw_b200.so is not built (run `python -c 'import ecw_cc_b200; ecw_cc_b200.build()'`); "
                           "there is no CPU fallback for the ECW-CC residual path")
        d = ctypes.CDLL(LIB_PATH)
        c_p, c_i, c_l, c_d, c_s = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_double, ctypes.c_char_p
        sig = {
            "ecw_ctx_create": (c_i, [ctypes.POINTER(c_p), c_i, c_i]),
            "ecw_ctx_destroy": (None, [c_p]),
            "ecw_last_error": (c_s, [c_p]),
            "ecw_version": (c_s, []),
            "ecw_ctx_set_shard": (c_i, [c_p, c_i, c_i]),
            "ecw_resume": (c_i, [c_p, c_p]),
            "ecw_nccl_unique_id": (c_i, [c_s, c_p]),
            "ecw_ctx_init_nccl": (c_i, [c_p, c_s, c_p, c_i, c_i]),
            "ecw_ctx_nccl_ops": (c_l, [c_p]),
            "ecw_ctx_set_gemm": (c_i, [c_p, c_i, c_d]),
            "ecw_ctx_get_gemm": (c_i, [c_p]),
            "ecw_int8_error_bound": (c_i, [c_p, ctypes.POINTER(c_d), c_p]),
            "ecw_ctx_set_engine_override": (c_i, [c_p, c_i]),
            "ecw_ctx_set_plan_variant": (c_i, [c_p, c_i]),
            "ecw_ctx_set_int8_splitk": (c_i, [c_p, c_l]),
            "ecw_ccs_t1inter": (c_i, [c_p, c_p, c_p, c_p, c_p]),
            "ecw_ccs_l1inter": (c_i, [c_p, c_p, c_p, c_i, c_p, c_p, c_p, c_p]),
            "ecw_ccs_r1inter": (c_i, [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p]),
            "ecw_ccs_esl1inter": (c_i, [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p]),
            "ecw_ctx_set_graphs": (c_i, [c_p, c_i]),
            "ecw_ctx_graph_stats": (c_i, [c_p, ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64)]),
            "ecw_ctx_test_assume_vvvv_planes": (c_i, [c_p]),
            "ecw_ctx_test_assume_ovvv_planes": (c_i, [c_p]),
            "ecw_ctx_test_cut_cache_min": (c_i, [c_p, c_l]),
            "ecw_eris_ovvv_planes": (c_i, [c_p, c_p]),
            "ecw_ozaki_plane_bytes2": (c_l, [c_l, c_l, c_l, c_i]),
            "ecw_ozaki_stat_elems2": (c_l, [c_l, c_l]),
            "ecw_ozaki_split2": (c_i, [c_p, c_l, c_l, c_l, c_l, c_l, c_l, c_i, c_p, c_p, c_p]),
            "ecw_ozaki_gemm_batched": (c_i, [c_p, c_p, c_l, c_p, c_p, c_l, c_l, c_l, c_l, c_p, c_l, c_l, c_d, c_d, c_i,
                                           ctypes.POINTER(c_l), c_p]),
            "ecw_eris_vvvv_planes": (c_i, [c_p, c_p, c_l, c_l, c_p]),
            "ecw_pending_collective": (c_i, [c_p, ctypes.POINTER(c_l)]),
            "ecw_slot_elems": (c_l, [c_p, c_s]),
            "ecw_bind": (c_i, [c_p, c_s, c_p]),
            "ecw_eris_pack_from_dense": (c_i, [c_p, c_p, c_p, c_p]),
            "ecw_eris_synthetic": (c_i, [c_p, c_d, c_p]),
            "ecw_synth_tensor": (c_i, [c_i, c_p, c_i, c_i, c_l, c_l, c_d, c_p]),
            "ecw_workspace_bytes": (c_l, [c_p, c_s, c_i]),
            "ecw_set_workspace": (c_i, [c_p, c_p, c_l]),
            "ecw_ccsd_tupdate": (c_i, [c_p, c_p, c_p, c_p, c_p, c_i, c_d, c_p, c_p, c_p]),
            "ecw_ccsd_lupdate": (c_i, [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_d, c_p, c_p, c_p]),
            "ecw_ccsd_gamma": (c_i, [c_p, c_p, c_p, c_p, c_p, c_p, c_p]),
            "ecw_ccsd_energy": (c_i, [c_p, c_p, c_p, c_p, c_p, c_p]),
            "ecw_subdiff": (c_i, [c_p, c_p, c_d, c_p, c_l, c_p]),
            "ecw_antisym_defect": (c_i, [c_p, c_i, c_i, c_p, c_p]),
            "ecw_plan_dump": (c_l, [c_p, c_s, c_i, c_p, c_l]),
            "ecw_plan_dump_contract": (c_l, [c_p, c_d, c_p, c_s, c_p, c_s, c_d, c_p, c_s, c_p, c_l]),
            "ecw_plan_flops": (c_d, [c_p, c_s, c_i]),
            "ecw_plan_launches": (c_l, [c_p, c_s, c_i]),
            "ecw_dgemm": (c_i, [c_i, c_i, c_l, c_l, c_l, c_d, c_p, c_l, c_p, c_l, c_d, c_p, c_l, c_i, c_p]),
            "ecw_ozaki_plane_bytes": (c_l, [c_l, c_l, c_i]),
            "ecw_ozaki_padded_rows": (c_l, [c_l]),
            "ecw_ozaki_stat_elems": (c_l, [c_l]),
            "ecw_ozaki_tile_n": (c_i, [c_i]),
            "ecw_ozaki_split": (c_i, [c_p, c_l, c_l, c_l, c_l, c_i, c_p, c_p, c_p]),
            "ecw_ozaki_split_rows": (c_i, [c_p, c_l, c_l, c_l, c_l, c_i, c_p, c_p, c_l, c_l, c_p]),
            "ecw_ozaki_gemm": (c_i, [c_p, c_p, c_p, c_p, c_l, c_l, c_l, c_p, c_l, c_l, c_d, c_d, c_i, c_p]),
            "ecw_op_contract": (c_i, [c_p, c_d, c_p, c_s, c_p, c_s, c_d, c_p, c_s, c_p]),
            "ecw_op_axpby": (c_i, [c_p, c_d, c_p, c_s, c_d, c_p, c_s, c_p]),
            "ecw_op_mul": (c_i, [c_p, c_d, c_p, c_p, c_d, c_p, c_p]),
            "ecw_op_unpack": (c_i, [c_p, c_d, c_p, c_i, c_d, c_p, c_p]),
            "ecw_op_diag_shift": (c_i, [c_p, c_p, c_d, c_p, c_l, c_p]),
            "ecw_op_denom": (c_i, [c_p, c_p, c_p, c_p, c_i, c_i, c_d, c_d, c_p, c_p]),
            "ecw_op_dot": (c_i, [c_p, c_d, c_p, c_p, c_d, c_p, c_p]),
            "ecw_op_workspace_needed": (c_l, [c_p]),
            "ecw_conv_check": (c_i, [c_p, c_p, c_p, c_p, c_l, c_p, c_p, c_i, c_p]),
            "ecw_vexp_mat": (c_i, [c_p, c_p, c_p, c_d, c_p, c_p, c_p, c_l, c_p]),
            "ecw_ft_aopair": (c_i, [c_p, c_l, c_p, c_i, c_p, c_l, c_p, c_p]),
            "ecw_vexp_sf": (c_i, [c_p, c_i, c_p, c_i, c_p, c_l, c_p, c_d, c_p, c_p, c_p, c_p, c_p, c_p, c_p]),
            "ecw_vexp_sf_workspace_bytes": (c_l, [c_i, c_i, c_l]),
            "ecw_ft_aopair_cryst": (c_i, [c_p, c_l, c_p, c_p, c_i, c_p, c_i, c_p, c_p, c_i, c_l, c_p, c_p]),
            "ecw_vexp_sfobs": (c_i, [c_p, c_i, c_p, c_i, c_p, c_l, c_p, c_p, c_d, c_d, c_p, c_p, c_p, c_p, c_p, c_p,
                                     c_p]),
            "ecw_vexp_sfobs_workspace_bytes": (c_l, [c_i, c_i, c_l]),
            "ecw_density_grid": (c_i, [c_p, c_l, c_p, c_i, c_p, ctypes.POINTER(c_d), c_i, c_i, c_i, c_p, c_p, c_p]),
            "ecw_density_grid_workspace_bytes": (c_l, [c_i, c_l]),
            "ecw_fourier_map": (c_i, [c_p, c_p, c_l, c_d, c_d, c_i, c_i, c_i, c_p, c_p]),
            "ecw_profile_enable": (c_i, [c_p, c_i]),
            "ecw_profile_dump": (c_l, [c_p, c_p, c_l]),
        }
        for name, (res, args) in sig.items():
            fn = getattr(d, name)
            fn.restype = res
            fn.argtypes = args
        self._dll = d
        self.symbols = sorted(sig)
        return d

    def __getattr__(self, name):
        return getattr(self._load(), name)


lib = _Lib()
