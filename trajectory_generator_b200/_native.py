"""ctypes binding of the CUDA library (include/trajectory_generator_b200.h).

The library is built in-tree by ``build_native()`` (also called from ``__graft_entry__.build``):
``trajectory_generator_b200/lib/libTrajectoryConstraints.so`` -- the same file name the
reference's ctypes wrappers load (CF/turning_constraints.py:12-15), because it also exports the
reference's 24 legacy symbols.  There is no CPU fallback: if the library is missing, importing
any compute entry point raises.
"""
import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libTrajectoryConstraints.so")
CSRC = os.path.join(HERE, "csrc")

# field order of struct TgLayout (csrc/tg_spec.h)
LAYOUT_FIELDS = ("d N nint n ia is0 is1 it0 nws niw meq mineq m r_start n_start r_end n_end r_sder n_sder "
                 "r_eder n_eder r_iwl n_iwl r_iwv n_iwv r_db n_db r_tanl r_tanu n_tan r_turn n_turn r_sfcl r_sfcu "
                 "n_sfc r_obs n_obs m_nl m_lin turn_first turn_ncp p_start_loc p_end_loc p_target_vel p_sdir p_svel "
                 "p_sacc p_edir p_evel p_eacc p_iwl p_iwv p_minv p_maxv p_up p_horiz p_maxa p_grav p_jerk p_tanmin "
                 "p_tanmax p_turn p_sfc p_obs_c p_obs_r P").split()

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC"]
# translation units: the host API (+ legacy single-problem kernels) and one unit per (kernel family, lanes per problem)
UNITS = ["tg_api.cu", "tg_sample.cu", "tg_build.cu", "tg_smooth.cu", "tg_multistart.cu", "tg_solve_fused.cu", "tg_solve_g64.cu"] + ["tg_%s_g%d.cu" % (fam, gs) for fam in ("eval", "solve", "solve_fd", "polish", "sens") for gs in (8, 16, 32)]
HEADERS = ["tg_sqp.h", "tg_eval.h", "tg_spec.h", "tg_shape.h", "tg_smooth.h", "tg_kernels_eval.inc", "tg_kernels_solve.inc", "tg_polish.h",
           "tg_kernels_polish.inc", "tg_sens.h", "tg_kernels_sens.inc"]


def build_native(force=False, verbose=False, variant=None, extra_flags=()):
    """Compile csrc/*.cu for sm_100a into lib/libTrajectoryConstraints.so (nvcc cross-compiles without a GPU).
    Units are compiled in parallel into lib/obj/ and linked into one shared library.
    `variant` (tuning experiments only): build lib/variants/<variant>.so with `extra_flags`; select it at run time
    with the environment variable TG_LIB=<path>."""
    from concurrent.futures import ThreadPoolExecutor
    deps = [os.path.join(CSRC, f) for f in HEADERS]
    deps.append(os.path.join(os.path.dirname(HERE), "include", "trajectory_generator_b200.h"))
    objdir = os.path.join(HERE, "lib", "obj" if not variant else os.path.join("variants", variant + "_obj"))
    os.makedirs(objdir, exist_ok=True)
    lib_path = LIB_PATH if not variant else os.path.join(HERE, "lib", "variants", variant + ".so")
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    newest_dep = max(os.path.getmtime(d) for d in deps)

    def compile_unit(unit):
        src = os.path.join(CSRC, unit)
        obj = os.path.join(objdir, unit.replace(".cu", ".o"))
        if not force and os.path.exists(obj) and os.path.getmtime(obj) >= max(newest_dep, os.path.getmtime(src)):
            return obj, False, ""
        cmd = [nvcc] + NVCC_FLAGS + list(extra_flags) + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, src]
        proc = subprocess.run(cmd, capture_output=True, text=True)
        if proc.returncode != 0:
            raise RuntimeError("nvcc failed:\n%s\n%s" % (" ".join(cmd), proc.stderr))
        return obj, True, proc.stderr

    with ThreadPoolExecutor(max_workers=min(len(UNITS), os.cpu_count() or 1)) as pool:
        results = list(pool.map(compile_unit, UNITS))
    if verbose:
        for _, _, log in results:
            print(log)
    objs = [r[0] for r in results]
    if force or any(r[1] for r in results) or not os.path.exists(lib_path):
        cmd = [nvcc, "-shared", "-o", lib_path] + objs
        proc = subprocess.run(cmd, capture_output=True, text=True)
        if proc.returncode != 0:
            raise RuntimeError("link failed:\n%s\n%s" % (" ".join(cmd), proc.stderr))
    return lib_path


_LIB = None
_F64 = ctypes.POINTER(ctypes.c_double)
_I32 = ctypes.POINTER(ctypes.c_int)


def lib():
    """The loaded CUDA library; raises if it has not been built (no fallback)."""
    global _LIB
    if _LIB is None:
        path = os.environ.get("TG_LIB", LIB_PATH)         # TG_LIB: a tuning variant built by build_native(variant=...)
        if not os.path.exists(path):
            raise RuntimeError("CUDA library %s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(there is no CPU fallback)" % path)
        L = ctypes.CDLL(path)
        L.tg_spec_count.restype = ctypes.c_int
        L.tg_layout.argtypes = [_I32, _I32, ctypes.c_int]
        L.tg_layout.restype = ctypes.c_int
        L.tg_last_error.restype = ctypes.c_char_p
        L.tg_device_check.restype = ctypes.c_int
        L.tg_launch_count.restype = ctypes.c_ulonglong
        vp, sz = ctypes.c_void_p, ctypes.c_size_t
        L.tg_eval_batch.argtypes = [_I32, ctypes.c_int, vp, vp, vp, vp, vp, vp, vp]
        L.tg_linear_rows_batch.argtypes = [_I32, ctypes.c_int, vp, vp, vp]
        L.tg_solve_workspace_bytes.argtypes = [_I32, ctypes.c_int]
        L.tg_solve_workspace_bytes.restype = sz
        L.tg_solve_plan_info.argtypes = [_I32, ctypes.c_int, _I32, ctypes.c_int]
        L.tg_solve_plan_info.restype = ctypes.c_int
        L.tg_solve_batch.argtypes = [_I32, ctypes.c_int, vp, vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_double,
                                     ctypes.c_int, vp, sz, vp]
        L.tg_solve_batch_kkt.argtypes = list(L.tg_solve_batch.argtypes) + [vp, vp]
        L.tg_eval_host.argtypes = [_I32, ctypes.c_int, vp, vp, vp, vp, vp, vp]
        L.tg_solve_host.argtypes = [_I32, ctypes.c_int, vp, vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_double,
                                    ctypes.c_int]
        L.tg_set_stage_timing.argtypes = [ctypes.c_int]
        L.tg_set_stage_timing.restype = None
        L.tg_last_solve_stats.argtypes = [_F64, ctypes.c_int]
        L.tg_last_solve_stats.restype = ctypes.c_int
        L.tg_measure_fp64_peak.argtypes = [_F64]
        L.tg_measure_fp64_peak.restype = ctypes.c_int
        L.tg_sample_batch.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, ctypes.c_long, vp, ctypes.c_long,
                                      ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, ctypes.c_double, vp, ctypes.c_long,
                                      vp, vp, vp]
        L.tg_sample_batch.restype = ctypes.c_int
        L.tg_sample_batch_order.argtypes = [ctypes.c_int] + list(L.tg_sample_batch.argtypes)
        L.tg_sample_batch_order.restype = ctypes.c_int
        L.tg_interval_points_batch.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp, ctypes.c_int, vp, vp]
        L.tg_interval_points_batch.restype = ctypes.c_int
        L.tg_sfc_intervals_batch.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, ctypes.c_int, vp, vp, vp]
        L.tg_sfc_intervals_batch.restype = ctypes.c_int
        L.tg_smooth_workspace_bytes.argtypes = [ctypes.c_int] * 5
        L.tg_smooth_workspace_bytes.restype = sz
        L.tg_smooth_batch.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_int,
                                      vp, vp, vp, vp, vp, ctypes.c_int, ctypes.c_double, vp, sz, vp]
        L.tg_smooth_batch.restype = ctypes.c_int
        L.tg_smooth_initial_batch.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp]
        L.tg_smooth_initial_batch.restype = ctypes.c_int
        L.tg_initial_guess_batch.argtypes = [_I32, ctypes.c_int, vp, ctypes.c_int, vp, ctypes.c_int, ctypes.c_double, vp, vp]
        L.tg_initial_guess_batch.restype = ctypes.c_int
        L.tg_sfc_boxes_batch.argtypes = [_I32, ctypes.c_int, vp, vp, vp, vp, vp]
        L.tg_sfc_boxes_batch.restype = ctypes.c_int
        L.tg_multistart_expand.argtypes = [_I32, ctypes.c_int, ctypes.c_int, vp, vp, ctypes.c_uint64, ctypes.c_double, vp, vp, vp]
        L.tg_multistart_expand.restype = ctypes.c_int
        L.tg_multistart_select.argtypes = [_I32, ctypes.c_int, ctypes.c_int] + [vp] * 6 + [ctypes.c_double] + [vp] * 8
        L.tg_multistart_select.restype = ctypes.c_int
        L.tg_polish_batch.argtypes = [_I32, ctypes.c_int] + [vp] * 9 + [ctypes.c_int, ctypes.c_double, vp, sz, vp]
        L.tg_polish_batch.restype = ctypes.c_int
        L.tg_polish_workspace_bytes.argtypes = [_I32, ctypes.c_int]
        L.tg_polish_workspace_bytes.restype = sz
        L.tg_polish_plan_info.argtypes = [_I32, ctypes.c_int, _I32, ctypes.c_int]
        L.tg_polish_plan_info.restype = ctypes.c_int
        L.tg_sens_batch.argtypes = [_I32, ctypes.c_int] + [vp] * 8 + [ctypes.c_double, vp, sz, vp]
        L.tg_sens_batch.restype = ctypes.c_int
        L.tg_sens_workspace_bytes.argtypes = [_I32, ctypes.c_int]
        L.tg_sens_workspace_bytes.restype = sz
        L.tg_sens_plan_info.argtypes = [_I32, ctypes.c_int, _I32, ctypes.c_int]
        L.tg_sens_plan_info.restype = ctypes.c_int
        for name in ("tg_eval_batch", "tg_linear_rows_batch", "tg_solve_batch", "tg_solve_batch_kkt", "tg_eval_host", "tg_solve_host"):
            getattr(L, name).restype = ctypes.c_int
        _LIB = L
    return _LIB


def check(rc, what):
    if rc != 0:
        raise RuntimeError("%s failed (code %d): %s" % (what, rc, lib().tg_last_error().decode()))


def spec_ptr(spec):
    spec = np.ascontiguousarray(spec, dtype=np.int32)
    if spec.size != lib().tg_spec_count():
        raise ValueError("spec must have %d entries" % lib().tg_spec_count())
    return spec, spec.ctypes.data_as(_I32)


def layout_ints(spec):
    spec, sp = spec_ptr(spec)
    out = np.zeros(len(LAYOUT_FIELDS), dtype=np.int32)
    cnt = lib().tg_layout(sp, out.ctypes.data_as(_I32), out.size)
    if cnt != len(LAYOUT_FIELDS):
        raise RuntimeError("TgLayout has %d fields, the Python mirror lists %d" % (cnt, len(LAYOUT_FIELDS)))
    return out
