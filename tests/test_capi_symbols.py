"""CPU-side checks of the drop-in boundary: libpsulvsb_b200.so loads without a GPU, exports every
symbol include/psulvsb.h declares, reports errors as codes, and the ctypes structs match the header."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import psulvsb_b200  # noqa: F401
from psulvsb_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    src = open(os.path.join(ROOT, "include", "psulvsb.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(psulvsb_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    names = header_functions()
    assert len(names) >= 25
    lib = C.CDLL(capi.LIB_PATH)
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing
    assert sorted(capi.SYMBOLS) == names          # the Python binding covers the whole header
    # include/psulvsb_io.h (host-side helpers) as well
    src = open(os.path.join(ROOT, "include", "psulvsb_io.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    io_names = sorted(set(re.findall(r"\b(psulvsb_[a-z0-9_]+)\s*\(", src)))
    from psulvsb_b200 import io
    assert io_names == sorted(io.IO_SYMBOLS)
    assert not [n for n in io_names if not hasattr(lib, n)]


def test_version_defaults_and_no_device_behaviour():
    L = capi.lib()
    assert L.psulvsb_version() == 100
    p = capi.default_params()
    # RobustRegistrationSolver::Params defaults (registration.h:383-426) and the lifted constants
    assert p.noise_bound == 0.01 and p.cbar2 == 1 and p.estimate_scaling == 1
    assert p.rotation_max_iterations == 100 and p.rotation_gnc_factor == 1.4 and p.rotation_cost_threshold == 1e-6
    assert p.inloop_noise_bound == 0.05 and p.inloop_cost_threshold == 0.005 and p.host_round_limit == 5
    assert p.tpro_host == 0.99 and p.tpro_local == 0.99 and p.local_max_iter == 10 and p.wallclock_cap_s == 60.0
    if L.psulvsb_device_count() == 0:
        # no CPU fallback: every compute entry point fails loudly with PSULVSB_ERR_NO_DEVICE
        h = C.c_void_p()
        assert L.psulvsb_create(C.byref(h), 0) == capi.ERR_NO_DEVICE
        assert b"no CUDA device" in L.psulvsb_last_error()
        assert L.psulvsb_philox_fill(None, 0, 1, 0, 0, 4, None) == capi.ERR_NO_DEVICE
        with pytest.raises(capi.PsulvsbError):
            capi.Handle(0)


def test_struct_layouts_match_the_oracle_mirror():
    """psulvsb_params_t / solution prefix / trace records are field-for-field the oracle's structs, so a
    trace from either solver can be compared directly."""
    from oracle import oracle as O

    assert [f[0] for f in capi.Params._fields_] == [f[0] for f in O.Params._fields_]
    assert C.sizeof(capi.Params) == C.sizeof(O.Params)
    n = len(O.Solution._fields_)
    assert [f[0] for f in capi.Solution._fields_][:n] == [f[0] for f in O.Solution._fields_]
    assert C.sizeof(capi.LocalTrace) == C.sizeof(O.LocalTrace) == 176
    assert C.sizeof(capi.HostTrace) == C.sizeof(O.HostTrace) == 32


def test_host_problem_layout():
    src = np.arange(12, dtype=np.float64).reshape(3, 4)
    hp = capi.HostProblem(src, src + 1)
    ps = hp.c_struct()
    assert ps.C == 4 and ps.M == 4
    assert [ps.src[i] for i in range(6)] == [0, 4, 8, 1, 5, 9]      # column-major 3xN, as Eigen stores it
    assert list(hp.keep_mask) == [1, 1, 1, 1] and list(hp.reduce_map) == [0, 1, 2, 3]
    with pytest.raises(ValueError):
        capi.HostProblem(np.zeros((4, 3)), np.zeros((4, 3)))
    with pytest.raises(ValueError):
        capi.HostProblem(np.zeros((3, 4)), np.zeros((3, 4)), np.zeros((3, 9)), np.zeros((3, 9)))


def test_mirror_params_defaults():
    from psulvsb_b200 import RobustRegistrationSolver as S

    p = S.Params()
    assert p.noise_bound == 0.01 and p.estimate_scaling is True and p.rotation_gnc_factor == 1.4
    assert p.rotation_estimation_algorithm == S.ROTATION_ESTIMATION_ALGORITHM.GNC_TLS
    assert p.inlier_selection_mode == S.INLIER_SELECTION_MODE.PMC_EXACT
    assert int(S.INLIER_SELECTION_MODE.NONE) == 3


def test_argument_validation_without_device():
    """Bad arguments are refused with PSULVSB_ERR_INVALID before any device work (so this runs without a GPU)."""
    L = capi.lib()
    assert L.psulvsb_solve(None, None, None, None, None) == capi.ERR_INVALID
    assert L.psulvsb_solve_batch(None, None, None, 0, None, None) == capi.ERR_INVALID
    assert L.psulvsb_batch_upload(None, None, 0) == capi.ERR_INVALID
    assert L.psulvsb_destroy(None) == capi.OK
    assert L.psulvsb_launch_count(None) == 0 and L.psulvsb_last_ticks(None) == 0
    n = C.c_longlong(0)
    assert L.psulvsb_ply_vertex_count(b"/nonexistent/file.ply", C.byref(n)) == capi.ERR_INVALID
    assert b"cannot open" in L.psulvsb_last_error()


def test_debug_switches_accept_only_the_coverage_switches():
    """psulvsb_debug_set (no device needed) knows four switches and "reset"; the launch-shape tuning switches are gone
    and are refused like any unknown name, as is a k1_variant the launcher has no kernel for."""
    L = capi.lib()
    try:
        for name in ("gnc_cluster", "gnc_cps", "gnc_prefetch", "gnc_park_pct", "gnc_grid_lv", "upload_prof"):
            assert L.psulvsb_debug_set(name.encode(), 1.0) == capi.ERR_INVALID, name
            assert b"unknown switch" in L.psulvsb_last_error()
        for value in (3.0, 5.0, -1.0, 1.5):
            assert L.psulvsb_debug_set(b"k1_variant", value) == capi.ERR_INVALID, value
        for name, value in (("gnc_deep_margin", 1e-4), ("sample_list_cap_test", 4.0), ("edge_wide", 1.0),
                            ("k1_variant", 0.0), ("k1_variant", 1.0), ("k1_variant", 2.0), ("k1_variant", 4.0)):
            assert L.psulvsb_debug_set(name.encode(), value) == capi.OK, (name, value)
    finally:
        assert L.psulvsb_debug_set(b"reset", 0.0) == capi.OK


def test_fp32_pipe_kernels_are_packed_and_tma_staged():
    """The SASS of the consistency-mask and scoring kernels carries what DESIGN.md section 6 says they are built on:
    packed FP32 (FFMA2) in the pair / score loops, their 64-bit operand kept in the operand-reuse cache, and 1-D TMA
    bulk copies (UBLKCP) for the tile rings."""
    import shutil
    import subprocess

    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    sass = subprocess.run([cuobjdump, "-sass", capi.LIB_PATH], capture_output=True, text=True, timeout=300).stdout
    per_fn, name = {}, None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1)
            per_fn[name] = {"FFMA2": 0, "UBLKCP": 0, "FFMA": 0, "REUSE64": 0}
        elif name:
            for op in ("FFMA2", "UBLKCP"):
                if re.search(r"\b%s\b" % op, line):
                    per_fn[name][op] += 1
            if re.search(r"\bFFMA\b", line):
                per_fn[name]["FFMA"] += 1
            if "FFMA2" in line and "reuse.F32x2" in line:
                per_fn[name]["REUSE64"] += 1
    k1 = {k: v for k, v in per_fn.items() if "k1_mask_kernelILi4ELi256ELb1" in k}
    k4 = {k: v for k, v in per_fn.items() if "score_batch_kernel" in k}
    assert len(k1) == 1 and len(k4) == 1, (list(k1), list(k4))
    for ops in list(k1.values()) + list(k4.values()):
        assert ops["UBLKCP"] >= 2, ops          # both tile arrays come by bulk copy
        assert ops["FFMA2"] >= 100, ops         # the unrolled loops are packed ...
        assert ops["FFMA2"] > ops["FFMA"], ops  # ... what is left scalar is the rare slow / fix-up / odd-tail code
        # r2: two columns (K1) / two points (K4) in the halves -- the 64-bit operand is the one consecutive FFMA2 share
        assert ops["REUSE64"] >= 40, ops
