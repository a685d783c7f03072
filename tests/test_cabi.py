"""The C-ABI library loads and exports every entry point include/dsp_lp.h declares (no compute, no GPU)."""
import re
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def declared_functions():
    h = (ROOT / "include" / "dsp_lp.h").read_text()
    h = re.sub(r"/\*.*?\*/", "", h, flags=re.S)
    return sorted(set(re.findall(r"\b(dsp_lp_\w+)\s*\(", h)))


def test_header_declares_the_boundary():
    f = declared_functions()
    for name in ("dsp_lp_template_create", "dsp_lp_solve_batch", "dsp_lp_solve_batch_host", "dsp_lp_template_destroy"):
        assert name in f


def test_library_exports_every_declared_symbol(cuda_solver_lib):
    from dispatches_b200 import solver
    for name in declared_functions():
        assert hasattr(cuda_solver_lib, name), name
    assert sorted(solver.EXPORTS) == declared_functions()
    assert b"sm_100a" in cuda_solver_lib.dsp_lp_version()


def test_sass_is_sm100a_with_tma_staging():
    """The built library carries sm_100a SASS with the TMA bulk copy (UBLKCP) and FP64 FMAs."""
    import shutil
    import subprocess
    if shutil.which("cuobjdump") is None:
        import pytest
        pytest.skip("cuobjdump not on PATH")
    from dispatches_b200.csrc import build
    lib = build.build()
    sass = subprocess.run(["cuobjdump", "-sass", str(lib)], capture_output=True, text=True).stdout
    assert "sm_100a" in sass and "UBLKCP" in sass and "DFMA" in sass


def test_no_cpu_fallback_in_product():
    """The product package never imports the oracle and the solver refuses non-CUDA tensors."""
    for p in list((ROOT / "dispatches_b200").rglob("*.py")) + list((ROOT / "tools").rglob("*.py")):
        src = p.read_text()
        assert "import oracle" not in src and "from oracle" not in src, p
    import numpy as np
    import pytest
    import torch
    from dispatches_b200 import solver, templates as TP
    if torch.cuda.is_available():
        pytest.skip("checks the no-GPU failure mode")
    with pytest.raises(RuntimeError):
        solver.BatchLPSolver(TP.nuclear(4)).solve_host(np.zeros((1, 4)))


def test_argument_errors_are_reported_without_a_gpu(cuda_solver_lib):
    """Bad descriptors / null handles come back as DSP_E_ARG with a message (no CUDA call is made before the checks)."""
    import ctypes as C
    from dispatches_b200 import solver
    lib = cuda_solver_lib
    d = solver._Desc(m=0, n=5, nb=0, w=0, Pc=1, Pr=0)
    h = C.c_void_p()
    assert lib.dsp_lp_template_create(C.byref(d), C.byref(h)) == -1
    assert b"bad dimensions" in lib.dsp_lp_last_error()
    assert lib.dsp_lp_solve_batch(None, 4, None, None, 0, None, None, None, None, None, None, None) == -1
    assert lib.dsp_lp_solve_batch_host(None, 4, None, None, 0, None, None, None, None, None, None) == -1
    o = solver._Opts()
    lib.dsp_lp_default_opts(C.byref(o))
    assert (o.tol, o.feas_tol, o.max_iter, o.kernel) == (1e-9, 1e-9, 60, solver.KERNEL_AUTO) and o.reg_primal == 1e-8
    sd = solver._StageWB(T=40)
    assert lib.dsp_lp_template_set_stage_wb(None, C.byref(sd)) == -1


def test_forced_rebuild_from_source():
    """build(force=True) recompiles libdsp_lp.so from the sources for sm_100a (nvcc cross-compiles without a GPU) -- the
    round-end check must not depend on a stale prebuilt library."""
    import time
    from dispatches_b200.csrc import build
    t0 = time.time()
    lib = build.build(force=True)
    assert lib.exists() and lib.stat().st_mtime >= t0 - 1.0


def test_up_to_date_build_writes_nothing(cuda_solver_lib):
    """bench.py calls build() and may run from a read-only tree: with the library current, build() creates or changes no file"""
    from dispatches_b200.csrc import build
    lib = build.build()
    (lib.parent / ".build.lock").unlink(missing_ok=True)
    before = {p: p.stat().st_mtime_ns for p in lib.parent.iterdir()}
    assert build.build() == lib
    assert {p: p.stat().st_mtime_ns for p in lib.parent.iterdir()} == before


def build_c_example(tmp_path):
    import shutil
    import subprocess
    from dispatches_b200.csrc import build
    lib = build.build()
    exe = tmp_path / "c_abi_example"
    cmd = [shutil.which("gcc") or "gcc", "-std=c99", "-O1", "-Wall", f"-I{ROOT / 'include'}", str(ROOT / "tests" / "c_abi_example.c"),
           f"-L{lib.parent}", "-ldsp_lp", f"-Wl,-rpath,{lib.parent}", "-lm", "-o", str(exe)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def test_the_c_abi_compiles_and_links_from_plain_c(tmp_path):
    """include/dsp_lp.h is C99-clean and a C program links against libdsp_lp.so with nothing but the header (INTEGRATION.md 1b)"""
    exe = build_c_example(tmp_path)
    assert exe.exists()
