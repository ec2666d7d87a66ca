"""CPU-side checks of the drop-in boundary: the shared library loads, exports every symbol include/isdf.h declares,
struct layouts agree, and the product refuses to run without a GPU (no CPU fallback, no oracle on the product path)."""
import ctypes as C
import os
import re
import subprocess
import pytest
import isdf_b200 as I

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    txt = open(os.path.join(ROOT, "include", "isdf.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(isdf_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    import __graft_entry__ as G   # noqa: F401  (repo root is on sys.path through pytest rootdir)
    if not os.path.exists(I.LIB_PATH):
        G.build()
    syms = header_symbols()
    assert set(syms) == set(I.ABI_SYMBOLS), (set(syms) ^ set(I.ABI_SYMBOLS))
    out = subprocess.check_output(["nm", "-D", "--defined-only", I.LIB_PATH]).decode()
    exported = set(re.findall(r"\bT (isdf_[a-z0-9_]+)\b", out))
    assert set(syms) <= exported, set(syms) - exported
    lib = I.load_library()
    for s in syms:
        assert getattr(lib, s) is not None


def test_no_torch_or_oracle_linked_into_product():
    out = subprocess.check_output(["ldd", I.LIB_PATH]).decode()
    out = re.sub(r"\(0x[0-9a-f]+\)", "", out)            # load addresses are random hex and can spell "c10"
    assert "torch" not in out and "oracle" not in out and "c10" not in out
    # the product sources never include the oracle
    for dirpath, _, files in os.walk(os.path.join(ROOT, "implicit-sdf-planner_b200")):
        for f in files:
            if f.endswith((".cu", ".cuh", ".hpp", ".h", ".cpp", ".py")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "oracle_" not in txt and "liboracle" not in txt, os.path.join(dirpath, f)


def test_default_config_matches_python_mirror():
    lib = I.load_library()
    c = I.Config()
    assert lib.isdf_default_config(C.byref(c)) == 0
    d = I.default_config_values()
    for name, _ in I.Config._fields_:
        assert getattr(c, name) == getattr(d, name), name
    assert C.sizeof(I.Config) == 144


def test_shape_kind_ids_match_oracle():
    import oracle_lib as O
    for name in I.NAMED_SHAPES:
        sh = O.Shape.named(name)
        assert 0 <= sh.kind() < I.SHAPE_KINDS["MESH"]


def test_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(I.IsdfError) as e:
        I.Evaluator(I.default_config_values(), device=0)
    assert e.value.code == -3   # ISDF_ERR_CUDA — never a silent CPU path


def test_argument_validation_without_gpu_calls():
    lib = I.load_library()
    assert lib.isdf_default_config(None) == -1
    assert lib.isdf_create(None, 0, None) == -1
    bad = I.default_config_values()
    bad.integral_intervs = 0
    h = C.c_void_p()
    assert lib.isdf_create(C.byref(bad), 0, C.byref(h)) == -1
    assert b"config" in lib.isdf_last_error()


def test_header_is_plain_c99():
    src = '#include "isdf.h"\nint main(void) { isdf_config c; isdf_kernel_config k = {45, 45, 9, 0}; (void)c; (void)k; return 0; }\n'
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), "-x", "c", "-"],
                       input=src.encode(), capture_output=True)
    assert r.returncode == 0, r.stderr.decode()
    assert C.sizeof(I.KernelConfig) == 32


def test_new_entry_points_validate_arguments_without_gpu_calls():
    import numpy as np
    lib = I.load_library()
    cost = np.zeros(3)
    x, g, bc = np.zeros(3 * 13), np.zeros(3 * 13), np.zeros(9)
    dp = C.POINTER(C.c_double)
    r = lib.isdf_callback_batch(None, 3, 4, bc.ctypes.data_as(dp), bc.ctypes.data_as(dp), 0, 20.0, x.ctypes.data_as(dp), cost.ctypes.data_as(dp), g.ctypes.data_as(dp))
    assert r == -1 and np.all(np.isnan(cost))            # every cost poisoned: either optimiser driver stops
    assert lib.isdf_frontend_build_kernels(None, None, None, None) == -1
    assert lib.isdf_frontend_feasibility(None, None) == -1
    assert lib.isdf_frontend_check_batch(None, 0, None, None, None, None) == -1
    assert lib.isdf_peer_export(None, 2, 10, None) == -1
    assert lib.isdf_peer_connect(None, 2, 0, None, 1) == -1
    assert lib.isdf_peer_allreduce_device(None, None, 0, None) == -1
    assert lib.isdf_peer_status(None) == -1 and lib.isdf_peer_disconnect(None) == -1
    assert lib.isdf_get_batch_trajectories(None, None, None, None) == -1


def test_plain_c_client_links_and_fails_loudly_without_a_gpu(tmp_path):
    """examples/minimal.c: a C99 program against include/isdf.h + libisdf_b200.so only (no torch, no C++ runtime on its side)."""
    import torch
    exe = str(tmp_path / "minimal")
    libdir = os.path.dirname(I.LIB_PATH)
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "examples", "minimal.c"), "-o", exe, I.LIB_PATH, f"-Wl,-rpath,{libdir}", "-lm"], capture_output=True)
    assert r.returncode == 0, r.stderr.decode()
    run = subprocess.run([exe], capture_output=True, timeout=120)
    if torch.cuda.is_available():
        assert run.returncode == 0 and b"cost" in run.stdout, (run.stdout, run.stderr)
    else:
        assert run.returncode == 3 and b"isdf_create: -3" in run.stderr      # ISDF_ERR_CUDA, never a silent CPU path
