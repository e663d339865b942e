"""CPU tests (`-m "not gpu"`): host logic, wire formats and the C-ABI boundary (no compute calls).

* the shared libraries load and export every symbol include/spectral.h declares; libtrp.so / libcub.so export
  exactly the reference's plugin symbol `find_traj` (trp_wrapper.cpp:16-20);
* struct layouts match the reference's (Params 88 B: py_cpp_.h:6-21; Cube 112 B: cube_type.h:2-24);
* without a CUDA device the product fails loudly (no CPU fallback, the oracle is never loaded);
* c_road_*.txt reader/writer round trip (trp_wrapper.cpp:39-144 grammar) and the %.3f trajectory reader.
"""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import helpers as H
from spectral_b200 import api
from spectral_b200.scenarios import WEIGHTS_FILE, config2, load_fixture
from spectral_b200.wire import (ScenarioBatch, read_scenario_text, read_trajectory_text, write_scenario_text)


def _header_symbols():
    hdr = open(os.path.join(H.ROOT, "include", "spectral.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(spectral_[a-z0-9_]+)\s*\(", hdr)))


def test_libspectral_exports_every_declared_symbol():
    lib = api.load_library()
    syms = _header_symbols()
    assert len(syms) >= 12
    for s in syms:
        assert hasattr(lib, s), "libspectral.so does not export %s" % s


@pytest.mark.parametrize("variant", ("trp", "cub"))
def test_plugin_libraries_export_find_traj_only(variant):
    path = api.lib_path("lib%s.so" % variant)
    out = subprocess.run(["nm", "-D", "--defined-only", path], capture_output=True, text=True).stdout
    exported = [ln.split()[-1] for ln in out.splitlines() if " T " in ln]
    assert "find_traj" in exported
    # the reference's libtrp.so exports find_traj as its only C symbol (SURVEY.md 8b)
    assert [s for s in exported if not s.startswith("_")] == ["find_traj"]
    cdll = ctypes.CDLL(path)
    assert hasattr(cdll, "find_traj")


def test_struct_layouts_match_reference():
    assert ctypes.sizeof(api.Params) == 88
    assert api.Params.iteration.offset == 80
    assert api.CUBE_DTYPE.itemsize == 112
    off = {n: api.CUBE_DTYPE.fields[n][1] for n in api.CUBE_DTYPE.names}
    assert (off["beg_t"], off["end_t"], off["t"], off["t_dif"], off["beg_l"], off["end_l"]) == (0, 4, 8, 16, 24, 32)
    assert (off["upp_skew"], off["upp_bias"], off["down_skew"], off["down_bias"]) == (40, 48, 56, 64)
    assert (off["l_upp_skew"], off["l_upp_bias"], off["l_down_skew"], off["l_down_bias"]) == (72, 80, 88, 96)
    assert (off["merge"], off["split"], off["count"]) == (104, 105, 108)
    o = api.default_options()
    assert (o.max_iter, o.scaling, o.check_termination) == (5000, 4, 25)          # trp_wrapper.cpp:191, solve_3d.cc:1242
    assert (o.eps_abs, o.eps_rel, o.eps_prim_inf) == (1e-5, 1e-5, 2.5e-5)         # solve_3d.cc:1238-1239,1454
    assert (o.rho, o.sigma, o.alpha) == (0.1, 1e-6, 1.6)                          # OSQP defaults


def _cuda_available():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


@pytest.mark.skipif(_cuda_available(), reason="this checks the no-GPU failure mode")
def test_product_fails_loudly_without_a_gpu(tmp_path):
    with pytest.raises(RuntimeError, match="no CPU path"):
        api.SpectralPlanner(device=0, max_batch=4)
    # find_traj through the plugin: the reference's failure sentinel, no output file, and no oracle involved
    os.environ["SPECTRAL_IO_DIR"] = str(tmp_path)
    try:
        write_scenario_text(str(tmp_path / "c_road_s1_2.txt"), load_fixture("c1"))
        assert api._run_btrapz(api.Params(*WEIGHTS_FILE, 5), "trp") == api.FAIL_COST
        assert not (tmp_path / "s1_slt_3d_5.txt").exists()
    finally:
        os.environ.pop("SPECTRAL_IO_DIR", None)


def test_product_never_links_or_imports_the_oracle():
    for lib in ("libspectral.so", "libtrp.so", "libcub.so"):
        out = subprocess.run(["ldd", api.lib_path(lib)], capture_output=True, text=True).stdout
        assert "oracle" not in out
    for root, _, files in os.walk(os.path.join(H.ROOT, "spectral_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                src = open(os.path.join(root, f), errors="ignore").read()
                assert "pyoracle" not in src and "liboracle" not in src and "oracle/" not in src.replace("oracle/gen_golden.py", ""), f


@pytest.mark.parametrize("name", ("c1", "c7", "c_road_s1_2"))
def test_scenario_text_round_trip(tmp_path, name):
    sc = load_fixture(name)
    p = str(tmp_path / "in.txt")
    write_scenario_text(p, sc)
    back = read_scenario_text(p)
    assert back.n_knots == sc.n_knots and back.delta_t == sc.delta_t and back.n_regions == sc.n_regions
    for f in ("init_s", "init_l", "scalars", "s_bounds", "l_bounds", "ds_bounds", "dl_bounds", "s_ref", "l_ref"):
        assert np.array_equal(getattr(back, f), getattr(sc, f)), f
    # token count of the grammar: 19 + 4RN + 8N (SURVEY.md Appendix A; our writer emits zero kappas)
    ntok = len(open(p).read().split())
    assert ntok == 19 + 4 * sc.n_regions * sc.n_knots + 8 * sc.n_knots


def test_trajectory_text_reader_on_shipped_outputs():
    t = read_trajectory_text(os.path.join(H.GOLDEN, "s1_slt_3d_31.txt"))
    c = read_trajectory_text(os.path.join(H.GOLDEN, "s1_cub_3d_31.txt"))
    assert t.shape == (70, 7) and c.shape == (74, 7)
    assert np.allclose(t[:, 0], 0.1 * np.arange(70)) and t[0, 1] == 0.0 and t[0, 3] == 7.0


def test_scenario_batch_pack_slice_save_load(tmp_path):
    b = config2(12)
    assert b.batch == 12 and b.n_knots == 71 and b.n_regions == 2
    s = b.slice(3, 9)
    assert s.batch == 6 and np.array_equal(s.s_bounds, b.s_bounds[3:9])
    shapes = [a.shape for a in b.arrays()]
    assert shapes == [(12, 2, 71, 2), (12, 2, 71, 2), (12, 71, 2), (12, 71, 2), (12, 71), (12, 71), (12, 6), (12, 10)]
    p = str(tmp_path / "batch.npz")
    b.save(p)
    back = ScenarioBatch.load(p)
    for x, y in zip(b.arrays(), back.arrays()):
        assert np.array_equal(x, y)
    one = ScenarioBatch.from_scenarios([load_fixture("c1"), load_fixture("c3")])
    assert one.batch == 2


def test_reference_wrapper_surface_is_mirrored():
    """Same names / argument meaning as src/trp_wrapper.py:19-32,56-121."""
    names = [f[0] for f in api.Params._fields_]
    assert names == ["s_acc_weight", "s_jerk_weight", "l_acc_weight", "l_jerk_weight", "weight_s_ref", "weight_ds_ref",
                     "weight_l_ref", "weight_dl_ref", "weight_end_s", "weight_end_l", "iteration"]
    # the wrapper's Params field by field (ten c_double, then the c_int iteration) and its binding of the plugin symbol,
    # find_traj(POINTER(Params)) -> c_double (trp_wrapper.py:19-32,45-54): what an unchanged wrapper module relies on
    assert [f[1] for f in api.Params._fields_] == [ctypes.c_double] * 10 + [ctypes.c_int]
    assert [getattr(api.Params, n).offset for n in names] == [8 * i for i in range(11)]
    for variant in ("trp", "cub"):
        fn = api._plugin(variant).find_traj
        assert fn.argtypes == (ctypes.POINTER(api.Params),) and fn.restype is ctypes.c_double
    for fn in ("find_traj", "run_btrapz", "_run_btrapz"):
        assert callable(getattr(api, fn))

    class Trial:  # the Optuna trial protocol used by run_btrapz (trp_wrapper.py:69-80)
        def __init__(self):
            self.asked = []

        def suggest_float(self, name, lo, hi):
            self.asked.append((name, lo, hi))
            return 1.0

    if not _cuda_available():
        tr = Trial()
        os.environ["SPECTRAL_IO_DIR"] = "/nonexistent-dir"
        try:
            assert api.run_btrapz(tr, "trp") == api.FAIL_COST  # unreadable input -> sentinel, not a crash
        finally:
            os.environ.pop("SPECTRAL_IO_DIR", None)
        assert [a[0] for a in tr.asked] == names[:10] and all(a[1:] == (0, 50) for a in tr.asked)


def test_config3_groups_share_one_kkt_structure():
    """BASELINE configs[2] generator: within a group every scenario has the same segment count and time allocation (the
    KKT structure), only bounds / initial state / references differ; groups differ in their time allocation; scenario b
    does not depend on the batch it is generated in."""
    import pyoracle as po
    from spectral_b200.scenarios import WEIGHTS_FILE, config3
    G, B = 8, 256
    batch = config3(B, groups=G)
    r = po.solve_batch("trp", batch, WEIGHTS_FILE, mode=0, nthreads=0)
    sig = [(int(r["K"][b]),) + tuple(np.round(r["segs"][b, :r["K"][b]]["t"], 9)) for b in range(B)]
    per_group = [set(sig[b] for b in range(B) if b % G == g) for g in range(G)]
    assert all(len(x) == 1 for x in per_group), per_group
    assert len(set.union(*per_group)) >= G - 1
    assert not np.array_equal(batch.s_bounds[G], batch.s_bounds[2 * G])  # same group, different bounds
    tail = config3(16, groups=G, first=B - 16)
    for a, b in zip(tail.arrays(), batch.arrays()):
        assert np.array_equal(a, b[B - 16:])


# ---------------------------------------------------------------- the reference's OWN wrapper modules, unchanged
REF_SRC = "/root/reference/src"
REF_PYC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "wrappers")   # oracle/Makefile
REF_LIB_DIR = "/home/srujan_d/RISS/code/btrapz/src"   # the literal path the wrappers CDLL() (trp_wrapper.py:45, cub_wrapper.py)


def _stage_reference_wrapper(tmp_path, monkeypatch, module):
    """Installs OUR libtrp.so / libcub.so / libspectral.so at the literal path the reference's wrapper loads from, puts a
    stub `optuna` on sys.path (the wrappers import it at module top, trp_wrapper.py:3; it is not installed here) and imports
    the reference's module from /root/reference/src WITHOUT editing it (on the GPU box, which has no /root/reference: from the
    byte-compiled modules oracle/Makefile made of those files, oracle/_ref/wrappers/*.pyc -- same code objects, no source)."""
    import importlib
    import shutil
    import sys
    pyc = os.path.join(REF_PYC, module + ".pyc.bin")
    if not os.path.isdir(REF_SRC) and not os.path.exists(pyc):
        pytest.skip("neither /root/reference nor oracle/_ref/wrappers (built by oracle/Makefile) is present on this machine")
    try:
        os.makedirs(REF_LIB_DIR, exist_ok=True)
    except OSError:
        pytest.skip("cannot create " + REF_LIB_DIR)
    for name in ("libspectral.so", "libtrp.so", "libcub.so"):
        # (copy + rename: an earlier test of this process may still have the old file mapped; writing into it in place crashes)
        shutil.copy(api.lib_path(name), os.path.join(REF_LIB_DIR, name + ".new"))
        os.replace(os.path.join(REF_LIB_DIR, name + ".new"), os.path.join(REF_LIB_DIR, name))
    stub = tmp_path / "stub"
    stub.mkdir()
    (stub / "optuna.py").write_text("def create_study(*a, **k):\n    raise RuntimeError('stub')\n")
    monkeypatch.syspath_prepend(str(stub))
    sys.modules.pop(module, None)
    if os.path.isdir(REF_SRC):     # the sources where they lie
        monkeypatch.syspath_prepend(REF_SRC)
        return importlib.import_module(module)
    import importlib.machinery     # their byte-compiled form (same code objects)
    import importlib.util
    loader = importlib.machinery.SourcelessFileLoader(module, pyc)
    mod = importlib.util.module_from_spec(importlib.util.spec_from_loader(module, loader))
    loader.exec_module(mod)
    return mod


@pytest.mark.parametrize("module", ["trp_wrapper", "cub_wrapper"])
def test_unchanged_reference_wrapper_binds_our_library(tmp_path, monkeypatch, module):
    """src/trp_wrapper.py / src/cub_wrapper.py (unmodified) load our drop-in .so from their hard-coded path and bind
    find_traj(POINTER(Params)) -> c_double (trp_wrapper.py:45-54); their Params is our SpectralParams byte for byte.
    Without a GPU the call itself must FAIL LOUDLY (sentinel 1e11 -> the wrapper's find_traj() returns False), never
    compute on the CPU.  The numerical comparison through the same modules is the GPU test
    test_gpu_parity.py::test_unchanged_reference_wrapper_reproduces_shipped_output."""
    w = _stage_reference_wrapper(tmp_path, monkeypatch, module)
    assert w.cdll._name == os.path.join(REF_LIB_DIR, "libtrp.so" if module == "trp_wrapper" else "libcub.so")
    assert ctypes.sizeof(w.Params) == ctypes.sizeof(api.Params) == 88
    for (n0, t0), (n1, t1) in zip(w.Params._fields_, api.Params._fields_):
        assert n0 == n1 and t0 is t1 and getattr(w.Params, n0).offset == getattr(api.Params, n1).offset
    assert w._run_btrapz.restype is ctypes.c_double and w._run_btrapz.argtypes == (ctypes.POINTER(w.Params),)
    import torch
    if not torch.cuda.is_available():
        from spectral_b200.scenarios import load_fixture
        from spectral_b200.wire import write_scenario_text
        write_scenario_text(os.path.join(REF_LIB_DIR, "c_road_s1_2.txt" if module == "trp_wrapper" else "c_road_s1_3.txt"),
                            load_fixture("c1"))
        assert w._run_btrapz(w.Params(35.73, 41.61, 25.57, 41.59, 0.12, 10.04, 0.0, 0.0, 7.27, 32.13, 31)) == 100000000000
