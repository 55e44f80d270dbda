"""The C-ABI library builds, loads, and exports every symbol include/dgp_b200.h declares (no compute without a GPU)."""
import os
import re

import pytest


def header_symbols():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    text = open(os.path.join(root, "include", "dgp_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(dgp_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_header(lib_built):
    from deepgraphpose_b200 import _lib
    lib = _lib.load()
    syms = header_symbols()
    assert len(syms) >= 15
    for s in syms:
        assert hasattr(lib, s), "missing export %s" % s
        assert s in _lib.SIGNATURES, "no ctypes signature for %s" % s
    assert sorted(_lib.SIGNATURES) == syms


def test_output_dims_closed_form(lib_built):
    from deepgraphpose_b200.engine import output_dims
    assert output_dims(747, 832) == ((47, 52), (94, 104))
    assert output_dims(470, 640) == ((30, 40), (60, 80))
    assert output_dims(1024, 1280) == ((64, 80), (128, 160))


def test_no_gpu_fails_loudly(lib_built):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from deepgraphpose_b200._lib import DgpError
    from deepgraphpose_b200.engine import Engine
    with pytest.raises(DgpError):
        Engine(4)
    # and at the C level: dgp_create reports the missing device instead of falling back
    import ctypes as C
    from deepgraphpose_b200 import _lib
    lib = _lib.load()
    cfg = _lib.DgpConfig()
    cfg.num_joints = 4
    h = C.c_void_p()
    rc = lib.dgp_create(C.byref(cfg), C.byref(h))
    assert rc != 0 and b"no CPU fallback" in lib.dgp_last_error(None)


def test_product_never_imports_oracle():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pkg = os.path.join(root, "deepgraphpose_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle", src, flags=re.M), fn


def test_library_reads_only_the_plan_printing_env_var():
    """What the library computes depends on its inputs alone: the one environment variable it reads prints the plan."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    csrc = os.path.join(root, "deepgraphpose_b200", "csrc")
    args = []
    for fn in sorted(os.listdir(csrc)):
        src = open(os.path.join(csrc, fn)).read()
        args += [(fn, a.strip()) for a in re.findall(r"\bgetenv\s*\(([^)]*)\)", src)]
    assert [a for _, a in args] == ['"DGP_DEBUG_PLAN"'], args


def test_ctypes_structs_match_the_header(tmp_path):
    """sizeof / offsetof of every struct of include/dgp_b200.h (compiled with gcc) against the ctypes mirrors in _lib.py."""
    import ctypes as C
    import shutil
    import subprocess
    from deepgraphpose_b200 import _lib
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pairs = {"dgp_config": _lib.DgpConfig, "dgp_loss_cfg": _lib.DgpLossCfg, "dgp_loss_batch": _lib.DgpLossBatch,
             "dgp_cyclic_source": _lib.DgpCyclicSource}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "dgp_b200.h"', "int main(void) {"]
    for cname, ct in pairs.items():
        lines.append('  printf("%s %%zu\\n", sizeof(%s));' % (cname, cname))
        for fname, _ in ct._fields_:
            lines.append('  printf("%s.%s %%zu\\n", offsetof(%s, %s));' % (cname, fname, cname, fname))
    lines += ["  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for cname, ct in pairs.items():
        assert int(got[cname]) == C.sizeof(ct), (cname, got[cname], C.sizeof(ct))
        for fname, _ in ct._fields_:
            assert int(got["%s.%s" % (cname, fname)]) == getattr(ct, fname).offset, (cname, fname)
