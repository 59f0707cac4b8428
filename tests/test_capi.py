"""CPU-side checks of the drop-in boundary: the shared library loads and exports every symbol that
include/ia2c_b200.h declares, and the ctypes mirror of ia2c_episode_desc has the C layout."""
import os
import re
import subprocess
import sys

import pytest

from tests.conftest import ROOT

HEADER = os.path.join(ROOT, "include", "ia2c_b200.h")


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(ia2c_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from ia2c_b200 import _lib
    lib = _lib.load()
    names = declared_symbols()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/ia2c_b200.h but not exported"
    assert set(names) == set(_lib.SIGNATURES), set(names) ^ set(_lib.SIGNATURES)
    assert lib.ia2c_abi_version() == _lib.ABI_VERSION and lib.ia2c_last_error() is not None


def test_episode_desc_layout_matches_c(tmp_path):
    import ctypes
    from ia2c_b200 import _lib
    fields = [f[0] for f in _lib.EpisodeDesc._fields_]
    prog = '#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu", sizeof(ia2c_episode_desc));' % HEADER
    for f in fields:
        prog += 'printf(" %%zu", offsetof(ia2c_episode_desc, %s));' % f
    prog += "return 0;}\n"
    c = tmp_path / "layout.c"
    c.write_text(prog)
    exe = tmp_path / "layout"
    subprocess.run(["gcc", str(c), "-o", str(exe)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert out[0] == ctypes.sizeof(_lib.EpisodeDesc)
    assert out[1:] == [getattr(_lib.EpisodeDesc, f).offset for f in fields]


def test_no_cpu_fallback_without_cuda():
    import torch
    from ia2c_b200 import _lib
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    with pytest.raises(_lib.IA2CError, match="no CPU fallback"):
        from ia2c_b200.org_env import OrgVecEnv
        OrgVecEnv(4)
    with pytest.raises(_lib.IA2CError):
        from ia2c_b200.trainer import IA2CTrainer
        IA2CTrainer(4)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "ia2c_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f


def test_compat_modules_export_reference_names():
    sys.path.insert(0, os.path.join(ROOT, "ia2c_b200", "compat"))
    try:
        import ac_nets
        for n in ("torch", "nn", "F", "np", "Adam", "Categorical", "hidden_size", "NeuralNet", "CriticNetwork", "ActorNetwork"):
            assert hasattr(ac_nets, n), n
        assert ac_nets.hidden_size == 6
        import belief_filter
        import Org as org_mod
        assert hasattr(belief_filter, "BeliefFilter") and hasattr(org_mod, "Org")
        assert (org_mod.MEM, org_mod.MEM_SIZE, org_mod.STATE_VISIBLE) == (True, 1, False)
    finally:
        sys.path.pop(0)
        for m in ("ac_nets", "belief_filter", "Org"):
            sys.modules.pop(m, None)


@pytest.mark.parametrize("script", ["a2c_org_test.py", "ia2c.py"])
def test_unmodified_reference_scripts_resolve_against_the_drop_in_modules(script, tmp_path):
    """Without a GPU: the reference's scripts, unmodified and run from where they lie, must import the drop-in
    modules and reach the first CUDA call — where the product raises its loud no-fallback error."""
    import torch
    from oracle import ref_runner
    ref, origin = ref_runner.find_reference()
    if ref is None:
        pytest.skip(f"reference sources not staged: {origin}")
    if torch.cuda.is_available():
        pytest.skip("CUDA present: the scripts would train for hours")
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([ROOT, os.path.join(ROOT, "ia2c_b200", "compat"), os.path.join(ROOT, "ia2c_b200", "compat_gym")])
    # -P: do not put the script's own directory (which holds the reference modules) in front of PYTHONPATH
    r = subprocess.run([sys.executable, "-P", os.path.join(ref, script)], capture_output=True, text=True, env=env, cwd=str(tmp_path), timeout=300)
    assert r.returncode != 0
    assert "no CPU fallback" in r.stderr, r.stderr[-2000:]
    assert "ModuleNotFoundError" not in r.stderr and "ImportError" not in r.stderr


def test_changed_hidden_size_is_refused_not_ignored(monkeypatch):
    """ac_nets re-exports hidden_size (the scripts star-import it); the kernels are compiled for 6 — anything else must raise."""
    import pytest
    from ia2c_b200 import _lib, nets

    monkeypatch.setattr(nets, "hidden_size", 8)
    with pytest.raises(_lib.IA2CError, match="hidden_size"):
        nets._check_hidden_size()
    monkeypatch.setattr(nets, "hidden_size", 6)
    nets._check_hidden_size()
