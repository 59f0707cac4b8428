"""CPU tests of the host-side helpers added in round 2: the script launcher's constant substitution, the staged-reference
manifest, the NUMA helper's parsing and bench.py's block statistics."""
import json
import os

import pytest

from tests.conftest import ROOT


def test_launcher_substitutes_module_level_constants_only():
    from ia2c_b200 import launcher

    src = "import x\nNUM_EPISODES = 5000\nn_envs=10  # comment\nfor i in range(NUM_EPISODES):\n    n_envs_local = 3\n"
    out = launcher.substitute(src, {"NUM_EPISODES": "3", "n_envs": "64"})
    assert "NUM_EPISODES = 3\n" in out and "n_envs = 64  # comment" in out and "range(NUM_EPISODES)" in out and "n_envs_local = 3" in out
    with pytest.raises(ValueError, match="no module-level assignment"):
        launcher.substitute(src, {"n_updates": "4"})
    paths = launcher.dropin_paths()
    assert paths[-1].endswith(os.path.join("ia2c_b200", "compat")) and all(os.path.isdir(p) for p in paths)


def test_staged_reference_manifest_detects_modification(tmp_path):
    from oracle import make_ref

    src = tmp_path / "ref"
    src.mkdir()
    for f in make_ref.FILES:
        (src / f).write_text(f"# {f}\n")
    dst = tmp_path / "staged"
    m = make_ref.stage(str(src), str(dst))
    assert set(m["files"]) == set(make_ref.FILES) and make_ref.verify(str(dst))["files"] == m["files"]
    (dst / "ia2c.py").write_text("# tampered\n")
    with pytest.raises(RuntimeError, match="modified after staging"):
        make_ref.verify(str(dst))
    with pytest.raises(FileNotFoundError):
        make_ref.stage(str(tmp_path / "missing"), str(dst))


def test_staged_reference_is_git_ignored():
    from oracle import make_ref

    ignore = open(os.path.join(ROOT, ".gitignore")).read().split()
    assert make_ref.REF_DST == os.path.join(ROOT, "oracle", "_ref") and "oracle/_ref/" in ignore


def test_hostmem_cpulist_parsing_and_bind_never_raises():
    from ia2c_b200 import hostmem

    assert hostmem._parse_cpulist("0-3,8,10-11\n") == {0, 1, 2, 3, 8, 10, 11} and hostmem._parse_cpulist("") == set()
    before = os.sched_getaffinity(0)
    hostmem.unbind(before)
    assert os.sched_getaffinity(0) == before


def test_bench_block_statistics_and_reference_budget():
    import bench

    s = bench.med_spread([3.0, 1.0, 2.0])
    assert s == {"median": 2.0, "min": 1.0, "max": 3.0, "blocks": 3}
    assert "4096 envs per GPU" in bench.headline_workload(2, 4096, 8192)
    # the ours-arm and reference-arm lines quote the same workload string
    assert bench.headline_workload(2, 4096, 4096) == bench.headline_workload(2, 4096, 32768)
    json.dumps(s)
