"""CPU-side checks of frozen seats: the ctypes mirror of ia2c_frozen_seats has the C layout, ia2c_train_episode_frozen is
exported, and every refusal of the entry point happens before any device work (all descriptor pointers below point
nowhere)."""
import ctypes as C
import os
import re
import subprocess

import pytest

from tests.conftest import ROOT

HEADER = os.path.join(ROOT, "include", "ia2c_b200.h")
INVALID, UNSUPPORTED = -1, -3
_PTRS = ("actor_params", "critic_params", "obs", "reward", "act", "partner_true", "partner_pred", "env_state", "env_hist",
         "env_cls", "env_elapsed", "ep_return", "belief_records", "filter_action", "critic_grad", "actor_grad", "critic_m",
         "critic_v", "actor_m", "actor_v", "actor_grad_accum", "critic_step", "actor_step", "loss_out", "partials")


def test_frozen_seats_layout_and_export(tmp_path):
    from ia2c_b200 import _lib
    prog = ('#include <stdio.h>\n#include <stddef.h>\n#include "%s"\nint main(){printf("%%zu %%zu", sizeof(ia2c_frozen_seats),'
            ' offsetof(ia2c_frozen_seats, mask));return 0;}\n' % HEADER)
    c = tmp_path / "layout.c"
    c.write_text(prog)
    exe = tmp_path / "layout"
    subprocess.run(["gcc", str(c), "-o", str(exe)], check=True)
    size, off = (int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split())
    assert (size, off) == (C.sizeof(_lib.FrozenSeats), _lib.FrozenSeats.mask.offset) == (32, 0)
    lib = _lib.load()
    assert hasattr(lib, "ia2c_train_episode_frozen") and "ia2c_train_episode_frozen" in _lib.SIGNATURES
    assert re.search(r"\bint ia2c_train_episode_frozen\(", open(HEADER).read())


def _descs(N=2, M=5, flags=None):
    from ia2c_b200 import _lib
    lib = _lib.load()
    d = _lib.EpisodeDesc()
    d.E, d.E_total, d.env_offset, d.N, d.T, d.M = 10, 10, 0, N, 30, M
    d.flags = flags if flags is not None else (_lib.FLAG_FUSED_ROLLOUT | _lib.FLAG_FUSED_CRITIC if N <= 8 else 0) | _lib.FLAG_ACTOR_COLUMNS
    for name in _PTRS:
        setattr(d, name, 0x1000)
    d.partials_floats = 1 << 40
    r = _lib.RunsDesc()
    r.runs, r.seed = 4, 0x1000
    f = _lib.FrozenSeats()
    f.mask[0] = 1 << (N - 1)
    return lib, d, r, f


def _call(lib, d, r, f, p=None, w=None):
    return lib.ia2c_train_episode_frozen(C.byref(d), C.byref(r) if r is not None else None, p, w,
                                         C.byref(f) if f is not None else None, None)


def _mask(f, seats):
    for k in range(4):
        f.mask[k] = 0
    for s in seats:
        f.mask[s >> 6] |= 1 << (s & 63)


def _case(name):
    from ia2c_b200 import _lib
    N = 16 if name in ("no ACTOR_COLUMNS at N > 8", "tapes in a batch N=16") else (300 if name == "N=300" else 2)
    lib, d, r, f = _descs(N=N)
    runs = None
    if name == "null mask":
        f = None
    elif name == "bit at N":
        _mask(f, [0, 2])
    elif name == "bit in a high word":
        _mask(f, [0, 200])
    elif name == "no seat frozen":
        _mask(f, [])
    elif name == "every seat frozen":
        _mask(f, [0, 1])
    elif name == "SKIP_ADAM":
        d.flags |= _lib.FLAG_SKIP_ADAM
    elif name == "GRAD_ONLY":
        d.flags |= _lib.FLAG_GRAD_ONLY
    elif name == "env_offset":
        d.env_offset, d.E_total = 10, 20
    elif name == "ROLLOUT_PER_STEP":
        d.flags |= _lib.FLAG_ROLLOUT_PER_STEP
    elif name == "BELIEF_PER_STEP":
        d.flags |= _lib.FLAG_BELIEF_PER_STEP
    elif name == "no FUSED_ROLLOUT at N <= 8":
        d.flags &= ~(_lib.FLAG_FUSED_ROLLOUT | _lib.FLAG_FUSED_CRITIC)
    elif name == "no ACTOR_COLUMNS at N <= 8":
        d.flags &= ~_lib.FLAG_ACTOR_COLUMNS
    elif name == "no ACTOR_COLUMNS at N > 8":
        d.flags &= ~_lib.FLAG_ACTOR_COLUMNS
    elif name == "N=300":
        pass
    elif name == "tapes in a batch":
        d.inj_u_action, runs = 0x1000, r
    elif name == "tapes in a batch N=16":
        d.inj_u_belief, runs = 0x1000, r
    elif name == "priority without pool":
        return lib, d, runs, f, C.byref(_lib.PartnerPriorityDesc())
    return lib, d, runs, f, None


CASES = [
    ("null mask", INVALID, "null frozen-seat mask"),
    ("bit at N", INVALID, "at or above N"),
    ("bit in a high word", INVALID, "at or above N"),
    ("no seat frozen", INVALID, "at least one seat must be frozen and one trained"),
    ("every seat frozen", INVALID, "at least one seat must be frozen and one trained"),
    ("SKIP_ADAM", UNSUPPORTED, "SKIP_ADAM"),
    ("GRAD_ONLY", UNSUPPORTED, "GRAD_ONLY"),
    ("env_offset", UNSUPPORTED, "env_offset"),
    ("ROLLOUT_PER_STEP", UNSUPPORTED, "per-step"),
    ("BELIEF_PER_STEP", UNSUPPORTED, "per-step"),
    ("no FUSED_ROLLOUT at N <= 8", UNSUPPORTED, "fused rollout"),
    ("no ACTOR_COLUMNS at N <= 8", UNSUPPORTED, 'actor_kernel="columns"'),
    ("no ACTOR_COLUMNS at N > 8", UNSUPPORTED, 'actor_kernel="columns"'),
    ("N=300", UNSUPPORTED, "N above 256"),
    ("tapes in a batch", UNSUPPORTED, "injected replay tapes"),
    ("tapes in a batch N=16", UNSUPPORTED, "injected replay tapes"),
    ("priority without pool", INVALID, "need the per-env pool"),
]


@pytest.mark.parametrize("name,status,msg", CASES, ids=[c[0] for c in CASES])
def test_frozen_refusals_before_any_device_work(name, status, msg):
    from ia2c_b200 import _lib
    lib, d, runs, f, w = _case(name)
    assert _call(lib, d, runs, f, w=w) == status
    assert msg in lib.ia2c_last_error().decode()


def test_frozen_launch_count_unchanged_by_refusals():
    from ia2c_b200 import _lib
    before = _lib.launch_count()
    for name, _, _ in CASES:
        lib, d, runs, f, w = _case(name)
        _call(lib, d, runs, f, w=w)
    assert _lib.launch_count() == before


def test_frozen_set_accepts_every_form_of_seats():
    """freeze_seats' host-side parsing: a set, a list, a numpy array and a tensor (PartnerPool.seats is one) give the same
    set, and every malformed set is refused."""
    import numpy as np
    import torch

    from ia2c_b200.partners import SeatsPartners

    class Stub(SeatsPartners):
        N = 5

    s = Stub()
    for seats in ({0, 3}, [3, 0], (0, 3, 3), np.array([0, 3], dtype=np.int32), torch.tensor([0, 3], dtype=torch.int32)):
        assert s._frozen_set(seats) == frozenset({0, 3})
    for bad in (1, {5}, {-1}, set(), {0, 1, 2, 3, 4}, np.array([0.5])):
        with pytest.raises(ValueError):
            s._frozen_set(bad)
