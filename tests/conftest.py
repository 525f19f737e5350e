import hashlib
import importlib
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


def golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def pkg_module(name):
    import _b200_alias
    _b200_alias.load_package()
    return importlib.import_module(_b200_alias.PKG + "." + name)


@pytest.fixture(scope="session")
def built():
    """Everything compiled (no-op when up to date)."""
    import __graft_entry__ as g
    g.build()
    return True


@pytest.fixture(scope="session")
def he_sd():
    from oracle import net_port
    return net_port.he_state_dict(1234)


POST_CASES = {
    "p1": lambda s: s.stick_figures(1, 1)[:2], "p3": lambda s: s.stick_figures(3, 3)[:2],
    "p8": lambda s: s.stick_figures(8, 8)[:2], "p30": lambda s: s.stick_figures(30, 30)[:2],
    "noise0": lambda s: s.noise_maps(0),
    "empty": lambda s: (np.zeros((46, 46, 19), np.float32), np.zeros((46, 46, 38), np.float32)),
    "p5_40x52": lambda s: s.stick_figures(5, 55, h=40, w=52)[:2],
}


class RecordedPafprocess:
    """The getters of the reference's own pafprocess.cpp (the SWIG module's surface) as it answered on the scenarios of
    oracle/synth.fuzz_scenario (golden pafprocess_ref, written by tests/golden/make_golden.py)."""

    def __init__(self):
        g = golden("pafprocess_ref")
        self._digest, self._count = g["fuzz_digest"], g["fuzz_humans"]
        self._score, self._cid, self._part = g["fuzz_score"], g["fuzz_cid"], g["fuzz_part"]
        self._start = np.concatenate([[0], np.cumsum(np.maximum(self._count, 0))])

    def select(self, t, jl, paf):
        """Stands for process_paf on scenario t; jl / paf must be the inputs the recording was made from."""
        h = hashlib.sha256()
        for a in (jl, paf):
            h.update(np.ascontiguousarray(a).tobytes())
        assert h.hexdigest()[:16] == str(self._digest[t]), "scenario %d differs from the recorded input" % t
        assert self._count[t] >= 0, "scenario %d was not recorded" % t
        self._lo, self._n = int(self._start[t]), int(self._count[t])
        self._peaks = {int(c): tuple(self._part[self._lo + hid, p]) for hid in range(self._n) for p, c in
                       enumerate(self._cid[self._lo + hid]) if c >= 0}

    def get_num_humans(self):
        return self._n

    def get_score(self, hid):
        return float(self._score[self._lo + hid])

    def get_part_cid(self, hid, part):
        return int(self._cid[self._lo + hid, part])

    def get_part_x(self, cid):
        return int(self._peaks[cid][0])

    def get_part_y(self, cid):
        return int(self._peaks[cid][1])

    def get_part_score(self, cid):
        return float(np.float32(self._peaks[cid][2]))


def humans_rows_to_dicts(rows):
    """golden `humans` array [k, 1+18*3] -> [(score, {part: (x, y, s)})]"""
    out = []
    for r in rows:
        parts = {p: tuple(float(v) for v in r[1 + 3 * p: 4 + 3 * p]) for p in range(18) if r[1 + 3 * p] >= 0}
        out.append((float(r[0]), parts))
    return out


def assert_humans_equal(got, want, coord_tol=0.0, score_tol=2e-6):
    assert len(got) == len(want), "human count %d vs %d" % (len(got), len(want))
    for i, ((gs, gp), (ws, wp)) in enumerate(zip(got, want)):
        assert sorted(gp) == sorted(wp), "human %d parts differ: %s vs %s" % (i, sorted(gp), sorted(wp))
        for p in gp:
            assert abs(gp[p][0] - wp[p][0]) <= coord_tol and abs(gp[p][1] - wp[p][1]) <= coord_tol, (i, p, gp[p], wp[p])
            assert abs(gp[p][2] - wp[p][2]) <= score_tol, (i, p, gp[p], wp[p])
        assert abs(gs - ws) <= 1e-5, (i, gs, ws)
