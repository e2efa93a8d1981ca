"""CPU suite: the seed-exact spawn of csrc/spawn_core.h (the scenes mm_reset_seeded builds on the device) against
spawn.spawn_scene, through the g++ build of its host harness, and the argument checks of mm_reset_seeded."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT

TRAFFIC = ("cav", "mixed", "av", "hdv")
EDGE_SEEDS = (0, 1, 2 ** 31 - 1, 2 ** 31, 2 ** 32 - 1)


@pytest.fixture(scope="module")
def spawn_host(tmp_path_factory):
    src = os.path.join(ROOT, "marl-mass_b200", "csrc", "spawn_host.cpp")
    lib_path = str(tmp_path_factory.mktemp("spawn_host") / "libspawn_host.so")
    subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-std=c++17", "-shared", "-fPIC", src, "-o", lib_path])
    lib = ctypes.CDLL(lib_path)
    lib.mm_spawn_host.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int] + \
                                 [ctypes.c_void_p] * 9

    def run(seeds, num_cav, density, traffic):
        n = len(seeds)
        seeds = np.ascontiguousarray(seeds, np.uint32)
        num_cav = np.ascontiguousarray(num_cav, np.int32)
        out = {k: np.zeros(n, np.int32) for k in ("status", "n_veh", "n_cav", "n_merge")}
        out["fits"] = np.zeros(n, np.uint8)
        out["kind"] = np.zeros((n, 12), np.int32)
        out.update({k: np.zeros((n, 12), np.float64) for k in ("x", "y", "speed")})
        rc = lib.mm_spawn_host(seeds.ctypes.data, num_cav.ctypes.data, n, density, TRAFFIC.index(traffic),
                               *[out[k].ctypes.data for k in ("status", "fits", "n_veh", "n_cav", "n_merge", "kind", "x", "y",
                                                              "speed")])
        assert rc == 0
        return out
    return run


def _reference(seeds, num_cav, density, traffic):
    """spawn.spawn_scene per seed: (status, scene) with status 0 ok, 1 raises, 2 more than 11 vehicles."""
    from marl_mass_b200 import spawn
    res = []
    for s, c in zip(seeds, num_cav):
        try:
            v, n_merge = spawn.spawn_scene(int(s), density, traffic, int(c))
        except ValueError:
            res.append((1, None, None))
            continue
        res.append((2 if len(v) > 11 else 0, v, n_merge))
    return res


def _compare(got, want, seeds, num_cav):
    for i, (status, v, n_merge) in enumerate(want):
        what = "seed %d num_CAV %d" % (seeds[i], num_cav[i])
        assert got["status"][i] == status, what
        assert bool(got["fits"][i]) == (status == 0), what
        if status == 1:
            continue
        n = len(v)
        assert got["n_veh"][i] == n and got["n_merge"][i] == n_merge, what
        assert got["n_cav"][i] == sum(1 for k, *_ in v if k == 1), what
        assert got["kind"][i, :n].tolist() == [k for k, *_ in v], what
        for j, key in ((1, "x"), (2, "y"), (3, "speed")):
            want_col = np.array([veh[j] for veh in v], np.float64)
            assert np.array_equal(got[key][i, :n], want_col), (what, key)      # bit for bit
        assert not got["kind"][i, n:].any()


@pytest.mark.parametrize("density", (1, 2, 3))
@pytest.mark.parametrize("traffic", TRAFFIC)
def test_spawn_core_equals_spawn_scene(spawn_host, density, traffic):
    """17 000 seeds per (density, traffic type), 204 000 in all: random seeds over [0, 2^32) and the edge seeds, each with
    num_CAV cycling through 0 (drawn) and every value 1..11 - the valid ones must give the reference's scene bit for bit
    (kinds, x, y, speed, n_merge), the others must be reported as the reference fails them (ValueError, or a scene of
    12 vehicles that no env holds), and spawn_fits must agree."""
    rng = np.random.RandomState(1000 * density + TRAFFIC.index(traffic))
    n = 17000
    seeds = np.concatenate([np.array(EDGE_SEEDS, np.int64), rng.randint(0, 2 ** 32, size=n - len(EDGE_SEEDS), dtype=np.int64)])
    num_cav = np.arange(n) % 12
    got = spawn_host(seeds, num_cav, density, traffic)
    _compare(got, _reference(seeds, num_cav, density, traffic), seeds, num_cav)


def test_spawn_core_covers_the_evaluation_rule(spawn_host):
    """The per-episode num_CAV of the training-time evaluation (eval_num_cav) on every density: always a valid scene."""
    from marl_mass_b200.evaluation import eval_num_cav
    for density in (1, 2, 3):
        seeds = np.arange(3000, dtype=np.int64) * 7919
        num_cav = np.array([eval_num_cav(i, density) for i in range(len(seeds))])
        for traffic in TRAFFIC:
            got = spawn_host(seeds, num_cav, density, traffic)
            assert (got["status"] == 0).all() and got["fits"].all()
            _compare(got, _reference(seeds, num_cav, density, traffic), seeds, num_cav)


def test_reset_seeded_rejects_bad_arguments_before_any_cuda_call():
    """mm_reset_seeded refuses a null handle and null seeds; mm_check_seeds - the checks it runs first, for a handle of a
    given config, with no device involved - refuses seeds outside [0, 2^32) (numpy raises ValueError there), a num_CAV
    outside 0..11 and a num_CAV for which spawn_scene would raise or build more than 11 vehicles."""
    import marl_mass_b200 as mm
    from marl_mass_b200 import _lib
    L = mm.lib()
    seeds = np.array([0, 1, 2 ** 32 - 1], np.int64)
    assert L.mm_reset_seeded(None, seeds.ctypes.data, None, None) == -1
    assert b"env is null" in L.mm_last_error()

    def check(cfg, seeds, num_cav=None):
        seeds = np.ascontiguousarray(seeds, np.int64)
        nc = None if num_cav is None else np.ascontiguousarray(num_cav, np.int32)
        return L.mm_check_seeds(ctypes.byref(mm.make_mm_config(cfg)), len(seeds), seeds.ctypes.data,
                                None if nc is None else nc.ctypes.data)

    cfg = dict(mm.DEFAULT_CONFIG, traffic_density=3, traffic_type="mixed")
    assert check(cfg, seeds) == 0
    assert check(cfg, seeds, [5, 0, 4]) == 0
    for bad in (-1, 2 ** 32, 2 ** 40):
        assert check(cfg, [0, bad]) == -1
        assert b"seed" in L.mm_last_error() and b"[0, 2^32)" in L.mm_last_error()
    for bad in (-1, 12):
        assert check(cfg, [3, 4], [0, bad]) == -1
        assert b"num_CAV" in L.mm_last_error()
    # density 3 draws 3..5 HDVs: num_CAV 9 never fits (12 or more vehicles), 7 fits or not depending on the seed
    assert check(cfg, [3], [9]) == -1 and b"num_CAV" in L.mm_last_error()
    from marl_mass_b200 import spawn
    verdict = []
    for s in range(40):
        try:
            ok = len(spawn.spawn_scene(s, 3, "mixed", 7)[0]) <= 11
        except ValueError:
            ok = False
        verdict.append(ok)
        assert (check(cfg, [s], [7]) == 0) == ok, s
    assert any(verdict) and not all(verdict)
    assert check(cfg, [0], None) == 0 and check(cfg, np.zeros(0, np.int64)) == -1
    with pytest.raises(_lib.MMError):
        _lib.check(check(cfg, [2 ** 32]))
