"""CPU suite for the evaluation's shield records (mm_eval_shield_record): the C ABI, its ctypes mirror and the argument
checks that come before any device work."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT

HEADER = os.path.join(ROOT, "include", "marl_mass_b200.h")
INI = os.path.join(ROOT, "examples", "mass_td3_srew.ini")


def test_header_declares_and_library_exports_the_entry_point():
    import marl_mass_b200 as mm
    from marl_mass_b200 import _lib
    src = open(HEADER).read()
    assert re.search(r"int mm_eval_shield_record\(mm_env \*env, const mm_eval_shield_records \*rec, int t, void \*stream\);",
                     src)
    assert "mm_eval_shield_record" in _lib.EXPORTS
    assert mm.lib().mm_eval_shield_record is not None
    assert re.search(r"#define MM_ABI_VERSION 9\b", src)


def test_ctypes_struct_matches_the_header(tmp_path):
    """Every field's offset and the struct's size, as g++ lays out the header's mm_eval_shield_records."""
    from marl_mass_b200 import _lib
    S = _lib.MMEvalShieldRecords
    names = [f for f, _ in S._fields_]
    prog = tmp_path / "layout.cpp"
    prog.write_text('#include <cstdio>\n#include <cstddef>\n#include "marl_mass_b200.h"\nint main() {\n' +
                    'printf("%zu\\n", sizeof(mm_eval_shield_records));\n' +
                    "".join('printf("%%zu\\n", offsetof(mm_eval_shield_records, %s));\n' % f for f in names) + "}\n")
    exe = tmp_path / "layout"
    subprocess.check_call(["g++", "-std=c++17", "-I", os.path.dirname(HEADER), str(prog), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert got[0] == ctypes.sizeof(S)
    assert got[1:] == [getattr(S, f).offset for f in names]
    # every pointer of the header is in the mirror: nothing left out between fields
    fields = open(HEADER).read().split("} mm_eval_shield_records;")[0].rsplit("typedef struct {", 1)[1]
    fields = re.sub(r"/\*.*?\*/", "", fields, flags=re.S)
    assert sorted(re.findall(r"\*(\w+)", fields) + ["T"]) == sorted(names)


def _records(**kw):
    """Records with every required pointer set to a dummy non-null address (never dereferenced: the checks fail first)."""
    from marl_mass_b200 import _lib
    req = ("n_agents", "active") + _lib.SHIELD_COUNTS + _lib.SHIELD_F64
    return _lib.MMEvalShieldRecords(**dict({k: 0x1000 for k in req}, **dict({"T": 100}, **kw)))


def test_argument_checks_come_before_any_cuda_call():
    import marl_mass_b200 as mm
    L = mm.lib()
    ERR_ARG = -1

    def call(rec, t):
        rc = L.mm_eval_shield_record(None, None if rec is None else ctypes.byref(rec), t, None)
        return rc, L.mm_last_error().decode()

    rc, msg = call(None, 0)
    assert rc == ERR_ARG and "records are null" in msg
    for k in ("n_agents", "active", "shield_interventions", "min_agent_acc"):
        rc, msg = call(_records(**{k: 0}), 0)
        assert rc == ERR_ARG and "required" in msg, k
    rc, msg = call(_records(T=0), 0)
    assert rc == ERR_ARG and "T must be >= 1" in msg
    for t in (-1, 100):
        rc, msg = call(_records(), t)
        assert rc == ERR_ARG and "t must be in [0, T)" in msg, t
    rc, msg = call(_records(), 99)                     # valid records: the null handle is what is refused
    assert rc == ERR_ARG and "env is null" in msg
    rc, msg = call(_records(profile_slot=0x1000, profile_x=0x1000), 0)
    assert rc == ERR_ARG and "env is null" in msg


def test_evaluate_seeds_refuses_bad_control_profiles_before_device_work():
    import marl_mass_b200 as mm
    from marl_mass_b200 import evaluation as ev

    def never(obs, n_agents):
        raise AssertionError("no step may run")
    cfg = dict(mm.DEFAULT_CONFIG, safety_guarantee="cbf-cav")
    seeds = np.arange(10)
    with pytest.raises(ValueError, match="more than once"):
        ev.evaluate_seeds(never, cfg, seeds, control_profiles=[3, 1, 3])
    for bad in ([10], [-1], [0, 12]):
        with pytest.raises(ValueError, match=r"\[0, 10\)"):
            ev.evaluate_seeds(never, cfg, seeds, control_profiles=bad)
    with pytest.raises(ValueError, match=r"\[0, 4\)"):        # the range is that of the episodes evaluated
        ev.evaluate_seeds(never, cfg, seeds, eval_episodes=4, control_profiles=[4])
    with pytest.raises(TypeError):
        ev.evaluate_seeds(never, cfg, seeds, control_profiles=[1.5])


def test_train_refuses_eval_shield_without_eval_seeds():
    from marl_mass_b200.train import train
    for n in (0, -5):
        with pytest.raises(ValueError, match="eval_seeds"):
            train(INI, n_envs=4, iterations=1, eval_seeds=n, eval_shield=True)
