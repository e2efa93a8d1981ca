"""Host side of the batched merge environment: the reference's gym-style surface over the C ABI.

Two classes:

* `MergeEnvBatched` — E independent merge envs on one GPU, one kernel launch per policy step.
  `reset()` / `step()` mirror `MergeEnv.reset/step` (highway_env/envs/merge_env_v1.py:126-166,
  envs/common/abstract.py:176-209, 443-510) with a leading env axis; outputs are zero-copy torch views of the
  device buffers the handle owns.
* `MergeEnvLCMARL` — single-env adapter with the exact reference surface MAPPO drives
  (marl/mappo.py:44,104-135,281-342): `reset(is_training, testing_seeds, num_CAV) -> (obs, mask)`,
  `step(tuple) -> (obs, reward, done, info)`, `controlled_vehicles`, `config`, `n_s`, `n_a`, `T`, `is_crashed()`.

Config keys are the reference's ENV_CONFIG keys (run_mappo.py:145-171); as there, mutating `env.config[...]`
takes effect at the next `reset()`.  CBF eta/tau — class globals `CBFType.GAMMA_B/TAU` in the reference
(run_mappo.py:137-139) — are the keys `cbf_eta` and `HEADWAY_TIME`.

There is no CPU path: every call goes to libmarl_mass_b200.so and raises if it is missing.
"""
import ctypes as C

import numpy as np

from . import _lib
from . import spawn as _spawn
from ._lib import ENV_FIELDS, F64_FIELDS, I32_FIELDS, MAXV, NA, NS, SH_F, SH_I

SHIELD = {"none": 0, "cbf-hss": 1, "cbf-av": 1, "cbf-avs": 1, "cbf-avs_cint": 1, "cbf-mass": 2, "cbf-cav": 2,
          # the look-ahead baselines act on the action tuple before _simulate (abstract.py:459-464); the vehicles themselves
          # run un-shielded (safe_controller.py:232-239)
          "priority": 0, "dmc": 0}
SUPERVISOR = {"priority": 1, "dmc": 2}
REWARD = {"default": 0, "srew": 1, "mrew": 2}
TRAFFIC = {"cav": 0, "mixed": 1, "av": 2, "hdv": 3}

DEFAULT_CONFIG = {
    # merge_env_v1.py:32-57, 415-437 and abstract.py:106-130, with the values the shipped MASS ini uses
    "simulation_frequency": 15, "policy_frequency": 5, "duration": 20,
    "COLLISION_REWARD": 200, "HIGH_SPEED_REWARD": 1, "HEADWAY_COST": 4, "HEADWAY_TIME": 1.2,
    "MERGING_LANE_COST": 4, "traffic_density": 1, "safety_guarantee": "none", "lateral_control": "steer",
    "mixed_traffic": None, "traffic_type": "cav", "agent_reward": "default", "cbf_eta": 0.0,
    "action_masking": False, "seed": 0, "env_name": "merge-multi-agent-v1",
}
ENV_IDS = ("merge-multi-agent-v1", "merge-multi-agent-v0", "merge-multi-agent-v05", "merge-multi-agent-hdv-v1")


def traffic_type_of(cfg):
    """cav | mixed as the env class resolves it (merge_env_v1.py:206-209 for v0, 476-495 for v1)."""
    if cfg.get("env_name", "merge-multi-agent-v1") == "merge-multi-agent-v0":
        return "cav" if cfg.get("mixed_traffic", True) is False else "mixed"
    return cfg.get("traffic_type", "cav")


def make_mm_config(cfg):
    """Reference config dict -> mm_config.  Raises ValueError exactly where the reference would
    (decentral_layer.py:817 unknown safety type; safe_controller.py:174 unsupported lateral control)."""
    env_name = cfg.get("env_name", "merge-multi-agent-v1")
    if env_name not in ENV_IDS:
        raise KeyError("env id %r is not provided by marl_mass_b200 (available: %s)" % (env_name, list(ENV_IDS)))
    v0 = env_name == "merge-multi-agent-v0"
    sg = cfg.get("safety_guarantee", "none")
    supervisor = SUPERVISOR.get(sg, 0)
    if sg not in SHIELD:
        raise ValueError("Undefined safety_type:{0}".format(sg.split("-")[-1]))
    lat = cfg.get("lateral_control", "steer")
    if lat not in ("steer", "steer_vel") and not v0:
        raise AttributeError("Lateral control: {0} is not supported".format(lat))   # safe_controller.py:173-176
    if v0:
        # MergeEnvMARL (merge_env_v1.py:389-408): MDPVehicle ignores safety_guarantee / lateral_control /
        # agent_reward / traffic_type; vehicle counts follow `mixed_traffic` alone (merge_env_v1.py:206-209)
        tt = "cav" if cfg.get("mixed_traffic", True) is False else "mixed"
        sg, rk = "none", "default"
    else:
        tt = cfg.get("traffic_type", "cav")
        rk = cfg.get("agent_reward", "default")
    if tt not in TRAFFIC:
        raise ValueError("traffic_type %r is not supported (cav | mixed | av | hdv)" % (tt,))
    hdv_env = env_name == "merge-multi-agent-hdv-v1"
    if hdv_env != (tt == "hdv"):
        # MergeEnvLCHDV is the all-HDV evaluation env (merge_env_v1.py:552-674, test-idm-td3.ini); the other env classes
        # divide by the number of controlled vehicles
        raise ValueError("traffic_type 'hdv' and env id merge-multi-agent-hdv-v1 go together (got %r with %r)" % (tt, env_name))
    sim, pol = int(cfg["simulation_frequency"]), int(cfg["policy_frequency"])
    return _lib.MMConfig(
        shield=SHIELD[sg], reward_kind=REWARD[rk], env_v0=int(v0), steer_vel=int(lat == "steer_vel" and not v0),
        traffic_density=int(cfg["traffic_density"]), traffic_type=TRAFFIC[tt],
        duration_steps=int(cfg["duration"] * pol), substeps=sim // pol, dt=1 / sim,
        eta=float(cfg.get("cbf_eta", 0.0)), tau=float(cfg["HEADWAY_TIME"]),
        collision_reward=float(cfg["COLLISION_REWARD"]), high_speed_reward=float(cfg["HIGH_SPEED_REWARD"]),
        headway_cost=float(cfg["HEADWAY_COST"]), headway_time=float(cfg["HEADWAY_TIME"]),
        merging_lane_cost=float(cfg["MERGING_LANE_COST"]),
        couple_counts=int(bool(cfg.get("couple_vehicle_counts", False))), env_hdv=int(hdv_env), supervisor=supervisor)


class _DevArray(object):
    """Minimal __cuda_array_interface__ carrier so torch can view handle-owned device memory."""

    def __init__(self, ptr, shape, typestr, owner):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2, "strides": None}
        self._owner = owner


class MergeEnvBatched(object):
    n_s = NS
    n_a = NA

    def __init__(self, n_envs, config=None, device=0, record_diag=False):
        self.config = dict(DEFAULT_CONFIG)
        if config:
            self.config.update(config)
        self.n_envs = int(n_envs)
        self.device = int(device)
        self.record_diag = bool(record_diag)
        self.T = int(self.config["duration"] * self.config["policy_frequency"])
        self.v0 = self.config.get("env_name", "merge-multi-agent-v1") == "merge-multi-agent-v0"
        # Kinematics 5x5 (v0, v05: merge_env_v1.py:389-408, 527-550) vs KinematicLC 5x6 (v1)
        # KinematicLC 5x6 for the LC envs (v1, hdv-v1), Kinematics 5x5 for v0 / v05
        self.n_s = NS if self.config.get("env_name", "merge-multi-agent-v1") in ("merge-multi-agent-v1", "merge-multi-agent-hdv-v1") else 25
        self._L = _lib.lib()
        self._h = C.c_void_p()
        _lib.check(self._L.mm_create(C.byref(make_mm_config(self.config)), self.n_envs, self.device,
                                     int(self.record_diag), C.byref(self._h)))
        self._views = None
        self._reset_count = 0

    # ------------------------------------------------------------------ lifetime
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._L.mm_destroy(self._h)
            self._h = C.c_void_p()
            self._views = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ device views
    def buffers(self):
        """dict of torch tensors aliasing the handle's device buffers (valid until close())."""
        if self._views is None:
            import torch
            b = _lib.MMBuffers()
            _lib.check(self._L.mm_buffers_get(self._h, C.byref(b)))
            E = self.n_envs
            spec = {"obs": ((E, MAXV, NS), "<f4"), "reward": ((E,), "<f4"), "done": ((E,), "|u1"),
                    "agents_rewards": ((E, MAXV), "<f4"), "regional_rewards": ((E, MAXV), "<f4"),
                    "agents_dones": ((E, MAXV), "|u1"), "average_speed": ((E,), "<f4"),
                    "traffic_speed": ((E,), "<f4"), "min_headway": ((E,), "<f4"), "merge_percent": ((E,), "<f4"),
                    "n_agents": ((E,), "<i4"), "actions": ((E, MAXV), "|i1"), "action_mask": ((E, MAXV), "|u1"),
                    "new_actions": ((E, MAXV), "|i1")}
            dev = "cuda:%d" % self.device
            self._views = {k: torch.as_tensor(_DevArray(getattr(b, k), shp, ts, self), device=dev)
                           for k, (shp, ts) in spec.items()}
        return self._views

    @staticmethod
    def _stream_ptr(stream):
        if stream is None:
            import torch
            return C.c_void_p(torch.cuda.current_stream().cuda_stream)
        return C.c_void_p(getattr(stream, "cuda_stream", stream))

    # ------------------------------------------------------------------ reference surface, batched
    def _apply_config(self):
        self.T = int(self.config["duration"] * self.config["policy_frequency"])
        _lib.check(self._L.mm_set_config(self._h, C.byref(make_mm_config(self.config))))

    def reset(self, seed=None, mask=None, num_CAV=0, stream=None):
        """Device-side spawn of every env (or those with mask != 0); returns (obs, action_mask).

        seed=None continues the reference's habit of `self.seed += 1` per reset (abstract.py:183-190)."""
        self._apply_config()
        if seed is None:
            seed = int(self.config.get("seed", 0)) + self._reset_count
        self._reset_count += 1
        mptr = C.c_void_p(0)
        if mask is not None:
            assert mask.is_cuda and mask.dtype.itemsize == 1 and mask.numel() == self.n_envs
            mptr = C.c_void_p(mask.data_ptr())
        _lib.check(self._L.mm_reset(self._h, C.c_uint64(int(seed) & (2 ** 64 - 1)), mptr, int(num_CAV),
                                    self._stream_ptr(stream)))
        v = self.buffers()
        return v["obs"], self.action_mask()

    def reset_from_seeds(self, seeds, num_CAV=0):
        """Exactly the reference's scenes for `testing_seeds` (host replay of its MT19937 stream)."""
        self._apply_config()
        seeds = list(seeds)
        assert len(seeds) == self.n_envs
        self.spawn_rngs = []       # one MT19937 replay per env, positioned after the spawn draws (supervisor draws follow)
        st = _spawn.spawn_state(seeds, self.config["traffic_density"], traffic_type_of(self.config), num_CAV,
                                rngs=self.spawn_rngs)
        self.set_state(st)
        v = self.buffers()
        return v["obs"], self.action_mask()

    def reset_from_seeds_device(self, seeds, num_CAV=0, stream=None):
        """The scenes of `reset_from_seeds`, built on the device (mm_reset_seeded: the reference's MT19937 draws per env,
        one thread each) and left as `set_state` leaves them; nothing is synchronised.  num_CAV: one value or one per
        seed.  Unlike `reset_from_seeds` it keeps no `spawn_rngs` (the single-env adapter continues that stream on the
        host for the supervisors' draws).  Raises MMError, before anything is enqueued, for a seed outside [0, 2^32) or a
        num_CAV for which the reference's spawn raises or builds more than 11 vehicles."""
        self._apply_config()
        seeds = np.ascontiguousarray(seeds, np.int64).reshape(-1)
        assert len(seeds) == self.n_envs
        nc = np.ascontiguousarray(np.broadcast_to(np.asarray(num_CAV, np.int32), (self.n_envs,)))
        _lib.check(self._L.mm_reset_seeded(self._h, C.c_void_p(seeds.ctypes.data),
                                           C.c_void_p(nc.ctypes.data if nc.any() else 0), self._stream_ptr(stream)))
        v = self.buffers()
        return v["obs"], self.action_mask()

    def action_mask(self):
        """[E, MAXV, 5] int32.  action_masking False: all ones, as the reference returns (abstract.py:207-209).
        True: `_get_available_actions` per agent (abstract.py:219-240), unpacked from the kernel's bitmask.
        (The reference builds its mask as `[[0] * n_a] * n`, so its rows alias one list and every agent ends up
        with the union over agents; `MergeEnvLCMARL` reproduces that, this batched view is per agent.)"""
        import torch
        dev = "cuda:%d" % self.device
        if not self.config.get("action_masking", False):
            return torch.ones((self.n_envs, MAXV, NA), dtype=torch.int32, device=dev)
        bits = self.buffers()["action_mask"].to(torch.int32)
        return (bits[:, :, None] >> torch.arange(NA, device=dev, dtype=torch.int32)[None, None, :]) & 1

    def obs_view(self, obs=None):
        """The observation as the env id defines it: [E, MAXV, 30] for v1; for v0 (Kinematics, no heading column)
        columns 0..4 of each of the 5 rows, [E, MAXV, 25] (a copy); same for v05."""
        obs = self.buffers()["obs"] if obs is None else obs
        if self.n_s == NS:
            return obs
        return obs.view(self.n_envs, MAXV, 5, 6)[..., :5].reshape(self.n_envs, MAXV, 25)

    def step(self, actions=None, auto_reset=False, stream=None):
        """One policy step for every env.  actions: int8 CUDA tensor [E, MAXV] (None: the `actions` view).

        Returns (obs [E,MAXV,30] f32, reward [E] f32, done [E] u8, info) where info holds the device views
        named as the reference's info keys.  Nothing is synchronised."""
        aptr = C.c_void_p(0)
        if actions is not None:
            assert actions.is_cuda and actions.dtype.itemsize == 1 and actions.is_contiguous()
            assert actions.numel() == self.n_envs * MAXV
            aptr = C.c_void_p(actions.data_ptr())
        _lib.check(self._L.mm_step(self._h, aptr, int(bool(auto_reset)), self._stream_ptr(stream)))
        v = self.buffers()
        return v["obs"], v["reward"], v["done"], v

    def step_host(self, actions, auto_reset=False, out=None):
        """Same step through HOST arrays (numpy or pinned torch tensors): actions [E,MAXV] int8 in,
        obs/reward/done/regional_rewards/n_agents out.  Returns when the results are in `out`."""
        a = actions if isinstance(actions, np.ndarray) else actions.numpy()
        assert a.dtype == np.int8 and a.flags.c_contiguous and a.size == self.n_envs * MAXV
        if out is None:
            out = self.alloc_host_out()
        ptr = {k: (out[k].ctypes.data if isinstance(out[k], np.ndarray) else out[k].data_ptr()) for k in out}
        _lib.check(self._L.mm_step_host(self._h, C.c_void_p(a.ctypes.data), int(bool(auto_reset)),
                                        C.c_void_p(ptr.get("obs", 0)), C.c_void_p(ptr.get("reward", 0)),
                                        C.c_void_p(ptr.get("done", 0)), C.c_void_p(ptr.get("regional_rewards", 0)),
                                        C.c_void_p(ptr.get("n_agents", 0))))
        return out

    def step_host_ragged(self, actions, auto_reset=False, out=None):
        """`step_host` with the observations packed the way the reference returns them (an [A, n_s] array per env):
        out["obs_rows"][out["row_offset"][e] : out["row_offset"][e] + out["n_agents"][e]] are env e's rows.  `out` comes
        from `alloc_host_out(ragged=True)`."""
        a = actions if isinstance(actions, np.ndarray) else actions.numpy()
        assert a.dtype == np.int8 and a.flags.c_contiguous and a.size == self.n_envs * MAXV
        if out is None:
            out = self.alloc_host_out(ragged=True)
        ptr = {k: (out[k].ctypes.data if isinstance(out[k], np.ndarray) else out[k].data_ptr()) for k in out}
        _lib.check(self._L.mm_step_host_ragged(self._h, C.c_void_p(a.ctypes.data), int(bool(auto_reset)),
                                               C.c_void_p(ptr["obs_rows"]), C.c_void_p(ptr["row_offset"]),
                                               C.c_void_p(ptr.get("reward", 0)), C.c_void_p(ptr.get("done", 0)),
                                               C.c_void_p(ptr.get("regional_rewards", 0)), C.c_void_p(ptr.get("n_agents", 0))))
        return out

    def step_host_packed(self, actions, auto_reset=False, out=None):
        """`step_host` with the observation in packed form (mm_step_host_packed): per vehicle x, y, heading, speed
        (float32) and per agent the slots of the vehicles its observation rows show, plus reward / done / regional
        rewards - about 215 bytes per env-step instead of 1.1 KB of observation rows.  out["veh"][V0:V0 + n_veh[e]] are
        env e's vehicles (V0 = n_veh[:e].sum()), out["nbr"][A0:A0 + n_agents[e]] its agents' neighbour words.
        `expand_obs_rows(out)` rebuilds the [A, 30] rows on the host.  `out` comes from `alloc_host_out(packed=True)`."""
        a = actions if isinstance(actions, np.ndarray) else actions.numpy()
        assert a.dtype == np.int8 and a.flags.c_contiguous and a.size == self.n_envs * MAXV
        if out is None:
            out = self.alloc_host_out(packed=True)
        _lib.check(self._L.mm_step_host_packed(self._h, C.c_void_p(a.ctypes.data), int(bool(auto_reset)),
                                               C.byref(self._packed_struct(out))))
        return out

    @staticmethod
    def _packed_struct(out):
        ptr = lambda k: C.c_void_p(out[k].ctypes.data) if out.get(k) is not None else C.c_void_p(0)
        return _lib.MMPackedHost(veh=ptr("veh"), nbr=ptr("nbr"), n_veh=ptr("n_veh"), n_agents=ptr("n_agents"),
                                 reward=ptr("reward"), done=ptr("done"), regional_rewards=ptr("regional_rewards"))

    def expand_obs_rows(self, out, n_threads=0, obs_rows=None, row_offset=None):
        """Observation rows of a packed step, rebuilt on the host (mm_expand_obs_rows; no device involved):
        -> (obs_rows [sum n_agents, 30] f32, row_offset [E + 1] int64); env e's rows are obs_rows[row_offset[e]:row_offset[e + 1]]."""
        import os
        E = self.n_envs
        rows = int(out["n_agents"].sum(dtype=np.int64))
        if obs_rows is None:
            obs_rows = np.empty((rows, NS), np.float32)
        if row_offset is None:
            row_offset = np.empty((E + 1,), np.int64)
        assert obs_rows.dtype == np.float32 and obs_rows.flags.c_contiguous and obs_rows.shape[0] >= rows
        steer_vel = int(self.config.get("lateral_control", "steer") == "steer_vel" and not self.v0)
        _lib.check(self._L.mm_expand_obs_rows(C.byref(self._packed_struct(out)), E, steer_vel, C.c_void_p(obs_rows.ctypes.data),
                                              C.c_void_p(row_offset.ctypes.data), int(n_threads or len(os.sched_getaffinity(0)))))
        return obs_rows[:rows], row_offset

    def packed_bytes(self, out):
        """Device-to-host bytes of one mm_step_host_packed call that filled `out`."""
        E = self.n_envs
        return (int(out["n_veh"].sum(dtype=np.int64)) * 16 + int(out["n_agents"].sum(dtype=np.int64)) * 2 +
                E * (1 + 1 + 4 + 1 + MAXV * 4))

    def alloc_host_out(self, pinned=True, ragged=False, packed=False):
        import torch
        E = self.n_envs
        mk = lambda shape, dt: torch.empty(shape, dtype=dt, pin_memory=pinned).numpy()
        if packed:
            return {"veh": mk((E * 11, 4), torch.float32), "nbr": mk((E * MAXV,), torch.uint16),
                    "n_veh": mk((E,), torch.uint8), "n_agents": mk((E,), torch.uint8), "reward": mk((E,), torch.float32),
                    "done": mk((E,), torch.uint8), "regional_rewards": mk((E, MAXV), torch.float32)}
        out = {"reward": mk((E,), torch.float32), "done": mk((E,), torch.uint8),
               "regional_rewards": mk((E, MAXV), torch.float32), "n_agents": mk((E,), torch.int32)}
        if ragged:
            out["obs_rows"] = mk((E * MAXV, NS), torch.float32)
            out["row_offset"] = mk((E + 1,), torch.int64)
        else:
            out["obs"] = mk((E, MAXV, NS), torch.float32)
        return out

    # ------------------------------------------------------------------ state (teacher forcing / checkpoint)
    def _host_state_struct(self, st):
        kw = {}
        for k in F64_FIELDS:
            assert st[k].dtype == np.float64 and st[k].flags.c_contiguous and st[k].shape == (self.n_envs, MAXV), k
            kw[k] = st[k].ctypes.data_as(C.POINTER(C.c_double))
        for k in I32_FIELDS:
            assert st[k].dtype == np.int32 and st[k].flags.c_contiguous and st[k].shape == (self.n_envs, MAXV), k
            kw[k] = st[k].ctypes.data_as(C.POINTER(C.c_int32))
        for k in ENV_FIELDS:
            assert st[k].dtype == np.int32 and st[k].flags.c_contiguous and st[k].shape == (self.n_envs,), k
            kw[k] = st[k].ctypes.data_as(C.POINTER(C.c_int32))
        return _lib.MMStateHost(**kw)

    def get_state(self):
        st = _spawn.empty_state(self.n_envs)
        _lib.check(self._L.mm_get_state(self._h, C.byref(self._host_state_struct(st))))
        return st

    def set_state(self, st):
        _lib.check(self._L.mm_set_state(self._h, C.byref(self._host_state_struct(st))))

    def save(self, path):
        """Checkpoint: the full env-major state (every vehicle field, env counters) plus the config, as one .npz.
        (The reference cannot checkpoint an env; a batched rollout of hours needs it.)  The device-side spawn streams
        (per-env episode counters) are not part of it: after `load`, auto-reset draws new scenes from fresh streams."""
        import json
        st = self.get_state()
        np.savez_compressed(path, __config__=np.frombuffer(json.dumps(self.config).encode(), dtype=np.uint8),
                            __reset_count__=np.int64(self._reset_count), **st)

    def load(self, path):
        """Resume from `save`: same number of envs; the config stored with the state takes effect."""
        import json
        z = np.load(path)
        st = {k: np.ascontiguousarray(z[k]) for k in z.files if not k.startswith("__")}
        assert st["n_veh"].shape[0] == self.n_envs, "checkpoint holds %d envs, this handle %d" % (st["n_veh"].shape[0], self.n_envs)
        self.config.update(json.loads(bytes(z["__config__"]).decode()))
        self._reset_count = int(z["__reset_count__"])
        self._apply_config()
        self.set_state(st)
        v = self.buffers()
        return v["obs"], self.action_mask()

    def eval_record(self, records, t, stream=None):
        """mm_eval_record: the evaluation records (`_lib.MMEvalRecords`) of policy step t, taken on the device."""
        _lib.check(self._L.mm_eval_record(self._h, C.byref(records), int(t), self._stream_ptr(stream)))

    def eval_shield_record(self, records, t, stream=None):
        """mm_eval_shield_record: the shield records and control profiles (`_lib.MMEvalShieldRecords`) of policy step t,
        reduced on the device from the diagnostic record (needs record_diag).  Call it before `eval_record(t)`."""
        _lib.check(self._L.mm_eval_shield_record(self._h, C.byref(records), int(t), self._stream_ptr(stream)))

    def shield_diag(self):
        E = self.n_envs
        d = {k: np.zeros((E, 3, MAXV), np.int32) for k in SH_I}
        d.update({k: np.zeros((E, 3, MAXV), np.float64) for k in SH_F})
        s = _lib.MMShieldDiagHost(**{k: d[k].ctypes.data_as(C.POINTER(C.c_int32)) for k in SH_I},
                                  **{k: d[k].ctypes.data_as(C.POINTER(C.c_double)) for k in SH_F})
        _lib.check(self._L.mm_get_shield_diag(self._h, C.byref(s)))
        return d

    def shield_query(self, nom_steer, nom_acc, stream=None):
        """The shield alone (mm_shield_query): `safety_layer(...)` (decentral_layer.py:767-817) for every CAV of the
        current scenes, nothing stepped, no state written.  nom_steer / nom_acc: [E, 12] float64 cuda (the clipped
        low-level action per CAV).  -> dict of [E, 12] cuda tensors: safe_steer, safe_acc, min_headway (f64), ran,
        leader, front_adj, rear_adj, constrain_adj, active, is_lc_safe (int32)."""
        import torch
        dev = torch.device("cuda", self.device)
        ns = nom_steer.to(device=dev, dtype=torch.float64).contiguous()
        na = nom_acc.to(device=dev, dtype=torch.float64).contiguous()
        assert ns.shape == (self.n_envs, MAXV) and na.shape == (self.n_envs, MAXV)
        out = {k: torch.empty((self.n_envs, MAXV), dtype=torch.float64, device=dev) for k in ("safe_steer", "safe_acc", "min_headway")}
        out.update({k: torch.empty((self.n_envs, MAXV), dtype=torch.int32, device=dev)
                    for k in ("ran", "leader", "front_adj", "rear_adj", "constrain_adj", "active", "is_lc_safe")})
        s = _lib.MMShieldQueryOut(**{k: C.c_void_p(v.data_ptr()) for k, v in out.items()})
        _lib.check(self._L.mm_shield_query(self._h, C.c_void_p(ns.data_ptr()), C.c_void_p(na.data_ptr()), C.byref(s),
                                           self._stream_ptr(stream)))
        return out

    def stats(self, reset=False):
        s = _lib.MMStats()
        _lib.check(self._L.mm_stats(self._h, C.byref(s), int(reset)))
        return {k: getattr(s, k) for k, _ in _lib.MMStats._fields_}

    def kernel_launches(self):
        return int(self._L.mm_kernel_launches(self._h))

    def step_build(self):
        """Which build of the step kernel the last step launched (marl_mass_b200.h MM_BUILD_*: 3 / 4 generic, 31 / 32
        specialised for all-CAV envs under HSS / MASS)."""
        return int(self._L.mm_step_build(self._h))

    def supervise(self, actions, kind, draws=None, return_used=False):
        """The reference's baseline supervisors alone (mm_supervise) - `priority` (central_layer.py:16-178) or `dmc`
        (decentralised_dmc.py:70-198) - applied to the current scenes: returns the action tuples the reference would hand
        to _simulate.  actions [E, 12] integer cuda tensor; draws [E, 32] float64 cuda = the uniform numbers the reference
        takes from np.random.rand() in consumption order (None: Philox draws keyed (seed, env, episode, step)).
        With safety_guarantee = "priority" / "dmc" in the config, step() does this itself on every policy step."""
        import torch
        k = {"priority": 0, "dmc": 1}[kind]
        dev = torch.device("cuda", self.device)
        out = actions.to(device=dev, dtype=torch.int8).contiguous().clone()
        dptr = C.c_void_p(0)
        if draws is not None:
            draws = draws.to(device=dev, dtype=torch.float64).contiguous()
            assert draws.shape == (self.n_envs, _lib.SUPERVISOR_DRAWS)
            dptr = C.c_void_p(draws.data_ptr())
        used = torch.zeros(self.n_envs, dtype=torch.int32, device=dev)
        assert out.shape == (self.n_envs, MAXV)
        _lib.check(self._L.mm_supervise(self._h, k, C.c_void_p(out.data_ptr()), dptr, C.c_void_p(used.data_ptr()),
                                        C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        return (out, used) if return_used else out

    def set_supervisor_draws(self, draws=None):
        """Draws for the supervisors inside the following step() calls (mm_set_supervisor_draws): [E, 32] float64 cuda,
        consumed in order; None returns to the Philox stream.  The tensor is kept alive by the env."""
        import torch
        if draws is not None:
            draws = draws.to(device=torch.device("cuda", self.device), dtype=torch.float64).contiguous()
            assert draws.shape == (self.n_envs, _lib.SUPERVISOR_DRAWS)
        self._sup_draws = draws
        _lib.check(self._L.mm_set_supervisor_draws(self._h, C.c_void_p(0 if draws is None else draws.data_ptr())))

    def supervisor_draws_used(self):
        """[E] int32: how many draws each env's supervisor consumed in the last step."""
        used = np.zeros(self.n_envs, np.int32)
        _lib.check(self._L.mm_supervisor_draws_used(self._h, C.c_void_p(used.ctypes.data)))
        return used


def set_step_variant(variant=0):
    """0: automatic choice among the builds of the step kernel (marl_mass_b200.h mm_set_step_variant); 3 / 4: force a
    generic build; 5: automatic among the generic builds only; 6: 4 CTAs per SM, specialised builds allowed; 7: the
    warp-cooperative build where it applies; 8: automatic among the one-thread-per-env builds."""
    _lib.check(_lib.lib().mm_set_step_variant(int(variant)))


def shield_qp(a, c_lead, c_adj, has_adj, lo, hi, stream=None):
    """n independent CBF-QP solves on CUDA tensors (f64 inputs, uint8 has_adj).  Returns (u f64, active u8)."""
    import torch
    n = a.numel()
    for t in (a, c_lead, c_adj, lo, hi):
        assert t.is_cuda and t.dtype == torch.float64 and t.is_contiguous() and t.numel() == n
    assert has_adj.is_cuda and has_adj.dtype == torch.uint8 and has_adj.numel() == n
    u = torch.empty_like(a)
    active = torch.empty(n, dtype=torch.uint8, device=a.device)
    sp = C.c_void_p(torch.cuda.current_stream().cuda_stream if stream is None else stream.cuda_stream)
    _lib.check(_lib.lib().mm_shield_qp(*[C.c_void_p(t.data_ptr()) for t in (a, c_lead, c_adj, has_adj, lo, hi)],
                                       C.c_int64(n), C.c_void_p(u.data_ptr()), C.c_void_p(active.data_ptr()), sp))
    return u, active


# --------------------------------------------------------------------------------------------------
# single-env adapter with the reference surface
# --------------------------------------------------------------------------------------------------
class _VehicleView(object):
    """What MAPPO reads from env.controlled_vehicles[i] (mappo.py:329-346): crashed, position, speed."""

    def __init__(self, env, slot):
        self._env, self._slot = env, slot
        self.state_hist, self.action_hist, self.t_step = [], [], 0.0

    def _st(self):
        return self._env._state()

    @property
    def crashed(self):
        return bool(self._st()["crashed"][0, self._slot])

    @property
    def position(self):
        st = self._st()
        return np.array([st["x"][0, self._slot], st["y"][0, self._slot]])

    @property
    def speed(self):
        return float(self._st()["speed"][0, self._slot])

    @property
    def heading(self):
        return float(self._st()["heading"][0, self._slot])

    @property
    def id(self):
        return self._slot


class _RoadView(object):
    """env.road as mappo.py:425-435 / control_eval_mappo.py read it: `.vehicles`, each with `.id`, `.state_hist`,
    `.action_hist` (the per-sub-step control profile of safe_controller.py:187-227, when store_profile is on)."""

    def __init__(self):
        self.vehicles = []


class MergeEnvLCMARL(object):
    """Drop-in for gym.make('merge-multi-agent-v1') on the step path (merge_env_v1.py:410-525)."""
    n_a = NA
    n_s = NS

    ENV_NAME = "merge-multi-agent-v1"

    def __init__(self, config=None, device=0):
        config = dict(config or {}, env_name=self.ENV_NAME)
        # store_profile (MDPLCVehicle(store_profile=...), safe_controller.py:31,187-189): keep every vehicle's per-sub-step
        # state / action records in env.road.vehicles[i].state_hist / .action_hist (needs the kernel's diagnostic record)
        self.store_profile = bool(config.pop("store_profile", False))
        self.road = _RoadView()
        self._b = MergeEnvBatched(1, config, device=device, record_diag=self.store_profile)
        self.n_s = self._b.n_s
        self.config = self._b.config
        self.seed = self.config.get("seed", 0)
        self.T = self._b.T
        self.steps = 0
        self.controlled_vehicles = []
        self.vehicle_speed, self.vehicle_pos = [], []
        self._cache = None
        self.reset()

    @property
    def unwrapped(self):
        return self

    def _state(self):
        if self._cache is None:
            self._cache = self._b.get_state()
        return self._cache

    def reset(self, is_training=True, testing_seeds=0, num_CAV=0):
        seed = self.seed if is_training else testing_seeds
        self.seed += 1  # abstract.py:190
        self._b.reset_from_seeds([seed], num_CAV=num_CAV)
        self.T = self._b.T
        self._cache = None
        self.steps = 0
        self.vehicle_speed, self.vehicle_pos = [], []
        n = int(self._state()["n_cav"][0])
        self.road.vehicles = [_VehicleView(self, i) for i in range(int(self._state()["n_veh"][0]))]
        self.controlled_vehicles = self.road.vehicles[:n]
        import torch
        torch.cuda.synchronize(self._b.device)
        obs = self._b.obs_view()[0, :n].double().cpu().numpy()
        return obs, self._mask(n)

    def step(self, action):
        import torch
        n = len(self.controlled_vehicles)
        a = np.full((1, MAXV), 1, np.int8)
        a[0, :n] = np.asarray(tuple(action), np.int64)[:n]
        v = self._b.buffers()
        v["actions"].copy_(torch.from_numpy(a))
        new_action = action
        if self.config.get("safety_guarantee") in ("priority", "dmc"):
            # abstract.py:459-464.  The supervisor's np.random.rand() numbers are the next draws of the stream the spawn
            # left behind: hand the kernel a look-ahead of that stream, then advance the replay by what it consumed
            rs = self._b.spawn_rngs[0]
            peek = np.random.RandomState()
            peek.set_state(rs.get_state())
            self._b.set_supervisor_draws(torch.from_numpy(peek.rand(1, _lib.SUPERVISOR_DRAWS)))
            self._b.step(None)
            rs.rand(int(self._b.supervisor_draws_used()[0]))
            new_action = tuple(int(x) for x in v["new_actions"][0, :n].cpu().numpy())
        else:
            self._b.step(None)
        torch.cuda.synchronize(self._b.device)
        self._cache = None
        self.steps += 1
        if self.store_profile:
            self._log_profiles()
        st = self._state()
        obs = self._b.obs_view()[0, :n].double().cpu().numpy()
        reward = float(v["reward"][0])
        done = bool(v["done"][0])
        speeds = [float(st["speed"][0, i]) for i in range(n)]
        self.vehicle_speed.append(speeds)
        self.vehicle_pos.append([float(st["x"][0, i]) for i in range(n)])
        info = {
            "speed": speeds[0], "crashed": bool(st["crashed"][0, 0]), "action": action, "new_action": new_action,
            "action_mask": self._mask(n), "average_speed": float(v["average_speed"][0]),
            "vehicle_speed": np.array(self.vehicle_speed), "vehicle_position": np.array(self.vehicle_pos),
            "agents_dones": tuple(bool(x) for x in v["agents_dones"][0, :n].cpu().numpy()),
            "agents_info": [[float(st["x"][0, i]), float(st["y"][0, i]), speeds[i]] for i in range(n)],
            "agents_rewards": tuple(float(x) for x in v["agents_rewards"][0, :n].cpu().numpy()),
            "regional_rewards": tuple(float(x) for x in v["regional_rewards"][0, :n].cpu().numpy()),
            "traffic_speed": float(v["traffic_speed"][0]), "min_headway": float(v["min_headway"][0]),
        }
        if done:
            info["merge_percent"] = float(v["merge_percent"][0])
        return obs, reward, done, info

    def _log_profiles(self):
        """log_step (safe_controller.py:187-227) for every vehicle and sub-step of the policy step just taken."""
        d = self._b.shield_diag()
        dt = 1.0 / self.config["simulation_frequency"]
        steer_vel = self.config.get("lateral_control", "steer") == "steer_vel"
        for sub in range(3):
            for v in self.road.vehicles:
                i = v._slot
                if not d["moved"][0, sub, i]:
                    continue
                v.t_step += dt
                h, sp = float(d["heading"][0, sub, i]), float(d["speed"][0, sub, i])
                rec = {"presence": 1, "x": float(d["x"][0, sub, i]), "y": float(d["y"][0, sub, i]),
                       "vx": sp * np.cos(h), "vy": sp * np.sin(h), "heading": h, "cos_h": np.cos(h), "sin_h": np.sin(h),
                       "speed": sp, "t_step": v.t_step, "headway": float(d["min_headway"][0, sub, i])}
                if not steer_vel:
                    rec["steering_angle"] = float(d["nom_steer"][0, sub, i])
                ran = bool(d["ran"][0, sub, i])
                if ran:
                    rec["safe_status"] = {"active_set": int(d["active"][0, sub, i]), "is_lc_safe": bool(d["is_lc_safe"][0, sub, i])}
                v.state_hist.append(rec)
                hl = int(d["hl_action"][0, sub, i])
                act = {"acceleration": float(d["safe_acc"][0, sub, i]), "steering": float(d["safe_steer"][0, sub, i]),
                       "ull_acceleration": float(d["nom_acc"][0, sub, i]), "ull_steering": float(d["nom_steer"][0, sub, i]),
                       "lc_action": hl if hl >= 0 else None, "t_step": v.t_step}
                if ran:
                    act["safe_diff"] = {"acceleration": act["acceleration"] - act["ull_acceleration"],
                                        "steering": act["steering"] - act["ull_steering"]}
                v.action_hist.append(act)

    def _mask(self, n):
        """action mask as the reference returns it (abstract.py:201-209, 474-481): all ones without masking; with
        masking the reference's rows alias ONE list (`[[0] * n_a] * n`), i.e. the union over the agents."""
        if not self.config.get("action_masking", False):
            return np.array([[1] * self.n_a] * n)
        bits = self._b.buffers()["action_mask"][0, :n].cpu().numpy()
        union = int(np.bitwise_or.reduce(bits)) if n else 0
        return np.array([[(union >> a) & 1 for a in range(self.n_a)]] * n)

    def is_crashed(self):
        st = self._state()
        return bool(st["crashed"][0, :len(self.controlled_vehicles)].any())

    def render(self, mode="human"):
        """abstract.py:512-556.  'rgb_array': the frame MAPPO.evaluation records (mappo.py:292-322), rasterised on the
        CPU from the device state (render.py); 'human' would open a pygame window in the reference - there is no
        display surface here, nothing is shown and None is returned."""
        if mode == "rgb_array":
            from .render import render_scene
            return render_scene(self._state(), 0, self.config)
        return None

    def close(self):
        self._b.close()


class MergeEnvMARL(MergeEnvLCMARL):
    """Drop-in for gym.make('merge-multi-agent-v0') (merge_env_v1.py:389-408): un-shielded MDPVehicle CAVs,
    IDMVehicle HDVs unless mixed_traffic is False, Kinematics 5x5 observation (n_s = 25)."""
    ENV_NAME = "merge-multi-agent-v0"
    n_s = 25


class MergeEnvMARLSteerVel(MergeEnvLCMARL):
    """Drop-in for gym.make('merge-multi-agent-v05') (merge_env_v1.py:527-550): MDPLCVehicle dynamics (shields and
    lateral_control apply) with the 5x5 Kinematics observation."""
    ENV_NAME = "merge-multi-agent-v05"
    n_s = 25


class MergeEnvLCHDV(MergeEnvLCMARL):
    """Drop-in for gym.make('merge-multi-agent-hdv-v1') (merge_env_v1.py:552-674; eval_idm.py, test-idm-td3.ini): IDM /
    MOBIL vehicles only.  Nobody is controlled: `step(action)` ignores its argument, the observation has one row per
    vehicle, the reward is the mean of the per-vehicle reward over all vehicles, any crash ends the episode."""
    ENV_NAME = "merge-multi-agent-hdv-v1"

    def __init__(self, config=None, device=0):
        super().__init__(dict({"traffic_type": "hdv"}, **(config or {})), device=device)

    @property
    def vehicle(self):
        return self.road.vehicles[0] if self.road.vehicles else None

    def reset(self, is_training=True, testing_seeds=0, num_CAV=0):
        super().reset(is_training, testing_seeds, num_CAV)
        n = len(self.road.vehicles)
        return self._b.obs_view()[0, :n].double().cpu().numpy(), np.array([[1] * self.n_a] * n)

    def step(self, action=()):
        import torch
        v = self._b.buffers()
        self._b.step(None)
        torch.cuda.synchronize(self._b.device)
        self._cache = None
        self.steps += 1
        if self.store_profile:
            self._log_profiles()
        st = self._state()
        n = len(self.road.vehicles)
        obs = self._b.obs_view()[0, :n].double().cpu().numpy()
        self.vehicle_speed.append([float(x) for x in st["speed"][0, :n]])
        self.vehicle_pos.append([float(x) for x in st["x"][0, :n]])
        done = bool(v["done"][0])
        info = {"speed": float(st["speed"][0, 0]), "crashed": bool(st["crashed"][0, 0]),
                "average_speed": float(v["average_speed"][0]), "traffic_speed": float(v["traffic_speed"][0]),
                "min_headway": float(v["min_headway"][0])}
        if done:
            info["merge_percent"] = float(v["merge_percent"][0])
        return obs, float(v["reward"][0]), done, info

    def is_crashed(self):
        st = self._state()
        return bool(st["crashed"][0, :len(self.road.vehicles)].any())


_REGISTRY = {"merge-multi-agent-v1": MergeEnvLCMARL, "merge-multi-agent-v0": MergeEnvMARL,
             "merge-multi-agent-v05": MergeEnvMARLSteerVel, "merge-multi-agent-hdv-v1": MergeEnvLCHDV}


def make(env_id, **kwargs):
    """gym.make stand-in for the env ids on the hot path (merge_env_v1.py:686-689)."""
    if env_id not in _REGISTRY:
        raise KeyError("env id %r is not provided by marl_mass_b200 (available: %s)" % (env_id, sorted(_REGISTRY)))
    return _REGISTRY[env_id](**kwargs)
