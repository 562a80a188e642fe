"""The reference's own env-cfg objects lower to exactly the restated TaskSpec.  The objects are replayed from their
record (tests/golden/cfg_blobs/reference_cfgs.json, written by tests/golden/make_cfg_blobs.py from the reference tree),
so the comparison runs on every machine."""
import importlib.util
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


def _make_cfg_blobs():
    spec = importlib.util.spec_from_file_location("make_cfg_blobs", ROOT / "tests" / "golden" / "make_cfg_blobs.py")
    mk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mk)
    return mk


@pytest.fixture(scope="module")
def ref_cfgs():
    """{reference cfg class name: constructor of its default instance}, with shims/ (isaaclab) importable."""
    if str(ROOT / "shims") not in sys.path:
        sys.path.insert(0, str(ROOT / "shims"))
    return _make_cfg_blobs().recorded_cfg_classes()


def _cfg_dict(c):
    out = {}
    for name, _ in c._fields_:
        v = getattr(c, name)
        out[name] = list(v) if hasattr(v, "__len__") else v
    return out


def test_drift_cfg_lowers_to_restated_spec(ref_cfgs):
    import wheeledlab_b200 as wl
    from wheeledlab_b200.compat import spec_from_reference_cfg
    cfg = ref_cfgs["MushrDriftRLEnvCfg"]()
    cfg.scene.num_envs = 64
    got = spec_from_reference_cfg(cfg)
    exp = wl.drift_task(num_envs=64, seed=42)
    a, b = _cfg_dict(got.cfg), _cfg_dict(exp.cfg)
    diff = {k: (a[k], b[k]) for k in a if a[k] != b[k]}
    assert not diff, diff
    assert got.reward_names == exp.reward_names
    assert [(t.reward_term_name, t.increase, t.episodes_per_increase, t.max_increases) for t in got.curriculum] == \
           [(t.reward_term_name, t.increase, t.episodes_per_increase, t.max_increases) for t in exp.curriculum]
    assert got.cfg.max_episode_length == 250


def test_f1tenth_and_elevation_cfgs_lower(ref_cfgs):
    from wheeledlab_b200.compat import spec_from_reference_cfg
    f = ref_cfgs["F1TenthDriftRLEnvCfg"](); f.scene.num_envs = 8
    s = spec_from_reference_cfg(f)
    assert s.cfg.action_kind == 2 and abs(s.cfg.base_length - 0.365) < 1e-6 and abs(s.cfg.base_width - 0.284) < 1e-6
    e = ref_cfgs["MushrElevationRLEnvCfg"](); e.scene.num_envs = 8
    s = spec_from_reference_cfg(e)
    assert s.cfg.task == 1 and s.cfg.max_episode_length == 200 and s.cfg.decimation == 10 and s.cfg.substeps == 2
    assert s.reward_names == ["vel_towards_goal", "height_z", "falling_penalty", "termination_penalty"]
    assert list(s.cfg.rew_weight)[:4] == [200.0, 5000.0, 0.0, -200.0] and s.obs_dim == 689


def test_unknown_term_fails_loudly(ref_cfgs):
    from wheeledlab_b200.compat import spec_from_reference_cfg
    from isaaclab.managers import RewardTermCfg
    cfg = ref_cfgs["MushrDriftRLEnvCfg"]()
    cfg.rewards.side_slip = RewardTermCfg(func=lambda env: 0, weight=1.0)
    with pytest.raises(NotImplementedError):
        spec_from_reference_cfg(cfg)


def test_unknown_term_becomes_host_side_term_when_allowed(ref_cfgs):
    """allow_python_terms: the cfg's own function is kept and registered as a Python term of the staged step."""
    from wheeledlab_b200.compat import spec_from_reference_cfg
    from isaaclab.managers import RewardTermCfg, TerminationTermCfg
    cfg = ref_cfgs["MushrDriftRLEnvCfg"]()
    f = lambda env, k=1.0: 0
    g = lambda env: 0
    cfg.rewards.my_bonus = RewardTermCfg(func=f, weight=3.0, params={"k": 2.0})
    cfg.terminations.my_stop = TerminationTermCfg(func=g)
    cfg.rewards._cfg_fields = list(getattr(cfg.rewards, "_cfg_fields", [])) + ["my_bonus"] if hasattr(cfg.rewards, "_cfg_fields") else None
    cfg.terminations._cfg_fields = list(getattr(cfg.terminations, "_cfg_fields", [])) + ["my_stop"] if hasattr(cfg.terminations, "_cfg_fields") else None
    with pytest.raises(NotImplementedError):
        spec_from_reference_cfg(cfg)
    s = spec_from_reference_cfg(cfg, allow_python_terms=True)
    assert s.python_reward_terms == [("my_bonus", f, 3.0, {"k": 2.0})]
    assert s.python_termination_terms == [("my_stop", g, False, {})]
    assert "my_bonus" not in s.reward_names and len(s.reward_names) == 7      # built-in slots untouched


# ---- the registration path: the reference's four register() calls, replayed through the gymnasium stand-in in shims/ ----
def _cfg_blob(c):
    import ctypes as C
    return C.string_at(C.addressof(c), C.sizeof(c))


def test_unmodified_registration_and_all_cfgs_lower_to_the_committed_blobs():
    """The recorded registration of `import wheeledlab_tasks` (reference source, untouched) registers the four gym ids
    through the gymnasium stand-in; every train and play cfg lowers through compat.spec_from_reference_cfg to exactly the
    committed fixture, and the train cfgs equal make_task(id) byte for byte."""
    import wheeledlab_b200 as wl
    from wheeledlab_b200.compat import spec_from_reference_cfg
    gym = _make_cfg_blobs().import_recorded_tasks()
    assert sorted(gym.registry) == sorted(wl.GYM_IDS)
    for gid in gym.registry:
        s = gym.spec(gid)
        assert s.entry_point == "isaaclab.envs:ManagerBasedRLEnv" and s.kwargs["rsl_rl_cfg_entry_point"].count(":") == 1
        for key, suffix in (("env_cfg_entry_point", "ref"), ("play_env_cfg_entry_point", "play.ref")):
            cls = s.kwargs.get(key)
            if cls is None:
                continue
            cfg = cls(); cfg.scene.num_envs = 4096
            got = spec_from_reference_cfg(cfg)
            fixture = (ROOT / "tests" / "golden" / "cfg_blobs" / f"{gid}.{suffix}.bin").read_bytes()
            assert _cfg_blob(got.cfg) == fixture, (gid, key)
            if suffix == "play.ref":                 # play cfgs: "no terminations" (Drift / Visual also drop rewards and curriculum)
                assert got.cfg.term_enable == 0
                if "Elevation" not in gid:
                    assert got.cfg.curr_n == 0 and not any(got.cfg.rew_weight)
    # a modified observation group is rejected, not silently replaced by the built-in one (ADVICE r1)
    bad = gym.spec("Isaac-MushrDriftRL-v0").kwargs["env_cfg_entry_point"]()
    bad.observations.policy.base_lin_vel_term = None
    with pytest.raises(NotImplementedError):
        spec_from_reference_cfg(bad)


def test_make_task_reproduces_the_lowered_reference_cfgs():
    """The package's own restatement of the four registered tasks equals the blobs lowered from the reference's cfg
    objects, byte for byte."""
    import numpy as np
    import wheeledlab_b200 as wl
    blobs = ROOT / "tests" / "golden" / "cfg_blobs"
    ref_map = np.load(blobs / "visual_ref_map.npz")["map"]
    for gid in wl.GYM_IDS:
        kw = {"traversability": ref_map} if "Visual" in gid else {}
        spec = wl.make_task(gid, num_envs=4096, seed=42, **kw)
        assert _cfg_blob(spec.cfg) == (blobs / f"{gid}.ref.bin").read_bytes(), gid


def test_torch_ops_front_registers_and_rejects_cpu_tensors():
    """torch.ops.wheeledlab_b200.* (csrc/wl_torch_ops.cpp): the schemas the PyTorch-extension boundary declares exist, outputs
    are declared as written in place, and a CPU tensor fails loudly (CUDA dispatch key only: no CPU path)."""
    import torch
    from wheeledlab_b200 import torch_ops
    ops = torch_ops.load()
    sch = {name: str(getattr(ops, name).default._schema) for name in ("step", "step_out", "observe_out", "reset")}
    assert "Tensor(a!) obs" in sch["step_out"] and "Tensor(d!) truncated" in sch["step_out"] and "Tensor(e!)? log" in sch["step_out"]
    assert sch["step"].endswith("-> (Tensor, Tensor, Tensor, Tensor)")
    assert "Tensor? env_ids" in sch["reset"] and "Tensor(a!) obs" in sch["observe_out"]
    import pytest
    with pytest.raises(NotImplementedError):
        ops.step(1, torch.zeros(4, 2), 0)
