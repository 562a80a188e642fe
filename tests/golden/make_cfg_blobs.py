#!/usr/bin/env python
"""Write the lowered wl_config of every registered task as a binary blob (tests/golden/cfg_blobs/<name>.bin).

Two producers must agree byte for byte (tests/test_compat_cpu.py, tests/test_gpu_parity.py):
  * the package's own restatement of the reference configuration (wheeledlab_b200.tasks.make_task), and
  * the lowering of the REFERENCE'S OWN cfg objects (wheeledlab_b200.compat.spec_from_reference_cfg), imported from
    /root/reference in the authoring container (this script records them as <name>.ref.bin when the tree is present).
The blobs also let non-Python hosts (examples/c_host) and bench.py's reference arm build a task without importing the package.
num_envs = 4096, seed = 42, env_id_offset = 0 in every blob (the first fields of wl_config; consumers patch them).

The reference's registry and cfg objects are also recorded as data (cfg_blobs/reference_cfgs.json: field values, class
names, term functions by name -- everything the lowering reads), so that tests/test_compat_cpu.py lowers the same objects
on machines that do not have the reference tree (import_recorded_tasks).
"""
import ctypes as C
import json
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
sys.path.insert(0, str(ROOT))
OUT = HERE / "cfg_blobs"
RECORD = OUT / "reference_cfgs.json"
VISUAL_MAP = OUT / "visual_ref_map.npz"

TASKS = {"drift": "Isaac-MushrDriftRL-v0", "f1tenth_drift": "Isaac-F1TenthDriftRL-v0", "elevation": "Isaac-MushrElevationRL-v0",
         "visual": "Isaac-MushrVisualRL-v0", "hound_4wd": "hound_4wd"}


def blob(cfg) -> bytes:
    return C.string_at(C.addressof(cfg), C.sizeof(cfg))


def import_reference_tasks():
    """Import the UNMODIFIED wheeledlab_tasks package of /root/reference against the stand-ins in shims/ (gymnasium, isaaclab,
    pxr, matplotlib).  Importing it registers the four gym ids (wheeledlab_tasks/__init__.py:14-63) and -- quirk Q10 -- builds the
    Visual traversability map and tries to create <assets>/data/rgb_maps: the reference tree is read-only here, so that one
    makedirs is skipped."""
    import os
    ref = Path("/root/reference/source")
    sys.path[:0] = [str(ROOT / "shims"), str(ref / "wheeledlab"), str(ref / "wheeledlab_assets"), str(ref / "wheeledlab_tasks")]
    real = os.makedirs

    def makedirs(path, *a, **k):
        if str(path).startswith(str(ref)):
            return None
        return real(path, *a, **k)

    top = sys.modules.get("wheeledlab_tasks")
    if top is not None and getattr(top, "__file__", None) is None:       # a path-only stub of another test (skips __init__): drop it
        for k in [k for k in sys.modules if k == "wheeledlab_tasks" or k.startswith("wheeledlab_tasks.")]:
            del sys.modules[k]
    os.makedirs = makedirs
    try:
        import wheeledlab_tasks  # noqa: F401
    finally:
        os.makedirs = real
    import gymnasium as gym
    return gym


def _encode(o, path, ref):
    """JSON form of a cfg object tree.  Every dict carries one tag, so that _decode can tell the kinds apart.  Paths
    into the reference tree `ref` are recorded relative to it, as "<reference>/..."."""
    if path.endswith(".traversability_hashmap"):      # drawn at random at every import (quirk Q10): recorded as VISUAL_MAP's map
        import numpy as np
        if np.asarray(o).shape != np.load(VISUAL_MAP)["map"].shape:
            raise ValueError(f"{path}: shape differs from {VISUAL_MAP.name}")
        return {"__map__": VISUAL_MAP.name}
    if hasattr(o, "_cfg_fields"):
        return {"__cfg__": [f"{type(o).__module__}:{type(o).__name__}",
                            {k: _encode(getattr(o, k), f"{path}.{k}", ref) for k in o._cfg_fields}]}
    if isinstance(o, dict):
        if not all(isinstance(k, str) for k in o):
            raise TypeError(f"{path}: non-string key")
        return {"__dict__": {k: _encode(v, f"{path}[{k}]", ref) for k, v in o.items()}}
    if isinstance(o, tuple):
        return {"__tuple__": [_encode(v, path, ref) for v in o]}
    if isinstance(o, list):
        return [_encode(v, path, ref) for v in o]
    if isinstance(o, slice):
        return {"__slice__": [o.start, o.stop, o.step]}
    if isinstance(o, type):
        return {"__type__": f"{o.__module__}:{o.__name__}"}
    if callable(o):
        return {"__func__": f"{o.__module__}:{o.__name__}"}
    if isinstance(o, str) and o.startswith(ref + "/"):       # asset paths; the Visual rgb_maps file name is a timestamp taken
        return "<reference>" + o[len(ref):]                  # at import, so it differs between records (the lowering ignores it)
    if o is None or isinstance(o, (bool, int, float, str)):
        return o
    raise TypeError(f"{path}: cannot record a {type(o).__name__}")


_NAMED = {}


def _named(kind, ref):
    """One stand-in per recorded class or function, with the recorded __module__ and __name__ (the lowering matches
    terms, action classes and noise cfgs by name)."""
    if (kind, ref) not in _NAMED:
        mod, name = ref.split(":")
        if kind == "__func__":
            def obj(*args, **kwargs):
                raise NotImplementedError(f"{ref} is recorded by name only")
            obj.__name__ = obj.__qualname__ = name
            obj.__module__ = mod
        else:
            obj = type(name, (), {"__module__": mod})
        _NAMED[(kind, ref)] = obj
    return _NAMED[(kind, ref)]


def _decode(n):
    if isinstance(n, list):
        return [_decode(v) for v in n]
    if not isinstance(n, dict):
        return n
    (tag, v), = n.items()
    if tag == "__cfg__":
        obj = _named(tag, v[0])()
        obj._cfg_fields = list(v[1])
        for k, x in v[1].items():
            setattr(obj, k, _decode(x))
        return obj
    if tag == "__dict__":
        return {k: _decode(x) for k, x in v.items()}
    if tag == "__tuple__":
        return tuple(_decode(x) for x in v)
    if tag == "__slice__":
        return slice(*v)
    if tag == "__map__":
        import numpy as np
        return np.load(OUT / v)["map"].tolist()
    return _named(tag, v)


def record_reference_tasks(gym):
    """Write RECORD from the registry import_reference_tasks() filled: each id's spec, and a default instance of each
    cfg class its kwargs name."""
    ref = str(Path(sys.modules["wheeledlab_tasks"].__file__).resolve().parents[2])      # <ref>/wheeledlab_tasks/wheeledlab_tasks/
    registry, cfgs = {}, {}
    for gid in gym.registry:
        s = gym.spec(gid)
        kwargs = {}
        for key, v in s.kwargs.items():
            if isinstance(v, str):
                kwargs[key] = v
            else:
                kwargs[key] = {"__cfg_class__": v.__name__}
                cfgs[v.__name__] = _encode(v(), v.__name__, ref)
        registry[gid] = {"entry_point": s.entry_point, "disable_env_checker": s.disable_env_checker, "kwargs": kwargs}
    RECORD.write_text(json.dumps({"registry": registry, "cfgs": cfgs}, separators=(",", ":")) + "\n")


def recorded_cfg_classes():
    """{cfg class name: callable returning a fresh object tree of that class's default instance}, from RECORD."""
    cfgs = json.loads(RECORD.read_text())["cfgs"]

    def cls(name):
        def make():
            return _decode(cfgs[name])
        make.__name__ = name
        return make
    return {name: cls(name) for name in cfgs}


def import_recorded_tasks():
    """import_reference_tasks() replayed from RECORD: the recorded ids are registered through the gymnasium stand-in,
    with every cfg entry point building a fresh object tree."""
    if str(ROOT / "shims") not in sys.path:
        sys.path.insert(0, str(ROOT / "shims"))
    import gymnasium as gym
    classes = recorded_cfg_classes()
    for gid, s in json.loads(RECORD.read_text())["registry"].items():
        kwargs = {k: classes[v["__cfg_class__"]] if isinstance(v, dict) else v for k, v in s["kwargs"].items()}
        gym.register(id=gid, entry_point=s["entry_point"], disable_env_checker=s["disable_env_checker"], kwargs=kwargs)
    return gym


def main():
    import numpy as np
    import wheeledlab_b200 as wl
    OUT.mkdir(exist_ok=True)
    for name, tid in TASKS.items():
        spec = wl.make_task(tid, num_envs=4096, seed=42)
        (OUT / f"{name}.bin").write_bytes(blob(spec.cfg))
        print(name, C.sizeof(spec.cfg), "bytes")
    if Path("/root/reference/source").exists():          # authoring container: lower the reference's own cfg objects
        from wheeledlab_b200.compat import spec_from_reference_cfg
        gym = import_reference_tasks()
        for gid in gym.registry:
            for key, suffix in (("env_cfg_entry_point", "ref"), ("play_env_cfg_entry_point", "play.ref")):
                cls = gym.spec(gid).kwargs.get(key)
                if cls is None:
                    continue
                cfg = cls()
                cfg.scene.num_envs = 4096
                got = spec_from_reference_cfg(cfg)
                (OUT / f"{gid}.{suffix}.bin").write_bytes(blob(got.cfg))
                if "Visual" in gid and suffix == "ref":
                    np.savez_compressed(OUT / "visual_ref_map.npz", map=np.asarray(cfg.scene.terrain.traversability_hashmap, dtype=bool))
                print(gid, suffix)
        record_reference_tasks(gym)
        print(RECORD.name)


if __name__ == "__main__":
    main()
