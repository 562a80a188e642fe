#!/usr/bin/env python
"""bench.py -- env-steps/s of the fused WheeledLab step (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload drift|elev|hound4wd] [--envs E] [--impl ours|reference]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one env.step() of the workload over E envs per GPU with synthetic U[-1,1]^2 actions from the counter-based
generator.  Workloads (BASELINE.json configs):
    drift     configs[1]  RSS_DRIFT_CONFIG  MushrDriftRL, 4096 envs, dt 5 ms x 4, DR + pushes + obs noise  (the headline metric)
    elev      configs[2]  RSS_ELEV_CONFIG   MushrElevationRL, 4096 envs, height-field terrain + 676-ray height scan
    hound4wd  configs[3]  "HOUND 4WD"       MuSHR + HOUND_SUS_ACTUATOR_CFG (4 driven wheels) + Mushr4WDActionCfg, 8192 envs
(configs[4] = drift at --gpus 8; configs[0] is the reference's CPU plumbing case, a parity-test size.)  Rank 0 prints ONE JSON line.

  value     whole-job env-steps/s, inputs resident in HBM.  Timed region = EXACTLY K steps issued back to back between two
            CUDA events (barrier + synchronize on both sides), max over ranks; the K steps are one CUDA graph (uploaded at
            set-up) that starts right behind the graph of the W warm-up steps, so the region holds no host launch latency.
            Cold caches WITHOUT a flush kernel: the working set is larger than L2 -- M independent env sets (state +
            parameters) are stepped round-robin and every step writes a fresh rollout-slab row, so no step finds its inputs
            in L2 (`config.l2`).  With N > 1 the run exchanges the rollout slab after every T_ROLL-th step, inside the timed
            region: fused into the step kernels as peer-memory stores + one device barrier ("fanout", Drift family), a
            copy-engine pull ("ce") or NCCL all-gather ("nccl") overlapped with the next rollout's steps; the ranks'
            clocks are aligned on the device before the warm-up steps.
  flush_protocol  the round-1 protocol kept for comparison: per-step events with a 256 MiB L2-flush fill between steps, and
            the same measurement around an EMPTY kernel (the floor of that protocol: ~6 us on B200).
  e2e       same metric through the public ManagerBasedRLEnv.step_host() with HOST (pinned) buffers: H2D of the actions and
            D2H of observations + reward + done masks inside the timed region, every step, stream-synchronised.
  roofline  algorithmic bytes of the step kernel(s) / average step duration in the timed region vs the measured HBM peak.
  cpu_baseline  the CPU oracle (oracle/wl_oracle.c, "port") timed on this box's host cores.
--impl reference times that same CPU implementation (all physical cores) as the reference arm: the reference's own PhysX
pipeline is a closed binary that is not in /root/reference (DESIGN.md).  It does not import the product package.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"
# algorithmic bytes per env-step (DESIGN.md "Kernels"):
#   drift / hound4wd: reads 13 state+param groups x16 B + action 8 B; writes 9 state groups x16 B + obs 56 + rew 4 + 2 masks
#   elev: reads 15 groups + action; writes 11 groups + the 689-float observation row + rew + masks
BYTES_PER_ENV_STEP = (13 * 16 + 8) + (9 * 16 + 56 + 4 + 2)
WORKLOADS = {
    "drift": {"task": "drift", "envs": 4096, "bytes": BYTES_PER_ENV_STEP, "obs_dim": 14, "blob": "drift.bin",
              "label": "RSS_DRIFT_CONFIG MushrDriftRL, dt 5ms x4, DR+push+noise on", "kernel": "wl_step_duo_kernel (Drift family, 8 envs per CTA)",
              "traffic_profile": "profiles/r02_ncu_step_drift_4096.txt"},
    "elev": {"task": "elevation", "envs": 4096, "bytes": (15 * 16 + 8) + (11 * 16 + 689 * 4 + 4 + 2), "obs_dim": 689, "blob": "elevation.bin",
             "label": "RSS_ELEV_CONFIG MushrElevationRL, dt 10ms x10 (5 ms sub-steps), reference terrain raster + 676-ray height scan",
             "kernel": "wl_step_quad_kernel<ELEVATION> + wl_scan_kernel<TMA>", "traffic_profile": "profiles/r02_ncu_step_elev_4096.txt"},
    "hound4wd": {"task": "hound_4wd", "envs": 8192, "bytes": BYTES_PER_ENV_STEP, "obs_dim": 14, "blob": "hound_4wd.bin",
                 "label": "HOUND 4WD: MuSHR + HOUND_SUS_ACTUATOR_CFG (4 driven wheels) + Mushr4WDActionCfg, mass/friction DR, dt 5ms x4",
                 "kernel": "wl_step_duo_kernel (4WD action map)", "traffic_profile": "profiles/r02_ncu_step_hound_8192.txt"},
}
L2_BYTES = 126 * 1024 * 1024
SET_BYTES_PER_ENV = 256                                        # state + parameters per env: 16 groups x 16 B (wl_state_bytes)
DUMP_BYTES = 64 * 10**6                                        # --dump-outputs: all files together, .npy headers included


def _peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def _traffic(path):
    """dram bytes per launch recorded in the committed `ncu --set full` summary of this workload (or None)."""
    p = ROOT / path
    if not p.exists():
        return None
    tot = 0.0
    for line in p.read_text().splitlines():
        for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            if line.strip().startswith(key + " ="):
                val, unit = line.split("=")[1].split()[:2]
                tot += float(val) * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(unit, 1)
    return tot or None


def dump_outputs(outdir, outputs):
    """--dump-outputs: what the last timed step returned ({name: torch or numpy array, one row per env}) as float32
    <outdir>/<name>.npy.  When the rows exceed DUMP_BYTES together, every array keeps the same fixed, seeded sample of
    envs (in env order)."""
    import numpy as np
    n = len(next(iter(outputs.values())))
    row_bytes = sum(4 * math.prod(a.shape[1:]) for a in outputs.values())
    keep = (DUMP_BYTES - 256 * len(outputs)) // row_bytes     # (256 B: more than an .npy header takes)
    rows = np.sort(np.random.default_rng(0).choice(n, keep, replace=False)) if n > keep else None
    Path(outdir).mkdir(parents=True, exist_ok=True)
    for name, a in outputs.items():
        if hasattr(a, "cpu"):                                  # a torch tensor: only the kept rows leave the device
            if rows is not None:
                import torch
                a = a[torch.from_numpy(rows).to(a.device)]
            a = a.cpu().numpy()
        elif rows is not None:
            a = a[rows]
        np.save(Path(outdir) / f"{name}.npy", np.ascontiguousarray(a, dtype=np.float32))


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_indices):
        self.gpu = ",".join(str(g) for g in (gpu_indices if isinstance(gpu_indices, (list, tuple, range)) else [gpu_indices]))
        self.rows, self.proc = [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", self.gpu], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, mx, reasons, per = [], [], set(), {}
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                per.setdefault(int(r[0]), []).append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        out = {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
               "reasons": sorted(reasons), "samples": len(sm)}
        if len(per) > 1:                                      # one median per GPU of the job
            out["per_gpu_sm_mhz"] = [statistics.median(per[g]) for g in sorted(per)]
        return out


# ---------------------------------------------------------------------------------------------------------------------
# CPU side (the oracle): test infrastructure used here as the reported CPU baseline / reference arm only
# ---------------------------------------------------------------------------------------------------------------------
_PHYS = None


def _physical_cores() -> int:
    """Physical cores this process may run on (SMT siblings counted once), capped by the cgroup CPU quota if there is one.
    Evaluated ONCE, before the OpenMP runtime binds the calling thread to a core (OMP_PROC_BIND)."""
    global _PHYS
    if _PHYS is None:
        _PHYS = _physical_cores_uncached()
    return _PHYS


def _physical_cores_uncached() -> int:
    try:
        allowed = os.sched_getaffinity(0)
    except Exception:
        allowed = set(range(os.cpu_count() or 1))
    cores = set()
    try:
        for cpu in allowed:
            base = Path(f"/sys/devices/system/cpu/cpu{cpu}/topology")
            cores.add((base.joinpath("physical_package_id").read_text().strip(), base.joinpath("core_id").read_text().strip()))
        n = max(1, len(cores))
    except Exception:
        n = max(1, len(allowed) // 2)
    try:                                                       # cgroup v2 quota: "max 100000" or "<quota> <period>"
        q, per = Path("/sys/fs/cgroup/cpu.max").read_text().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per))))
    except Exception:
        pass
    return n


def _pick_threads(workload: str, envs: int, seed: int):
    """'All the host threads it can use': the physical-core count, checked against half and a quarter of it on a 0.6 s probe
    each (shared / throttled boxes scale badly past their real allotment); returns (threads, {threads: env-steps/s})."""
    full = _physical_cores()
    probe = {}
    for th in sorted({max(1, full // 4), max(1, full // 2), full}):
        orc = _cpu_oracle(workload, envs, seed, th)
        steps, el = _time_oracle(orc, 2, 3, 0.6, 2.0)
        probe[th] = envs * steps / el
    best = max(probe, key=probe.get)
    return best, {str(k): round(v) for k, v in probe.items()}


def _cpu_oracle(workload: str, envs: int, seed: int, threads: int):
    """The oracle on `envs` envs of the workload, built from the committed config blob (no product import)."""
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
    sys.path.insert(0, str(ROOT / "tests"))
    import numpy as np
    import oracle_lib as O
    w = WORKLOADS[workload]
    O.get_lib("native")                                        # -O3 -march=native build (made on this box)
    cfg = O.cfg_from_blob(ROOT / "tests" / "golden" / "cfg_blobs" / w["blob"], num_envs=envs, seed=seed, env_id_offset=0)
    hf = None
    if w["task"] == "elevation":                               # the shipped raster of the reference's terrain mesh, padded like the product does
        d = np.load(ROOT / "wheeledlab_b200" / "data" / "terrain_huge_compact_0p1m.npz")
        h = d["heights"].astype(np.float32)
        pitch = (h.shape[1] + 3) & ~3
        hf = np.zeros((h.shape[0], pitch), np.float32); hf[:, :h.shape[1]] = h
        if pitch > h.shape[1]:
            hf[:, h.shape[1]:] = h[:, -1:]
    orc = O.Oracle(cfg, heightfield=hf, kind="native", threads=threads)
    orc.startup(); orc.reset(None, 0)
    return orc


def _time_oracle(orc, warm: int, min_steps: int, min_s: float, max_s: float):
    acts = [orc.synth_actions(t) for t in range(8)]
    for t in range(warm):
        orc.step(acts[t % 8], t)
    t0 = time.perf_counter(); steps = 0
    while True:
        orc.step(acts[steps % 8], warm + steps); steps += 1
        el = time.perf_counter() - t0
        if (steps >= min_steps and el >= min_s) or el > max_s:
            break
    return steps, el


def cpu_baseline(workload: str, envs: int, seed: int, budget_s: float = 12.0):
    """Time the CPU oracle on a bounded sample: `envs` envs, as many steps as fit in ~budget_s, all physical cores."""
    threads, probe = _pick_threads(workload, envs, seed)
    orc = _cpu_oracle(workload, envs, seed, threads)
    steps, el = _time_oracle(orc, 3, 20, budget_s, budget_s)
    return {"value": envs * steps / el, "unit": UNIT, "cores": threads, "kind": "port", "thread_probe": probe,
            "sample": f"{envs} envs x {steps} env-steps of {workload} (oracle/wl_oracle.c -O3 -march=native, OpenMP {threads} threads: best of "
                      f"{{1/4, 1/2, 1}} x {_physical_cores()} physical cores, OMP_PROC_BIND=close), {el:.1f} s"}


def run_reference(args):
    """Reference arm: the CPU implementation of the path on this box's host cores (rank 0 only), same workload and the same
    GLOBAL env count as the GPU arm at this N."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = WORKLOADS[args.workload]
    envs = (args.envs or w["envs"]) * max(1, args.gpus)
    threads, probe = _pick_threads(args.workload, envs, args.seed)
    orc = _cpu_oracle(args.workload, envs, args.seed, threads)
    acts = [orc.synth_actions(t) for t in range(8)]
    for t in range(args.warmup):
        orc.step(acts[t % 8], t)
    t0 = time.perf_counter()
    for k in range(args.steps):
        out = orc.step(acts[k % 8], args.warmup + k)
    el = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(zip(("obs", "rewards", "terminated", "truncated"), out)))
    val = envs * args.steps / el
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{w['label']}: {envs} envs (CPU, one box)", "envs_per_step": envs, "same_config": True,
                   "note": "PhysX is not runnable here; this is the CPU restatement of the same step (oracle/wl_oracle.c)"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "thread_probe": probe,
                         "sample": f"{envs} envs x {args.steps} steps, OpenMP {threads} threads (best of 1/4, 1/2, 1 x "
                                   f"{_physical_cores()} physical cores; {os.cpu_count()} logical), OMP_PROC_BIND=close, {el:.2f} s timed"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


class _StdoutGuard:
    """Everything any library prints to fd 1 (e.g. NCCL's version banner) goes to stderr; emit() writes the ONE JSON line
    to the real stdout."""

    def __init__(self):
        sys.stdout.flush()
        self._real = os.dup(1)
        os.dup2(2, 1)

    def emit(self, text: str):
        os.write(self._real, (text + "\n").encode())


def run_ours(args):
    guard = _StdoutGuard()
    import torch
    import torch.distributed as dist
    import wheeledlab_b200 as wl
    from wheeledlab_b200.distributed import RolloutSlab
    from wheeledlab_b200.sim import _stream_ptr

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")     # NCCL's version/warn lines must not pollute the ONE JSON line
        dist.init_process_group("nccl", device_id=torch.device(dev))

    w = WORKLOADS[args.workload]
    E, K, W = args.envs or w["envs"], args.steps, args.warmup
    mk = lambda seed_off=0: wl.make_task(w["task"], num_envs=E, seed=args.seed + seed_off, env_id_offset=rank * E)
    peak, peak_src = _peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        tt = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    # ---- M independent env sets: the working set (state + parameters) exceeds L2, so round-robin stepping is cold ----
    # M follows the nominal SET_BYTES_PER_ENV, not this build's buffer size: which env set runs step k, with which seed
    # and history, then depends on the arguments only, and --dump-outputs of two builds can be compared
    sim0 = wl.WheeledSim(mk(), dev)
    set_bytes = sim0._buf.numel() * 4
    M = max(4, math.ceil(2.2 * L2_BYTES / (SET_BYTES_PER_ENV * E)))
    sims = [sim0] + [wl.WheeledSim(mk(1000 * m), dev) for m in range(1, M)]
    for s in sims:
        s.startup(); s.reset(None, 0)
    # rollout length: rsl_rl num_steps_per_env is 128 (rsl_rl_ppo_cfg.py:6), shortened so that the driver's short runs still hold
    # exchanges inside the K steps.  The run is continuous: step k (warm-up steps included) fills row k % T_ROLL of slab
    # (k // T_ROLL) % 2 and an exchange follows every T_ROLL-th step, so a window of K steps holds ~K / T_ROLL of them
    fam = w["task"] in ("drift", "hound_4wd")
    want = args.gather if args.gather != "auto" else ("mcast" if fam else "ce")   # mcast falls back to per-peer stores, then NCCL
    if want in ("fanout", "mcast") and not fam:
        want = "ce"                                           # the height-scan rows are written by wl_scan_kernel (no fan-out)
    T_ROLL = min(128, max(4, K // 2))
    n_slabs = 2
    gather_mode, syms = "nccl", []
    use_mc = False
    if world > 1 and want in ("fanout", "mcast", "ce"):
        try:                                                  # symmetric (P2P-mapped) slabs: the fused fan-out, or a copy-engine pull
            from wheeledlab_b200.distributed import SymmetricRolloutSlab
            syms = [SymmetricRolloutSlab(T_ROLL, E, sim0.obs_dim, 2, dev) for _ in range(n_slabs)]
            gather_mode = "fanout" if want == "mcast" else want
            use_mc = want == "mcast" and all(sy.mc_delta != 0 for sy in syms)
            if want == "mcast" and not use_mc:
                print("[bench] no NVSwitch multicast alias for the symmetric buffers; per-peer stores", file=sys.stderr)
        except Exception as ex:
            if args.gather != "auto":
                raise
            syms = []
            print(f"[bench] symmetric memory unavailable ({ex!r}); using the NCCL all-gather", file=sys.stderr)
    slabs = [sy.slab for sy in syms] if syms else [RolloutSlab(T_ROLL, E, sim0.obs_dim, 2, dev) for _ in range(n_slabs)]
    acts = torch.stack([sim0.synth_actions(t) for t in range(max(8, min(W + K, 64)))])   # resident in HBM
    NA = acts.shape[0]
    tcount = [0] * M

    def make_bound(k):                                        # step k of the run: env set k % M, slab (k // T_ROLL) % 2, row k % T_ROLL
        fn = sims[k % M].bind_step(acts[k % NA], slabs[(k // T_ROLL) % n_slabs].step_outputs(k % T_ROLL))
        if not syms:
            return fn
        if gather_mode != "fanout":
            return fn
        sim_k, sy_k = sims[k % M], syms[(k // T_ROLL) % n_slabs]
        deltas, mcd = sy_k.peer_deltas, (sy_k.mc_delta if use_mc else 0)

        def fan(tc, _fn=fn, _sim=sim_k, _d=deltas, _m=mcd):   # this step's rows also go to the same slab slot of every peer
            _sim.set_peer_fanout(_d)
            _sim.set_multicast_fanout(_m)
            _fn(tc)
        return fan

    bound_w = [make_bound(k) for k in range(W)]
    bound = [make_bound(W + k) for k in range(K)]
    gstream = torch.cuda.Stream(device=dev) if world > 1 else None
    main = torch.cuda.current_stream()

    def run_steps(fns, k0, timed):
        """Issue the steps back to back on the current stream; with N > 1, ONE exchange of the filled slab per T_ROLL steps:
        gather mode "nccl": all_gather_into_tensor on its own stream (overlaps the next steps; the step stream only waits when
        a slab is about to be refilled before its gather is done); mode "fanout": the steps have already stored their rows
        into every peer's symmetric buffer -- only a device-side barrier remains."""
        cur_stream = torch.cuda.current_stream()
        gev, gdone = [], [None] * n_slabs
        for j, fn in enumerate(fns):
            k = k0 + j
            row, cur = k % T_ROLL, (k // T_ROLL) % n_slabs
            if world > 1 and row == 0 and gdone[cur] is not None:
                cur_stream.wait_event(gdone[cur])             # this slab's previous exchange must be over before it is refilled
            m = k % M
            fn(tcount[m]); tcount[m] += 1
            if world > 1 and row == T_ROLL - 1:
                filled = torch.cuda.Event(); filled.record()
                with torch.cuda.stream(gstream):              # the exchange runs beside the next rollout's steps
                    gstream.wait_event(filled)
                    g0, g1 = torch.cuda.Event(enable_timing=timed), torch.cuda.Event(enable_timing=timed)
                    g0.record()
                    if gather_mode == "fanout":
                        syms[cur].barrier()                   # the rows are already in every peer's buffer: completion barrier only
                    elif gather_mode == "ce":
                        syms[cur].gather_ce()
                    else:
                        slabs[cur].all_gather()
                    g1.record(); gev.append((g0, g1))
                    gdone[cur] = g1
        for g in gdone:                                       # the last gathers must be finished before the clock stops
            if g is not None:
                cur_stream.wait_event(g)
        return gev

    if world > 1:                                             # untimed set-up: one exchange per slab (NCCL channels / receive
        for i_s in range(n_slabs):                            # buffers, the barrier kernel's module load, peer mappings touched)
            if gather_mode == "fanout":
                syms[i_s].barrier()
            elif gather_mode == "ce":
                syms[i_s].gather_ce()
            else:
                slabs[i_s].all_gather()
    # Both the W warm-up steps and the K timed steps are captured into CUDA graphs (how a rollout is meant to be driven: the
    # Python + driver launch path costs ~8 us per step here, more than the kernel), instantiated and uploaded at set-up.  On the
    # device the sequence is  [spin][rank alignment][W warm-up steps] e0 [K steps] e1 : the warm-up runs IMMEDIATELY before the
    # clock starts (caches, clocks and -- N > 1 -- the NVLink lanes are in their steady state: idle lanes take ~0.1 ms to wake),
    # and the spin keeps the GPU busy while the host enqueues everything, so e0..e1 holds no host launch latency.
    sim_x = wl.WheeledSim(mk(777), dev); sim_x.startup(); sim_x.reset(None, 0)        # loads the step kernels' module before capture
    sim_x.bind_step(acts[0], RolloutSlab(1, E, sim0.obs_dim, 2, dev).step_outputs(0))(0)
    torch.cuda.synchronize()
    del sim_x
    graph, graph_w, timing_mode, gev = None, None, "eager stream launches", []

    def capture(fns, k0):
        g = torch.cuda.CUDAGraph()
        cs_ = torch.cuda.Stream(device=dev)
        cs_.wait_stream(main)
        with torch.cuda.stream(cs_):
            with torch.cuda.graph(g, stream=cs_):
                ev = run_steps(fns, k0, False)
        main.wait_stream(cs_)
        wl.upload_graph(g, main)                              # set-up, not steps: the first replay would otherwise pay the upload
        return g, ev

    if not args.eager:
        keep = list(tcount)
        try:
            graph_w, _ = capture(bound_w, 0)
            graph, gev = capture(bound, W)
            timing_mode = "one CUDA graph of the K steps (instantiated + uploaded at set-up), replayed once right after the graph of the W warm-up steps"
        except Exception as ex:
            print(f"[bench] graph capture failed ({ex!r}); timing eager launches", file=sys.stderr)
            graph = graph_w = None
            tcount[:] = keep
    sampler = ClockSampler(list(range(world)) if world > 1 else local)
    barrier()
    if rank == 0:
        sampler.start()
    l0 = sum(s.launch_count for s in sims)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_tok = torch.zeros(1, device=dev)
    if world > 1:
        dist.all_reduce(sync_tok)                             # (untimed: first use of this buffer)
    barrier()
    torch.cuda._sleep(400_000 if world == 1 else 800_000)
    if world > 1:                                             # device-side alignment of the ranks: the hosts leave dist.barrier()
        dist.all_reduce(sync_tok)                             # up to ~0.1 ms apart, which the first exchange would otherwise absorb
    if graph is not None:
        graph_w.replay()
        e0.record()
        graph.replay()
    else:
        run_steps(bound_w, 0, False)
        l0 = sum(s.launch_count for s in sims)
        e0.record()
        gev = run_steps(bound, W, True)
    e1.record()
    barrier()
    tot_ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:                      # before anything else writes into the slabs
        last = W + K - 1
        obs, rew, term, trunc = slabs[(last // T_ROLL) % n_slabs].step_outputs(last % T_ROLL)
        dump_outputs(args.dump_outputs, {"obs": obs, "rewards": rew, "terminated": term, "truncated": trunc})
    launches = (sum(s.launch_count for s in sims) - l0) if graph is None else K
    n_exchanges = len(gev)
    # duration of one exchange on its own (eager, outside the timed region): all-gather ms / barrier ms
    gather_each = []
    if world > 1:
        for _ in range(3):
            a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            a_.record()
            if gather_mode == "fanout":
                syms[0].barrier()
            elif gather_mode == "ce":
                syms[0].gather_ce()
            else:
                slabs[0].all_gather()
            b_.record(); torch.cuda.synchronize()
            gather_each.append(a_.elapsed_time(b_))
    gather_ms = sum(gather_each)
    if gather_each and rank == 0:
        print(f"[bench] slab exchange ({gather_mode}) ms per call, measured alone: {[round(x, 3) for x in gather_each]}", file=sys.stderr)

    # ---- round-1 protocol for comparison: per-step events, 256 MiB flush fill between steps; and its floor (empty kernel) ----
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    KF = min(K, 50)
    outs = slabs[0].step_outputs(0)
    t = tcount[0]
    fn0 = sim0.bind_step(acts[0], outs)
    for _ in range(3):
        fn0(t); flush.fill_(0.0); t += 1
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(KF)]
    for a, b in ev:
        a.record(); fn0(t); b.record(); flush.fill_(0.0); t += 1
    torch.cuda.synchronize()
    flush_us = [a.elapsed_time(b) * 1e3 for a, b in ev]
    evn = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(30)]
    for a, b in evn:
        a.record(); wl.lib.wl_test_null((4 * E + 31) // 32, 32, _stream_ptr(sim0.device)); b.record(); flush.fill_(0.0)
    torch.cuda.synchronize()
    null_us = statistics.median(a.elapsed_time(b) * 1e3 for a, b in evn)
    del flush
    # ---- warm-L2, CUDA-graph replay of K steps on ONE env set (supplementary: how a rollout is meant to be driven) ----
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    sim0.set_step_counter(t)
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            for k in range(K):
                sim0.step(acts[k % NA], sim0.device_counter_plus(k), out=outs)
            sim0.advance_counter(K)
    torch.cuda.current_stream().wait_stream(s)
    sim0.set_step_counter(t)
    g.replay(); barrier()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda._sleep(200_000)                                # (as above: the host's graph-launch latency stays outside g0..g1)
    g0.record(); g.replay(); g1.record(); barrier()
    graph_ms = g0.elapsed_time(g1)
    sim0.note_device_counter(t + 2 * K)
    # ---- end-to-end through the public API with host buffers: actions H2D, observations + reward + dones D2H, every step ----
    env = wl.ManagerBasedRLEnv(mk(), device=dev)
    env.reset()
    env.host_obs = True
    h_act = acts.cpu().pin_memory()
    h_rows = [h_act[k] for k in range(NA)]                    # row views of the pinned block (what a host-side policy hands over)

    def time_e2e(transport, host_obs=True):
        env.host_transport, env.host_obs = transport, host_obs
        for k in range(max(W, 5)):
            env.step_host(h_rows[k % NA])
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        a.record()
        for k in range(K):
            obs, rew, term, trunc, extras = env.step_host(h_rows[k % NA])      # returns after the stream sync: results are on the host
        b.record(); barrier()
        return max(a.elapsed_time(b), 1e3 * (time.perf_counter() - t0) * 0.0)

    e2e_variants = {"zero_copy_obs_host": time_e2e("zero_copy"), "staged_copy_obs_host": time_e2e("copy"),
                    "zero_copy_obs_on_device": time_e2e("zero_copy", host_obs=False)}
    best = min(("zero_copy_obs_host", "staged_copy_obs_host"), key=lambda k2: e2e_variants[k2])
    e2e_ms = e2e_variants[best]
    # ---- supplementary figures (drift only): policy in the loop, fused policy, fused K-step rollout ----
    pil = pfu = fused = None
    if args.workload == "drift" and not args.no_extras:
        try:
            from wheeledlab_b200.rollout import GraphedRollout
            torch.manual_seed(0)
            mlp = torch.nn.Sequential(torch.nn.Linear(sim0.obs_dim, 64), torch.nn.ELU(), torch.nn.Linear(64, 64), torch.nn.ELU(),
                                      torch.nn.Linear(64, 2)).to(dev)
            sim_p = wl.WheeledSim(mk(), dev); sim_p.startup(); sim_p.reset(None, 0)
            with torch.no_grad():
                roll = GraphedRollout(sim_p, lambda o: mlp(o), 128).capture(0)
                roll.run(); barrier()
                R = 4
                p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                p0.record()
                for _ in range(R):
                    roll.run()
                p1.record(); barrier()
            pil_ms = max_over_ranks(p0.elapsed_time(p1))
            pil = {"value": E * world * 128 * R / (pil_ms * 1e-3), "unit": UNIT, "ms_per_step": pil_ms / (128 * R),
                   "note": "rsl_rl-sized actor (14-64-64-2 ELU, torch/cuBLAS) + fused env step, 128 steps per CUDA-graph launch"}
        except Exception as ex:
            pil = {"error": repr(ex)[:200]}
        try:
            from wheeledlab_b200.policy import FusedPolicyRollout, pack_actor_critic
            torch.manual_seed(0)
            mkn = lambda out: torch.nn.Sequential(torch.nn.Linear(sim0.obs_dim, 64), torch.nn.ELU(), torch.nn.Linear(64, 64), torch.nn.ELU(),
                                                  torch.nn.Linear(64, out)).to(dev)
            blob = pack_actor_critic(mkn(2), mkn(1), torch.ones(2), sim0.obs_dim, dev)
            sim_q = wl.WheeledSim(mk(), dev); sim_q.startup(); sim_q.reset(None, 0)
            froll = FusedPolicyRollout(sim_q, blob, 128).capture(0)
            froll.run(); barrier()
            R = 4
            q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            q0.record()
            for _ in range(R):
                froll.run()
            q1.record(); barrier()
            pfu_ms = max_over_ranks(q0.elapsed_time(q1))
            pfu = {"value": E * world * 128 * R / (pfu_ms * 1e-3), "unit": UNIT, "ms_per_step": pfu_ms / (128 * R),
                   "note": "rsl_rl actor AND critic (14-64-64-2/1 ELU), Gaussian sample + log-prob, and the env step in ONE kernel; "
                           "128 launches per CUDA graph"}
        except Exception as ex:
            pfu = {"error": repr(ex)[:200]}
        try:
            KFR = 125                                         # divides the 250-step episode: windows end on curriculum boundaries
            sim_f = wl.WheeledSim(mk(), dev); sim_f.startup(); sim_f.reset(None, 0)
            slab_f = RolloutSlab(KFR, E, sim_f.obs_dim, 2, dev)
            logs_f = torch.empty((KFR, 16), dtype=torch.float32, device=dev)
            sim_f.rollout(KFR, 0, slab_f, logs_f); barrier()
            RF = 8
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record()
            for r in range(RF):
                sim_f.rollout(KFR, KFR * (1 + r), slab_f, logs_f)
            f1.record(); barrier()
            f_ms = max_over_ranks(f0.elapsed_time(f1))
            fused = {"value": E * world * KFR * RF / (f_ms * 1e-3), "unit": UNIT, "ms_per_step": f_ms / (KFR * RF), "K": KFR,
                     "note": "wl_rollout: K env.steps per launch, state in registers, in-kernel U[-1,1]^2 actions; every step still "
                             "writes its obs/action/reward/done slab rows and episode-log row; bit-identical to K wl_step calls"}
        except Exception as ex:
            fused = {"error": repr(ex)[:200]}
    # The timed region lasts ~0.1 ms and nvidia-smi needs up to a second to deliver its first row: keep every GPU of the job under
    # the same step load (a scratch env set, no exchange) until rank 0 has read two rows per GPU, so that the clocks line is never
    # empty or sampled on an idle (down-clocked) device.
    def _need_rows():
        return rank == 0 and sampler.proc is not None and len(sampler.rows) < 2 * world
    flag = torch.tensor([1.0 if _need_rows() else 0.0], device=dev)
    if world > 1:
        dist.all_reduce(flag, op=dist.ReduceOp.MAX)
    if float(flag.item()) > 0:
        sim_l = wl.WheeledSim(mk(555), dev); sim_l.startup(); sim_l.reset(None, 0)
        fn_l = sim_l.bind_step(acts[0], RolloutSlab(1, E, sim0.obs_dim, 2, dev).step_outputs(0))
        t_l, t_end = 0, time.time() + 4.0
        while True:
            for _ in range(500):
                fn_l(t_l); t_l += 1
            flag.fill_(1.0 if (_need_rows() and time.time() < t_end) else 0.0)
            if world > 1:
                dist.all_reduce(flag, op=dist.ReduceOp.MAX)
            if float(flag.item()) == 0:
                break
        del sim_l
    clocks = sampler.stop() if rank == 0 else None

    tot_ms_own = tot_ms
    tot_ms, graph_ms, e2e_ms = max_over_ranks(tot_ms), max_over_ranks(graph_ms), max_over_ranks(e2e_ms)
    gather_ms = max_over_ranks(gather_ms)
    per_rank = None
    if world > 1:                                             # diagnostics: which rank sets the max
        st = torch.tensor([tot_ms_own / K, statistics.median(flush_us) * 1e-3], dtype=torch.float64, device=dev)
        allst = [torch.zeros_like(st) for _ in range(world)]
        dist.all_gather(allst, st)
        per_rank = {"step_us_mean": [round(float(x[0]) * 1e3, 3) for x in allst],
                    "flush_protocol_step_us_median": [round(float(x[1]) * 1e3, 3) for x in allst]}
    if rank == 0:
        total_envs = E * world
        value = total_envs * K / (tot_ms * 1e-3)
        kern_s = tot_ms * 1e-3 / K
        achieved = w["bytes"] * E / kern_s / 1e9
        cpu = cpu_baseline(args.workload, E, args.seed, budget_s=args.cpu_budget) if world == 1 else None
        slab_bytes = slabs[0].nbytes
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": tot_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{w['label']}: {E} envs/GPU x {world} GPU", "envs_per_gpu": E, "global_envs": total_envs,
                       "actions": "U[-1,1]^2 philox(seed,env,step)",
                       "l2": f"inputs larger than L2, no flush kernel: {M} independent {E}-env sets ({M * set_bytes / 1e6:.0f} MB of state + "
                             f"parameters) stepped round-robin, every step writes a fresh rollout-slab row ({n_slabs} x {slab_bytes / 1e6:.0f} MB)",
                       "parallelism": f"env-shard x{world}", "timing": f"2 CUDA events around the K back-to-back steps ({timing_mode})"},
            "clocks": clocks,
            "e2e": {"value": total_envs * K / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": E * 8,
                    "d2h_bytes_per_step": E * (6 + 4 * sim0.obs_dim), "ms_per_step": e2e_ms / K, "transport": best,
                    "variants_ms_per_step": {k2: v / K for k2, v in e2e_variants.items()},
                    "api": "ManagerBasedRLEnv.step_host(pinned actions), host_obs=True: actions H2D, observations + reward + dones D2H "
                           "(zero_copy: the kernel reads / writes pinned host memory over PCIe; staged_copy: cudaMemcpyAsync both ways), "
                           "stream sync, every step.  zero_copy_obs_on_device (round 1's figure: obs left on the GPU) is listed for comparison"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": _traffic(w["traffic_profile"]) if E == w["envs"] else None, "traffic_unit": "bytes/launch (dram read + write, ncu --set full)",
                         "traffic_source": w["traffic_profile"], "peak_source": peak_src, "kernel": w["kernel"],
                         "bytes_per_env_step": w["bytes"], "avg_step_us": kern_s * 1e6,
                         "kernel_variant": ("duo (8 envs per 64-thread CTA: env warp 4 lanes/env + aux warp)" if (fam and E <= 37888)
                                            else "quad (4 lanes/env)" if E <= 148 * 4 * 32 * 2 else "thread-per-env"),
                         "note": f"{E} envs move {w['bytes'] * E / 1e6:.1f} MB per launch: latency-bound at this size, see profiles/ for the N sweep"},
            "cpu_baseline": cpu,
            "flush_protocol": {"step_us_median": statistics.median(flush_us), "step_us_mean": statistics.mean(flush_us),
                               "value": total_envs / (statistics.mean(flush_us) * 1e-6) if world == 1 else None,
                               "empty_kernel_us": null_us,
                               "note": "round-1 protocol: per-step events, 256 MiB L2-flush fill between steps; empty_kernel_us is the same "
                                       "measurement around an EMPTY kernel of the same geometry (the protocol's own floor)"},
            "collective": {"kind": {"fanout": ("fused NVSwitch-multicast fan-out: every step stores its slab rows ONCE to the multicast alias of the "
                                               "symmetric buffers (multimem.st; the switch replicates them into every rank's copy); one device-side "
                                               "barrier per iteration") if use_mc else
                                              "fused peer-memory fan-out: every step stores its slab rows into each peer's symmetric buffer over NVLink; "
                                              "one device-side barrier per iteration",
                                    "ce": "copy-engine pull: barrier, world-1 P2P memcpys of the peers' slabs over NVLink (no SM), barrier",
                                    "nccl": "all_gather_into_tensor(rollout slab)"}[gather_mode],
                           "mode": ("mcast" if use_mc else gather_mode), "per_iteration_steps": T_ROLL, "bytes_per_rank": slab_bytes, "count": n_exchanges,
                           "ms_each_measured_alone": [round(x, 3) for x in gather_each],
                           "nvlink_bytes_per_step_per_rank": (E * (4 * sim0.obs_dim + 6) * (1 if use_mc else world - 1)) if gather_mode == "fanout" else None,
                           "bus_GBps": (slab_bytes * (world - 1) / (statistics.mean(gather_each) * 1e-3) / 1e9) if (gather_each and gather_mode != "fanout") else None,
                           "inside_timed_region": True,
                           "note": "every exchange of the K steps (count) completes before the clock stops; nccl mode: double-buffered slabs, the "
                                   "gather of iteration i runs on its own stream under the steps of iteration i+1"}
            if world > 1 else None,
            "per_rank": per_rank,
            "policy_in_loop_graph": pil,
            "policy_fused_in_step": pfu,
            "rollout_fused": fused,
            "warm_l2_graph": {"value": total_envs * K / (graph_ms * 1e-3), "unit": UNIT, "ms_per_step": graph_ms / K,
                              "note": "K steps of ONE env set captured in one CUDA graph (PDL edges), state L2-resident (supplementary)"},
        }
        guard.emit(json.dumps(line))
    if world > 1:                                             # (symmetric-memory / graph teardown can stall at interpreter exit: leave at once)
        dist.barrier()
        sys.stdout.flush(); sys.stderr.flush()
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--workload", default="drift", choices=sorted(WORKLOADS))
    ap.add_argument("--envs", type=int, default=0, help="envs per GPU (default: the workload's BASELINE size)")
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-budget", type=float, default=12.0)
    ap.add_argument("--no-extras", action="store_true", help="skip the supplementary figures (policy-in-loop, fused rollout)")
    ap.add_argument("--eager", action="store_true", help="time eager stream launches instead of one CUDA graph of the K steps")
    ap.add_argument("--gather", default="auto", choices=["auto", "nccl", "ce", "fanout", "mcast"],
                    help="N > 1 slab exchange: fused into the step kernel as NVSwitch-multicast stores (mcast; auto for the Drift family, "
                         "falling back to per-peer stores = fanout, then to NCCL), copy-engine pull over symmetric memory (ce; auto "
                         "for Elevation), or NCCL all-gather")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one returned (observations, "
                    "rewards, terminated, truncated) as float32 DIR/<name>.npy (<= 64 MB: a seeded sample of envs when larger).  "
                    "Compares builds run with the same arguments and --impl; the two --impl arms step different env sets, "
                    "so their dumps are not comparable with each other")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
