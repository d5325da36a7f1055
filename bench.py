#!/usr/bin/env python
"""SAC gradient steps/s on B200 (BASELINE.json metric), with roofline, CPU baseline, e2e and the other BASELINE configs.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload LL|VS|MS|C10|C10O] [--replicas R] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference ...      # the reference's CPU learner path on the host cores

One "step" = one full SAC gradient step (target, twin-critic update, actor update, temperature update, Polyak) of every
learner replica on the GPU.

`value`  learner-steps/s with the replay ring resident in HBM: index sampling + gather + step all on the device, CUDA
         graphs of 8/4/2/1 steps.  Every graph is instantiated BEFORE the clock starts (b200sac_prepare) and >= 16 warm-up
         steps run first.  The timed region is EXACTLY K steps, run as a train of back-to-back windows (multiples of 8 steps,
         so each window is whole 8-step graphs), a CUDA event between windows, barrier + synchronize on both sides of the
         train; `ms_per_step` is the MEDIAN over windows of the window's time per step (per window: max over ranks); all
         window statistics and per-rank medians are in `timing`.
         --dump-outputs DIR writes what the timed region computed in its last step (rank 0): the losses of every replica and
         each replica's parameters, target networks and Adam moments, as DIR/<name>.npy (float32; Adam step counts and the
         GEMM back-end used, `precision`, float64).  Inputs are seeded, so the same arguments give the same inputs on every
         run; pin --precision 0 or 1 to compare dumps, since the default -1 picks the back-end by a timing probe.  Above
         64 MB in all, every large tensor is replaced by a fixed seeded sample of its elements (flattened).  The library
         must have been built (__graft_entry__.build()) from the sources in the tree: the benchmark refuses a missing or
         stale one, and compiles nothing and writes nothing in the source tree.
`e2e`    the same metric through the reference-shaped `Learner.update()` with the replay ring in pinned HOST memory: per
         step a host-side sample + gather, an H2D copy of the minibatch and a D2H read of the losses, synchronously --
         the reference's update() contract.
`configs` short legs of the other BASELINE.json configs (VS, MS, C10), config 4's 10-learner placement over the GPUs of
         this run, and the learners-per-GPU sweep; same timing protocol.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark leaves the source tree untouched (it may be read-only)

import numpy as np  # noqa: E402
import torch  # noqa: E402

# ring sizes, declared once: `value` samples the device ring (BASELINE config 2: 1M transitions resident in HBM);
# the e2e leg, the cpu_baseline and the --impl reference arm all use the SAME host-side buffer size (BASELINE.md §3).
DEVICE_RING = 1 << 20
HOST_RING = 20000

# SURVEY.md §8(d): algorithmic work per gradient step (streaming model)
WORK = {
    "LL": dict(gflop=0.557, mbytes=6.087),
    "VS": dict(gflop=10.970, mbytes=30.188),
    "MS": dict(gflop=13.846, mbytes=30.728),
    "C10": dict(gflop=17.088, mbytes=37.377),
    # CARE(O): same consumer MLPs and mixture as C10; the context path is per-task (10 rows) in both, so the per-step
    # streaming-model work differs only by the 89.6 k trainable context-encoder parameters (SURVEY §8(f) rank 4)
    "C10O": dict(gflop=17.088, mbytes=37.377 + 89600 * 24e-6),
}
WORKLOAD_DESC = {
    "LL": "LunarLanderContinuous-v2 SAC learner (obs 8, act 2, MLP 256-256, batch 256)",
    "VS": "MT1 VSAC-shape SAC learner (obs 39, act 4, MLP 400x3, batch 1024, twin-Q)",
    "MS": "MT10 MTSAC learner (mtobs 49, act 4, MLP 400x3, batch 1280, 10 tasks one-hot, weighted loss)",
    "C10": "MT10 CARE(M) learner (mtobs 49, act 4, K=6 mixture encoders 39-50-50, 768-d context, MLP 400x3 over the 100-d encoded state, batch 1280)",
    "C10O": "MT10 CARE(O) learner (use_modified_care=false: trainable context encoder 768-100-50-50-50-50 with its own Adam, "
            "K=6 mixture encoders, MLP 400x3, batch 1280, unweighted losses)",
}
REF_VARIANT = {"LL": "LL", "VS": "VS", "MS": "MS", "C10": "C10", "C10O": "C10"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm=float(d["hbm_gbs"]), tf=float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), src="measured")
    return dict(hbm=6650.0, tf=1590.0, src="fallback")


def core_config(workload, replicas, precision=1):
    from distributed_sac_b200.core import CoreConfig
    if workload == "LL":
        return CoreConfig(replicas=replicas, precision=precision)
    if workload == "VS":
        return CoreConfig(state_dim=39, act_dim=4, actor_hidden=[400] * 3, critic_hidden=[400] * 3, batch=1024,
                          replicas=replicas, precision=precision)
    if workload == "MS":
        return CoreConfig(state_dim=39, act_dim=4, actor_hidden=[400] * 3, critic_hidden=[400] * 3, batch=1280,
                          num_tasks=10, weighted_loss=True, replicas=replicas, precision=precision)
    if workload == "C10":
        return CoreConfig(state_dim=39, act_dim=4, actor_hidden=[400] * 3, critic_hidden=[400] * 3, batch=1280,
                          num_tasks=10, weighted_loss=True, replicas=replicas, precision=precision, care=True)
    if workload == "C10O":
        return CoreConfig(state_dim=39, act_dim=4, actor_hidden=[400] * 3, critic_hidden=[400] * 3, batch=1280,
                          num_tasks=10, weighted_loss=False, replicas=replicas, precision=precision, care=True,
                          care_original=True, emb_dim=50, lr_ctx=3e-4)
    raise ValueError(workload)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons (B200_PROFILING.md recipe).  Started before the warm-up; lines that arrive
    between mark_begin() and mark_end() are the timed region's."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []
        self.t0 = self.t1 = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "50"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        time.sleep(0.06)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, sm_timed, mx, reasons = [], [], [], set()
        for ts, ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                v = float(f[1]); mx.append(float(f[2]))
            except ValueError:
                continue
            sm.append(v)
            if self.t0 is not None and self.t1 is not None and self.t0 <= ts <= self.t1 + 0.05:
                sm_timed.append(v)
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        use = sorted(sm_timed) if sm_timed else sorted(sm)
        return {"sm_mhz": use[len(use) // 2] if use else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "samples_in_timed_region": len(sm_timed),
                "window": "warm-up + timed region of the headline leg (50 ms period)"}


# --------------------------------------------------------------------------------------------------
# CPU side: the reference's own learner (kind "reference") when a checkout is reachable, else the oracle port ("port")
# --------------------------------------------------------------------------------------------------
def reference_available():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_harness as rh
    return rh.available()


def cpu_learner(workload, n_buffer=HOST_RING, seed=0, prefer_reference=True):
    """(kind, update_fn): update_fn() = one reference-shaped update() (sample + update_SAC) on the host."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import sac_port as sp
    if prefer_reference and reference_available():
        import ref_harness as rh
        over = {"use_modified_care": workload == "C10"} if workload in ("C10", "C10O") else None
        lrn, _ = rh.make_learner(REF_VARIANT[workload], over, seed=seed)
        spec = {"LL": sp.ll_spec, "VS": sp.vs_spec}.get(workload, sp.ms_spec)()
        rh.fill_memory(lrn, REF_VARIANT[workload], sp.synthetic_batch(spec, seed=1234, batch=n_buffer))
        return "reference", lrn.update
    if workload in ("C10", "C10O"):
        import care_port as cp
        spec = cp.CareSpec() if workload == "C10" else cp.CareSpec(modified=False, weighted_loss=False)
        lrn = cp.CarePortLearner(spec, cp.init_params(spec, seed=seed))
        rspec = sp.ms_spec()                       # same replay layout as MTSAC: mtobs rows, B/T per task
    else:
        spec = rspec = {"LL": sp.ll_spec, "VS": sp.vs_spec, "MS": sp.ms_spec}[workload]()
        lrn = sp.PortLearner(spec, sp.init_params(spec, seed=seed))
    rb = sp.PortReplay(rspec, n_buffer, seed=seed)
    rb.push_many(*[t.numpy() for t in sp.synthetic_batch(rspec, seed=1234, batch=n_buffer)])
    return "port", (lambda: lrn.update_SAC(*rb.sample()))      # (CarePortLearner.update_SAC is its update())


def best_cpu_threads(update, ncpu=None):
    """Eager PyTorch on many cores is slower than on a few for these tiny ops (and a 128-thread probe of the larger
    learners costs minutes): probe 1 / 4 / 8 / 16 threads briefly and use the fastest, so the CPU arm is the reference path at
    its best on this host."""
    ncpu = ncpu or os.cpu_count() or 1
    cands = [t for t in (4, 8, 16, 1) if t <= ncpu] or [1]
    best, best_v = cands[0], 0.0
    for t in cands:
        torch.set_num_threads(t)
        update()
        t0 = time.perf_counter()
        n = 0
        while n < 3 and (n == 0 or time.perf_counter() - t0 < 1.5):
            update()
            n += 1
        v = n / (time.perf_counter() - t0)
        if v > best_v:
            best, best_v = t, v
    return best, best_v


def time_cpu(workload, budget_s=15.0, max_steps=2000, steps=None, warmup=5):
    """steps/s of update() on the host cores over a bounded sample: `steps` if given, else as many as fit `budget_s`."""
    kind, update = cpu_learner(workload)
    threads, probe_v = best_cpu_threads(update)
    torch.set_num_threads(threads)
    n = steps if steps else int(max(10, min(max_steps, budget_s * probe_v)))
    for _ in range(warmup):
        update()
    t0 = time.perf_counter()
    for _ in range(n):
        update()
    dt = time.perf_counter() - t0
    return dict(value=n / dt, steps=n, seconds=dt, cores=threads, kind=kind)


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.startswith("model name"):
                    return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def cpu_baseline_block(workload, budget_s):
    c = time_cpu(workload, budget_s=budget_s)
    what = ("the UNMODIFIED reference Learner.update() (Redis stubbed, device cpu)" if c["kind"] == "reference"
            else "the CPU oracle port (same eager-PyTorch op sequence as the reference's update(); no reference checkout on this box)")
    return {"value": c["value"], "unit": "steps/s", "cores": c["cores"], "kind": c["kind"],
            "sample": f"{c['steps']} update() calls (sample from a {HOST_RING}-transition host buffer + update_SAC) of {what} after 5 warm-up, "
                      f"{c['seconds']:.1f} s, torch {torch.__version__} CPU, {os.cpu_count()} logical CPUs, {cpu_model()}"}


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU learner path on the host cores, rank 0 only."""
    if rank != 0:
        return
    kind, update = cpu_learner(args.workload)
    threads, probe_v = best_cpu_threads(update)
    torch.set_num_threads(threads)
    # bounded sample: keep the whole run within ~2 minutes of CPU time whatever K the driver passes
    steps = max(10, min(args.steps, int(100 * probe_v)))
    warmup = min(max(args.warmup, 3), max(3, int(10 * probe_v)))
    for _ in range(warmup):
        update()
    t0 = time.perf_counter()
    for _ in range(steps):
        update()
    dt = time.perf_counter() - t0
    v = steps / dt
    line = {
        "impl": "reference", "metric": "SAC gradient steps/sec", "value": v, "unit": "steps/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD_DESC[args.workload], "host_replay": f"{HOST_RING}-transition host buffer, uniform sampling w/o replacement",
                   "learners": 1},
        "cpu_baseline": {"value": v, "unit": "steps/s", "cores": threads, "kind": kind,
                         "sample": f"{steps} update() calls (sample + update_SAC) after {warmup} warm-up, torch {torch.__version__} CPU, "
                                   f"{os.cpu_count()} logical CPUs, {cpu_model()}; "
                                   + ("unmodified reference Learner" if kind == "reference" else "oracle port of the reference learner (no reference checkout on this box)")},
        "e2e": {"value": v, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# GPU side
# --------------------------------------------------------------------------------------------------
def write_cfg(workload, tmp):
    """cfg JSON in the reference's own format (cfg/*.json) for the drop-in Learner."""
    base = {"device": "cuda", "buffer_size": 1e6, "reward_scale": 1, "gamma": 0.99, "log_alpha": 0, "tau": 0.005,
            "start_memory_len": 5000, "random_step": 5000}
    if workload == "LL":
        cfg = dict(base, num_tasks=10, batch_size=256, lr_actor=3e-4, lr_critic=3e-4, num_learn=1, num_time_step=1)
    elif workload == "VS":
        cfg = dict(base, batch_size=1024, lr_actor=3e-4, lr_critic=3e-4, update_delay=5, print_period_player=2,
                   print_period_learner=5, actor_hidden_dim=[400] * 3, critic_hidden_dim=[400] * 3)
    elif workload in ("C10", "C10O"):
        names = [f"task-{i}" for i in range(10)]
        g = torch.Generator().manual_seed(7)
        emb = {n: (torch.randn(768, generator=g) * 0.3).tolist() for n in names}     # synthetic stand-in for the RoBERTa rows
        with open(os.path.join(tmp, "emb.json"), "w") as f:
            json.dump(emb, f)
        with open(os.path.join(tmp, "names.json"), "w") as f:
            json.dump(names, f)
        cfg = dict(base, use_modified_care=(workload == "C10"), num_tasks=10, batch_size=1280, update_delay=6, print_period_player=2,
                   print_period_learner=10, max_episode_time=500,
                   actor={"state_dim": 39, "action_dim": 4, "action_bound": [-1.0, 1.0], "lr_actor": 3e-4,
                          "actor_hidden_dim": [400] * 3},
                   critic={"state_dim": 39, "action_dim": 4, "lr_critic": 3e-4, "critic_hidden_dim": [400] * 3},
                   encoder={"state_dim": 39, "pretrained_embedding_json_path": os.path.join(tmp, "emb.json"),
                            "task_name_json_path": os.path.join(tmp, "names.json"), "hidden_dims_contextEnc": [50, 50],
                            "embedding_dim_contextEnc": 50, "output_dim_contextEnc": 50, "RoBERTa_embedding_dim": 768,
                            "lr_contextEnc": 3e-4, "hidden_dims_mixtureEnc": [50], "output_dim_mixtureEnc": 50,
                            "num_encoders": 6, "num_tasks": 10, "state_encoder_tau": 0.05})
    else:
        cfg = dict(base, use_weighted_loss=True, num_tasks=10, batch_size=1280, update_delay=6, print_period_player=2,
                   print_period_learner=10, max_episode_time=500,
                   actor={"state_dim": 39, "action_dim": 4, "action_bound": [-1.0, 1.0], "lr_actor": 3e-4,
                          "actor_hidden_dim": [400] * 3},
                   critic={"state_dim": 39, "action_dim": 4, "lr_critic": 3e-4, "critic_hidden_dim": [400] * 3})
    path = os.path.join(tmp, "cfg.json")
    with open(path, "w") as f:
        json.dump(cfg, f)
    return path


class _NullServer:
    """The Redis server is IPC, not part of the measured path; the bench feeds the ring directly."""

    def __init__(self): self.kv = {}
    def scan_iter(self): return []
    def delete(self, k): pass
    def set(self, k, v): self.kv[k] = v            # keeps the value alive like a server would (no copy)
    def get(self, k): return self.kv.get(k)
    def rpush(self, k, v): pass

    def pipeline(self):
        class _P:
            def lrange(self, *a): return self
            def ltrim(self, *a): return self
            def execute(self): return [[], True]
        return _P()


def make_learner(workload, cfg_path, device_index, buffer_size, precision=1):
    from distributed_sac_b200 import learner as L
    srv = _NullServer()
    if workload == "LL":
        return L.LunarLanderLearner(cfg_path, write_mode=False, server=srv, device_index=device_index, buffer_size=buffer_size,
                                    precision=precision)
    if workload == "VS":
        return L.VSACLearner(cfg_path, write_mode=False, server=srv, device_index=device_index, precision=precision)
    if workload in ("C10", "C10O"):
        return L.CARELearner(None, None, cfg_path, write_mode=False, server=srv, device_index=device_index, precision=precision)
    return L.MTSACLearner(None, None, cfg_path, write_mode=False, server=srv, device_index=device_index, precision=precision)


DUMP_BYTES = 60 << 20        # array payload; with the .npy headers the dump stays under 64 MB


def dump_outputs(core, out_dir):
    """The state the last step left, as a caller reads it back (read_losses, get_named, get_steps), to out_dir/<name>.npy:
    `losses` [R][4] (critic, actor, alpha, entropy), `param.<tensor>` / `adam_m.<tensor>` / `adam_v.<tensor>` [R][shape] for
    every tensor of the layout (targets included), `adam_steps` [R][n] and `precision` [1] (the GEMM back-end that computed
    them: 0 = fp32 FFMA, 1 = 3xTF32 tcgen05).  If the arrays exceed DUMP_BYTES, each one of more
    than 4096 elements is replaced by the same fraction of its (flattened) elements at indices drawn with a fixed seed."""
    from distributed_sac_b200 import _lib
    R = core.cfg.replicas
    arrays = {"losses": core.read_losses(1)[0].numpy()}
    for tag, which in (("param", _lib.PARAMS), ("adam_m", _lib.ADAM_M), ("adam_v", _lib.ADAM_V)):
        per_replica = [core.get_named(which, r) for r in range(R)]
        for name in per_replica[0]:
            arrays[f"{tag}.{name}"] = np.stack([p[name].numpy() for p in per_replica])
    arrays["adam_steps"] = np.array([core.get_steps(r) for r in range(R)], dtype=np.float64)
    arrays["precision"] = np.array([core.cfg.precision], dtype=np.float64)
    big = sum(a.nbytes for a in arrays.values() if a.size > 4096)
    small = sum(a.nbytes for a in arrays.values()) - big
    frac = min(1.0, (DUMP_BYTES - small) / max(big, 1))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if frac < 1.0 and a.size > 4096:
            flat = a.reshape(-1)
            idx = np.random.default_rng(0).choice(flat.size, max(1, int(flat.size * frac)), replace=False)
            a = flat[np.sort(idx)]
        np.save(os.path.join(out_dir, name + ".npy"), a)


class Bench:
    def __init__(self, args):
        self.args = args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist
        self.stream = torch.cuda.Stream()
        self.pk = peaks()

    def barrier(self):
        torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize()

    def gather_ranks(self, vals):
        """[world][len(vals)] of a per-rank float list."""
        t = torch.tensor(vals, dtype=torch.float64, device="cuda")
        if self.dist is None:
            return t.reshape(1, -1).cpu()
        out = [torch.empty_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return torch.stack(out).cpu()

    # ---- the timing protocol ------------------------------------------------------------------------------------
    def timed_windows(self, core, ring, steps, W, clocks=None):
        """Train of back-to-back windows that together run exactly `steps` steps; returns (median over windows of the window's
        ms per step [max over ranks per window], info)."""
        w = 8 * max(1, math.ceil(steps / 128))           # ~16 windows, each whole 8-step graphs but (maybe) the last
        sizes = [w] * (steps // w) + ([steps % w] if steps % w else [])
        n = len(sizes)
        warm = max(W, 16)
        with torch.cuda.stream(self.stream):
            core.prepare(ring)                            # every graph instantiated before the clock starts
            core.step_sampled(ring, warm)
            self.barrier()
            evs = [torch.cuda.Event(enable_timing=True) for _ in range(n + 1)]
            if clocks:
                clocks.mark_begin()
            evs[0].record()
            for i, k in enumerate(sizes):
                core.step_sampled(ring, k)
                evs[i + 1].record()
            self.barrier()
            if clocks:
                clocks.mark_end()
        ms = [evs[i].elapsed_time(evs[i + 1]) for i in range(n)]
        allr = self.gather_ranks(ms)                      # [world][n]
        per_window = allr.max(dim=0).values               # max over ranks, per window
        per_step = per_window / torch.tensor(sizes, dtype=per_window.dtype)
        med = float(per_step.median())
        info = {"windows": n, "timed_steps": steps, "steps_per_window": sizes, "warmup_steps": warm,
                "window_ms": {"min": float(per_window.min()), "median": float(per_window.median()), "max": float(per_window.max()),
                              "first": float(per_window[0])},
                "step_ms": {"min": float(per_step.min()), "median": med, "max": float(per_step.max()), "first": float(per_step[0])},
                "per_rank_median_step_ms": [float(x) for x in (allr / torch.tensor(sizes, dtype=allr.dtype)).median(dim=1).values],
                "train_ms": float(allr.sum(dim=1).max()),
                "rule": "ms_per_step = median over windows of (max over ranks of the window's device time) / (the window's steps)"}
        return med, info

    def gpu_leg(self, workload, R, precision, steps, W, ring_n, seed0=1234, detail=False, clocks=None, bcast=False, dump=None):
        from distributed_sac_b200.core import Replay, SacCore
        from distributed_sac_b200.replicas import broadcast_initial_params
        core = SacCore(core_config(workload, R, precision), self.local, seed=seed0 + self.rank)
        if bcast and self.dist is not None:
            broadcast_initial_params(core, src=0)         # independent replicas: ONE collective (SURVEY 8(e))
        ring = Replay(core, ring_n, where="device", seed=99 + self.rank)
        ring.fill_synthetic(ring_n, seed=seed0 + self.rank)
        ms, info = self.timed_windows(core, ring, steps, W, clocks)
        losses = core.read_losses(min(steps, 64))
        assert torch.isfinite(losses).all(), f"non-finite losses in the timed region ({workload})"
        if dump:                                          # before the detail runs below step the core further
            dump_outputs(core, dump)
        total = self.gather_ranks([float(R)]).sum().item()                 # learners over all ranks
        out = {"value": total / (ms * 1e-3), "ms_per_step": ms, "learners": int(total), "timing": info,
               "launches_per_step": core.launches_per_step + 1,
               "gemm_backend": ("layer-chained fp32 FFMA (chain.cuh)" if (precision == 0 and workload == "LL") else
                                "fp32 FFMA" if precision == 0 else "tcgen05 3xTF32")}
        work = WORK[workload]
        step_s = ms * 1e-3
        out["hbm_frac"] = R * work["mbytes"] * 1e6 / step_s / 1e9 / self.pk["hbm"]
        out["tensor_frac"] = R * work["gflop"] * 1e9 / step_s / 1e12 / self.pk["tf"]
        if detail:
            with torch.cuda.stream(self.stream):
                prof = core.profile_step(ring, iters=10)
            torch.cuda.synchronize()
            with torch.cuda.stream(self.stream):
                tl = core.graph_timeline(ring, iters=200)          # true in-graph start-to-start times (us)
            torch.cuda.synchronize()
            names = ["sample_indices", "ingest"] + [n for n, _ in prof][1:]
            out["timeline"] = list(zip(names, tl))
        ring.close()
        core.close()
        return out

    def e2e_leg(self, workload, precision, Ke, W, with_publication=False):
        """Learner.update() per step, pinned-host ring of HOST_RING transitions."""
        res = {}
        with tempfile.TemporaryDirectory() as tmp:
            old = os.getcwd()
            os.chdir(tmp)
            try:
                lrn = make_learner(workload, write_cfg(workload, tmp), self.local, buffer_size=HOST_RING, precision=precision)
                lrn.memory.ring.fill_synthetic(HOST_RING, seed=4321 + self.rank)
                row_bytes = 4 * ((2 * lrn.core.cfg.obs_dim + lrn.core.cfg.act_dim + 2 + 31) // 32 * 32)
                with torch.cuda.stream(self.stream):
                    lrn.soft_update(None, None, 1.0)
                    lrn.core.prepare(lrn.memory.ring)
                    for _ in range(max(W, 16)):
                        lrn.update()
                    self.barrier()
                    t0 = time.perf_counter()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    last = None
                    for _ in range(Ke):
                        last = lrn.update()
                    e1.record()
                    self.barrier()
                    wall = time.perf_counter() - t0
                assert all(map(lambda x: x == x, last)), "NaN loss in e2e leg"
                t_e2e = max(wall, e0.elapsed_time(e1) * 1e-3)
                t_e2e = float(self.gather_ranks([t_e2e]).max())
                res = {"value": self.world * Ke / t_e2e, "unit": "steps/s", "h2d_bytes_per_step": lrn.core.cfg.batch * row_bytes,
                       "d2h_bytes_per_step": 16, "steps": Ke,
                       "api": "Learner.update() per step (host sample+gather from the pinned ring -> pinned staging -> cudaMemcpyAsync on a "
                              "side stream -> graph launch -> losses written to mapped pinned memory -> stream sync)",
                       "host_replay": f"{HOST_RING}-transition pinned-host ring"}
                if with_publication:
                    with torch.cuda.stream(self.stream):      # pipelined variant: no per-step host sync
                        lrn.update_many(max(W, 16))
                        self.barrier()
                        t0 = time.perf_counter()
                        lrn.update_many(Ke)
                        self.barrier()
                        res["pipelined_update_many"] = {"value": self.world * Ke / (time.perf_counter() - t0), "unit": "steps/s"}
                    # run()-loop body: update + publication of the actor blob (LL/learner.py:296-299), two ways:
                    #   blocking   = update(); get_parameters(); pickle
                    #   overlapped = Learner.run() itself (max_updates = Kp): step k+1 and the device-side assembly of its blob are
                    #                enqueued before blob k is handed to Redis; the checkpoint write of iteration 0 is stubbed out
                    import pickle as _pk
                    Kp = max(50, min(Ke, 500))
                    with torch.cuda.stream(self.stream):
                        t0 = time.perf_counter()
                        for _ in range(Kp):
                            lrn.update()
                            blob = lrn.parameters_blob(blocking=True)
                        t_block = time.perf_counter() - t0
                        lrn.save_checkpoint = lambda idx: None
                        lrn.my_print = lambda content: None
                        lrn.update_delay = 1
                        lrn.start_memory_len = -1                    # the ring was filled directly (per-task sub-rings hold HOST_RING / T rows)
                        lrn.run(max_updates=16)
                        t0 = time.perf_counter()
                        done = lrn.run(max_updates=Kp)
                        t_over = time.perf_counter() - t0
                        assert done == Kp
                        blob = lrn.server.get("parameters")
                    pub_bytes = 4 * sum(v.numel() for m in _pk.loads(blob).values() for v in m.values())
                    res["with_publication"] = {"unit": "steps/s", "d2h_bytes_per_step": len(blob) + 16, "steps": Kp,
                                               "payload_bytes_per_step": pub_bytes,
                                               "update_then_get_parameters": self.world * Kp / t_block,
                                               "overlapped_run_loop": self.world * Kp / t_over,
                                               "note": "per step: update + the pickled {'actor': state_dict} blob Learner.run() sets in Redis "
                                                       "(payload floats gathered into a device image of the pickle stream by a kernel -> one D2H "
                                                       "copy -> bytes); overlapped_run_loop times Learner.run(max_updates) as shipped"}
                lrn.memory.stop()
            finally:
                os.chdir(old)
        return res


def roofline_block(b, leg, workload, R, traffic=None, traffic_src=None):
    work = WORK[workload]
    step_s = leg["ms_per_step"] * 1e-3
    ach_gbs = R * work["mbytes"] * 1e6 / step_s / 1e9
    ach_tf = R * work["gflop"] * 1e9 / step_s / 1e12
    tl = leg.get("timeline") or []
    tot = sum(t for _, t in tl) or 1.0
    fam = {}
    for name, t in tl:
        f = name.split("{")[0].split("(")[0] if "tcgen05" not in name else "gemm_tc"
        f = "gemm_ffma" if f.startswith("gemm_") and f != "gemm_tc" else f
        fam[f] = fam.get(f, 0.0) + t
    top = max(fam.items(), key=lambda kv: kv[1]) if fam else ("n/a", 0.0)
    return {
        "bound": "hbm", "achieved": ach_gbs, "peak": b.pk["hbm"], "unit": "GB/s", "frac": ach_gbs / b.pk["hbm"],
        "traffic": traffic, "traffic_unit": "bytes of DRAM read+write per step", "traffic_source": traffic_src,
        "peak_source": b.pk["src"],
        "launch": f"one gradient step of {R} learner(s) = {leg['launches_per_step']} kernel launches inside a CUDA graph",
        "algorithmic_bytes_per_step": work["mbytes"] * 1e6 * R, "algorithmic_flop_per_step": work["gflop"] * 1e9 * R,
        "tensor": {"achieved": ach_tf, "peak": b.pk["tf"], "unit": "TFLOP/s", "frac": ach_tf / b.pk["tf"],
                   "note": "denominator = measured dense bf16 cuBLAS; the fp32-exact paths issue FFMA or 3 tensor-core MACs per algorithmic MAC"},
        "dominant_kernel": {"name": top[0], "share_of_step": top[1] / tot, "us_per_step_in_graph": top[1],
                            "launches_per_step": sum(1 for n, _ in tl if (n.split("{")[0].split("(")[0] == top[0]) or
                                                     (top[0] == "gemm_tc" and "tcgen05" in n) or
                                                     (top[0] == "gemm_ffma" and n.startswith("gemm_") and "tcgen05" not in n))},
        "per_launch_us_in_graph": [[n, round(t, 2)] for n, t in tl],
        "note": ("neither roof binds: the step runs out of L2 (`traffic` = measured DRAM bytes per step with the caches left alone vs "
                 "`algorithmic_bytes_per_step`) as %d dependent launches; what bounds it is the per-SM TMA request cadence inside the "
                 "chained / tcgen05 kernels (~675 cycles per bulk request, ~105 cycles per tf32 MMA) and the kernel boundaries "
                 "(DESIGN.md 4, profiles/README.md)") % leg["launches_per_step"],
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="LL", choices=["LL", "VS", "MS", "C10", "C10O"])
    ap.add_argument("--replicas", type=int, default=1, help="independent learners co-scheduled per GPU")
    ap.add_argument("--ring", type=int, default=DEVICE_RING, help="transitions in the device replay ring (per learner)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="timed update() calls for the e2e leg (default: max(steps, 1000) capped at 2000)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU time budget of the headline cpu_baseline sample")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--precision", type=int, default=-1,
                    help="0 = fp32 FFMA (layer-chained kernels for LL-class shapes), 1 = 3xTF32 tcgen05 GEMMs, -1 = probe both, headline = faster")
    ap.add_argument("--configs", default="auto", help="'auto' = short legs of VS, MS, C10 + config 4 placement + learners-per-GPU sweep; 'none' = headline only")
    ap.add_argument("--sweep", default="4,16,64", help="learners-per-GPU values of the sweep (headline workload, short legs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's losses, parameters and Adam state as DIR/<name>.npy "
                         "(pin --precision when comparing dumps: -1 picks the back-end by timing)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import __graft_entry__ as ge
    if ge.library_is_stale():
        raise SystemExit(f"{ge.LIB} is missing or older than its sources: build it with "
                         "`python -c 'import __graft_entry__ as g; g.build()'` (the benchmark compiles nothing)")
    from distributed_sac_b200 import _lib
    _lib.load()
    from distributed_sac_b200.replicas import shard_replicas

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the product path)")
    b = Bench(args)
    t_mark = [time.perf_counter()]

    def log(what):
        if b.rank == 0:
            now = time.perf_counter()
            print(f"[bench] {what}: {now - t_mark[0]:.1f} s", file=sys.stderr, flush=True)
            t_mark[0] = now
    W = max(args.warmup, 3)
    K = args.steps
    R = args.replicas
    wl = args.workload
    t_start = time.perf_counter()

    clocks = ClockSampler(b.local)
    clocks.start()

    # ---- headline: device-resident leg (value) -----------------------------------------------------------------
    by_precision = {"probe": {}, "final": {}}
    cands = [0, 1] if args.precision < 0 else [args.precision]
    if len(cands) > 1:            # short probe of both back-ends; the full timed run uses the faster one
        for pr in cands:
            leg = b.gpu_leg(wl, R, pr, 600, 16, 1 << 16)
            by_precision["probe"]["fp32" if pr == 0 else "tc3xtf32"] = leg["value"]
        args.precision = 0 if by_precision["probe"]["fp32"] >= by_precision["probe"]["tc3xtf32"] else 1
    log("back-end probe")
    head = b.gpu_leg(wl, R, args.precision, K, W, args.ring, detail=True, clocks=clocks, bcast=True,
                     dump=args.dump_outputs if b.rank == 0 else None)
    clk = clocks.stop()
    by_precision["final"]["fp32" if args.precision == 0 else "tc3xtf32"] = head["value"]
    row_bytes = 4 * ((2 * core_config(wl, 1).obs_dim + core_config(wl, 1).act_dim + 2 + 31) // 32 * 32)
    ring_mib = args.ring * row_bytes / 2 ** 20

    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if os.path.exists(tpath) and R == 1:
        with open(tpath) as f:
            tj = json.load(f).get(f"{wl}_p{args.precision}")
        if tj:
            traffic = tj["dram_read_bytes_per_step"] + tj["dram_write_bytes_per_step"]
            traffic_src = "profiles/r2_traffic.json: " + tj["source"]
    roofline = roofline_block(b, head, wl, R, traffic, traffic_src)

    log("headline device-resident leg")
    # ---- e2e leg ---------------------------------------------------------------------------------------------------
    Ke = args.e2e_steps or min(max(K, 1000), 2000)
    e2e = b.e2e_leg(wl, args.precision, Ke, W, with_publication=True)

    log("e2e leg")
    # ---- the other BASELINE configs, config 4's placement, learners-per-GPU sweep -------------------------------------
    configs, sweep = {}, {}
    if args.configs == "auto":
        for w2 in [w for w in ("VS", "MS", "C10") if w != wl]:
            leg = b.gpu_leg(w2, 1, 1, 400, 16, 1 << 17)
            e2 = b.e2e_leg(w2, 1, 200, 16)
            configs[w2] = {"workload": WORKLOAD_DESC[w2], "value": leg["value"], "unit": "steps/s", "ms_per_step": leg["ms_per_step"],
                           "n_gpus": world, "learners": leg["learners"], "e2e": {k: e2[k] for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step", "steps")},
                           "roofline": {"hbm_frac": leg["hbm_frac"], "tensor_frac": leg["tensor_frac"],
                                        "algorithmic_bytes_per_step": WORK[w2]["mbytes"] * 1e6, "algorithmic_flop_per_step": WORK[w2]["gflop"] * 1e9},
                           "gemm_backend": leg["gemm_backend"], "launches_per_step": leg["launches_per_step"], "timing": leg["timing"]["step_ms"]}
            log(f"config leg {w2}")
        # BASELINE config 4: 10 independent MTSAC learners over the GPUs of this run (8 GPUs: 2,2,1,1,1,1,1,1)
        place = shard_replicas(10, world)
        mine = len(place[b.rank])
        leg = b.gpu_leg("MS", max(mine, 1), 1, 300, 16, 1 << 16)
        configs["cfg4_10_learners"] = {"workload": "10 independent " + WORKLOAD_DESC["MS"] + " replicas, no gradient all-reduce",
                                       "placement_learners_per_gpu": [len(p) for p in place], "value": leg["value"], "unit": "steps/s (sum over the 10 learners)",
                                       "ms_per_step": leg["ms_per_step"], "n_gpus": world, "learners": leg["learners"],
                                       "roofline": {"hbm_frac_of_rank0": leg["hbm_frac"], "tensor_frac_of_rank0": leg["tensor_frac"]},
                                       "timing": leg["timing"]["step_ms"]}
        log("config 4 placement")
        for r_extra in [int(x) for x in args.sweep.split(",") if x]:
            sweep[str(r_extra)] = {}
            for pr in (0, 1):
                leg = b.gpu_leg(wl, r_extra, pr, 200, 16, max(1 << 14, (1 << 19) // r_extra), seed0=77)
                sweep[str(r_extra)]["fp32" if pr == 0 else "tc3xtf32"] = {"value": leg["value"], "hbm_frac": leg["hbm_frac"]}

    log("learners-per-GPU sweep")
    cpu = None
    if b.rank == 0 and world == 1 and not args.no_cpu:
        cpu = cpu_baseline_block(wl, args.cpu_seconds)
        log("cpu_baseline headline")
        if args.configs == "auto":
            for w2 in configs:
                if w2 in WORK:
                    configs[w2]["cpu_baseline"] = cpu_baseline_block(w2, 4.0)
                    log(f"cpu_baseline {w2}")

    if b.rank == 0:
        line = {
            "metric": "SAC gradient steps/sec", "value": head["value"], "unit": "steps/s", "n_gpus": world, "steps": K, "warmup": head["timing"]["warmup_steps"],
            "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": WORKLOAD_DESC[wl], "learners_per_gpu": R,
                       "replay": f"{args.ring}-transition device-resident ring per learner, {row_bytes} B rows = {ring_mib:.0f} MiB",
                       "host_replay": f"e2e, cpu_baseline and --impl reference: {HOST_RING}-transition host buffer",
                       "l2": "inputs larger than L2: minibatches are gathered from the %.0f MiB ring (> 126 MB L2); no explicit flush" % (ring_mib * R),
                       "parallelism": f"{world} x independent learner replicas, NCCL broadcast of initial weights only",
                       "precision": ("hidden-layer GEMMs 3xTF32 on tcgen05 (fp32-class, <=2e-6 of fp64), rest fp32 FFMA" if args.precision == 1
                                     else "exact fp32 (FFMA), layer-chained kernels") + ", fp64-evaluated transcendentals",
                       "gemm_backend": head["gemm_backend"]},
            "timing": head["timing"], "clocks": clk, "e2e": e2e,
            "gpu_launches": K * head["launches_per_step"],
            "roofline": roofline, "cpu_baseline": cpu, "by_precision": by_precision,
            "configs": configs, "replicas_per_gpu_sweep": sweep,
            "bench_wall_s": round(time.perf_counter() - t_start, 1),
        }
        print(json.dumps(line), flush=True)
    if b.dist is not None:
        b.dist.destroy_process_group()


if __name__ == "__main__":
    main()
