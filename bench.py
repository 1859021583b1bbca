#!/usr/bin/env python
"""bench.py — env-steps/s of the fused GEM step on B200 (BASELINE.json metric), with roofline + CPU baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config pmsm|pmsm_64k|fin_sc_pmsm|scim|eesm|mixed] [--envs-per-gpu E]
                    [--dump-outputs DIR]

Default workload (BASELINE.json metric / configs[1] at the size the metric is quoted on): Cont-CC-PMSM-v0, RK4 (one step per
tau = 1e-4), 2^20 envs per GPU, synthetic U(-1,1)^3 actions, Wiener references, in-kernel auto-reset; weak scaling: every rank steps its
own 2^20-env shard (keyed by global env index), no data-path collective (SURVEY.md §8e).  `--config` selects the other BASELINE
configs (configs[1] at N=65536, configs[2] Finite-SC-PMSM, configs[3] SCIM, configs[4] mixed PMSM+SynRM+EESM); the default run also times
them briefly and reports them under `other_configs`, so that the driver's 1/2/4/8-GPU records hold them too.

One "step" = one batched env.step over the rank's shard = one pass of the hot path (core.py:328-371).
 * value    : whole-job env-steps/s with the actions resident in HBM, through `env.rollout` (gemb200_rollout_record): the K timed steps are
              issued as fused launches of <= 32 steps each (rollout_kernel: the persistent records stay in registers across the steps of a
              launch), and EVERY step's obs / next reference / reward / terminated is written to HBM (record_every = 1) — the same
              outputs, bit for bit, as K env.step calls (tests/test_gpu_rollout.py).  One CUDA-event pair on the launching stream around
              all K steps; ms_per_step = event time / K, max over ranks.  Inputs larger than L2: a launch reads K x 12.6 MB of actions and
              writes K x 72.4 MB of outputs, nothing is re-read.
 * per_step_launch : the same K steps as K separate gemb200_step launches (step_kernel; the closed-loop shape, round 1's `value`),
              rotating over 4 replicas of the batch so that every launch finds its records in HBM, not in L2.
 * e2e      : same metric through the public host-buffer entry point (gemb200_step_host): pinned host actions -> H2D ->
              launch -> D2H of obs/ref/reward/terminated -> sync, every step.
 * roofline : for the dominant kernel of `value` (rollout_kernel): algorithmic bytes per env-step (SURVEY.md §8d bookkeeping: action in,
              obs/ref/reward/terminated out every step, record read + written once per launch) x envs / mean kernel time per step vs the
              measured HBM copy bandwidth in MEASURED_PEAKS.json.  `per_step_launch.roofline` is the same for step_kernel with the
              canonical 129 B/env-step.
 * cpu_baseline : the float64 C oracle (a port of the reference's algorithm, oracle/gem_oracle.c) on this box's host
              cores, bounded sample.  `--impl reference` runs only that arm.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "env-steps/sec at N=2^20 PMSM, 1/2/4/8 GPU; HBM GB/s vs roofline"
UNIT = "env-steps/s"
ROLL_MAX = 32  # steps per fused launch (bounds the size of the recorded trajectory: 32 x 72 MB at N = 2^20)
DUMP_ENVS = 1 << 16  # envs per array written by --dump-outputs: a fixed sample keeps the default 2^20-env workload at ~5 MB

# BASELINE.json configs; n_* feed the algorithmic-bytes bookkeeping of SURVEY.md §8(d)
CONFIGS = {
    "pmsm": dict(env_id="Cont-CC-PMSM-v0", n_act=3, n_ode=4, n_obs=14, n_ref=2, envs=1 << 20,
                 what="ContB6 + IdealSupply + ConstantSpeedLoad(100 rad/s), Wiener refs (i_sd,i_sq) + WSE reward + SquaredConstraint fused"),
    "pmsm_64k": dict(env_id="Cont-CC-PMSM-v0", n_act=3, n_ode=4, n_obs=14, n_ref=2, envs=1 << 16, what="BASELINE configs[1]: N=65536"),
    "fin_sc_pmsm": dict(env_id="Finite-SC-PMSM-v0", n_act=1, n_ode=4, n_obs=14, n_ref=1, envs=1 << 20, n_finite=8,
                        what="BASELINE configs[2]: FiniteB6 (8 switching states) + PolynomialStaticLoad, tau=1e-5, Wiener omega reference"),
    "fin_sc_pmsm_il": dict(env_id="Finite-SC-PMSM-v0", n_act=1, n_ode=4, n_obs=14, n_ref=1, envs=1 << 20, n_finite=8, interlock=1e-6,
                           what="configs[2] variant: interlocking time 1 us (two switching segments per step, general kernel instantiation)"),
    "scim": dict(env_id="Cont-CC-SCIM-v0", n_act=3, n_ode=6, n_obs=14, n_ref=2, envs=1 << 20, what="BASELINE configs[3]: 5-state induction motor"),
    "eesm": dict(env_id="Cont-CC-EESM-v0", n_act=4, n_ode=5, n_obs=16, n_ref=3, envs=1 << 20, what="B6 + 4QC excitation converter"),
    "synrm": dict(env_id="Cont-CC-SynRM-v0", n_act=3, n_ode=4, n_obs=14, n_ref=2, envs=1 << 20, what="reluctance motor"),
    "mixed": dict(types=("pmsm", "synrm", "eesm"), envs=(1 << 20) // 3 * 3,
                  what="BASELINE configs[4]: env g of type g mod 3 in {PMSM, SynRM, EESM}, physically segmented per type, one fused launch per type "
                       "on its own stream"),
}
for _c in CONFIGS.values():
    if "types" not in _c:
        _c["record_bytes"] = 8 * _c["n_ode"] + 8 * _c["n_ref"]


def b_alg(c):
    """canonical algorithmic bytes per env-step of ONE single-step launch (SURVEY.md §8d)"""
    if "types" in c:
        return sum(b_alg(CONFIGS[t]) for t in c["types"]) / len(c["types"])
    return 4 * c["n_act"] + 8 * c["n_ode"] + 4 * c["n_obs"] + 4 * c["n_ref"] + 8 * c["n_ref"] + 5


def b_alg_rollout(c, k, every=1):
    """same bookkeeping for a fused launch of k steps: action in every step, outputs every `every` steps, record once per launch"""
    if "types" in c:
        return sum(b_alg_rollout(CONFIGS[t], k, every) for t in c["types"]) / len(c["types"])
    return 4 * c["n_act"] + (4 * c["n_obs"] + 4 * c["n_ref"] + 5) / every + (8 * c["n_ode"] + 8 * c["n_ref"]) / k


def make_env(cfg_name, n_envs, device=0, rank=0):
    import gym_electric_motor_b200 as gem

    c = CONFIGS[cfg_name]
    if "types" in c:
        from gym_electric_motor_b200.mixed import MixedEnvBatch

        return MixedEnvBatch([CONFIGS[t]["env_id"] for t in c["types"]], n_envs, device=device, dtype="float32", ode_solver=gem.physical_systems.RK4Solver(),
                             autoreset="same_step", seed=0, env_index_offset=rank * n_envs)
    extra = dict(converter=dict(interlocking_time=c["interlock"])) if "interlock" in c else {}
    return gem.make(c["env_id"], num_envs=n_envs, device=device, dtype="float32", ode_solver=gem.physical_systems.RK4Solver(),
                    autoreset="same_step", seed=0, env_index_offset=rank * n_envs, **extra)


def workload_config(cfg_name, n_envs, n_gpus):
    c = CONFIGS[cfg_name]
    ids = c["env_id"] if "types" not in c else "+".join(CONFIGS[t]["env_id"] for t in c["types"])
    tau = 1e-5 if cfg_name.startswith("fin_sc_pmsm") else 1e-4
    return {"workload": f"{ids} x {n_envs} envs/GPU, RK4 x1 per tau={tau:g}, {c['what']}, same-step auto-reset",
            "name": cfg_name, "env_id": ids, "envs_per_gpu": n_envs, "global_envs": n_envs * n_gpus, "solver": "rk4x1", "tau": tau,
            "parallelism": f"env-shard x{n_gpus} (no collective)",
            "l2": "inputs larger than L2: fused launches stream K x (actions + outputs) through HBM once, nothing is re-read; the per-step-launch arm "
                  "rotates over 4 replicas of the env batch",
            "layout": "obs [K,N,n_obs] row-per-env (AoS), persistent state SoA of 16-byte chunks"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(key):
    """dram bytes per launch from the committed ncu captures (profiles/ncu_traffic.json), or None."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(key)
        except Exception:
            return None
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        """Start early (nvidia-smi needs ~100 ms before its first row); rows are stamped on arrival, mark()/stop() bracket the timed region."""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(self.gpu)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def wait_first(self, timeout=5.0):
        t0 = time.perf_counter()
        while self.proc is not None and not self.rows and time.perf_counter() - t0 < timeout:
            time.sleep(0.01)

    def mark(self):
        self.t_begin = time.perf_counter()

    def mark_end(self):
        self.t_end = time.perf_counter()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t_end = getattr(self, "t_end", time.perf_counter())
        time.sleep(0.03)  # let the last row of the region arrive
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        t_begin = getattr(self, "t_begin", 0.0)
        inside = [r for (t, r) in self.rows if t_begin <= t <= t_end + 0.03]
        window = "timed regions (all arms)"
        if not inside:  # region shorter than the sampling period: take the rows closest to it
            inside = [r for (t, r) in self.rows if t_begin - 0.25 <= t <= t_end + 0.25]
            window = "timed regions +-250 ms"
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in inside:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm), "window": window}


# ----------------------------------------------------------------------------------------------------------------------
# CPU arm (the oracle = C port of the reference's algorithm; bench.py's only use of oracle/)
# ----------------------------------------------------------------------------------------------------------------------
def cpu_arm(cfg_name, n_envs, steps, warmup, min_seconds=2.0, max_seconds=None):
    """Oracle on all host cores: `steps` timed steps over `n_envs` envs, the block repeated until >= min_seconds have been timed (or, with
    max_seconds, as many 16-step blocks as fit).  Returns (env-steps/s, cores, sample description)."""
    import numpy as np

    from oracle.gem_oracle import Oracle
    from gym_electric_motor_b200 import _cabi as K

    c = CONFIGS[cfg_name]
    if "types" in c:
        c, cfg_name = CONFIGS["pmsm"], "pmsm"
    cores = os.cpu_count() or 1
    env = make_env(cfg_name, n_envs)  # host-side spec only; no device handle is created until the env is used
    cfg = env.build_config()
    cfg.dtype = K.F64
    ora = Oracle(cfg, nthreads=cores)
    ora.reset()
    rng = np.random.default_rng(0)
    if "n_finite" in c:
        acts = rng.integers(0, c["n_finite"], size=(4, n_envs, c["n_act"])).astype(np.int32)
    else:
        acts = rng.uniform(-1, 1, size=(4, n_envs, c["n_act"]))
    chunk = 16  # steps per rollout call: the oracle's worker threads persist over a call (two barriers per step, no thread creation)
    ora.rollout(acts, max(1, warmup))
    t0 = time.perf_counter()
    done, blocks = 0, 0
    while True:
        todo = steps if max_seconds is None else chunk
        k = 0
        while k < todo:
            cnt = min(chunk, todo - k)
            ora.rollout(acts, cnt)
            k += cnt
        done += todo
        blocks += 1
        el = time.perf_counter() - t0
        if max_seconds is not None:
            if el >= max_seconds:
                break
        elif el >= min_seconds:
            break
    el = time.perf_counter() - t0
    how = f"{blocks} x {steps} steps" if max_seconds is None else f"{done} steps"
    return n_envs * done / el, cores, f"{c['env_id']}, {n_envs} envs x {how}, RK4 x1, float64 C oracle (gem_oracle_rollout), {cores} threads, {el:.1f} s timed"


def run_reference(args, rank):
    """--impl reference: the reference's CPU algorithm for the same path on the host cores (oracle port; the Python
    reference itself cannot travel to this box and runs ~1e4 steps/s/core, BASELINE.md §2).  Steps the SAME number of envs per step as the
    GPU arm's config says (envs_per_gpu); K timed steps, repeated as a block until >= 2 s have been timed."""
    if rank != 0:
        return
    n = args.envs_per_gpu or CONFIGS[args.config]["envs"]
    v, cores, sample = cpu_arm(args.config, n, max(args.steps, 1), max(args.warmup, 1), min_seconds=2.0)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * n / v, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args.config, n, args.gpus),
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------------------
# GPU arms
# ----------------------------------------------------------------------------------------------------------------------
class Workload:
    """One config on this rank: env (or mixed batch), action pools, recorded-output buffers; `rollout(k)` issues k fused steps."""

    def __init__(self, cfg_name, n, device, rank, torch):
        self.torch, self.name, self.c, self.n = torch, cfg_name, CONFIGS[cfg_name], n
        self.env = make_env(cfg_name, n, device=device, rank=rank)
        self.mixed = "types" in self.c
        self.sims = [e.sim for e in self.env.envs] if self.mixed else [self.env.sim]
        self.dev = self.sims[0].device
        self.env.reset()
        gen = torch.Generator(device=self.dev).manual_seed(1234 + rank)
        self.acts, self.outs = [], []
        for s in self.sims:
            if s.finite:
                a = torch.randint(0, 8, (ROLL_MAX, s.n, s.n_act), generator=gen, device=self.dev, dtype=torch.int32)
            else:
                a = torch.rand((ROLL_MAX, s.n, s.n_act), generator=gen, device=self.dev, dtype=torch.float32) * 2 - 1
            self.acts.append(a)
            self.outs.append((torch.empty((ROLL_MAX, s.n, s.n_state), device=self.dev), torch.empty((ROLL_MAX, s.n, max(s.n_ref, 1)), device=self.dev),
                              torch.empty((ROLL_MAX, s.n), device=self.dev), torch.empty((ROLL_MAX, s.n), dtype=torch.uint8, device=self.dev)))
        if self.mixed:
            self.env._ensure_streams()

    def launches(self):
        return sum(s.launch_count for s in self.sims)

    def rollout(self, k, every=1):
        """k fused steps (k <= ROLL_MAX) on the current stream (mixed: one launch per type on its own stream, joined by events)"""
        torch = self.torch
        if not self.mixed:
            self.sims[0].rollout_into(self.acts[0], k, every, *self.outs[0])
            return
        cur = torch.cuda.current_stream(self.dev)
        self.env._start.record(cur)
        for s, a, o, st, ev in zip(self.sims, self.acts, self.outs, self.env._streams, self.env._events):
            st.wait_event(self.env._start)
            with torch.cuda.stream(st):
                s.rollout_into(a, k, every, *o)
            ev.record(st)
        for ev in self.env._events:
            cur.wait_event(ev)

    def steps(self, total, every=1):
        done = 0
        while done < total:
            k = min(ROLL_MAX, total - done)
            self.rollout(k, every)
            done += k

    def close(self):
        self.env.close()


def dump_outputs(wl, K, out_dir):
    """Write what the timed path returned for its last step — obs, reference, reward and terminated of the last of the K fused steps — as
    <out_dir>/<name>.npy in float32 (mixed batch: <type>_<name>.npy), for a fixed sample of DUMP_ENVS envs drawn with seed 0 (sorted env
    indices), so that two builds run with the same arguments can be compared output for output."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    last = (K - 1) % ROLL_MAX  # slot of the last step in the last fused launch (Workload.steps issues launches of ROLL_MAX steps first)
    for i, (s, outs) in enumerate(zip(wl.sims, wl.outs)):
        idx = np.sort(np.random.default_rng(0).choice(s.n, size=min(s.n, DUMP_ENVS), replace=False))
        sel = wl.torch.as_tensor(idx, device=wl.dev)
        prefix = f"{wl.c['types'][i]}_" if wl.mixed else ""
        for name, t in zip(("obs", "reference", "reward", "terminated"), outs):
            if name == "reference" and not s.n_ref:
                continue
            np.save(os.path.join(out_dir, f"{prefix}{name}.npy"), t[last].index_select(0, sel).float().cpu().numpy())


def gate(torch):
    """Keep the GPU busy for ~0.15 ms right before a timed region starts: the start event is recorded BEHIND this spin kernel, so the host
    has queued the timed launches by the time the event fires and the event-to-event time is device time of the K steps only — no host
    launch latency inside (at 0.4 ms per 20-step launch a 15 us submission gap would be 4 %; it also differs per rank under torchrun)."""
    torch.cuda._sleep(300000)


def time_rollout(wl, K, W, barrier, torch):
    wl.rollout(ROLL_MAX)  # untimed: every slice of the output buffers has been written once before the timed region
    wl.steps(max(W, 3))
    barrier()
    l0 = wl.launches()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    gate(torch)
    ev0.record()
    wl.steps(K)
    ev1.record()
    barrier()
    return ev0.elapsed_time(ev1), wl.launches() - l0, (time.perf_counter() - t0) * 1e3


def time_closed_loop(torch, device, barrier, n=1 << 16, k=32, reps=24):
    """BASELINE configs[1] (N = 65 536) in CLOSED loop — action = controller(state, reference) between the steps, the reference's control
    loop (core.py:328-371 per step).  eager: policy kernels + ONE gemb200_step launch per step, issued from Python; graph: the same k steps
    captured once in a CUDA graph (env.capture_steps: device-resident clock of the C-ABI) and replayed.  Two policies: `hold` (a constant
    action tensor: what is left is the env step itself — step_kernel + the one-thread clock tick per step) and `linear` (state feedback
    a = clamp(state Ws + ref Wr): two small GEMMs + clamp = 3 kernels per step).  Device time per step (CUDA events around reps x k steps
    with the queue kept full) and wall time per step."""
    out = {"envs": n, "steps_per_graph": k}
    for pname in ("hold", "linear"):
        env = make_env("pmsm_64k", n, device=device, rank=77)
        (st, rf), _ = env.reset()
        dev = st.device
        idx = [env.physical_system.state_names.index(nm) for nm in env.reference_names]
        ws = torch.zeros((st.shape[1], 3), device=dev)
        wr = torch.zeros((rf.shape[1], 3), device=dev)
        for j, col in enumerate(idx):  # P controller on the referenced currents, spread over the three phases
            for ph, g in enumerate((1.0, -0.5, -0.5) if j == 0 else (0.0, 0.866, -0.866)):
                ws[col, ph] -= 3.0 * g
                wr[j, ph] += 3.0 * g
        hold = torch.rand((n, 3), device=dev) * 0.4 - 0.2

        def policy(state, ref):
            if pname == "hold":
                return hold
            return torch.addmm(state @ ws, ref, wr).clamp_(-1.0, 1.0)

        for _ in range(k):
            (st, rf), _, _, _, _ = env.step(policy(st, rf))
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(reps * k):
            (st, rf), _, _, _, _ = env.step(policy(st, rf))
        e1.record()
        barrier()
        r = {"eager_us_per_step": 1e3 * e0.elapsed_time(e1) / (reps * k), "eager_wall_us_per_step": 1e6 * (time.perf_counter() - t0) / (reps * k)}
        cap = env.capture_steps(policy, k)
        l0 = env.sim.launch_count
        for _ in range(3):
            cap.replay()
        barrier()
        t0 = time.perf_counter()
        e0.record()
        for _ in range(reps):
            cap.replay()
        e1.record()
        barrier()
        r["graph_us_per_step"] = 1e3 * e0.elapsed_time(e1) / (reps * k)
        r["graph_wall_us_per_step"] = 1e6 * (time.perf_counter() - t0) / (reps * k)
        r["graph_env_steps_per_s"] = n / (r["graph_us_per_step"] * 1e-6)
        r["eager_env_steps_per_s"] = n / (r["eager_us_per_step"] * 1e-6)
        r["library_calls_during_replays"] = env.sim.launch_count - l0
        out[pname] = r
        cap.release()
        env.close()
    out["note"] = ("kernel nodes per captured step: policy kernels (hold: 0, linear: 3) + step_kernel + the one-thread clock tick; the open-loop "
                   "equivalent (pre-computed actions, one fused launch) is other_configs.pmsm_64k")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--config", default="pmsm", choices=sorted(CONFIGS))
    ap.add_argument("--envs-per-gpu", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the brief timings of the other BASELINE configs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last step's outputs (a fixed sample of envs) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    from gym_electric_motor_b200 import hostmem

    torch.cuda.set_device(local_rank)  # first: nothing may create a context on device 0 from the other ranks
    dev = torch.device("cuda", local_rank)
    hostmem.bind_to_device_numa_node(local_rank)  # pinned buffers of the e2e arm must sit on the GPU's NUMA node (first touch follows the thread)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    cfg_name = args.config
    c = CONFIGS[cfg_name]
    n = args.envs_per_gpu or c["envs"]
    K, W = args.steps, args.warmup

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- primary arm: K steps as fused launches, every step's outputs recorded ----------------
    wl = Workload(cfg_name, n, local_rank, rank, torch)
    if rank == 0:
        sampler.wait_first()
        sampler.mark()
    ms, launches, t_wall = time_rollout(wl, K, W, barrier, torch)
    if args.dump_outputs and rank == 0:
        dump_outputs(wl, K, args.dump_outputs)
    # the same K steps with only the LAST step's outputs written (what an open-loop consumer of the final state pays)
    wl.steps(3, every=0)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    gate(torch)
    e0.record()
    wl.steps(K, every=0)
    e1.record()
    barrier()
    ms_last = e0.elapsed_time(e1)

    # ---------------- per-step launches (closed-loop shape): K x gemb200_step rotating over R replicas ----------------
    ms_step, step_launches = None, 0
    if not wl.mixed:
        R = 4 if n >= (1 << 18) else 16
        envs = [wl.env] + [make_env(cfg_name, n, device=local_rank, rank=rank * R + r + 1000) for r in range(1, R)]
        for e in envs[1:]:
            e.reset()
        pool = [wl.acts[0][j] for j in range(8)]
        for k in range(max(W, R)):
            envs[k % R].step(pool[k % 8])
        barrier()
        l0 = sum(e.sim.launch_count for e in envs)
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        gate(torch)
        s0.record()
        for k in range(K):
            envs[k % R].step(pool[k % 8])
        s1.record()
        barrier()
        ms_step = s0.elapsed_time(s1)
        step_launches = sum(e.sim.launch_count for e in envs) - l0
        for e in envs[1:]:
            e.close()

    # ---------------- N > 1 only: the sharded layout's ONE collective — a single NCCL all-gather of the packed (obs, ref, reward,
    # terminated) buffer after every step, double-buffered so that gather(k) overlaps step(k+1) ----------------
    ms_gather, gather_bytes, ms_peer, peer_error = None, 0, None, None
    if world > 1 and not wl.mixed:
        from gym_electric_motor_b200.distributed import OverlappedGather

        sim = wl.sims[0]
        og = OverlappedGather(sim, torch.float32)
        gather_bytes = og.nbytes
        pool = [wl.acts[0][j] for j in range(8)]
        for k in range(3):
            og.step(pool[k % 8])
        og.finish()
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        gate(torch)
        g0.record()
        for k in range(K):
            og.step(pool[k % 8])
        og.finish()
        g1.record()
        barrier()
        ms_gather = g0.elapsed_time(g1)
        og.release()
        # the same aggregated return FUSED into the step: the kernel stores its outputs into every rank's gather buffer over NVLink
        # (distributed.PeerGather, gemb200_bind_peers) — no collective call, a flag per (buffer, source) instead
        try:
            from gym_electric_motor_b200.distributed import PeerGather

            pg = PeerGather(sim, torch.float32)
            for k in range(3):
                pg.step(pool[k % 8])
            pg.finish()
            barrier()
            p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            gate(torch)
            p0.record()
            for k in range(K):
                pg.step(pool[k % 8])
            pg.finish()
            p1.record()
            barrier()
            ms_peer = p0.elapsed_time(p1)
            pg.check()
            pg.release()
        except Exception as exc:  # e.g. CUDA IPC not permitted in this container: keep the NCCL figure, say why
            ms_peer, peer_error = None, f"{type(exc).__name__}: {exc}"[:300]

    # ---------------- e2e arm: host buffers through the C-ABI ----------------
    ms_e2e, ke, h2d, d2h = None, 0, 0, 0
    if not wl.mixed:
        sim = wl.sims[0]
        adt = torch.int32 if sim.finite else torch.float32
        h_act = []
        for _ in range(2):
            t = hostmem.pinned_empty((n, sim.n_act), adt, local_rank)
            t.copy_(wl.acts[0][len(h_act)].cpu())
            h_act.append(t)
        h_obs = hostmem.pinned_empty((n, sim.n_state), torch.float32, local_rank)
        h_ref = hostmem.pinned_empty((n, max(sim.n_ref, 1)), torch.float32, local_rank)
        h_rew = hostmem.pinned_empty((n,), torch.float32, local_rank)
        h_term = hostmem.pinned_empty((n,), torch.uint8, local_rank)
        ke = max(1, min(K, 50))
        for k in range(3):
            sim.step_host_ptr(h_act[k % 2].data_ptr(), h_obs.data_ptr(), h_ref.data_ptr(), h_rew.data_ptr(), h_term.data_ptr())
        barrier()
        t0 = time.perf_counter()
        for k in range(ke):
            sim.step_host_ptr(h_act[k % 2].data_ptr(), h_obs.data_ptr(), h_ref.data_ptr(), h_rew.data_ptr(), h_term.data_ptr())
        barrier()
        ms_e2e = (time.perf_counter() - t0) * 1e3
        h2d, d2h = n * sim.n_act * 4, n * (sim.n_state + sim.n_ref + 1) * 4 + n
    if rank == 0:
        sampler.mark_end()

    # ---------------- the other BASELINE configs, briefly (fused launches, every step recorded) ----------------
    others = {}
    wl.close()
    del wl
    torch.cuda.empty_cache()
    if not args.no_extra and cfg_name == "pmsm" and not args.envs_per_gpu:
        for name in ("pmsm_64k", "fin_sc_pmsm", "scim", "mixed"):
            oc = CONFIGS[name]
            w2 = Workload(name, oc["envs"], local_rank, rank, torch)
            k2 = max(K, 64) if name == "pmsm_64k" else min(max(K, 16), 64)
            m2, l2, _ = time_rollout(w2, k2, 3, barrier, torch)
            others[name] = (m2, k2, l2, oc["envs"])
            w2.close()
            del w2
            torch.cuda.empty_cache()
    closed = None
    if not args.no_extra and cfg_name == "pmsm" and not args.envs_per_gpu and world == 1:
        try:
            closed = time_closed_loop(torch, local_rank, barrier)
        except Exception as exc:  # a secondary arm must not take the bench line down with it
            closed = {"error": f"{type(exc).__name__}: {exc}"[:300]}
            torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None

    vals = [ms, ms_last, ms_step or 0.0, ms_gather or 0.0, ms_e2e or 0.0, ms_peer or 0.0] + [others[k][0] for k in sorted(others)]
    t = torch.tensor(vals, dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    vals = [float(x) for x in t.tolist()]
    ms, ms_last, ms_step, ms_gather, ms_e2e, ms_peer = vals[:6]
    for i, k in enumerate(sorted(others)):
        others[k] = (vals[6 + i],) + others[k][1:]
    if rank == 0:
        total_envs = n * world
        ms_per_step = ms / K
        value = total_envs / (ms_per_step * 1e-3)
        peak, peak_src = peaks()
        k_eff = min(K, ROLL_MAX)
        ba = b_alg_rollout(c, k_eff, 1)
        achieved = ba * n / (ms_per_step * 1e-3) / 1e9  # per GPU: this kernel's algorithmic GB/s
        traffic = ncu_traffic(f"rollout_kernel_{cfg_name}_f32_aos_bytes_per_step")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(cfg_name, n, world),
            "api": f"env.rollout / gemb200_rollout_record: {launches} fused launches of <= {ROLL_MAX} steps, outputs of every step recorded",
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "traffic_note": "DRAM bytes per env-batch step from profiles/ncu_traffic.json (ncu range replay over whole launches), or null",
                         "peak_source": peak_src, "alg_bytes_per_env_step": ba,
                         "alg_bytes_note": f"4*n_act + 4*n_obs + 4*n_ref + 5 per step + (8*n_ode + 8*n_ref)/{k_eff} (record read+written once per fused launch)",
                         "kernel": "rollout_kernel" + ("<SYNC,cont,f32,NREF=2,AoS,PLAIN>" if cfg_name.startswith("pmsm") else ""), "kernel_ms_per_step": ms_per_step},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "rollout_last_only": {"value": total_envs * K / (ms_last * 1e-3), "ms_per_step": ms_last / K,
                                  "note": "same fused launches writing only the last step's outputs (record_every = 0)"},
            "wall_ms_timed_region": t_wall,
        }
        if ms_step:
            a1 = b_alg(c) * n / (ms_step / K * 1e-3) / 1e9
            line["per_step_launch"] = {"value": total_envs * K / (ms_step * 1e-3), "ms_per_step": ms_step / K, "gpu_launches": int(step_launches),
                                       "roofline": {"bound": "hbm", "achieved": a1, "peak": peak, "unit": "GB/s", "frac": a1 / peak, "alg_bytes_per_env_step": b_alg(c),
                                                    "traffic": ncu_traffic(f"step_kernel_{cfg_name}_f32_aos_bytes_per_launch"), "kernel": "step_kernel"},
                                       "note": "K separate gemb200_step launches (one env.step per launch, closed-loop shape), rotating over replicas of the batch"}
        if closed:
            line["closed_loop_64k"] = closed
        if ms_e2e:
            line["e2e"] = {"value": total_envs * ke / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": ke,
                           "ms_per_step": ms_e2e / ke, "api": "gemb200_step_host via VectorSim.step_host_ptr (NUMA-local pinned host buffers)",
                           "host_placement": hostmem.placement.get(local_rank), "pcie_link": hostmem.pcie_link(local_rank),
                           "d2h_GBps": d2h * ke / (ms_e2e * 1e-3) / 1e9}
        if world > 1 and ms_gather:
            best = min(ms_gather, ms_peer) if ms_peer else ms_gather
            line["with_all_gather"] = {"value": total_envs * K / (best * 1e-3), "unit": UNIT, "ms_per_step": best / K,
                                       "bytes_per_rank_per_step": gather_bytes, "ingress_GBps_per_gpu": (world - 1) * gather_bytes / (best / K * 1e-3) / 1e9,
                                       "how": "peer_store" if (ms_peer and ms_peer <= ms_gather) else "nccl_overlapped",
                                       "nccl_overlapped": {"value": total_envs * K / (ms_gather * 1e-3), "ms_per_step": ms_gather / K,
                                                           "note": "every step followed by ONE NCCL all_gather_into_tensor of the packed (obs, ref, reward, "
                                                                   "terminated) buffer the kernel writes into, double-buffered on a side stream: gather(k) "
                                                                   "overlaps step(k+1)"},
                                       "peer_store": ({"value": total_envs * K / (ms_peer * 1e-3), "ms_per_step": ms_peer / K,
                                                       "note": "fused step + gather: the step kernel stores obs / ref / reward / terminated into every rank's "
                                                               "gather buffer over NVLink (gemb200_bind_peers), flags instead of a collective call"}
                                                      if ms_peer else {"unavailable": peer_error}),
                                       "note": "`value` above is the sharded layout without the aggregated return (rank-local consumers)"}
        if others:
            line["other_configs"] = {}
            for name, (m2, k2, l2, n2) in others.items():
                oc = CONFIGS[name]
                ba2 = b_alg_rollout(oc, min(k2, ROLL_MAX), 1)
                ach2 = ba2 * n2 / (m2 / k2 * 1e-3) / 1e9
                line["other_configs"][name] = {"value": n2 * world * k2 / (m2 * 1e-3), "unit": UNIT, "envs_per_gpu": n2, "steps": k2, "ms_per_step": m2 / k2,
                                               "gpu_launches": int(l2), "alg_bytes_per_env_step": ba2, "roofline_frac": ach2 / peak, "what": oc["what"]}
        if world == 1 and not args.no_cpu_baseline:
            v, cores, sample = cpu_arm(cfg_name, 1 << 16, 16, 2, max_seconds=12.0)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                                    "note": "python reference itself: ~8.6e3 env.step/s/core (BASELINE.md §2, survey container)"}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
