#!/usr/bin/env python
"""Benchmark of the hot path named by BASELINE.json: differentiable env-steps/s (forward + adjoint).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|reference-cuda] [--env AntEnv] [--num-envs 4096]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one short-horizon rollout of the workload: ``horizon`` env-steps forward for ``num_envs`` environments
per GPU, then the adjoint of all of them.  Every timed loop (kernel path, end-to-end graphed and eager, each config) runs
K steps.  ``--dump-outputs DIR`` writes what the last timed step of the headline workload computed, as float32
``DIR/<name>.npy``: ``kernel_*`` (final q / qd, gradients w.r.t. the initial state and every step's joint_act) and
``e2e_loss`` / ``e2e_grad_actions`` (what the graphed rollout hands back); inputs are seeded, so two builds can be
compared output for output.  Headline workload = BASELINE.json configs[1]: AntEnv, 4096 envs, SHAC
horizon 32 (SURVEY.md section 8d).  Prints ONE JSON line (rank 0):

* ``e2e``      THE HEADLINE: env-steps/s through the reference-facing API -- ``envs.<Env>.step`` (action map, ``dflex.sim.
               SemiImplicitIntegrator.forward``, observation, reward, masked reset) + ``sum(rew).backward()`` -- with every
               rollout's actions copied from pinned HOST memory inside the timed region and the loss + action gradients
               read back (one CUDA graph per rollout; the eager loop is reported beside it).
* ``value``    the KERNEL PATH only (not section 8d's env-step): 2 x horizon launches of the simulation kernels through the
               C ABI on resident inputs (pre-scaled joint_act, random cotangents), CUDA events, max over ranks.  It explains
               ``e2e``; it is not the claim.
* ``roofline`` dominant kernel (the adjoint launch): ``frac`` = SURVEY.md section 8d's algorithmic bytes (state-only tape:
               2 200 B per Ant env-step adjoint) x environments / measured launch time / measured HBM peak.  ``design_frac`` =
               the same with the bytes this design really moves (tape rows incl. the forward intermediates + H^-1 blocks);
               ``fp32`` = executed fp32 FLOP against the CUDA-core peak: the path is issue / latency bound, not HBM bound.
* ``configs``  the other named configs of BASELINE.json, each with value / e2e / kernel_ms / section-8d roofline:
               ``humanoid8192`` (C2, fp32 tape) and ``humanoid8192_bf16_tape`` (C2 as named: "bf16 states" -- the tape stores the
               link velocities, bias accelerations and wrenches of every row as bf16; arithmetic and the state stay fp32),
               ``snu4096_bptt128`` (C3), ``cartpole64`` (C0's shape on the GPU); under torchrun also
               ``c4``: Ant at 8192 envs per GPU with the policy-gradient all-reduce (C4).
* ``cpu_baseline`` / ``gpu_baseline``  the UNMODIFIED reference through its own public API (``oracle/ref_gpu_arm.py`` on the
               install under ``baseline/_ref``): its CPU path on one host core, and its CUDA codegen path (rebuilt for
               sm_100, one flag edit) on this GPU at the headline config -- the only pre-existing GPU implementation.
* ``--impl reference`` times the reference CPU path on all host cores (one single-threaded process per core, wall-clocked);
  ``--impl reference-cuda`` the reference CUDA path; both print the same line shape with ``"impl": "reference"``.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries exactly ONE JSON line: keep NCCL's version banner (NCCL_DEBUG unset / VERSION prints it when the first
# communicator comes up) off it.  Set before torch / NCCL are loaded: the library latches its debug level on first use.
if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"
# ... and whatever NCCL does log (recent versions print the banner at WARN as well) goes to a file, not to stdout
os.environ.setdefault("NCCL_DEBUG_FILE", "/tmp/dfx_bench_nccl.%h.%p.log")

MM_FREQ = {"AntEnv": 16, "HumanoidEnv": 48, "SNUHumanoidEnv": 8, "CartPoleSwingUpEnv": 4, "HopperEnv": 16, "CheetahEnv": 16}
SUBSTEPS = {"AntEnv": 16, "HumanoidEnv": 48, "SNUHumanoidEnv": 48, "CartPoleSwingUpEnv": 4, "HopperEnv": 16, "CheetahEnv": 16}
HORIZON = {"SNUHumanoidEnv": 128}
# reference CPU sample per process and step: (num_envs, env-steps), ~1-3 s of single-core work through the stock API
CPU_SAMPLE = {"AntEnv": (64, 8), "HumanoidEnv": (16, 2), "SNUHumanoidEnv": (8, 2), "CartPoleSwingUpEnv": (64, 32),
              "HopperEnv": (64, 8), "CheetahEnv": (64, 8)}
METRIC = "differentiable env-steps/s (fwd+bwd)"


def algorithmic_bytes(Q, D, A, substeps, row=None, nseg=1):
    """Bytes one env-step MUST move per environment, fp32.  With row=None: SURVEY.md section 8d's figure for a
    state-only tape (row = Q + D) -- the yardstick of ``roofline.frac``.  With the kernels' actual tape row (q, qd + the
    forward intermediates the adjoint reads back instead of recomputing, DESIGN.md section 2) and the D*D H^-1 block per
    mass-matrix update: the design's own traffic (``roofline.design_frac``).  Returns (forward, backward)."""
    row = (Q + D) if row is None else row
    hinv = 0 if row == Q + D else nseg * D * D
    fwd = 4 * (Q + D + A) + 4 * (Q + D) + 4 * (substeps * row + hinv)
    bwd = 4 * (substeps * row + hinv) + 4 * (Q + D) + 4 * A + 4 * (Q + D + A)
    return fwd, bwd


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for k, name in enumerate(names):
                if len(r) > 3 + k and r[3 + k].lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ reference arms
def _ref_arm_cmd(env, num_envs, horizon, rollouts, warmup, device):
    return [sys.executable, os.path.join(ROOT, "oracle", "ref_gpu_arm.py"), "--env", env, "--num-envs", str(num_envs),
            "--horizon", str(horizon), "--rollouts", str(rollouts), "--warmup", str(warmup), "--device", device]


def _run_ref_arm(cmd, timeout):
    """Run oracle/ref_gpu_arm.py (the reference through its stock API, own interpreter); returns its JSON or {"unavailable": ...}."""
    try:
        proc = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout)
    except subprocess.TimeoutExpired:
        return {"unavailable": "reference arm timed out after %d s" % timeout}
    lines = [l for l in proc.stdout.splitlines() if l.startswith("{")]
    if proc.returncode != 0 or not lines:
        return {"unavailable": "reference arm failed: " + (proc.stderr.strip().splitlines() or ["?"])[-1][:300]}
    return json.loads(lines[-1])


def cpu_reference_baseline(env_name):
    """The reference's CPU path through its stock API on ONE host core (it is a serial loop), bounded sample."""
    n, steps = CPU_SAMPLE[env_name]
    steps = steps * 6          # ~10-20 s of single-core work over the two timed rollouts
    r = _run_ref_arm(_ref_arm_cmd(env_name, n, steps, 2, 1, "cpu"), 900)
    if "unavailable" in r:
        return {"value": None, "unit": "env-steps/s", "cores": 0, "kind": "reference", "sample": r["unavailable"]}
    return {"value": r["env_steps_per_s"], "unit": "env-steps/s", "cores": 1, "kind": "reference",
            "sample": "%s: 2 rollouts of %d envs x %d env-steps (forward + sum(rew).backward()) through the UNMODIFIED reference's "
                      "envs.%s.step on its own generated CPU kernels, %.1f s; host has %d cores"
                      % (env_name, n, steps, env_name, r["forward_s"] + r["backward_s"], os.cpu_count()),
            "seconds": r["forward_s"] + r["backward_s"], "api": r["api"]}


def gpu_reference_baseline(env_name, num_envs, horizon, rollouts=2):
    """The reference's own CUDA codegen path (sm_100 rebuild) on this GPU at the same config: the GPU-vs-GPU bar."""
    r = _run_ref_arm(_ref_arm_cmd(env_name, num_envs, horizon, rollouts, 1, "cuda:0"), 900)
    if "unavailable" in r:
        return {"value": None, "unit": "env-steps/s", "kind": "reference-cuda", "unavailable": r["unavailable"]}
    return {"value": r["env_steps_per_s"], "unit": "env-steps/s", "kind": "reference-cuda", "api": r["api"],
            "config": "%s num_envs=%d horizon=%d, %d timed rollouts" % (env_name, num_envs, horizon, rollouts),
            "forward_s": r["forward_s"], "backward_s": r["backward_s"], "finite": r["finite"], "peak_mem_gb": r["peak_mem_gb"],
            "note": "reference CUDA codegen (dflex/dflex/adjoint.py:1247-1262) with the one flag edit compute_35 -> compute_100 "
                    "(adjoint.py:1861), driven through the reference's stock envs.%s.step; host-timed with synchronize "
                    "(Python launch overhead is part of the reference path)" % env_name}


def _cpu_pool_worker(env_name, n, horizon, rollouts, warmup, out_q):
    """One host process of the reference arm: builds the reference env once, then `rollouts` timed rollouts on one core."""
    try:
        t_launch = time.time()
        r = _run_ref_arm(_ref_arm_cmd(env_name, n, horizon, rollouts, warmup, "cpu") + ["--stamp"], 3000)
        r["t_launch"] = t_launch
        out_q.put(r)
    except Exception as exc:  # pragma: no cover
        out_q.put({"unavailable": repr(exc)})


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on this box's host cores.  Its kernels are a serial
    loop (adjoint.py:1271-1279), so "all the host threads it can use" = one single-threaded process per core of the affinity
    mask, all running the same bounded sample of the workload concurrently (environments are independent).  Throughput is
    WALL-CLOCKED over the pool: from the first worker entering its timed loop to the last one leaving it."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import multiprocessing as mp
    env = args.env
    n, steps = CPU_SAMPLE[env]
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        cores = os.cpu_count() or 1
    procs = max(1, args.cpu_procs or min(cores, 64))     # (64 torch processes are ~60 GB of host memory; more adds little on an SMT box)
    ctx = mp.get_context("spawn")
    out_q = ctx.Queue()
    workers = [ctx.Process(target=_cpu_pool_worker, args=(env, n, steps, args.steps, max(1, args.warmup), out_q)) for _ in range(procs)]
    for w in workers:
        w.start()
    results = [out_q.get() for _ in workers]
    for w in workers:
        w.join()
    bad = [r for r in results if "unavailable" in r]
    if bad:
        print(json.dumps({"impl": "reference", "unavailable": bad[0]["unavailable"]}))
        return
    wall = max(r["t_end"] for r in results) - min(r["t_start"] for r in results)
    value = procs * n * steps * args.steps / wall
    base = {"value": value, "unit": "env-steps/s", "cores": procs, "kind": "reference",
            "sample": "%s: %d single-threaded processes (affinity mask: %d cores, host: %d) x %d rollouts of (%d envs x %d env-steps, "
                      "forward + sum(rew).backward()) through the UNMODIFIED reference's envs.%s.step on its own generated CPU kernels; "
                      "wall clock over the pool %.1f s" % (env, procs, cores, os.cpu_count() or 0, args.steps, n, steps, env, wall)}
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "env-steps/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "%s reference dflex CPU path, bounded sample per step: %d processes x %d envs x %d env-steps" % (env, procs, n, steps)},
            "cpu_baseline": base,
            "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def run_reference_cuda(args):
    """--impl reference-cuda: the reference's CUDA codegen path on GPU 0 at the headline config."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    T = args.horizon or HORIZON.get(args.env, 32)
    g = gpu_reference_baseline(args.env, args.num_envs, T, rollouts=max(1, args.steps))
    if g.get("value") is None:
        print(json.dumps({"impl": "reference", "unavailable": g.get("unavailable", "?")}))
        return
    secs = g["forward_s"] + g["backward_s"]
    line = {"impl": "reference", "metric": METRIC, "value": g["value"], "unit": "env-steps/s", "n_gpus": 1,
            "steps": max(1, args.steps), "warmup": 1, "ms_per_step": 1e3 * secs / max(1, args.steps), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "%s num_envs=%d horizon=%d on the reference's CUDA codegen path (sm_100 rebuild)" % (args.env, args.num_envs, T)},
            "gpu_baseline": g,
            "e2e": {"value": g["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ our arm
DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays, num_envs):
    """Write ``arrays`` (name -> (tensor, axis of the environments or None)) as ``out_dir/<name>.npy`` in float32.  When they
    exceed DUMP_BYTES together, every array keeps the same fixed, seeded sample of environments (in index order)."""
    import numpy as np
    total = sum(t.numel() * 4 for t, _ in arrays.values())
    keep = None
    if total > DUMP_BYTES:
        k = max(1, num_envs * DUMP_BYTES // total)
        keep = np.sort(np.random.default_rng(0).choice(num_envs, k, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, (t, axis) in arrays.items():
        a = t.detach().float().cpu().numpy()
        if keep is not None and axis is not None:
            a = np.take(a, keep, axis=axis)
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32, copy=False))


def measure_config(env_name, N, T, steps, warmup, dev, rank, world, dist, e2e_mode="graph", comm_floats=0,
                   ncu_range=False, ncu_range_e2e=False, clocks=None, tape_dtype="fp32", dump_dir=None):
    """Kernel path + end-to-end numbers of one workload on this rank.  Returns a dict of raw timings and geometry.
    tape_dtype "bf16": the adjoint tape stores (v, a, f_tot) of every row as bf16 (BASELINE config C2 "bf16 states"; arithmetic
    and the state stay fp32).  dump_dir: write what the last timed step of each path computed there (``dump_outputs``)."""
    import torch
    import diffrl_b200
    from diffrl_b200 import _capi
    import diffrl_b200.envs as envs
    from diffrl_b200.dflex_api.sim import _engine_for

    S, mm = SUBSTEPS[env_name], MM_FREQ[env_name]
    torch.manual_seed(1234 + rank)
    env = getattr(envs, env_name)(num_envs=N, device=str(dev), render=False, seed=rank, stochastic_init=False,
                                  no_grad=False, MM_caching_frequency=mm)
    diffrl_b200.set_tape_dtype(tape_dtype)      # read when the pack is created (next line)
    try:
        eng = _engine_for(env.model)
    finally:
        diffrl_b200.set_tape_dtype("fp32")
    Q, D, M = eng.Q, eng.D, eng.M
    lib = _capi.lib()
    dt = env.sim_dt

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ------------------------------------------------------------ kernel path (inputs resident in HBM)
    g = torch.Generator(device=dev).manual_seed(1 + rank)
    env.clear_grad(); env.reset()
    q0, qd0 = env.state.joint_q.detach().clone(), env.state.joint_qd.detach().clone()
    acts = [torch.zeros(N * D, device=dev) for _ in range(T)]
    muscs = [None] * T
    for t in range(T):
        a = torch.rand((N, env.num_actions), generator=g, device=dev) * 2 - 1
        if env_name == "SNUHumanoidEnv":
            muscs[t] = ((a * 0.5 + 0.5).view(-1) * env.muscle_strengths).contiguous()
        else:
            env.state.joint_act.zero_()
            env._apply_actions(a)
            acts[t] = env.state.joint_act.detach().clone()
    gq_seed, gqd_seed = torch.randn(N * Q, device=dev), torch.randn(N * D, device=dev)
    phase_events = []      # (start, forward done, backward done) of every timed rollout, on the launching stream

    def kernel_rollout(record=False):
        ev3 = [torch.cuda.Event(enable_timing=True) for _ in range(3)] if record else None
        if record:
            ev3[0].record()
        q, qd, tapes = q0, qd0, []
        for t in range(T):
            q, qd, tape, _ = eng.forward(q, qd, acts[t], muscs[t], S, mm, dt)
            tapes.append(tape)
        if record:
            ev3[1].record()
        gq, gqd, gacts, gms = gq_seed, gqd_seed, [None] * T, [None] * T
        for t in reversed(range(T)):
            gq, gqd, gacts[t], gms[t] = eng.backward(acts[t], muscs[t], tapes[t], gq, gqd, S, mm, dt)
        if record:
            ev3[2].record()
            phase_events.append(ev3)
        return q, qd, gq, gqd, gacts, gms      # what a caller of this path receives

    for _ in range(warmup):
        kernel_rollout()
    barrier()
    if ncu_range:
        torch.cuda.profiler.start()
        kernel_rollout()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
    launches0 = lib.dfx_launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(steps):
        kernel_out = kernel_rollout(record=True)
    ev[1].record()
    barrier()
    kernel_ms = ev[0].elapsed_time(ev[1])
    launches = lib.dfx_launch_count() - launches0
    # average launch duration of the forward and of the adjoint kernel INSIDE the timed rollouts (every launch reads /
    # writes its own tape block, gigabytes per rollout, far beyond L2): the roofline denominators
    fwd_ms = sum(e[0].elapsed_time(e[1]) for e in phase_events) / (len(phase_events) * T)
    bwd_ms = sum(e[1].elapsed_time(e[2]) for e in phase_events) / (len(phase_events) * T)
    tape_mb = T * eng.tape_floats(S, mm) * 4 / 1e6

    # ------------------------------------------------------------ end to end through env.step + autograd
    host_actions = torch.empty((T, N, env.num_actions), dtype=torch.float32).pin_memory()
    host_actions.copy_(torch.rand(host_actions.shape) * 2 - 1)
    host_grad = torch.empty((T, N, env.num_actions), dtype=torch.float32).pin_memory()
    host_loss = torch.empty((), dtype=torch.float32).pin_memory()
    comm = torch.zeros(comm_floats, device=dev) if (world > 1 and comm_floats) else None

    def allreduce_policy_gradient(grad):
        # the one collective of a data-parallel SHAC actor update (SURVEY.md section 8e): the flattened policy gradient,
        # summed over ranks once per rollout.  The synthetic benchmark has no policy network; a buffer of the actor's
        # size (cfg/shac/ant.yaml: 128-64-32 MLP = 16 K floats) carries the action-gradient summary.
        if comm is not None:
            comm[: T * env.num_actions] = grad.mean(dim=1).reshape(-1)
            dist.all_reduce(comm)

    def e2e_rollout():
        env.clear_grad()
        env.reset()
        env.initialize_trajectory()
        a_dev = host_actions.to(dev, non_blocking=True).requires_grad_()
        loss = torch.zeros((), device=dev)
        for t in range(T):
            obs, rew, done, _ = env.step(a_dev[t])
            loss = loss + rew.sum()
        loss.backward()
        allreduce_policy_gradient(a_dev.grad)
        host_grad.copy_(a_dev.grad, non_blocking=True)
        host_loss.copy_(loss.detach(), non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return float(host_loss)

    e2e_steps = steps
    for _ in range(max(1, warmup // 2)):
        e2e_rollout()
    barrier()
    e3 = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    e3[0].record()
    for _ in range(e2e_steps):
        e2e_rollout()
    e3[1].record()
    barrier()
    eager_ms = e3[0].elapsed_time(e3[1])
    e2e_out = (host_loss, host_grad)

    # the same rollout through the package's graphed-rollout API (one CUDA graph per rollout: H2D actions,
    # horizon x env.step, loss.backward, D2H loss + action gradients)
    e2e_ms, e2e_api = eager_ms, "envs.%s.step -> dflex.sim.SemiImplicitIntegrator.forward -> autograd (eager)" % env_name
    if e2e_mode != "eager" and hasattr(env, "_start_state"):
        from diffrl_b200.rollout import GraphedRollout
        env.clear_grad(); env.reset(); env.initialize_trajectory()
        roll = GraphedRollout(env, T)
        roll.host_actions.copy_(host_actions)      # the pinned staging buffer the graph's H2D copy reads every rollout

        def graphed_rollout():
            env.clear_grad()
            env.reset()
            loss_h, grad_h = roll(None, sync=False)
            allreduce_policy_gradient(roll.actions.grad)
            torch.cuda.current_stream().synchronize()
            return float(loss_h)

        for _ in range(max(1, warmup // 2)):
            graphed_rollout()
        barrier()
        if ncu_range_e2e:          # launch list of ONE end-to-end rollout (profiles/): ncu --profile-from-start off
            torch.cuda.profiler.start()
            graphed_rollout()
            torch.cuda.synchronize()
            torch.cuda.profiler.stop()
        e3[0].record()
        for _ in range(e2e_steps):
            graphed_rollout()
        e3[1].record()
        barrier()
        e2e_ms = e3[0].elapsed_time(e3[1])
        e2e_api = "diffrl_b200.rollout.GraphedRollout(envs.%s): one CUDA graph = H2D actions + %d x env.step + backward + D2H" % (env_name, T)
        e2e_out = (roll.host_loss.clone(), roll.host_grad.clone())
        del roll

    if dump_dir:
        q, qd, gq, gqd, gacts, gms = kernel_out
        arrays = {"kernel_q": (q.view(N, Q), 0), "kernel_qd": (qd.view(N, D), 0), "kernel_grad_q0": (gq.view(N, Q), 0),
                  "kernel_grad_qd0": (gqd.view(N, D), 0), "kernel_grad_joint_act": (torch.stack(gacts).view(T, N, D), 1),
                  "e2e_loss": (e2e_out[0], None), "e2e_grad_actions": (e2e_out[1], 1)}
        if M:
            arrays["kernel_grad_muscle_act"] = (torch.stack(gms).view(T, N, M), 1)
        dump_outputs(dump_dir, arrays, N)
    del kernel_out, e2e_out

    tile = int(lib.dfx_pack_query(eng.pack, 9))
    row = int(lib.dfx_pack_query(eng.pack, 8))   # DFX_QUERY_TAPE_ROW_FLOATS
    out = dict(env=env_name, N=N, T=T, S=S, mm=mm, Q=Q, D=D, M=M, row=row, tile=tile, kernel_ms=kernel_ms, e2e_ms=e2e_ms,
               eager_ms=eager_ms, fwd_ms=fwd_ms, bwd_ms=bwd_ms, launches=int(launches), steps=steps, e2e_steps=e2e_steps,
               tape_mb=tape_mb, tape_dtype=tape_dtype, e2e_api=e2e_api, h2d=int(host_actions.numel() * 4), d2h=int(host_grad.numel() * 4 + 4),
               comm_floats=comm_floats if comm is not None else 0)
    del env, eng, acts, muscs, host_actions, host_grad
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    return out


def roofline_record(m, peaks, peak_kind, traffic=None, fp32=None):
    """SURVEY.md section 8d roofline of the adjoint launch (+ the forward launch and the design's own bytes beside it)."""
    N, Q, D, A, S, mm = m["N"], m["Q"], m["D"], m["D"] + m["M"], m["S"], m["mm"]
    s_fwd, s_bwd = algorithmic_bytes(Q, D, A, S)
    d_fwd, d_bwd = algorithmic_bytes(Q, D, A, S, row=m["row"], nseg=(S + mm - 1) // mm)
    peak = peaks["hbm_gbs"]
    ach = N * s_bwd / (m["bwd_ms"] * 1e-3) / 1e9
    dach = N * d_bwd / (m["bwd_ms"] * 1e-3) / 1e9
    whole = N * (s_fwd + s_bwd) / ((m["fwd_ms"] + m["bwd_ms"]) * 1e-3) / 1e9
    family = ("dfx_tile_kernel<BWD=1> (adjoint of one env-step, %d-environment tiles, TMA bulk tape copies)" % m["tile"]) if m["tile"] \
        else "dfx_step_kernel<G,BWD=1> (adjoint of one env-step, lane groups)"
    return {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
            "peak_source": peak_kind, "kernel": family,
            "algorithmic_bytes_per_launch": N * s_bwd,
            "bytes_definition": "SURVEY.md section 8d, state-only tape: %d B forward + %d B adjoint per env-step" % (s_fwd, s_bwd),
            "forward_kernel": {"achieved": N * s_fwd / (m["fwd_ms"] * 1e-3) / 1e9, "frac": N * s_fwd / (m["fwd_ms"] * 1e-3) / 1e9 / peak,
                               "algorithmic_bytes_per_launch": N * s_fwd},
            "env_step_fwd_plus_adjoint": {"achieved": whole, "frac": whole / peak},
            "design_frac": dach / peak, "design_achieved": dach, "design_bytes_per_launch": N * d_bwd,
            "design_bytes_definition": "what this design moves: tape rows with the forward intermediates (4 x %d B per env-substep) + H^-1 blocks + state I/O" % m["row"],
            "fp32": fp32,
            "note": "the fused path is FP32-issue / latency bound, not HBM bound (profiles/, DESIGN.md section 3); launch durations are "
                    "averages over the timed rollouts (CUDA events on the launching stream)"}


def profile_numbers(env_name, N, m, sm_mhz):
    """(DRAM bytes per adjoint launch, fp32 record) from the committed ncu capture of this launch shape (profiles/r0X_traffic.json,
    tools/make_traffic_json.py), or (None, None) when no capture of this (env, num_envs) is committed."""
    for tname in ("r02_traffic.json", "r01_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", tname)
        if not os.path.exists(tpath):
            continue
        with open(tpath) as f:
            prof = json.load(f).get(env_name, {})
        if not prof or prof.get("num_envs", 4096) != N:
            continue
        fp32 = None
        if "bwd_fp32_flop_per_launch" in prof:
            # SURVEY.md 8d's second yardstick: fp32 FLOP actually executed (counted by ncu for this launch shape) per
            # second against the CUDA-core peak 148 SMs x 128 lanes x 2 FLOP x the SM clock sampled during the run
            flop = prof["fwd_fp32_flop_per_launch"] + prof["bwd_fp32_flop_per_launch"]
            peak = 148 * 128 * 2 * sm_mhz * 1e6
            secs = (m["fwd_ms"] + m["bwd_ms"]) * 1e-3
            fp32 = {"achieved_tflops": flop / secs / 1e12, "peak_tflops": peak / 1e12, "frac": flop / secs / peak,
                    "flop_per_env_step": flop / N, "source": "profiles/%s (ncu instruction counts)" % tname}
        return prof.get("bwd_dram_bytes_per_launch"), fp32
    return None, None


def config_record(m, world, peaks, peak_kind):
    value = world * m["N"] * m["T"] * m["steps"] / (m["kernel_ms"] * 1e-3)
    e2e = world * m["N"] * m["T"] * m["e2e_steps"] / (m["e2e_ms"] * 1e-3)
    return {"workload": "%s num_envs=%d/GPU horizon=%d substeps=%d mass_matrix_freq=%d" % (m["env"], m["N"], m["T"], m["S"], m["mm"]),
            "value": value, "unit": "env-steps/s", "value_is": "kernel path (simulation launches only)",
            "e2e": {"value": e2e, "unit": "env-steps/s", "api": m["e2e_api"], "h2d_bytes_per_step": m["h2d"], "d2h_bytes_per_step": m["d2h"],
                    "eager_env_step_loop": world * m["N"] * m["T"] * m["e2e_steps"] / (m["eager_ms"] * 1e-3)},
            "kernel_ms": {"forward_env_step": m["fwd_ms"], "backward_env_step": m["bwd_ms"]},
            "kernel_family": ("tile (%d envs per CTA)" % m["tile"]) if m["tile"] else "lane group",
            "tape_mb_per_rollout": m["tape_mb"], "tape_storage": "fp32" if m.get("tape_dtype", "fp32") == "fp32" else "bf16 for (v, a, f_tot) of every row, fp32 otherwise (arithmetic fp32)",
            "gpu_launches": m["launches"],
            "roofline": roofline_record(m, peaks, peak_kind, *profile_numbers(m["env"], m["N"], m, 1965.0))}


def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    env_name, N, T = args.env, args.num_envs, args.horizon or HORIZON.get(args.env, 32)
    comm_floats = 16384     # the Ant actor's flattened gradient (cfg/shac/ant.yaml); one all-reduce per rollout when world > 1
    with ClockSampler(local) as clocks:
        head = measure_config(env_name, N, T, args.steps, args.warmup, dev, rank, world, dist, e2e_mode=args.e2e,
                              comm_floats=comm_floats, ncu_range=args.ncu_range, ncu_range_e2e=args.ncu_range_e2e,
                              dump_dir=args.dump_outputs if rank == 0 else None)
    # ---- the other named configs (BASELINE.json): short runs, same measurement
    subs = {}
    if not args.no_configs:
        plan = []
        if world > 1:
            plan.append(("c4", "AntEnv", 8192, 32, args.steps, 2))
        else:
            plan += [("humanoid8192", "HumanoidEnv", 8192, 32, args.steps, 1), ("humanoid8192_bf16_tape", "HumanoidEnv", 8192, 32, args.steps, 1),
                     ("snu4096_bptt128", "SNUHumanoidEnv", 4096, 128, args.steps, 1), ("cartpole64", "CartPoleSwingUpEnv", 64, 32, args.steps, 2)]
        for key, e, n, t, k, w in plan:
            try:
                subs[key] = measure_config(e, n, t, k, w, dev, rank, world, dist, e2e_mode=args.e2e, comm_floats=comm_floats,
                                           tape_dtype="bf16" if key.endswith("bf16_tape") else "fp32")
            except Exception as exc:     # a sub-config must not take the headline down
                subs[key] = {"error": repr(exc)[:300]}

    # ------------------------------------------------------------ reduce over ranks (max time)
    def reduce_times(m):
        if "error" in m:
            return m
        times = torch.tensor([m["kernel_ms"], m["e2e_ms"], m["eager_ms"], m["fwd_ms"], m["bwd_ms"]], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(times, op=dist.ReduceOp.MAX)
        m["kernel_ms"], m["e2e_ms"], m["eager_ms"], m["fwd_ms"], m["bwd_ms"] = times.tolist()
        return m

    head = reduce_times(head)
    subs = {k: reduce_times(v) for k, v in subs.items()}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks, peak_kind = measured_peaks()
    value = world * N * T * args.steps / (head["kernel_ms"] * 1e-3)
    e2e_value = world * N * T * head["e2e_steps"] / (head["e2e_ms"] * 1e-3)
    traffic, fp32 = profile_numbers(env_name, N, head, clocks.summary().get("sm_mhz") or 1965.0)
    line = {
        "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": world,
        "value_is": "kernel path: simulation-kernel launches only, inputs resident (the headline is e2e)",
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": head["kernel_ms"] / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "%s num_envs=%d/GPU SHAC short-horizon=%d (rollout forward + adjoint), substeps=%d, "
                               "mass_matrix_freq=%d" % (env_name, N, T, head["S"], head["mm"]),
                   "parallelism": "env-sharded x%d, no data-path collective%s" % (world, "; one %d KB policy-gradient all-reduce per rollout (e2e)" % (comm_floats * 4 // 1024) if world > 1 else ""),
                   "cache": "per-rollout tape %.0f MB > 126 MB L2 (inputs larger than L2)" % head["tape_mb"],
                   "kernel_family": ("tile (%d envs per CTA, TMA tape copies)" % head["tile"]) if head["tile"] else "lane group"},
        "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": head["h2d"], "d2h_bytes_per_step": head["d2h"],
                "api": head["e2e_api"], "ms_per_step": head["e2e_ms"] / head["e2e_steps"],
                "eager_env_step_loop": {"value": world * N * T * head["e2e_steps"] / (head["eager_ms"] * 1e-3), "ms_per_step": head["eager_ms"] / head["e2e_steps"]}},
        "gpu_launches": head["launches"],
        "kernel_ms": {"forward_env_step": head["fwd_ms"], "backward_env_step": head["bwd_ms"]},
        "roofline": roofline_record(head, peaks, peak_kind, traffic, fp32),
        "clocks": clocks.summary(),
    }
    if subs:
        line["configs"] = {k: (v if "error" in v else config_record(v, world, peaks, peak_kind)) for k, v in subs.items()}
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_reference_baseline(env_name)
    if world == 1 and not args.no_gpu_baseline:
        torch.cuda.empty_cache()
        line["gpu_baseline"] = gpu_reference_baseline(env_name, N, T)
        if line["gpu_baseline"].get("value"):
            line["gpu_baseline"]["e2e_over_reference_cuda"] = e2e_value / line["gpu_baseline"]["value"]
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-cuda"])
    ap.add_argument("--env", default="AntEnv", choices=sorted(SUBSTEPS))
    ap.add_argument("--num-envs", type=int, default=4096)
    ap.add_argument("--horizon", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config sub-records (humanoid8192, snu4096_bptt128, cartpole64 / c4)")
    ap.add_argument("--e2e", default="graph", choices=["graph", "eager"])
    ap.add_argument("--cpu-procs", type=int, default=0, help="reference arm: host processes (default: one per core of the affinity mask)")
    ap.add_argument("--ncu-range-e2e", action="store_true",
                    help="wrap one graphed end-to-end rollout in cudaProfilerStart/Stop (for ncu --profile-from-start off)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step of the headline workload computed as DIR/<name>.npy "
                         "(float32; inputs are seeded, so two builds can be compared output for output)")
    ap.add_argument("--ncu-range", action="store_true",
                    help="wrap ONE kernel-path step in cudaProfilerStart/Stop (use with ncu --profile-from-start off)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "reference-cuda":
        run_reference_cuda(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
