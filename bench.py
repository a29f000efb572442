#!/usr/bin/env python
"""bench.py -- generations/sec of the ES hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one ES generation (estorch.py:214-248): evaluate the P = 4096 mirrored members of the
1M-parameter MLP over a synthetic observation batch, centred-rank the returns, reduce
sum_j w_j * noise_j, negate/clamp, Adam, post-update rollout.  Prints ONE JSON line on rank 0.

  value  device-resident throughput: inputs already in HBM, no host synchronisation inside the
         timed region (CUDA events, max over ranks); log() is not due inside the region
  e2e    the same through the public API with HOST buffers: every generation uploads the
         observation/target batch from pinned host memory, calls log() and reads
         population_returns + episode_reward back (host clock around K steps) -- the headline
  roofline / kernels   per-kernel achieved rate vs MEASURED_PEAKS.json
  cpu_baseline         the reference's CPU path on this box's host cores, bounded sample, rank 0 / N=1
  extra                the other BASELINE.json configs through the same public API (short runs)

`--dump-outputs DIR` writes, after the timed generations, what a caller of ES.train holds after the last
one (parameters, population returns, episode / best reward, best policy) as DIR/<name>.npy; the inputs are
seeded, so two builds run with the same arguments can be compared output for output.

`--impl reference` runs only the reference's CPU path (rank 0): the UNMODIFIED reference package from
baseline/_ref (installed by __graft_entry__.build()) when present, else the CPU port of its cost
structure (oracle/reference_port.py); same metric/config.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MLP_1M = [128, 512, 512, 512, 512, 288]
WORKLOADS = {
    # BASELINE.json metric: pop=4096, 1M-param MLP (SURVEY 8: obs 128, 4x512 hidden, 288 out)
    "north_star": dict(algo="es", dims=MLP_1M, population_size=4096, sigma=0.02, batch=256),
    # configs[1]: CartPole-shape 2x64 MLP, pop 4096, 1 GPU
    "cartpole": dict(algo="es", dims=[4, 64, 64, 2], population_size=4096, sigma=0.1, batch=256),
    # configs[2]: the 1M MLP at pop=8192, sigma=0.02, sharded over 8 GPUs (runs on however many there are)
    "config3": dict(algo="es", dims=MLP_1M, population_size=8192, sigma=0.02, batch=256),
    # configs[3]: NSRA-ES, BipedalWalker-shape MLP 24->4, pop 2048 (examples/nsra_es.py:61-67)
    "nsra_bipedal": dict(algo="nsra", dims=[24, 64, 64, 4], population_size=2048, sigma=0.02, batch=256,
                         bc_obs=64, bc_dim=256),
    # configs[4]: Atari conv policy 84x84x4 + VirtualBatchNorm, pop 1024 (examples/atari.py:14-37)
    "atari_vbn": dict(algo="es", conv=True, population_size=1024, sigma=0.02, batch=32, ref_batch=128, n_actions=4),
}
METRIC = "generations/sec at pop=4096, 1M-param MLP"


class MLP(torch.nn.Module):
    def __init__(self, dims):
        super().__init__()
        layers = []
        for i in range(len(dims) - 1):
            layers.append(torch.nn.Linear(dims[i], dims[i + 1]))
            if i + 2 < len(dims):
                layers.append(torch.nn.ReLU())
        self.net = torch.nn.Sequential(*layers)

    def forward(self, x):
        return self.net(x)


def n_params(wl):
    if wl.get("conv"):
        return 677268 if wl["n_actions"] == 4 else None
    dims = wl["dims"]
    return sum(dims[i] * dims[i + 1] + dims[i + 1] for i in range(len(dims) - 1))


def synthetic_batch(dims, batch):
    g = torch.Generator().manual_seed(1234)
    return torch.randn(batch, dims[0], generator=g), torch.randn(batch, dims[-1], generator=g)


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p["hbm_gbs"], tensor_burst=p["bf16_tflops"], tensor=p["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tensor_burst=1590.0, tensor=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def window(self, t0, t1):
        rows = [r for t, r in self.rows if t0 <= t <= t1] or [r for _, r in self.rows[-3:]]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": float(rows[0][1]) if rows[0][1].replace(".", "").isdigit() else None,
                "power_w_max": max((float(r[2]) for r in rows if r[2].replace(".", "").isdigit()), default=None),
                "samples": len(rows), "reasons": reasons}

    def stop(self):
        if self.proc:
            self.proc.terminate()


# ----------------------------------------------------------------------------- CPU reference arm
def _host_threads():
    """torchrun exports OMP_NUM_THREADS=1: give the CPU arm the cores it would have on its own."""
    n = max(1, min(os.cpu_count() or 1, 64))
    torch.set_num_threads(n)
    return n


def cpu_reference(wl, steps, warmup, budget_s=20.0):
    """Time the reference's CPU path for the workload on a bounded population sample and scale
    linearly in P (sample, cat, rollouts, mm are all O(P*n); SURVEY 8d).  Uses the unmodified
    reference (baseline/_ref) when it is installed, else the CPU port of its cost structure."""
    from oracle.ref_shim import import_reference
    from oracle.reference_port import time_reference
    from estorch_b200.agents import DeviceAgent
    cores = _host_threads()
    dims, P, sigma = wl["dims"], wl["population_size"], wl["sigma"]
    obs, tgt = synthetic_batch(dims, wl["batch"])
    ref = import_reference()
    torch.manual_seed(0)

    def run(sample_P, k, w):
        if ref is None:
            return time_reference(MLP, {"dims": dims}, DeviceAgent(obs, tgt), sample_P, sigma, steps=k, warmup=w)
        # the reference's own classes and loop: ES.__init__ (estorch.py:121-148) + ES.train(n_steps, n_proc=1)

        class Quiet(ref.ES):
            def log(self):
                pass
        es = Quiet(MLP, DeviceAgent, torch.optim.Adam, population_size=sample_P, sigma=sigma,
                   policy_kwargs={"dims": dims}, agent_kwargs=dict(obs=obs, target=tgt), optimizer_kwargs={"lr": 0.01})
        if w:
            es.train(w)
        t0 = time.perf_counter()
        es.train(k)
        return (time.perf_counter() - t0) / k, {}

    probe_P = 16
    dt, _ = run(probe_P, 1, 0)
    per_member = dt / probe_P
    sample_P = int(min(P, max(16, budget_s / max(1, steps + warmup) / per_member)))
    sample_P -= sample_P % 2
    dt, phases = run(sample_P, steps, warmup)
    scale = P / sample_P
    return dict(seconds_per_generation_full=dt * scale, value=1.0 / (dt * scale), sample_P=sample_P,
                extrapolation_factor=scale, seconds_per_generation_sample=dt, phases_sample_s=phases, cores=cores,
                kind="port" if ref is None else "reference")


def run_reference_arm(args, wl, rank, world):
    if rank != 0:
        return
    r = cpu_reference(wl, args.steps, min(args.warmup, 1), budget_s=60.0)
    what = ("the UNMODIFIED reference package (baseline/_ref, estorch.ES.train(n_proc=1) through a one-rank mpi4py shim)"
            if r["kind"] == "reference" else "CPU port of the reference's cost structure (oracle/reference_port.py)")
    cb = {"value": r["value"], "unit": "generations/s", "cores": r["cores"], "kind": r["kind"],
          "sample_P": r["sample_P"], "extrapolation_factor": r["extrapolation_factor"],
          "sample": f"{what}; population_size={r['sample_P']} of {wl['population_size']} per step, same policy/batch, "
                    f"the agent is this repo's DeviceAgent (plain torch rollout: it implements the reference's Agent "
                    f"protocol); time scaled linearly in P by {r['extrapolation_factor']:.1f} (all phases are O(P*n)); "
                    f"1 process, {r['cores']} torch threads of {os.cpu_count()} cpus"}
    line = {"impl": "reference", "metric": METRIC, "value": r["value"],
            "unit": "generations/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * r["seconds_per_generation_full"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, wl, world), "cpu_baseline": cb,
            "e2e": {"value": r["value"], "unit": "generations/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0}}
    emit(line)


def workload_config(args, wl, world, name=None):
    name = name or args.workload
    if wl.get("conv"):
        shape = (f"conv 4->16 k8 s4 / VirtualBatchNorm / conv 16->32 k4 s2 / VirtualBatchNorm / fc 2592->256->{wl['n_actions']}"
                 f" (n={n_params(wl)}), {wl['ref_batch']} reference frames")
    else:
        shape = f"MLP {wl['dims']} (n={n_params(wl)})"
    return {"workload": f"{name}: {wl['algo'].upper()} generation, population_size={wl['population_size']} "
                        f"({wl['population_size'] // 2} antithetic pairs), {shape}, synthetic obs batch "
                        f"B={wl['batch']}, sigma={wl['sigma']}, Adam lr=0.01, noise table 2^{args.table_log2} entries "
                        f"(fp32 values with an 11-bit significand; evaluate and reduction stream the exact 16-bit copy)",
            "population_size": wl["population_size"], "n_parameters": n_params(wl),
            "batch": wl["batch"], "parallelism": f"pairs sharded over {world} GPU(s)",
            "l2": "noise stream per step (>= 4 GB at north_star) exceeds L2; no flush needed"}


# ----------------------------------------------------------------------------- our arm
def build_es(wl, args, eval_precision, log_interval):
    """The workload through the public API (estorch_b200.ES / NSRA_ES)."""
    import estorch_b200 as E
    P, sigma, B = wl["population_size"], wl["sigma"], wl["batch"]

    class Streaming(E.DeviceAgent):
        """e2e: each generation's batch comes from pinned host memory."""
        stream_from_host = False

        def __init__(self, obs, target, **kw):
            super().__init__(obs, target, **kw)
            self.h_obs, self.h_tgt = self.obs.clone().pin_memory(), self.target.clone().pin_memory()

        def next_batch(self, step):
            return (self.h_obs, self.h_tgt) if self.stream_from_host else None

    base = E.NSRA_ES if wl["algo"] == "nsra" else E.ES

    class Bench(base):
        read_back = False

        def log(self):
            if self.read_back:   # the step's result, on the host (D2H of P returns + 32-byte state)
                self.last = (self.population_returns, self.episode_reward)

    torch.manual_seed(0)
    common = dict(population_size=P, sigma=sigma, optimizer_kwargs={"lr": 0.01}, noise_table_size=1 << args.table_log2,
                  noise_seed=42, log_interval=log_interval)
    if wl.get("conv"):
        from estorch_b200.vbn import VirtualBatchNorm

        class AtariPolicy(torch.nn.Module):          # architecture of the reference's examples/atari.py:14-37
            def __init__(self, n_actions, xref):
                super().__init__()
                self.xref = xref
                self.conv1 = torch.nn.Conv2d(4, 16, 8, 4)
                self.bn1 = VirtualBatchNorm(16)
                self.conv2 = torch.nn.Conv2d(16, 32, 4, 2)
                self.bn2 = VirtualBatchNorm(32)
                self.fc1 = torch.nn.Linear(2592, 256)
                self.fc2 = torch.nn.Linear(256, n_actions)

            def forward(self, x):
                F = torch.nn.functional
                r = F.relu(self.bn1(self.conv1(self.xref.to(x.device))))
                r = F.relu(self.bn2(self.conv2(r)))
                x = F.relu(self.bn1(self.conv1(x)))
                x = F.relu(self.bn2(self.conv2(x)))
                return self.fc2(F.relu(self.fc1(x.view(-1, 2592))))
        g = torch.Generator().manual_seed(1234)
        xref = torch.rand(wl["ref_batch"], 4, 84, 84, generator=g)
        obs, tgt = torch.rand(B, 4, 84, 84, generator=g), torch.randn(B, wl["n_actions"], generator=g)
        es = Bench(AtariPolicy, Streaming, torch.optim.Adam, policy_kwargs=dict(n_actions=wl["n_actions"], xref=xref),
                   agent_kwargs=dict(obs=obs, target=tgt), **common)
    else:
        obs, tgt = synthetic_batch(wl["dims"], B)
        akw = dict(obs=obs, target=tgt)
        if wl["algo"] == "nsra":
            akw.update(bc_obs=wl["bc_obs"], bc_dim=wl["bc_dim"])
        es = Bench(MLP, Streaming, torch.optim.Adam, policy_kwargs={"dims": wl["dims"]}, agent_kwargs=akw,
                   eval_precision=eval_precision, **common)
    assert es._fused, "bench: fused device path is not active"
    return es, obs, tgt


def capture_outputs(es):
    """What a caller of ES.train holds after the last generation, copied to the host (float32 arrays,
    float64 scalars)."""
    def flat(module):
        return torch.nn.utils.parameters_to_vector(module.parameters()).detach().float().cpu().numpy()
    out = {"population_returns": np.array(es.population_returns, dtype=np.float32),      # a copy: the host cache is reused
           "episode_reward": np.array([es.episode_reward], dtype=np.float64),
           "best_reward": np.array([es.best_reward], dtype=np.float64),
           "best_policy": np.concatenate([v.detach().float().cpu().reshape(-1).numpy()
                                          for v in es.best_policy_dict.values()])}
    if hasattr(es, "meta_population"):
        out["meta_population"] = np.stack([flat(policy) for policy, _ in es.meta_population])
    else:
        out["policy"] = flat(es.policy)
    return out


def dump_outputs(outputs, directory, limit=64 << 20):
    total = sum(a.nbytes for a in outputs.values())
    if total > limit:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs exceed the {limit}-byte limit")
    os.makedirs(directory, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def timed_region(es, steps, warmup, world, dev, sampler=None):
    """(ms, wall s, clocks, launches) of `steps` generations: CUDA events around the region,
    barrier + synchronize on both sides, max over ranks."""
    import torch.distributed as dist

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    es.train(warmup)
    barrier()
    launches0 = es._be.launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    ev0.record()
    es.train(steps)
    ev1.record()
    barrier()
    t1 = time.perf_counter()
    ms, wall = ev0.elapsed_time(ev1), t1 - t0
    if world > 1:
        t = torch.tensor([ms, wall], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, wall = float(t[0].item()), float(t[1].item())
    return ms, wall, (sampler.window(t0, t1) if sampler else None), es._be.launches - launches0


def run_extra(name, args, world, dev, steps=20):
    """One of the other BASELINE configs through the same public API: device-resident generations/s
    and the host-in / host-out e2e figure (short run)."""
    wl = WORKLOADS[name]
    try:
        es, obs, tgt = build_es(wl, args, "auto", 10 ** 9)
        ms, _, _, launches = timed_region(es, steps, 5, world, dev)
        es.agent.stream_from_host, es.read_back, es._log_interval = True, True, 1
        _, wall, _, _ = timed_region(es, steps, 5, world, dev)
        out = {"config": workload_config(args, wl, world, name)["workload"], "n_gpus": world, "steps": steps,
               "value": steps / (ms / 1e3), "e2e": steps / wall, "unit": "generations/s",
               "ms_per_step": ms / steps, "eval_precision": es._precision, "gpu_launches": launches}
        del es
        torch.cuda.empty_cache()
        return out
    except Exception as e:           # an extra must never cost the headline line
        return {"config": name, "error": repr(e)[:300]}


def run_ours(args, wl, rank, world, local_rank):
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)
    P = wl["population_size"]
    es, obs, tgt = build_es(wl, args, args.eval_precision, 10 ** 9)

    # ---- value: device-resident, no host sync in the loop
    sampler = ClockSampler(local_rank) if rank == 0 else None   # nvidia-smi needs ~1 s to start streaming
    ms, _, clocks, launches = timed_region(es, args.steps, args.warmup, world, dev, sampler)
    outputs = capture_outputs(es) if args.dump_outputs and rank == 0 else None

    # ---- e2e: host buffers in, log() + host results out, every generation
    es.agent.stream_from_host, es.read_back, es._log_interval = True, True, 1
    _, e2e_s, _, _ = timed_region(es, args.steps, args.warmup, world, dev)
    if sampler:
        sampler.stop()

    peaks = load_peaks()
    kern = {}
    if not wl.get("conv") and wl["algo"] == "es":
        kern = kernel_rooflines(es, wl, args, world, rank, peaks)
    precision = es._precision
    graphed = any(isinstance(v, tuple) for v in es.__dict__.get("_graphs", {}).values())
    del es
    torch.cuda.empty_cache()

    extras = None
    # (single-GPU runs only: the scaling runs stay lean; the other configs at their named GPU counts are
    #  recorded with `--workload NAME` under torchrun, see profiles/)
    names = ()
    if args.extras:                       # explicit list: also under torchrun (the configs named for N GPUs)
        names = tuple(x for x in args.extras.split(",") if x)
    elif not args.no_extras and args.workload == "north_star" and world == 1:
        names = ("cartpole", "nsra_bipedal", "config3", "atari_vbn")
    if names:
        extras = {}
        for name in names:
            extras[name] = run_extra(name, args, world, dev, steps=5 if name == "atari_vbn" else 20)

    if rank != 0:
        return
    if outputs is not None:
        dump_outputs(outputs, args.dump_outputs)
    line = {"metric": METRIC, "value": args.steps / (ms / 1e3),
            "unit": "generations/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None,
            "dtype": {"f16": "f32 (fp32-equivalent: evaluate GEMMs on tcgen05 with fp16 operands = 11-bit significand, "
                             "TF32 class, each weight formed in fp32 from fp32 theta + the exactly-16-bit noise value and "
                             "rounded once, f32 accumulate, f32 bias/loss; f32 ranks, reduction, Adam)",
                      "bf16": "bf16 operands / f32 accumulate (evaluate GEMMs); f32 noise, ranks, reduction, Adam",
                      "bf16s": "bf16 operands formed from bf16 shadows of theta/noise, f32 accumulate (evaluate "
                               "GEMMs); f32 noise table, ranks, reduction, Adam"}.get(precision, "f32"),
            "eval_precision": precision,
            "data": "synthetic", "config": workload_config(args, wl, world),
            "e2e": {"value": args.steps / e2e_s, "unit": "generations/s",
                    "h2d_bytes_per_step": int(obs.numel() * 4 + tgt.numel() * 4),
                    "d2h_bytes_per_step": int(4 * P + 32)},
            "gpu_launches": launches, "cuda_graph": graphed, "clocks": clocks}
    line.update(kern)
    line["cpu_baseline"] = None
    if world == 1 and not args.no_cpu_baseline and not wl.get("conv") and wl["algo"] == "es":
        r = cpu_reference(wl, steps=1, warmup=0, budget_s=15.0)
        line["cpu_baseline"] = {
            "value": r["value"], "unit": "generations/s", "cores": r["cores"], "kind": r["kind"],
            "sample_P": r["sample_P"], "extrapolation_factor": r["extrapolation_factor"],
            "sample": f"1 generation of {'the unmodified reference (baseline/_ref)' if r['kind'] == 'reference' else 'the CPU port'} "
                      f"at population_size={r['sample_P']} of {P}, scaled linearly in P; {r['cores']} torch threads of "
                      f"{os.cpu_count()} cpus; {r['seconds_per_generation_sample']:.2f} s/sample-generation"}
    if extras is not None:
        line["extra"] = extras
    emit(line)


def kernel_rooflines(es, wl, args, world, rank, peaks):
    """Per-kernel device time (CUDA events on the launching stream), geometry of this rank."""
    from estorch_b200.backend import adam_desc
    be, P, sigma, B, dims = es._be, wl["population_size"], wl["sigma"], wl["batch"], wl["dims"]
    n, pairs, pl, slot = n_params(wl), P // 2, es._pairs_local, es._slots[0]

    def timed(fn, iters=5):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
        for a, b in evs:
            a.record(); fn(); b.record()
        torch.cuda.synchronize()
        return sorted(a.elapsed_time(b) for a, b in evs)[iters // 2]

    R = es._returns if world == 1 else es._rm_buffers()[0]
    gt = es._grad_table()                       # the exact fp16 copy of the table when there is one
    tbytes = gt.element_size()
    rp, rm_ = (R[es._pair_begin: es._pair_begin + pl], R[pairs + es._pair_begin: pairs + es._pair_begin + pl]) \
        if world == 1 else (R[rank, 0], R[rank, 1])
    t_eval = timed(lambda: be.eval_mlp(es._spec.dims, slot.theta, es._table, es._offsets, es._order, pl, sigma,
                                       es._obs, es._tgt, rp, rm_, **es._eval_kw(slot)), iters=3)
    scratch = [t.clone() for t in (slot.theta, slot.m, slot.v)]
    ad = adam_desc(lr=0.01)
    if world == 1:
        st_scratch = slot.state.clone()
        t_grad = timed(lambda: be.rank_grad_adam(R, None, 1.0, 0.0, P, gt, es._offsets, es._order,
                                                 scratch[0], scratch[1], scratch[2], st_scratch, ad,
                                                 es._ranks, None, None))
    else:
        rmaj = gt.dtype == torch.float16
        peers = es.__dict__.get("_peer_ptrs")
        if peers is not None:       # the kernel the generation runs: every rank launches it here in lock-step
            st_scratch = slot.state.clone()
            import torch.distributed as dist
            dist.barrier()
            t_grad = timed(lambda: be.rank_grad_xr_adam(R.view(-1), None, 1.0, 0.0, P, world, rank, gt, es._offsets,
                                                        es._order, es._pair_begin, pl, peers, scratch[0], scratch[1],
                                                        scratch[2], st_scratch, ad, es._ranks, None, None))
        else:
            t_grad = timed(lambda: be.rank_grad(R.view(-1) if rmaj else es._returns, None, 1.0, 0.0, P, gt,
                                                es._offsets, es._order, es._pair_begin, pl, n, es._grad, es._ranks,
                                                None, world=world if rmaj else 1))
    # algorithmic bytes per launch on this rank (SURVEY 8d with the table's element size: the engine's
    # table entries are fp16-representable and both kernels stream the exact 16-bit copy)
    bytes_grad = tbytes * n * pl + 28 * n + 8 * P
    bytes_eval = tbytes * n * pl + 4 * n + 4 * B * (dims[0] + dims[-1]) + 4 * P
    flops_eval = 2.0 * n * B * 2 * pl
    # DRAM traffic per launch (dram__bytes_read.sum + dram__bytes_write.sum) from the committed
    # `ncu --set full` capture of exactly these kernels / shapes on one GPU (profiles/ncu_traffic.json)
    traffic = {}
    if args.workload == "north_star" and world == 1:
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        except (OSError, ValueError):
            traffic = {}
    kname_g = ("rank_grad_adam" if world == 1 else "rank_grad_xr_adam" if es.__dict__.get("_peer_ptrs") else
               "rank_grad") + ("_h" if tbytes == 2 else "")
    tr_g = traffic.get(kname_g)
    k_grad = {"kernel": kname_g, "bound": "l2",
              "achieved": bytes_grad / t_grad / 1e6, "peak": peaks["hbm"], "unit": "GB/s",
              "frac": bytes_grad / t_grad / 1e6 / peaks["hbm"],
              "frac_algorithmic_vs_hbm": bytes_grad / t_grad / 1e6 / peaks["hbm"],
              "frac_dram_vs_hbm": (tr_g / t_grad / 1e6 / peaks["hbm"]) if tr_g else None,
              "ms": t_grad, "traffic": tr_g,
              "traffic_source": "committed ncu capture (profiles/ncu_traffic.json)" if tr_g else None,
              "algorithmic_bytes": bytes_grad,
              "note": "algorithmic/HBM > 1 is L2 reuse: the rows of one generation overlap in the table and every CTA "
                      "walks the pairs in offset-sorted order, so the table is fetched from HBM about once per launch "
                      "and the rest of the algorithmic bytes are L2 hits; the binding resource is L2 bandwidth / "
                      "bytes in flight, not HBM"}
    kname_e = "eval_mlp_" + es._precision
    k_eval = {"kernel": kname_e, "bound": "tensor", "achieved": flops_eval / t_eval / 1e9,
              "peak": peaks["tensor_burst"], "peak_kind": "burst (the kernel is timed alone)", "unit": "TFLOP/s",
              "frac": flops_eval / t_eval / 1e9 / peaks["tensor_burst"],
              "frac_of_sustained_peak": flops_eval / t_eval / 1e9 / peaks["tensor"],
              "ms": t_eval, "traffic": traffic.get(kname_e),
              "traffic_source": "committed ncu capture (profiles/ncu_traffic.json)" if traffic.get(kname_e) else None,
              "algorithmic_bytes": bytes_eval, "flops": flops_eval,
              "hbm_frac_of_noise_stream": bytes_eval / t_eval / 1e6 / peaks["hbm"]}
    dominant = k_eval if t_eval >= t_grad else k_grad
    roofline = {k: dominant.get(k) for k in ("bound", "achieved", "peak", "unit", "frac", "traffic")}
    roofline["kernel"] = dominant["kernel"]
    roofline["peak_source"] = peaks["source"] + (", bf16 burst" if dominant is k_eval else "")
    return {"roofline": roofline, "kernels": [k_grad, k_eval]}


_JSON_FD = None


def emit(line):
    """The ONE JSON line, on the process's real stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="north_star", choices=sorted(WORKLOADS))
    ap.add_argument("--table-log2", type=int, default=28)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the short runs of the other BASELINE configs")
    ap.add_argument("--extras", default="", help="comma list of other workloads to run in the same process (any N)")
    ap.add_argument("--eval-precision", default="auto", choices=["auto", "fp32", "f16", "bf16", "bf16s"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed generation's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    # >= 5 warm-up generations on our arm: a generation configuration is captured into a CUDA graph at its third
    # sighting, so the capture (tens of ms) happens in the warm-up, never inside the timed region
    args.warmup = max(args.warmup, 5) if args.impl == "ours" else args.warmup
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    wl = WORKLOADS[args.workload]
    # stdout carries exactly one JSON line: anything a library prints there (NCCL's version
    # banner at communicator creation, ...) is sent to stderr instead
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference_arm(args, wl, rank, world)
        return
    if world != args.gpus:
        if args.gpus > 1:
            raise SystemExit(f"--gpus {args.gpus} needs torchrun with {args.gpus} processes (WORLD_SIZE={world})")
    run_ours(args, wl, rank, world, local_rank)
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
