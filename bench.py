#!/usr/bin/env python
"""bench.py -- GAE + PPO-loss transitions/s on the B200 hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config cfg2_atari_large] [--scaling weak|strong]
                    [--impl reference] [--dump-outputs DIR]

A "step" = one pass of the hot path over one synthetic batch (SURVEY.md §8d): GAE once, then
(epochs x minibatches) fused loss forward+backward covering every transition once per epoch.
`value` = transitions per step (all ranks) / device time with inputs resident in HBM; `e2e` = the same
through `HotPath.run_host` with pinned HOST buffers in and out (H2D + D2H inside the timed region).
N > 1 (torchrun): every rank owns its own slice of environments -- `--scaling weak`: the full config per GPU
(cfg5's sweep); `--scaling strong`: the config's B environments split over the ranks (cfg4: 2048 / 8 = 256 per GPU,
football.py:135,227-228).  The only data-path exchange is the SUM of the float64 statistics table (NVLink peer-memory
mailboxes, or NCCL); at N > 1 the line carries `parity_check`: the exchanged table against the rank-ordered float64 sum,
bit for bit on every rank, and one minibatch's loss / gradients against the oracle evaluated with the global sums.
Beside the headline the line reports `step_trainer_order` (the same work issued as a trainer must issue it: one loss
launch per minibatch, each behind the previous) and `trainer_step` (the drop-in `MultiAgentPPOB200.step` with a small
policy, host sample in, stats out).  `step.launch` says how the timed step was issued (`--launch graph`: one CUDA graph
replay, the default; `--launch plan`: the step's recorded C-ABI calls as plain stream launches) and
`step.ms_per_step_other_launch` the same step issued the other way.  `extra` holds the neighbours of the path, each with its
own roofline: K1 (`srl_batch_gather`), K4b (`srl_ppo_loss_from_logits`), `srl_rnn_chunk_prep`, and the native decode of a
compressed frame leaf into pinned memory (`wire_decode_native`, host GB/s).
`--impl reference` times the reference's OWN functions (`MultiAgentPPO._compute_adv_and_value_target`, `_compute_loss` +
backward, loaded unmodified through oracle/ref_loader.py from oracle/_ref) on the host cores, same config / metric / unit,
per stage; where a GPU is visible it adds the same functions on cuda (the ATen-eager path SRL users have today).
`--dump-outputs DIR` writes what the timed step computed in its last timed step as DIR/<name>.npy (see dump_step_outputs);
the inputs depend only on the arguments, so two builds of the library can be compared output for output.
"""
from __future__ import annotations

import argparse
import dataclasses
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
# bench.py writes nothing into the tree it runs from: no __pycache__/*.pyc next to the modules it imports either
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402

from srl_b200 import synth  # noqa: E402

METRIC = "gae_ppo_loss_transitions_per_sec"
UNIT = "transitions/s"
GAE_BYTES = 19  # SURVEY.md §8(d): 11 B read + 8 B written per scanned row-lane
LOSS_BYTES = {True: 41, False: 37}  # per transition per pass, with / without value clipping
DUMP_BYTES = 64_000_000 - 4096  # --dump-outputs: array data of all files together (the .npy headers fit in the rest)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md, 6.65 TB/s)"


def workload_name(cfg):
    return (f"{cfg.name}: T={cfg.T}, B={cfg.B} envs, A={cfg.A} agents, L={cfg.L} rows, {cfg.epochs} epochs x "
            f"{cfg.minibatches} minibatches, clip_value={cfg.clip_value}, dual_clip={cfg.dual_clip}, "
            f"value_loss={cfg.value_loss}, popart={cfg.popart}")


def hyper_kwargs(cfg):
    return dict(eps_clip=cfg.eps_clip, clip_value=cfg.clip_value, dual_clip=cfg.dual_clip, c_clip=cfg.c_clip,
                value_loss=cfg.value_loss, value_loss_weight=cfg.value_loss_weight,
                entropy_bonus_weight=cfg.entropy_bonus_weight,
                value_loss_config=({"delta": cfg.value_loss_delta} if cfg.value_loss == "huber" else
                                   {"beta": cfg.value_loss_delta} if cfg.value_loss == "smoothl1" else None))


def shard_config(cfg, world, scaling):
    """The slice of the workload one rank owns.  weak: the whole config per GPU; strong: B / world environments."""
    if scaling == "weak" or world == 1:
        return cfg
    if cfg.B % world != 0 or (cfg.B // world) % cfg.minibatches != 0:
        raise SystemExit(f"--scaling strong: B={cfg.B} environments do not split over {world} ranks x {cfg.minibatches} minibatches")
    return dataclasses.replace(cfg, B=cfg.B // world)


# ----------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's own functions (oracle/_ref), else the oracle port
# ----------------------------------------------------------------------------------------------------
def _minibatch_indices(cfg, seed=0):
    """The environment slices of every (epoch, minibatch), as int64 lane-index tensors (the reference has no minibatching:
    its loss runs on `sample[:, idx]`, the definition oracle/ref_trainer.py uses too)."""
    from oracle import ref_math as M
    out = []
    n_env = cfg.B // cfg.minibatches
    for e in range(cfg.epochs):
        if cfg.minibatches == 1:
            out.append([None])
            continue
        env = M.philox_perm_ref(seed, e, cfg.B).astype(np.int64)
        lanes = (env[:, None] * cfg.A + np.arange(cfg.A)[None]).reshape(-1) if cfg.A > 1 else env
        out.append([torch.from_numpy(np.ascontiguousarray(env[j * n_env:(j + 1) * n_env])) for j in range(cfg.minibatches)])
        del lanes
    return out


def reference_functions_run(cfg, steps, warmup, device="cpu", budget_s=None):
    """Times the UNMODIFIED reference: MultiAgentPPO._compute_adv_and_value_target (mappo.py:118-144; gae.py:8-97) once, then
    per (epoch, minibatch) the PopArt update (:263-264), _compute_loss (:146-217), loss.backward() to the three policy
    outputs and the .mean().item() reads of mappo.py:293-299 -- on `device` ('cpu': all host threads; 'cuda': the
    ATen-eager path).  Returns per-stage seconds per step."""
    from oracle import ref_loader
    R = ref_loader.load()
    dev = torch.device(device)
    if dev.type == "cpu":
        torch.set_num_threads(os.cpu_count() or 1)
    s = synth.make_sample_scalars(cfg, seed=0)
    pol = synth.make_policy_outputs(cfg, s, seed=1)
    t = {k: torch.from_numpy(v).float().to(dev) for k, v in s.items()}  # the prefetcher's .float() (api/trainer.py:217)
    head = None
    if cfg.popart:
        head = R.popart.PopArtValueHead(4, 1, beta=0.99999).to(dev)
        head.update(torch.randn(64, 1, device=dev) * 2.0 + 0.5, mask=None)
    fake = ref_loader.FakePolicy(popart_head=head)
    fake.device = str(dev)
    tr = R.mappo.MultiAgentPPO(fake, discount_rate=cfg.gamma, gae_lambda=cfg.lmbda, popart=cfg.popart,
                               bootstrap_steps=cfg.bootstrap_steps, burn_in_steps=cfg.burn_in_steps, **hyper_kwargs(cfg))
    NA = R.namedarray.NamedArray
    sample = R.trainer.SampleBatch(obs=None, on_reset=t["on_reset"], done=t["done"], truncated=t["truncated"],
                                   reward=t["reward"], analyzed_result=NA(value=t["value"], log_probs=t["old_logp"],
                                                                          adv=None, ret=None))
    lo, hi, L = cfg.burn_in_steps, cfg.L - cfg.bootstrap_steps, cfg.L
    idx = _minibatch_indices(cfg)
    idx = [[None if i is None else i.to(dev) for i in row] for row in idx]
    pol_t = {k: torch.from_numpy(v).to(dev) for k, v in pol.items()}  # [E, T, B, (A,) 1]
    sync = (lambda: torch.cuda.synchronize(dev)) if dev.type == "cuda" else (lambda: None)
    rapply = R.namedarray.recursive_apply

    def one():
        sync()
        t0 = time.perf_counter()
        adv, ret = tr._compute_adv_and_value_target(sample, None)
        dims = len(t["value"].shape)
        pad = (0,) * (dims * 2 - 1) + (1,)
        sample.analyzed_result.adv = torch.nn.functional.pad(adv, pad)  # mappo.py:254-257, host mirror included
        sample.analyzed_result.ret = torch.nn.functional.pad(ret, pad)
        _ = sample.analyzed_result.adv.cpu().numpy(), sample.analyzed_result.ret.cpu().numpy()
        sync()
        t1 = time.perf_counter()
        valid = sample[lo:hi]
        mask = 1 - t["on_reset"][lo + 1:hi + 1]
        for e in range(cfg.epochs):
            if cfg.popart:
                fake.update_popart(valid.analyzed_result.ret, mask=mask)
            for j, ii in enumerate(idx[e]):
                take = (lambda x: x) if ii is None else (lambda x: x.index_select(1, ii))
                vmb = valid if ii is None else rapply(valid, take)
                nl, vp, en = (take(pol_t[k][e]).detach().requires_grad_(True) for k in ("new_logp", "v_pred", "entropy"))
                analyzed = R.mappo.SampleAnalyzedResult(old_action_log_probs=vmb.analyzed_result.log_probs,
                                                        new_action_log_probs=nl, state_values=vp, entropy=en)
                loss, res = tr._compute_loss(vmb, analyzed, take(mask))
                loss.backward()
                _ = {f.name: getattr(res, f.name).detach().mean().item() for f in dataclasses.fields(res)
                     if getattr(res, f.name) is not None}  # mappo.py:293-299
        sync()
        t2 = time.perf_counter()
        sample.analyzed_result.adv = sample.analyzed_result.ret = None
        return t1 - t0, t2 - t1

    for _ in range(warmup):
        one()
    gae_s, loss_s = [], []
    t_begin = time.perf_counter()
    for _ in range(steps):
        a, b = one()
        gae_s.append(a)
        loss_s.append(b)
        if budget_s is not None and time.perf_counter() - t_begin > budget_s and len(gae_s) >= 3:
            break
    g, l_ = sum(gae_s) / len(gae_s), sum(loss_s) / len(loss_s)
    return dict(value=cfg.transitions / (g + l_), ms_per_step=(g + l_) * 1e3, steps=len(gae_s),
                cores=torch.get_num_threads() if dev.type == "cpu" else 0, kind="reference",
                stages=dict(gae_ms=g * 1e3, loss_bwd_ms=l_ * 1e3, gae_transitions_per_s=cfg.transitions / g,
                            loss_transitions_per_s=cfg.transitions * cfg.epochs / l_))


def reference_assembly_run(cfg, n_env=64, reps=3):
    """Stage 1 of the reference on the host: recursive_aggregate(np.stack(axis=1)) of per-environment samples
    (base/buffer.py:118-126, base/namedarray.py:598-633), one thread, on a bounded sample of n_env environments."""
    from oracle import ref_loader
    R = ref_loader.load()
    NA = R.namedarray.NamedArray
    rng = np.random.default_rng(0)
    L = cfg.L
    shape = tuple(cfg.obs_shape) if cfg.obs_shape else (64,)
    mk = lambda: R.trainer.SampleBatch(
        obs=NA(x=rng.integers(0, 255, (L,) + shape, dtype=np.uint8)), on_reset=np.zeros((L, 1), dtype=np.uint8),
        done=np.zeros((L, 1), dtype=np.uint8), truncated=np.zeros((L, 1), dtype=np.uint8),
        reward=rng.standard_normal((L, 1)).astype(np.float32),
        analyzed_result=NA(value=rng.standard_normal((L, 1)).astype(np.float32),
                           log_probs=-rng.random((L, 1)).astype(np.float32)))
    samples = [mk() for _ in range(n_env)]
    nbytes = int(R.namedarray.size_bytes(samples[0])) * n_env
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        R.namedarray.recursive_aggregate(list(samples), lambda xs: np.stack(xs, axis=1))
        ts.append(time.perf_counter() - t0)
    best = min(ts)
    return dict(what=f"recursive_aggregate(np.stack, axis=1) of {n_env} samples, L={L}, obs {shape} uint8, 1 thread",
                bytes=nbytes, ms=best * 1e3, gbs=nbytes / best / 1e9, transitions_per_s=n_env * (L - 1) / best)


def port_run(cfg, steps, warmup, budget_s=None):
    """Fallback when oracle/_ref is not staged: the oracle port (oracle/ref_math.py::hot_path_ref) on all host threads."""
    from oracle import ref_math as M  # checker / baseline only
    torch.set_num_threads(os.cpu_count() or 1)
    s = synth.make_sample_scalars(cfg, seed=0)
    pol = synth.make_policy_outputs(cfg, s, seed=1)
    batch = {k: torch.from_numpy(v).float() for k, v in s.items()}
    batch.update({k: torch.from_numpy(v) for k, v in pol.items()})
    hp = M.LossHyper(**hyper_kwargs(cfg))
    pa = M.RunningMeanStdRef((1,)) if cfg.popart else None
    one = lambda: M.hot_path_ref(batch, hp, cfg.gamma, cfg.lmbda, cfg.epochs, cfg.minibatches, seed=0, popart=pa,
                                 bootstrap_steps=cfg.bootstrap_steps, burn_in_steps=cfg.burn_in_steps)
    for _ in range(warmup):
        one()
    times = []
    t_begin = time.perf_counter()
    for _ in range(steps):
        t0 = time.perf_counter()
        one()
        times.append(time.perf_counter() - t0)
        if budget_s is not None and time.perf_counter() - t_begin > budget_s and len(times) >= 3:
            break
    mean = sum(times) / len(times)
    return dict(value=cfg.transitions / mean, ms_per_step=mean * 1e3, steps=len(times), cores=torch.get_num_threads(),
                kind="port", stages=None)


def cpu_reference_run(cfg, steps, warmup, budget_s=None):
    from oracle import ref_loader
    if ref_loader.available():
        return reference_functions_run(cfg, steps, warmup, "cpu", budget_s)
    return port_run(cfg, steps, warmup, budget_s)


def _sample_text(r, cfg):
    if r["kind"] == "reference":
        return (f"{r['steps']} full steps ({r['ms_per_step']:.1f} ms each) of {workload_name(cfg)} on {r['cores']} host threads: the "
                f"UNMODIFIED reference functions MultiAgentPPO._compute_adv_and_value_target + per minibatch _compute_loss, "
                f"backward and the .item() reads (oracle/_ref, torch-CPU, float64 GAE)")
    return (f"{r['steps']} full steps ({r['ms_per_step']:.1f} ms each) of {workload_name(cfg)} on {r['cores']} host threads "
            f"(oracle port of mappo.py:118-217 + gae.py:8-97; oracle/_ref not staged)")


def run_reference_arm(args, cfg, rank, world):
    if rank != 0:
        return  # rank 0 alone runs the CPU arm; the others exit 0 without work
    cfg = shard_config(cfg, args.gpus, args.scaling)  # the per-GPU slice of our arm, on the host cores
    r = cpu_reference_run(cfg, args.steps, args.warmup)
    extra = {}
    try:
        extra["assembly"] = reference_assembly_run(cfg)
    except Exception as e:  # noqa: BLE001
        extra["assembly"] = dict(error=str(e))
    if torch.cuda.is_available() and r["kind"] == "reference":
        try:  # "what SRL users get today on this GPU": the same unmodified functions, tensors on cuda (SURVEY.md §2.2)
            g = reference_functions_run(cfg, min(args.steps, 20), 2, "cuda:0")
            extra["reference_gpu_eager"] = dict(value=g["value"], unit=UNIT, ms_per_step=g["ms_per_step"], stages=g["stages"],
                                                what="the same unmodified reference functions with the batch on cuda:0 "
                                                     "(ATen eager kernels, python scan over T), inputs resident in HBM")
        except Exception as e:  # noqa: BLE001
            extra["reference_gpu_eager"] = dict(error=str(e))
    line = dict(metric=METRIC, value=r["value"], unit=UNIT, n_gpus=args.gpus, steps=r["steps"], warmup=args.warmup,
                ms_per_step=r["ms_per_step"], higher_is_better=True, scaling=args.scaling, vs_baseline=None, dtype="f32",
                data="synthetic", impl="reference", config=dict(workload=workload_name(cfg)),
                cpu_baseline=dict(value=r["value"], unit=UNIT, cores=r["cores"], kind=r["kind"], sample=_sample_text(r, cfg),
                                  stages=r["stages"]),
                e2e=dict(value=r["value"], unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0, **extra)
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------
# host placement
# ----------------------------------------------------------------------------------------------------
def bind_to_gpu_numa(device_index, local_rank=0, local_world=1):
    """Runs this process on ITS OWN share of the CPUs NVML reports as local to the GPU (the pinned staging buffers are then
    allocated on that NUMA node).  With several ranks whose GPUs report the same CPU set (SCALE_r01: all eight GPUs of the
    box list CPUs 0-31) every rank takes a disjoint slice of it instead of all ranks piling onto the same cores.
    Returns the previous affinity (restored for the CPU arm)."""
    try:
        import pynvml
        before = os.sched_getaffinity(0)
        pynvml.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(device_index).uuid)
        h = pynvml.nvmlDeviceGetHandleByUUID((uuid if uuid.startswith("GPU-") else "GPU-" + uuid).encode())
        words = (max(before) + 64) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = sorted(i for i in before if (mask[i // 64] >> (i % 64)) & 1)
        if cpus and local_world > 1:
            per = max(1, len(cpus) // local_world)
            mine = cpus[local_rank * per:(local_rank + 1) * per] or cpus
            cpus = mine
        if cpus:
            os.sched_setaffinity(0, set(cpus))
        return before
    except Exception:
        return None


# ----------------------------------------------------------------------------------------------------
# clocks: NVML polled in-process (a thread, ~1 kHz) around the timed regions
# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    _REASONS = (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40))

    def __init__(self, device_index, period_s=0.001):
        self.rows, self.ok, self._stop = [], False, False
        try:
            import pynvml
            pynvml.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(device_index).uuid)
            self.h = pynvml.nvmlDeviceGetHandleByUUID((uuid if uuid.startswith("GPU-") else "GPU-" + uuid).encode())
            self.nv = pynvml
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.period = period_s
            self.ok = True
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.ok = False

    def _pump(self):
        nv = self.nv
        while not self._stop:
            try:
                c = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((time.perf_counter(), c, r))
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self, windows=None):
        """windows: [(t0, t1)] perf_counter intervals of the timed regions; samples outside them are dropped."""
        if not self.ok:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvml unavailable"], samples=0)
        self._stop = True
        self.thread.join(timeout=1.0)
        rows = [r for r in self.rows if windows is None or any(a <= r[0] <= b for a, b in windows)]
        sm = [c for _, c, _ in rows]
        reasons = sorted({name for _, _, r in rows for name, bit in self._REASONS if r & bit})
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_min_mhz=min(sm) if sm else None,
                    sm_max_mhz=self.max_sm, reasons=reasons, samples=len(sm), sampler="pynvml in-process, 1 ms period, "
                    "samples inside the timed regions only")


# ----------------------------------------------------------------------------------------------------
# a small policy for the trainer_step line: what MultiAgentPPO calls on a policy (SURVEY.md §8b), a two-layer MLP
# ----------------------------------------------------------------------------------------------------
class _BenchPolicy:

    def __init__(self, obs_dim, num_actions, device, hidden=64):
        import torch.nn as nn
        torch.manual_seed(0)
        self.net = nn.Sequential(nn.Linear(obs_dim, hidden), nn.Tanh(), nn.Linear(hidden, num_actions + 1)).to(device)
        self.device, self._version, self.k = device, -1, num_actions
        self.denormalize_value_during_rollout = False

    version = property(lambda self: self._version)

    def inc_version(self):
        self._version += 1

    def parameters(self):
        return self.net.parameters()

    def train_mode(self):
        self.net.train()

    def analyze(self, sample, target="ppo", burn_in_steps=0, **kw):
        from types import SimpleNamespace
        out = self.net(sample.obs.vec[burn_in_steps:])
        dist = torch.distributions.Categorical(logits=out[..., :self.k])
        action = sample.action.x[burn_in_steps:, ..., 0].long()
        return SimpleNamespace(old_action_log_probs=sample.analyzed_result.log_probs[burn_in_steps:],
                               new_action_log_probs=dist.log_prob(action).unsqueeze(-1), state_values=out[..., self.k:],
                               entropy=dist.entropy().unsqueeze(-1))


def trainer_step_run(cfg, dev, steps=5):
    """The drop-in `MultiAgentPPOB200.step` end to end: host numpy sample in (scalar leaves of the workload + a 16-float
    observation vector per transition), prefetch on, policy forward / backward / optimizer in PyTorch, stats out."""
    from srl_b200 import api
    from srl_b200.namedarray import NamedArray, size_bytes
    from srl_b200.trainer import MultiAgentPPOB200
    if cfg.A != 1:
        return None
    obs_dim, K = 16, int(cfg.num_actions[0])
    rng = np.random.default_rng(5)
    pol = _BenchPolicy(obs_dim, K, f"cuda:{dev.index}")
    hk = hyper_kwargs(cfg)
    tr = MultiAgentPPOB200(pol, discount_rate=cfg.gamma, gae_lambda=cfg.lmbda, bootstrap_steps=cfg.bootstrap_steps,
                           burn_in_steps=cfg.burn_in_steps, ppo_epochs=cfg.epochs, num_minibatches=cfg.minibatches,
                           popart=False, optimizer="adam", optimizer_config=dict(lr=1e-4),
                           **{k: v for k, v in hk.items() if v is not None})

    def sample(seed):
        s = synth.make_sample_scalars(cfg, seed)
        lead = s["value"].shape[:-1]
        return api.SampleBatch(obs=NamedArray(vec=rng.standard_normal(lead + (obs_dim,)).astype(np.float32)),
                               on_reset=s["on_reset"], done=s["done"], truncated=s["truncated"],
                               action=NamedArray(x=rng.integers(0, K, lead + (1,)).astype(np.uint8)), reward=s["reward"],
                               analyzed_result=api.AnalyzedResult(value=s["value"], log_probs=s["old_logp"]))

    samples = [sample(100 + i) for i in range(3)]
    host_bytes = size_bytes(samples[0])
    for i in range(3):  # the first call primes the prefetcher; two warm-up steps
        tr.step(samples[i % 3])
    torch.cuda.synchronize()
    h2d0 = tr.h2d_bytes
    t0 = time.perf_counter()
    for i in range(steps):
        tr.step(samples[i % 3])
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / steps
    return dict(ms_per_step=dt * 1e3, value=cfg.transitions / dt, unit=UNIT, steps=steps,
                h2d_bytes_per_step=(tr.h2d_bytes - h2d0) // steps, host_sample_bytes=int(host_bytes),
                what=f"MultiAgentPPOB200.step: host numpy sample (scalars + a {obs_dim}-float observation) -> pinned H2D in the "
                     f"leaves' own dtypes -> per minibatch: K5 gather, a 2-layer MLP policy (PyTorch), K4, backward, Adam "
                     f"-> stats; {cfg.epochs} epochs x {cfg.minibatches} minibatches; wall clock per call, prefetch on")


# ----------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------
def event_ms(pairs):
    return [a.elapsed_time(b) for a, b in pairs]


def parity_check(hp, cfg, pol_np, sample_np, rank, world, dist, dev):
    """Before anything is timed: one eager step, then (1) on several ranks, the exchanged statistics table against the
    float64 sum of the ranks' local tables added in rank order -- bit for bit, on every rank; (2) the loss scalars and the
    gradients of minibatch (0, 0) against the oracle (oracle/ref_math.py::ppo_loss_ref) on this rank's data, normalised with
    the GLOBAL sums (the reference's semantics across ranks, utils.py:58-61), within 1e-5."""
    from oracle import ref_math as M  # the checker
    out = dict(ranks=world)
    hp.ensure_table()  # in the fused-statistics mode nothing on the step's path produces the table: made here, for the check
    if world > 1:
        tables = [torch.empty_like(hp.local_stats) for _ in range(world)]
        dist.all_gather(tables, hp.local_stats.contiguous())
        expect = torch.zeros_like(hp.local_stats)
        for t in tables:
            expect += t
        same = bool(torch.equal(expect, hp.global_stats))
        flag = torch.tensor([1 if same else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        out["stats_table_bit_exact_on_every_rank"] = bool(flag.item())
    e, j = hp.epochs - 1, 0  # the last epoch: with PopArt its statistics are the ones still in hp.popart_ms
    T, n = hp.T, hp.n_mb
    lo, hi = hp.row_lo, hp.row_hi
    idx = hp.minibatch_lanes(e, j)
    ii = torch.arange(hp.N) if idx is None else idx.cpu().long()
    flat = lambda x: torch.from_numpy(np.ascontiguousarray(x.reshape(x.shape[0], -1)))
    take = lambda x: x.index_select(1, ii).unsqueeze(-1)
    t = {k: flat(v).float() for k, v in sample_np.items()}
    adv, ret = hp.adv.cpu(), hp.ret.cpu()
    mask = 1 - t["on_reset"][lo + 1:hi + 1]
    nl, vp, en = (hp_t.cpu().unsqueeze(-1) for hp_t in pol_np)
    row = hp.stats_row(e, j)
    g = hp.global_stats[row].cpu()
    pa = None
    if cfg.popart:  # an oracle RunningMeanStd whose mean_std() is the device's current (mu, sigma)
        ms = hp.popart_ms.cpu()
        pa = M.RunningMeanStdRef((1,))
        pa.debias = torch.ones(1, dtype=torch.float64)
        pa.mean = ms[0:1].clone()
        pa.mean_sq = (ms[1:2] ** 2 + ms[0:1] ** 2).clone()
    ref = M.ppo_loss_ref(nl, take(t["old_logp"][lo:hi]), vp, take(t["value"][lo:hi]), take(ret[lo:hi]), take(adv[lo:hi]), en,
                         take(mask), M.LossHyper(**hyper_kwargs(cfg)), popart=pa,
                         global_sums=(g[0].clone(), g[1].clone(), g[2].clone()))
    got = hp.out[e * hp.minibatches + j].cpu()
    m = float(got[9])
    rel = lambda a, b: float(abs(a - b) / max(1.0, abs(b)))
    out["loss_err"] = rel(float(got[0]), float(ref["loss"]))
    # Elements that sit ON a decision boundary of the loss are excused and counted: the clipped surrogate switches between
    # "full gradient" and "no gradient" where ratio == 1 +- eps, and torch's CPU exp and the device's expf differ by an ulp
    # there (one such element in 4 M at cfg4: ratio = 1.2000001669 on the host, 1.2000000477 = float(1.2) on the device).
    # Likewise the value clamp at |v - v_old| == eps.  Everything else must agree within 1e-5.
    hk = hyper_kwargs(cfg)
    ratio = (nl - take(t["old_logp"][lo:hi])).double().exp()[..., 0]
    eps_c = float(hk["eps_clip"])
    near_clip = ((ratio - (1 - eps_c)).abs() <= 4e-7) | ((ratio - (1 + eps_c)).abs() <= 4e-7)
    dvv = (vp - take(t["value"][lo:hi])).double().abs()[..., 0]
    near_vclip = (dvv - eps_c).abs() <= 4e-7
    errs, flips = [], 0
    for q, (k, excuse) in enumerate((("g_logp", near_clip), ("g_value", near_vclip), ("g_entropy", None))):
        a = hp.grads[e][j][q].cpu().double() * m
        b = ref[k][..., 0].double() * m
        err = (a - b).abs() / b.abs().clamp(min=1.0)
        if excuse is not None:
            flips += int(((err > 1e-5) & excuse).sum())
            err = torch.where(excuse, torch.zeros_like(err), err)
        errs.append(float(err.max()))
        if errs[-1] > 1e-5:  # say where, so that a failure can be read off the line
            w = int(err.argmax())
            r_, c_ = divmod(w, err.shape[1])
            out[f"worst_{k}"] = dict(row=r_, lane=c_, got=float(a[r_, c_]), ref=float(b[r_, c_]), bad=int((err > 1e-5).sum()),
                                     mask=float(take(mask)[r_, c_, 0]), adv=float(take(adv[lo:hi])[r_, c_, 0]),
                                     new_logp=float(nl[r_, c_, 0]), old_logp=float(take(t["old_logp"][lo:hi])[r_, c_, 0]),
                                     v_pred=float(vp[r_, c_, 0]), old_value=float(take(t["value"][lo:hi])[r_, c_, 0]),
                                     ret=float(take(ret[lo:hi])[r_, c_, 0]))
    out["boundary_elements_excused"] = flips
    out["grad_err"] = max(errs)
    out["grad_errs"] = dict(zip(("g_logp", "g_value", "g_entropy"), errs))
    ok = out["loss_err"] <= 1e-5 and out["grad_err"] <= 1e-5 and out.get("stats_table_bit_exact_on_every_rank", True)
    flag = torch.tensor([1 if ok else 0], device=dev)
    if world > 1:
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    out["ok"] = bool(flag.item())
    out["what"] = ("eager step before the timed region: exchanged stats table == rank-ordered float64 sum (bit for bit, all ranks); "
                   "the last epoch's first minibatch: loss and gradients vs oracle.ppo_loss_ref with the global sums, |x-ref| <= 1e-5*max(1,|ref|), "
                   "gradients on the g*M scale; min over ranks")
    return out


def dump_step_outputs(out_dir, hp, shard):
    """--dump-outputs: what one step hands its caller -- adv and ret [L, N] float32, the loss / statistics rows
    [E*M, 16] float64 and the gradients w.r.t. new_logp, v_pred and entropy [E, M, T, n] float32 -- as
    out_dir/<name>.npy.  Where they hold more than DUMP_BYTES, the loss table stays whole and every other array keeps the
    same fraction k / n of its n elements, flattened: the array is cut into k stretches of n // k or n // k + 1 elements
    that cover all of it, and one element of each is kept, at an offset drawn from a fixed seed, so the same arguments give
    the same sample.  `shard` says whose step it is (with several GPUs: rank 0's slice of the workload)."""
    arrays = dict(adv=hp.adv, ret=hp.ret, loss_out=hp.out, g_logp=hp.grads_all[:, :, 0], g_value=hp.grads_all[:, :, 1],
                  g_entropy=hp.grads_all[:, :, 2])
    nbytes = lambda t: t.numel() * t.element_size()
    frac = min(1.0, (DUMP_BYTES - nbytes(hp.out)) / sum(nbytes(t) for k, t in arrays.items() if k != "loss_out"))
    os.makedirs(out_dir, exist_ok=True)
    info = {}
    for seed, (name, t) in enumerate(arrays.items()):
        x = t.contiguous().view(-1)
        n = x.numel()
        k = n if frac == 1.0 or name == "loss_out" else max(1, int(n * frac))
        if k < n:  # k strata [lo, hi) that tile the whole array; one element of each
            lo = np.arange(k, dtype=np.int64) * n // k
            hi = np.arange(1, k + 1, dtype=np.int64) * n // k
            idx = lo + np.random.default_rng(seed).integers(0, hi - lo)
            x = x.index_select(0, torch.from_numpy(idx).to(x.device))
        else:
            x = x.view(t.shape)
        np.save(os.path.join(out_dir, f"{name}.npy"), x.cpu().numpy())
        info[name] = dict(shape=list(t.shape), dtype=str(t.dtype).replace("torch.", ""),
                          stored="all" if k == n else f"{k} of {n} elements")
    return dict(dir=os.path.abspath(out_dir), shard=shard, arrays=info)


def run_ours(args, cfg_full, rank, world, local_rank):
    import torch.distributed as dist
    from srl_b200 import ops
    from srl_b200.hotpath import HotPath

    cfg = shard_config(cfg_full, world, args.scaling)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    affinity_before = bind_to_gpu_numa(local_rank, local_rank, int(os.environ.get("LOCAL_WORLD_SIZE", world)))
    pg = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD
    ops._lib.load_library()  # fail loudly if the CUDA library is missing

    # ---- synthetic batch for this rank's slice of environments -------------------------------------
    s = synth.make_sample_scalars(cfg, seed=1000 * rank)
    pol = synth.make_policy_outputs(cfg, s, seed=1000 * rank + 1)
    E, Mb, T, N = cfg.epochs, cfg.minibatches, cfg.T, cfg.N
    hp = HotPath(cfg.L, cfg.B, cfg.A, gamma=cfg.gamma, lmbda=cfg.lmbda, hyper=ops.LossHyper(**hyper_kwargs(cfg)),
                 bootstrap_steps=cfg.bootstrap_steps, burn_in_steps=cfg.burn_in_steps, epochs=E, minibatches=Mb, seed=0,
                 popart=cfg.popart, device=dev, process_group=pg, fuse_gather=not args.explicit_gather,
                 graph_branches=args.branches, shuffle_block=args.shuffle_block, use_pack=not args.no_pack,
                 batch_losses=not args.no_batch, stats_exchange=args.exchange, fuse_stats=not args.no_fuse_stats,
                 exchange_timeout_s=30.0)
    n = hp.n_mb
    pinned = {k: torch.from_numpy(np.ascontiguousarray(v.reshape(cfg.L, N))).pin_memory() for k, v in s.items()}
    hp.load_sample(pinned)
    # policy outputs as the policy would emit them: one contiguous [T, n] block per (epoch, minibatch)
    blk = args.shuffle_block
    perm = [ops.philox_perm(0, e, cfg.B // blk, cfg.A * blk).long() if Mb > 1 else None for e in range(E)]
    pol_all = torch.empty((E, Mb, 3, T, n), dtype=torch.float32, device=dev)
    for e in range(E):
        for q, k in enumerate(("new_logp", "v_pred", "entropy")):
            full = torch.from_numpy(pol[k][e].reshape(T, N)).to(dev)
            for j in range(Mb):
                pol_all[e, j, q] = full if Mb == 1 else full.index_select(1, perm[e][j * n:(j + 1) * n])
    pol_dev = [[tuple(pol_all[e, j, q] for q in range(3)) for j in range(Mb)] for e in range(E)]
    pol_host = pol_all.cpu().pin_memory()
    out_host = dict(adv=torch.empty((cfg.L, N), dtype=torch.float32).pin_memory(),
                    ret=torch.empty((cfg.L, N), dtype=torch.float32).pin_memory(),
                    out=torch.empty((E * Mb, 16), dtype=torch.float64).pin_memory())

    # ---- parity first: an eager step checked against the oracle (and, on several ranks, the exchange) --
    hp.run_device(pol_dev, use_graph=False)
    hp.step_count = 0
    torch.cuda.synchronize()
    hp.check_exchange()
    pc = None
    if not args.no_parity_check:
        pc = parity_check(hp, cfg, pol_dev[E - 1][0], s, rank, world, dist, dev)

    # L2 flush between timed iterations: write a 256 MiB buffer (> 126 MB L2), then READ a second one.  The write
    # alone leaves the L2 full of dirty lines whose write-back the timed kernels would then pay for (it showed as
    # ~20 us on a 65 us kernel); the read pass evicts them and leaves clean lines, so the step starts cold.
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    flush_rd = torch.zeros(64 << 20, dtype=torch.int32, device=dev)  # 256 MiB

    def flush_l2():
        flush.zero_()
        flush_rd.max()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # Several ranks: the flush kernels of two GPUs do not end at the same moment (a few microseconds apart), and the step's
    # statistics exchange makes the early rank wait for the late one -- inside the timed region.  An UNTIMED device-side
    # rendezvous (the peer-memory exchange of one number) between the flush and the start event lines the ranks up, so
    # that what is timed is the step, not the flush skew.  --no-align switches it off (A/B).
    align = None
    if world > 1 and hp.peer is not None and not args.no_align:
        align_in = torch.ones(1, dtype=torch.float64, device=dev)
        align_out = torch.zeros(1, dtype=torch.float64, device=dev)
        align = lambda: hp.peer.allreduce_sum(align_in, align_out)

    def timed_steps(k, fn, flush_first=True):
        pairs = []
        for _ in range(k):
            if flush_first:
                flush_l2()
            if align is not None:
                align()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            pairs.append((a, b))
        torch.cuda.synchronize()
        return event_ms(pairs)

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    windows = []
    launch = args.launch if hp.plan_supported() else "graph"
    steps_by_launch = {"graph": lambda: hp.run_device(pol_dev, use_graph=True),
                       "plan": lambda: hp.run_device(pol_dev, plan=True)}
    step = steps_by_launch[launch]
    for _ in range(max(args.warmup, 3)):
        flush_l2()
        step()
    barrier()
    w0 = time.perf_counter()
    ms = timed_steps(args.steps, step)
    barrier()
    windows.append((w0, time.perf_counter()))
    # before anything else runs on the step's buffers
    dumped = None
    if args.dump_outputs and rank == 0:
        dumped = dump_step_outputs(args.dump_outputs, hp, "the whole workload on one GPU" if world == 1 else
                                   f"rank 0 of {world}: {workload_name(cfg)} ({args.scaling} scaling), inputs seeded for rank 0")
    ms_per_step = max_over_ranks(sum(ms)) / args.steps
    total_transitions = cfg.transitions * world
    value = total_transitions / (ms_per_step * 1e-3)

    # ---- warm-L2 variant (no flush), informational ------------------------------------------------
    ms_warm = timed_steps(min(args.steps, 200), step, flush_first=False)
    # ---- the other way of issuing the same launches (CUDA graph <-> recorded plan of stream launches), informational
    other = "plan" if launch == "graph" else "graph"
    ms_other = None
    if hp.plan_supported():
        for _ in range(3):
            flush_l2()
            steps_by_launch[other]()
        ms_other = statistics.mean(timed_steps(min(args.steps, 300), steps_by_launch[other]))

    # ---- the same work in the order a trainer must issue it: one loss launch per minibatch, each behind the previous
    # (minibatch j+1's policy outputs do not exist before the optimizer step on minibatch j) -- one stream, a linear graph
    trainer_order = None
    if Mb > 1 or E > 1:
        for _ in range(3):
            flush_l2()
            hp.run_trainer_order(pol_dev)
        barrier()
        w0 = time.perf_counter()
        ms_to = timed_steps(min(args.steps, 500), lambda: hp.run_trainer_order(pol_dev))
        barrier()
        windows.append((w0, time.perf_counter()))
        to_ms = max_over_ranks(sum(ms_to)) / len(ms_to)
        g_chain = hp.loss_chain_graph(pol_dev)
        chain_ms = statistics.mean(timed_steps(50, g_chain.replay)) / (E * Mb)
        trainer_order = dict(ms_per_step=to_ms, value=total_transitions / (to_ms * 1e-3), unit=UNIT,
                             loss_launches_per_step=E * Mb, us_per_dependent_loss_launch=chain_ms * 1e3,
                             what="GAE once, then one loss launch per (epoch, minibatch), each waiting for the one before it, "
                                  "one stream (a linear CUDA graph); CUDA events, L2 flushed per step")

    # ---- e2e: pinned host buffers in / out through HotPath.run_host -------------------------------
    e2e_steps = max(3, min(args.steps, args.e2e_steps))

    def e2e_run(**kw):
        for _ in range(3):
            hp.run_host(pinned, pol_host, out_host, **kw)
        barrier()
        wall, nb = [], None
        w0_ = time.perf_counter()
        for _ in range(e2e_steps):
            flush_l2()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            nb = hp.run_host(pinned, pol_host, out_host, **kw)
            wall.append(time.perf_counter() - t0)
        windows.append((w0_, time.perf_counter()))
        return max_over_ranks(sum(wall)) / e2e_steps, nb

    e2e_s, nbytes = e2e_run()
    e2e_res_s, nbytes_res = e2e_run(pol_device=pol_all)  # policy outputs born on the GPU, as in production
    e2e_value = total_transitions / e2e_s

    # ---- per-kernel durations for the roofline: CUDA events around graphs of one kernel kind ------
    peak, peak_src = peaks()
    k_reps = 20

    def graph_of(fn):
        s_ = torch.cuda.Stream()
        s_.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s_):
            fn()
        torch.cuda.current_stream().wait_stream(s_)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            fn()
        return g

    pg_saved, hp.pg = hp.pg, None
    # the loss launches exactly as the step issues them (one batched launch, one per epoch with PopArt, or one per
    # minibatch with --no-batch); PopArt's tiny update kernels ride along in the per-epoch case
    loss_launches = (E if cfg.popart else -(-(E * Mb) // 32)) if hp._immediate else E * Mb
    # stand-alone there is no kernel ahead to overlap with: launched without the programmatic attribute
    pdl_was = ops.set_pdl(False)
    g_loss = graph_of(lambda: hp._run_losses(pol_dev))
    lf = hp.leaf
    pack_kw = dict(old_logp=lf["old_logp"], pack=hp.pack, lane_aos=hp.lane_aos) if hp.pack is not None else {}
    if hp._perm_fused:  # the scan as the step issues it: with the permutations (and the minibatch shares) computed on the side
        saved_count, hp.step_count = hp.step_count, 0
        pack_kw["perm_job"] = hp.perm_job(with_part=hp.lane_aos is not None)
        hp.step_count = saved_count
    g_gae = graph_of(lambda: ops.gae_scan(lf["reward"], lf["value"], lf["done"], lf["truncated"], lf["on_reset"], cfg.gamma,
                                          cfg.lmbda, row_lo=hp.row_lo, row_hi=hp.row_hi,
                                          popart_mean_std=hp.popart_mean_std(), adv=hp.adv, ret=hp.ret,
                                          lane_part=hp.lane_part, **pack_kw))
    ops.set_pdl(pdl_was)
    hp.pg = pg_saved
    w0 = time.perf_counter()
    loss_ms = statistics.mean(timed_steps(k_reps, g_loss.replay)) / loss_launches
    gae_ms = statistics.mean(timed_steps(k_reps, g_gae.replay))
    windows.append((w0, time.perf_counter()))
    loss_ms_warm = statistics.mean(timed_steps(k_reps, g_loss.replay, flush_first=False)) / loss_launches
    gae_ms_warm = statistics.mean(timed_steps(k_reps, g_gae.replay, flush_first=False))
    loss_bytes = LOSS_BYTES[bool(cfg.clip_value)] * T * n * (E * Mb // loss_launches)
    gae_bytes = GAE_BYTES * (cfg.L - 1) * N
    kern = {
        "ppo_loss_kernel": dict(launches_per_step=loss_launches, ms_per_launch=loss_ms, bytes_per_launch=loss_bytes,
                                gbs=loss_bytes / loss_ms / 1e6, gbs_l2_warm=loss_bytes / loss_ms_warm / 1e6,
                                step_share=loss_ms * loss_launches / ms_per_step),
        "gae_scan_kernel": dict(launches_per_step=1, ms_per_launch=gae_ms, bytes_per_launch=gae_bytes,
                                gbs=gae_bytes / gae_ms / 1e6, gbs_l2_warm=gae_bytes / gae_ms_warm / 1e6,
                                step_share=gae_ms / ms_per_step),
    }
    dom = max(kern, key=lambda k_: kern[k_]["step_share"])
    traffic = None  # DRAM bytes per launch of the dominant kernel from the committed ncu capture of this workload
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic = json.load(f).get(cfg.name, {}).get(dom)
    except Exception:
        pass
    roofline = dict(bound="hbm", kernel=dom, achieved=kern[dom]["gbs"], peak=peak, unit="GB/s",
                    frac=kern[dom]["gbs"] / peak, traffic=traffic, peak_source=peak_src,
                    algorithmic_bytes_per_launch=kern[dom]["bytes_per_launch"],
                    ms_per_launch=kern[dom]["ms_per_launch"])
    step_bytes = gae_bytes + LOSS_BYTES[bool(cfg.clip_value)] * T * N * E

    # ---- the neighbours of the path, each with its own roofline (rank 0, N = 1) --------------------
    extra = None
    if rank == 0 and world == 1 and not args.no_extras:
        extra = {}
        try:
            extra.update(extras_run(cfg_full, dev, peak, timed_steps))
        except Exception as e:  # noqa: BLE001
            extra["error"] = f"{type(e).__name__}: {e}"
    clocks = sampler.stop(windows) if sampler else None

    trainer_line = None
    if rank == 0 and world == 1 and not args.no_extras:
        try:
            del flush, flush_rd
            torch.cuda.empty_cache()
            trainer_line = trainer_step_run(cfg, dev)
        except Exception as e:  # noqa: BLE001
            trainer_line = dict(error=f"{type(e).__name__}: {e}")

    # ---- CPU baseline beside it (rank 0, N = 1 only) ----------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        if affinity_before:
            os.sched_setaffinity(0, affinity_before)  # the CPU arm gets every host core
        r = cpu_reference_run(cfg, steps=200, warmup=2, budget_s=args.cpu_budget_s)
        cpu = dict(value=r["value"], unit=UNIT, cores=r["cores"], kind=r["kind"], sample=_sample_text(r, cfg),
                   stages=r["stages"])
    if rank == 0:
        line = dict(
            metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3),
            ms_per_step=ms_per_step, higher_is_better=True, scaling=args.scaling, vs_baseline=None, dtype="f32",
            data="synthetic",
            config=dict(workload=workload_name(cfg_full), per_gpu=workload_name(cfg) if world > 1 else "the whole workload",
                        transitions_per_step_per_gpu=cfg.transitions,
                        l2="flushed between timed iterations (256 MiB device write, then 256 MiB device read, before each step; working set "
                           f"{step_bytes / 1e6:.0f} MB algorithmic)",
                        timing="CUDA events per step on the launch stream, sum over steps, max over ranks" +
                        ("; the ranks meet in an untimed device-side rendezvous between the L2 flush and each start event "
                         "(flush skew between GPUs is not part of a step)" if align is not None else ""),
                        launch="one CUDA graph per step" + ("" if world == 1 else (
                            f" ({hp.exchange_kind} exchange of the float64 stats table captured inside)"
                            if hp._graph_a is None else f" split in two around the {hp.exchange_kind} exchange of the float64 stats table")),
                        loss_launch=("batched: %d launch(es) per step covering %d minibatches each (every minibatch's policy outputs "
                                     "given up front; see step_trainer_order for the dependency order of a real trainer)" %
                                     (loss_launches, E * Mb // loss_launches)) if hp._immediate else "one launch per minibatch",
                        sample_side="K2 pack (float4 per transition, row pairs interleaved)" if hp.pack is not None else "separate leaves",
                        minibatch_stats=("added inside the loss kernel from K2's per-lane sums (table on a side branch)" +
                                         ("; the ranks' sums exchanged inside the loss kernel over NVLink peer memory"
                                          if hp.peer_loss is not None else ""))
                        if hp.fuse_stats else "srl_group_stats table between K2 and the loss",
                        minibatch_gather=("fused into the loss loads (lane_idx)" if hp.fuse_gather else "explicit K5 gather") +
                        f", Philox permutation of {hp.shuffle_block}-environment blocks",
                        graph_branches=hp.graph_branches,
                        programmatic_dependent_launch=bool(ops.pdl_enabled()),
                        kernel_timing="kernels[*]: each kernel alone in a graph, launched without the programmatic "
                                      "attribute, CUDA events, L2 flushed"),
            clocks=clocks, parity_check=pc,
            e2e=dict(value=e2e_value, unit=UNIT, h2d_bytes_per_step=nbytes["h2d_bytes"],
                     d2h_bytes_per_step=nbytes["d2h_bytes"], ms_per_step=e2e_s * 1e3, steps=e2e_steps,
                     what="HotPath.run_host: pinned host sample + policy outputs of every minibatch -> H2D -> step -> D2H of adv, "
                          "ret (the reference's host mirror, mappo.py:254-257) and the loss/stats table; gradients stay in HBM for "
                          "the policy's backward; one CUDA graph; wall clock incl. final stream sync",
                     policy_outputs_resident=dict(
                         value=total_transitions / e2e_res_s, ms_per_step=e2e_res_s * 1e3,
                         h2d_bytes_per_step=nbytes_res["h2d_bytes"], d2h_bytes_per_step=nbytes_res["d2h_bytes"],
                         what="the same call with the policy outputs already in HBM (where the policy network produces them in "
                              "production): only the sample crosses PCIe")),
            gpu_launches=hp.count_launches() * args.steps,
            gpu_launches_per_step=hp.count_launches(),
            roofline=roofline, kernels=kern,
            step=dict(algorithmic_bytes=step_bytes, gbs=step_bytes / ms_per_step / 1e6,
                      frac_of_peak=step_bytes / ms_per_step / 1e6 / peak,
                      launch=launch + (": one CUDA graph replay per step" if launch == "graph" else
                                       ": the step's recorded C-ABI calls issued as plain stream launches (HotPath.run_device(plan=True))"),
                      ms_per_step_other_launch={other: ms_other},
                      ms_per_step_l2_warm=statistics.mean(ms_warm),
                      value_l2_warm=total_transitions / (statistics.mean(ms_warm) * 1e-3)),
            step_trainer_order=trainer_order, trainer_step=trainer_line, extra=extra,
            cpu_baseline=cpu)
        if dumped is not None:
            line["dump_outputs"] = dumped
        print(json.dumps(line), flush=True)
    align = None
    del hp, g_loss, g_gae  # CUDA graphs and peer mailboxes go before the process group does
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def extras_run(cfg, dev, peak, timed_steps):
    """The callers either side of the path (SURVEY.md §8 rows A1 and A6), each against the same HBM roofline."""
    from srl_b200 import ops
    out = {}
    # ---- K1: the batch gather on frame-shaped rows: [L, slots, row] -> [L, B, row] through an index vector ------------
    L, slots, row = 32, 512, int(np.prod(cfg.obs_shape)) if cfg.obs_shape else 4096
    src = torch.randint(0, 255, (L, slots, row), dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    idx = torch.randperm(slots, device=dev).to(torch.int32)
    fn = lambda: ops.batch_gather([(src, dst)], idx)
    fn()
    ms = statistics.mean(timed_steps(10, fn))
    nbytes = 2 * src.numel()
    out["batch_gather_k1"] = dict(ms_per_launch=ms, bytes_per_launch=nbytes, what=f"srl_batch_gather of uint8 rows of {row} B, "
                                  f"[{L}, {slots}] items through a random permutation (read + write)",
                                  roofline=dict(bound="hbm", achieved=nbytes / ms / 1e6, peak=peak, unit="GB/s",
                                                frac=nbytes / ms / 1e6 / peak))
    del src, dst
    # ---- K4b: the loss from the actor head's logits (Categorical log-prob / entropy fused in) -----------------------
    T, N = cfg.T, min(cfg.N, 4096)
    c1 = dataclasses.replace(cfg, B=N // cfg.A, epochs=1, minibatches=1)
    s = synth.make_sample_scalars(c1, 7)
    d = {k: torch.from_numpy(np.ascontiguousarray(v.reshape(c1.L, -1))).to(dev) for k, v in s.items()}
    adv, ret, part = ops.gae_scan(d["reward"], d["value"], d["done"], d["truncated"], d["on_reset"], cfg.gamma, cfg.lmbda,
                                  row_lo=0, row_hi=T)
    stats = ops.group_stats(part, groups=1, per=c1.N)[0]
    logits_np, act_np = synth.make_logits_actions(c1, (T, c1.N), 3)
    logits, act = torch.from_numpy(logits_np).to(dev), torch.from_numpy(act_np).to(dev)
    vp = d["value"][:T].clone()
    hpk = ops.LossHyper(**hyper_kwargs(cfg))
    fn = lambda: ops.ppo_loss_from_logits(logits, act, list(cfg.num_actions), vp, d["old_logp"][:T], d["value"][:T], ret[:T],
                                          adv[:T], d["on_reset"][1:T + 1], stats, hpk)
    fn()
    ms = statistics.mean(timed_steps(10, fn))
    SK, heads = int(sum(cfg.num_actions)), len(cfg.num_actions)
    per = 8 * SK + 4 * heads + 25  # SURVEY.md §8(d)
    nbytes = per * T * c1.N
    out["loss_from_logits_k4b"] = dict(ms_per_launch=ms, bytes_per_launch=nbytes,
                                       what=f"srl_ppo_loss_from_logits, T={T}, N={c1.N}, heads {list(cfg.num_actions)}: "
                                            f"{per} B per transition (SURVEY.md §8d)",
                                       roofline=dict(bound="hbm", achieved=nbytes / ms / 1e6, peak=peak, unit="GB/s",
                                                     frac=nbytes / ms / 1e6 / peak))
    del logits, act
    # ---- (f)4: a recurrent policy's minibatch -- chunked reset flags, segment boundaries, masked chunk-start states ------
    try:
        Tq, Bq = cfg.T, min(cfg.N, 4096)
        nq, Cq, layers, H = max(2, Bq // max(cfg.minibatches, 1)), (8 if Tq % 8 == 0 else 1), 1, 256
        g = torch.Generator(device="cpu").manual_seed(3)
        on_reset = (torch.rand((Tq, Bq), generator=g) < 0.01).to(torch.uint8).to(dev)
        hx = torch.randn((Tq, Bq, layers, H), generator=g).to(dev)
        env_idx = torch.randperm(Bq, generator=g)[:nq].to(torch.int32).to(dev)
        fn = lambda: ops.rnn_chunk_prep(on_reset, env_idx, Cq, hx=hx)
        fn()
        ms = statistics.mean(timed_steps(10, fn))
        nbytes = 2 * Tq * nq + 2 * Cq * nq * layers * H * 4
        out["rnn_chunk_prep"] = dict(ms_per_launch=ms, bytes_per_launch=nbytes,
                                     what=f"srl_rnn_chunk_prep (+ three torch.empty): T={Tq}, B={Bq}, minibatch of {nq} lanes, {Cq} "
                                          f"chunks, hidden state [{layers}, {H}] float32 per lane and step; an {nbytes / 1e6:.1f} MB "
                                          "launch, latency-bound",
                                     roofline=dict(bound="hbm", achieved=nbytes / ms / 1e6, peak=peak, unit="GB/s",
                                                   frac=nbytes / ms / 1e6 / peak))
        del hx
    except Exception as e:  # noqa: BLE001
        out["rnn_chunk_prep"] = dict(error=f"{type(e).__name__}: {e}")
    # ---- (f)2: a compressed frame leaf decoded into pinned memory by the library's own Blosc-1 / LZ4 decoder (host code) ----
    try:
        from tests import blosc1_writer  # the only Blosc-1 WRITER here (test double; blosc itself is absent): liblz4 streams
        rng = np.random.default_rng(0)
        img = np.zeros((129 * 4, 84, 84), dtype=np.uint8)
        for k in range(img.shape[0]):
            img[k, 10:60, 20:70] = rng.integers(0, 256)
            img[k, rng.integers(0, 84, 20), rng.integers(0, 84, 20)] = rng.integers(0, 256, 20)
        payload = img.tobytes()
        frame = np.frombuffer(blosc1_writer.compress(payload, 4, 1 << 18), dtype=np.uint8)
        pin = torch.empty(len(payload), dtype=torch.uint8).pin_memory()
        res = {}
        for th in (1, 8):
            t0 = time.perf_counter()
            for _ in range(20):
                ops._lib.call("srl_blosc1_decompress", frame.ctypes.data, frame.size, pin.data_ptr(), len(payload), th)
            res[f"threads_{th}_gbs"] = len(payload) / ((time.perf_counter() - t0) / 20) / 1e9
        ok = pin.numpy().tobytes() == payload
        out["wire_decode_native"] = dict(decoded_bytes=len(payload), compressed_bytes=int(frame.size), bit_exact=ok, **res,
                                         what="srl_blosc1_decompress: one Atari-like frame leaf [129, 4, 84, 84] uint8 (byte-"
                                              "shuffled, split, LZ4 streams written by liblz4) into pinned host memory; host wall "
                                              "clock; the Blosc-1 framing is unpinned against blosc itself (DESIGN.md 7.5)")
    except Exception as e:  # noqa: BLE001
        out["wire_decode_native"] = dict(error=f"{type(e).__name__}: {e}")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default 2000; 50 with --impl reference, whose CPU step of cfg2 takes ~0.1 s)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2_atari_large", choices=sorted(synth.CONFIGS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N > 1: the full config per GPU (weak) or the config's environments split over the GPUs (strong)")
    ap.add_argument("--e2e-steps", type=int, default=100)
    ap.add_argument("--cpu-budget-s", type=float, default=15.0)
    ap.add_argument("--launch", default="graph", choices=["graph", "plan"],
                    help="how the timed step is issued: one CUDA graph replay, or the recorded plan of stream launches")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the K1 / K4b / trainer_step lines")
    ap.add_argument("--no-parity-check", action="store_true")
    ap.add_argument("--no-align", action="store_true",
                    help="N > 1: do not line the ranks up (untimed device-side rendezvous) before each timed step")
    ap.add_argument("--shuffle-block", type=int, default=1,
                    help="environments per shuffled block (1 = per-environment permutation; 8 = one 32-byte sector)")
    ap.add_argument("--branches", type=int, default=16, help="parallel CUDA-graph branches for the per-minibatch launches")
    ap.add_argument("--explicit-gather", action="store_true", help="separate K5 gather launch instead of gather-on-load")
    ap.add_argument("--exchange", default="auto", choices=["auto", "p2p", "nccl"],
                    help="statistics exchange across ranks: NVLink peer-memory mailboxes (p2p) or NCCL all-reduce")
    ap.add_argument("--no-fuse-stats", action="store_true",
                    help="A/B: minibatch statistics from the srl_group_stats table instead of inside the loss kernel")
    ap.add_argument("--no-pack", action="store_true", help="A/B: gather the five sample leaves instead of K2's pack")
    ap.add_argument("--no-batch", action="store_true", help="A/B: one loss launch per minibatch (parallel graph branches)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the timed step's outputs of its last step to DIR/<name>.npy (at most 64 MB in all); "
                         "with several GPUs, rank 0's step on its slice of the workload")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 50 if args.impl == "reference" else 2000
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    cfg = synth.CONFIGS[args.config]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, cfg, rank, world)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        # launched without torchrun: re-launch ourselves one process per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29531", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    run_ours(args, cfg, rank, world, local_rank)


if __name__ == "__main__":
    main()
