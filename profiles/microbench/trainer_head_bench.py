"""K4b / K4c reading K2's loss pack, and MultiAgentPPOB200.step through the head losses, at cfg2's shape.

    python profiles/microbench/trainer_head_bench.py [--reps 200] [--warmup 20] [--steps 10] [--out FILE.json]

(a) One minibatch launch at cfg2's minibatch shape, T = 128 rows of n = 512 lanes gathered through a permutation from a
    sample of N = 4096 lanes (8 minibatches): K4b with heads (18,), K4c with D = 6 (shared [D] log_std and per-transition),
    float32 and bfloat16 policy sides, each with the sample side in two forms on the same sample:
      pack:   srl_ppo_loss_from_*_pack on the pack the scan wrote (what the trainer's permuted minibatches now read);
      leaves: the leaf entry on old_logp / value / ret / adv / on_reset through lane_idx.
    The two forms' outputs are compared first (they must be bit-identical).  Timing: CUDA events per launch; before each
    the L2 is flushed (256 MiB write + 256 MiB read) and a device sleep is queued, so the events measure device time.  The
    forms alternate in two rounds of `reps` launches; the reported time is the median of the two rounds' medians.
    Sample-side bytes per transition: the useful bytes (pack: one 16-byte item; leaves: 4 x 4 bytes + 1 flag byte with
    clip_value) and the 32-byte sectors the gather touches -- an estimate from the access pattern, not a measurement: a
    permuted lane's leaf element shares its sector with no other element of the launch (5 sectors per transition), while a
    pack sector holds the same lane's two rows of a row pair, both read by the launch (0.5 per transition).
(b) MultiAgentPPOB200.step at cfg2 (L = 129, B = 4096 single-agent environments, 4 epochs x 8 minibatches, Atari's loss)
    with a small MLP categorical policy (obs 64 -> 64 -> 18 actions + value), the same policy through target="ppo_head"
    and through target="ppo" from the same initial parameters.  Host sample, prefetch off; a device synchronise ends every
    timed step; the two trainers alternate step by step after two warm-up steps each.

The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import statistics
import sys
import tempfile
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn as nn  # noqa: E402

from bf16_logits_bench import card  # noqa: E402

T_MB, N_ALL, MINIBATCHES, K, DG = 128, 4096, 8, 18, 6


def kernel_part(args, dev):
    from srl_b200 import ops
    n = N_ALL // MINIBATCHES
    L = T_MB + 1
    g = torch.Generator(device=dev).manual_seed(0)
    f = lambda *s: torch.randn(*s, device=dev, generator=g)
    reward, value, old_logp = f(L, N_ALL), f(L, N_ALL), f(L, N_ALL) * 0.3 - 2.5
    flags = [(torch.rand(L, N_ALL, device=dev, generator=g) < p).to(torch.uint8) for p in (0.01, 0.005, 0.01)]
    pack = ops.new_pack(L, N_ALL, dev)
    adv, ret, _ = ops.gae_scan(reward, value, *flags, 0.99, 0.95, row_lo=0, row_hi=L - 1, old_logp=old_logp, pack=pack)
    on_reset = flags[2]
    leaves = (old_logp[:T_MB], value[:T_MB], ret[:T_MB], adv[:T_MB], on_reset[1:])
    no_leaves = (None,) * 5
    idx = ops.philox_perm(3, 0, N_ALL)[:n].contiguous()
    stats = torch.tensor([T_MB * n, 10.0, 2.0 * T_MB * n], dtype=torch.float64, device=dev)
    hp = ops.LossHyper(clip_value=True, dual_clip=False, value_loss="huber", value_loss_config=dict(delta=10.0),
                       value_loss_weight=1.0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    flush_rd = torch.zeros(64 << 20, dtype=torch.int32, device=dev)

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        pairs = []
        for _ in range(args.reps):
            flush.zero_()
            flush_rd.max()
            torch.cuda._sleep(1_000_000)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            pairs.append((a, b))
        torch.cuda.synchronize()
        return 1e3 * statistics.median(a.elapsed_time(b) for a, b in pairs)

    results = []
    for dtype in (torch.float32, torch.bfloat16):
        logits = (2 * f(T_MB, n, K)).to(dtype)
        action = torch.randint(0, K, (T_MB, n, 1), device=dev, generator=g).to(torch.int32)
        mean = f(T_MB, n, DG).to(dtype)
        act_g = f(T_MB, n, DG)
        v_pred = f(T_MB, n).to(dtype)
        ls_shared, ls_row = f(DG) * 0.3, (f(T_MB, n, DG) * 0.3).to(dtype)
        cases = {
            "k4b_k18": lambda smp, **kw: ops.ppo_loss_from_logits(logits, action, [K], v_pred, *smp, stats, hp,
                                                                  lane_idx=idx, **kw),
            "k4c_d6_shared": lambda smp, **kw: ops.ppo_loss_from_gaussian(mean, ls_shared, act_g, v_pred, *smp, stats, hp,
                                                                          lane_idx=idx, **kw),
            "k4c_d6_per_row": lambda smp, **kw: ops.ppo_loss_from_gaussian(mean, ls_row, act_g, v_pred, *smp, stats, hp,
                                                                           lane_idx=idx, **kw),
        }
        for name, run in cases.items():
            a, b = run(leaves), run(no_leaves, pack=pack)
            torch.cuda.synchronize()
            identical = all(torch.equal(x, y) for x, y in zip(a, b) if x is not None)
            leaf_fn, pack_fn = (lambda: run(leaves)), (lambda: run(no_leaves, pack=pack))
            rounds = {"pack": [], "leaves": []}
            for _ in range(2):
                rounds["pack"].append(timed(pack_fn))
                rounds["leaves"].append(timed(leaf_fn))
            line = dict(kernel=name, dtype=str(dtype).replace("torch.", ""), T=T_MB, n=n, N=N_ALL, bit_identical=identical,
                        sample_side_bytes_per_transition=dict(pack=dict(useful=16, sectors_32b_est=0.5),
                                                              leaves=dict(useful=17, sectors_32b_est=5)),
                        pack_us=statistics.median(rounds["pack"]), leaves_us=statistics.median(rounds["leaves"]),
                        rounds_us=rounds)
            line["leaves_over_pack"] = line["leaves_us"] / line["pack_us"]
            print(json.dumps({k: v for k, v in line.items() if k != "rounds_us"}), flush=True)
            results.append(line)
    return results


class MLPPolicy:
    """obs.vec [..., 64] -> tanh MLP -> 18 logits + value; target="ppo" builds the Categorical in torch, target="ppo_head"
    returns the logits (srl_b200.api.PPOHeadAnalyzedResult)."""

    def __init__(self, head, device="cuda:0", obs_dim=64, hidden=64, seed=0):
        torch.manual_seed(seed)
        self.net = nn.ModuleDict(dict(body=nn.Sequential(nn.Linear(obs_dim, hidden), nn.Tanh()), actor=nn.Linear(hidden, K),
                                      critic=nn.Linear(hidden, 1))).to(device)
        self.ppo_head = head
        self.device, self.version = device, -1

    def parameters(self):
        return self.net.parameters()

    def inc_version(self):
        self.version += 1

    def analyze(self, sample, target="ppo", burn_in_steps=0, **kw):
        from srl_b200.api import PPOHeadAnalyzedResult
        from types import SimpleNamespace
        h = self.net["body"](sample.obs.vec[burn_in_steps:])
        logits, value = self.net["actor"](h), self.net["critic"](h)
        action = sample.action.x[burn_in_steps:]
        if target == "ppo_head":
            return PPOHeadAnalyzedResult(state_values=value, action=action, logits=logits, head_sizes=[K])
        d = torch.distributions.Categorical(logits=logits)
        return SimpleNamespace(new_action_log_probs=d.log_prob(action[..., 0].long()).unsqueeze(-1), state_values=value,
                               entropy=d.entropy().unsqueeze(-1))


def trainer_part(args):
    from srl_b200 import api, synth
    from srl_b200.namedarray import NamedArray
    from srl_b200.trainer import MultiAgentPPOB200
    cfg = synth.PathConfig("cfg2", T=T_MB, B=N_ALL, p_end=0.002)
    kw = dict(discount_rate=0.99, gae_lambda=0.95, clip_value=True, dual_clip=False, value_loss="huber",
              value_loss_config=dict(delta=10.0), value_loss_weight=1.0, ppo_epochs=4, num_minibatches=MINIBATCHES,
              optimizer="adam", optimizer_config=dict(lr=1e-4), prefetch=False)

    def sample(seed):
        s = synth.make_sample_scalars(cfg, seed)
        rng = np.random.default_rng(seed)
        lead = s["value"].shape[:-1]
        return api.SampleBatch(obs=NamedArray(vec=rng.standard_normal(lead + (64,)).astype(np.float32)),
                               on_reset=s["on_reset"], done=s["done"], truncated=s["truncated"],
                               action=NamedArray(x=rng.integers(0, K, lead + (1,)).astype(np.float32)), reward=s["reward"],
                               analyzed_result=api.AnalyzedResult(value=s["value"], log_probs=s["old_logp"]))

    trainers = {name: MultiAgentPPOB200(MLPPolicy(head=(name == "ppo_head")), **kw) for name in ("ppo_head", "ppo")}
    samples = [sample(s) for s in range(4)]
    times = {name: [] for name in trainers}
    stats = {}
    for it in range(2 + args.steps):
        for name, tr in trainers.items():
            s = samples[it % len(samples)]
            s.analyzed_result.adv = s.analyzed_result.ret = None
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            stats[name] = tr.step(s).stats
            torch.cuda.synchronize()
            if it >= 2:
                times[name].append(1e3 * (time.perf_counter() - t0))
    out = dict(L=T_MB + 1, B=N_ALL, epochs=4, minibatches=MINIBATCHES, policy="MLP 64-64-18 + value, float32",
               steps=args.steps, last_stats=stats)
    for name, ts in times.items():
        out[name] = dict(median_ms=statistics.median(ts), min_ms=min(ts), max_ms=max(ts), all_ms=ts)
    out["ppo_over_ppo_head"] = out["ppo"]["median_ms"] / out["ppo_head"]["median_ms"]
    print(json.dumps({k: v for k, v in out.items() if k not in ("ppo", "ppo_head", "last_stats")} |
                     {k: round(out[k]["median_ms"], 3) for k in ("ppo", "ppo_head")}), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "k4bc_pack_trainer.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device: nothing here is measured on the CPU")
    dev = torch.device("cuda")
    doc = dict(what="K4b / K4c sample side from K2's pack against leaves + lane_idx at cfg2's minibatch shape; "
                    "MultiAgentPPOB200.step at cfg2 with a ppo_head policy against target='ppo'",
               card=card(), reps=args.reps, warmup=args.warmup,
               timing="(a) CUDA events per launch, L2 flushed (256 MiB write + 256 MiB read) and a device sleep queued "
                      "before each, median over reps, two alternating rounds, median of the two; (b) host clock around "
                      "each step, device synchronise before and after, median over steps, trainers alternating",
               kernels=kernel_part(args, dev), trainer_step=trainer_part(args))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(doc, fh, indent=1)
    print(json.dumps(dict(card=doc["card"])), flush=True)


if __name__ == "__main__":
    main()
