"""K4b with an availability mask: srl_ppo_loss_from_logits_masked against srl_ppo_loss_from_logits (no mask) and against the
unfused path, on the same inputs.

    python profiles/microbench/masked_logits_bench.py [--reps 300] [--warmup 20] [--out FILE.json]

Shapes: T = 128, N = 4096 (cfg2's minibatch), heads (18,) (Atari), (36,) (SMAC 27m) and (11, 11, 11, 2, 2) (hide-and-seek);
30 % of the actions unavailable, action 0 of every head always available; cfg3's loss (PopArt, dual clip, huber).  The
unfused path is what a SMAC policy runs without the masked kernel: eager masked_fill + torch.distributions.Categorical per
head, srl_ppo_loss_fwd_bwd on their log-prob and entropy, and the autograd backward of those ops to the logits.

Timing: CUDA events around each launch (the fused call, or the whole unfused sequence), many launches after warm-up.  Before
each one the L2 is flushed (256 MiB device write, then 256 MiB device read, as bench.py does) and a ~0.5 ms device sleep is
queued, so the host has enqueued the timed work before the GPU reaches it: the events measure device time, not Python.
Algorithmic bytes per transition are bench.py's K4b accounting, 8 sum K + 4 heads + 25 (logits in, d logits out, actions,
v_pred, old_logp, old_value, ret, adv, on_reset_next in, d v_pred out), plus sum K for the mask.  The roofline denominator
is 6550 GB/s, the measured copy bandwidth of DESIGN.md.  Shared memory per CTA and the CTAs per SM it allows are computed
from the kernel's layout and the device's limits.  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

PEAK_GBS = 6550.0


def card():
    info = dict(name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["nvidia_smi"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
    except (OSError, subprocess.SubprocessError):
        info["nvidia_smi"] = None
    return info


def smem_per_cta(sk, masked):
    """ppo_loss_from_logits' shared-memory layout (srl_b200/csrc/ppo_loss.cu): [256, sum K] floats, a second such block
    when it fits (cached exponentials), the [256, sum K] mask bytes, the mbarrier."""
    row, mask = 256 * sk * 4, (256 * sk if masked else 0)
    cache_e = 2 * row + mask + 16 <= 200 * 1024
    return (2 * row if cache_e else row) + mask + 16, cache_e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "k4b_masked_logits.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device: nothing here is measured on the CPU")
    from oracle import ref_math as M
    from srl_b200 import ops, synth

    dev = torch.device("cuda")
    props = torch.cuda.get_device_properties(0)
    sm_smem = getattr(props, "shared_memory_per_multiprocessor", None)
    T, N = 128, 4096
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
        ms = [a.elapsed_time(b) for a, b in pairs]
        return dict(median_us=1e3 * statistics.median(ms), mean_us=1e3 * statistics.mean(ms), min_us=1e3 * min(ms),
                    max_us=1e3 * max(ms))

    rng = np.random.default_rng(0)
    f = lambda *s: torch.from_numpy(rng.standard_normal(s).astype(np.float32)).to(dev)
    old_value, ret, adv = f(T + 1, N), f(T + 1, N), f(T + 1, N)
    on_reset = torch.from_numpy((rng.random((T + 1, N)) < 0.01).astype(np.uint8)).to(dev)
    v_pred = (old_value[:T] + 0.1 * f(T, N)).contiguous()
    mask = 1.0 - on_reset[1:].double()
    x = adv[:T].double() * mask
    stats = torch.tensor([mask.sum().item(), x.sum().item(), x.square().sum().item(), 0, 0, 0, 0, 0], dtype=torch.float64,
                         device=dev)
    popart = torch.tensor([0.5, 2.0], dtype=torch.float64, device=dev)
    hp = ops.LossHyper(dual_clip=True, c_clip=3.0, value_loss="huber", value_loss_config=dict(delta=10.0),
                       value_loss_weight=1.0)
    smp = (old_value[:T], ret[:T], adv[:T], on_reset[1:])

    results = []
    for heads in ((18,), (36,), (11, 11, 11, 2, 2)):
        cfg = synth.PathConfig("bench", T=T, B=N, num_actions=heads)
        logits_np, actions_np, avail_np = synth.make_masked_logits_actions(cfg, (T, N), seed=1, p_unavailable=0.3)
        logits, actions, avail = (torch.from_numpy(a).to(dev) for a in (logits_np, actions_np, avail_np))
        with torch.no_grad():
            lp0, _ = M.logp_entropy_from_logits_ref(logits, actions.long(), heads, available=avail)
        old_logp = torch.cat([lp0[..., 0] + 0.15 * f(T, N), torch.zeros(1, N, device=dev)]).contiguous()
        args_smp = (old_logp[:T], smp[0], smp[1], smp[2], smp[3])

        def masked():
            return ops.ppo_loss_from_logits(logits, actions, heads, v_pred, *args_smp, stats, hp, popart_mean_std=popart,
                                            available=avail)

        def unmasked():
            return ops.ppo_loss_from_logits(logits, actions, heads, v_pred, *args_smp, stats, hp, popart_mean_std=popart)

        z_l = logits.clone().requires_grad_(True)
        act_l = actions.long()

        def unfused():
            z_l.grad = None
            z = z_l.masked_fill(avail == 0, -1e10)
            lps, ens, off = [], [], 0
            for h, k in enumerate(heads):
                dist = torch.distributions.Categorical(logits=z[..., off:off + k])
                lps.append(dist.log_prob(act_l[..., h]))
                ens.append(dist.entropy())
                off += k
            lp, en = torch.stack(lps, -1).sum(-1), torch.stack(ens, -1).sum(-1)
            g_lp, g_v, g_en, out, _ = ops.ppo_loss_fwd_bwd(lp.detach(), v_pred, en.detach(), *args_smp, stats, hp,
                                                          popart_mean_std=popart)
            torch.autograd.backward([lp, en], [g_lp, g_en])
            return z_l.grad, g_v, out

        # the masked kernel and the unfused path agree (same inputs): a sanity line next to the times.  Per transition,
        # outside 1e-5 on the g * sum(mask) scale; ratios within float32 noise of a clip edge are counted beside
        a, b = masked(), unfused()
        torch.cuda.synchronize()
        Ms = float(stats[0])
        off_ = lambda x, y: (((x.double() - y.double()).abs() * Ms) > 1e-5 * (y.double().abs() * Ms).clamp(min=1.0))
        with torch.no_grad():
            r = (lp0[..., 0] - old_logp[:T]).exp()
            edge = ((r - (1 - hp.eps_clip)).abs() < 1e-5) | ((r - (1 + hp.eps_clip)).abs() < 1e-5)
        agree = dict(loss_abs=abs(float(a[2][0]) - float(b[2][0])),
                     g_logits_transitions_off=int(off_(a[0], b[0]).any(-1).sum()),
                     g_logits_nonzero_where_unavailable=int((a[0][avail == 0] != 0).sum()),
                     g_value_off=int(off_(a[1], b[1]).sum()), clip_edge_transitions=int(edge.sum()))
        sk = sum(heads)
        bpt = 8 * sk + 4 * len(heads) + 25
        line = dict(T=T, N=N, heads=list(heads), sum_k=sk, unavailable_fraction=float((avail == 0).float().mean()),
                    agreement=agree)
        # alternate the three paths twice: another tenant's load shows up as a spread between the two rounds
        runs = {"masked": [], "unmasked": [], "unfused": []}
        for _ in range(2):
            for name, fn in (("masked", masked), ("unmasked", unmasked), ("unfused", unfused)):
                runs[name].append(timed(fn))
        for name, ts in runs.items():
            nbytes = (bpt + (sk if name != "unmasked" else 0)) * T * N
            med = statistics.median(t["median_us"] for t in ts)
            entry = dict(median_us=med, rounds=ts, algorithmic_bytes=nbytes, gbs=nbytes / (med * 1e3),
                         of_6550=nbytes / (med * 1e3) / PEAK_GBS)
            if name != "unfused":
                smem, cache_e = smem_per_cta(sk, name == "masked")
                entry.update(smem_per_cta=smem, cache_e=cache_e,
                             ctas_per_sm_by_smem=None if sm_smem is None else int(sm_smem // (smem + 1024)))
            line[name] = entry
        line["masked_over_unmasked"] = line["masked"]["median_us"] / line["unmasked"]["median_us"]
        line["unfused_over_masked"] = line["unfused"]["median_us"] / line["masked"]["median_us"]
        print(json.dumps(line), flush=True)
        results.append(line)
    doc = dict(what="K4b srl_ppo_loss_from_logits_masked vs srl_ppo_loss_from_logits (no mask) vs unfused (eager masked_fill + "
                    "Categorical + srl_ppo_loss_fwd_bwd + autograd backward)",
               card=card(), shared_memory_per_sm=sm_smem, reps=args.reps, warmup=args.warmup,
               timing="CUDA events per launch; L2 flushed (256 MiB write + 256 MiB read) and a device sleep queued before "
                      "each; median over reps, two alternating rounds per path, median of the two", roofline_gbs=PEAK_GBS,
               results=results)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(doc, fh, indent=1)
    print(json.dumps(dict(card=doc["card"])), flush=True)


if __name__ == "__main__":
    main()
