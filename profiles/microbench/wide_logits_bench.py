"""K4b-wide (srl_ppo_loss_from_logits_wide) against the unfused path on wide categorical heads, and against K4b at widths
both take.

    python profiles/microbench/wide_logits_bench.py [--reps 50] [--warmup 5] [--out FILE.json]

Shapes (T x N transitions, heads, policy dtype, mask): 128 x 4096 at (200,), (362,) and (1024, 512, 256, 128, 64, 32, 16, 8)
in float32; 65536 transitions of (4672,) with about 1 % of the actions available; 8192 of (32000,) and 4096 of (151936,) in
bfloat16.  cfg3's loss (PopArt, dual clip, huber).  The unfused path is what such a policy runs without the kernel: eager
masked_fill (with a mask) + torch.distributions.Categorical per head on the float32 logits (a bfloat16 head's logits are
cast once, as the fused kernel widens them), srl_ppo_loss_fwd_bwd on their log-prob and entropy, and the autograd backward
to the logits.  The overlap rows time K4b-wide (routing thresholds lowered) against K4b itself at (18,), (36,) with a mask,
(11, 11, 11, 2, 2) and (199,), 128 x 4096 float32: for information, the routing of those widths does not change.

Timing: CUDA events around each launch (the fused call, or the whole unfused sequence), many launches after warm-up.  Before
each one the L2 is flushed (256 MiB device write, then 256 MiB device read, as bench.py does) and a ~0.5 ms device sleep is
queued, so that the events measure device time.  Algorithmic bytes per transition are K4b's accounting: 2 e sum K + 4 heads
+ 25 (bfloat16: + 21; e the element size: logits in, d logits out, actions, v_pred, old_logp, old_value, ret, adv,
on_reset_next in, d v_pred out), + sum K with a mask.  K4b-wide reads each row a second time for the gradient pass; that
read is not in the algorithmic bytes (`second_read_bytes` states it).  The roofline denominator is 6550 GB/s, the measured
copy bandwidth of DESIGN.md.  The card's name and power limit are read in the same run.
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
SHAPES = [((200,), 128 * 4096, torch.float32, None), ((362,), 128 * 4096, torch.float32, None),
          ((1024, 512, 256, 128, 64, 32, 16, 8), 128 * 4096, torch.float32, None),
          ((4672,), 65536, torch.float32, 0.01), ((32000,), 8192, torch.bfloat16, None),
          ((151936,), 4096, torch.bfloat16, None)]
OVERLAP = [((18,), None), ((36,), 0.7), ((11, 11, 11, 2, 2), None), ((199,), None)]


def card():
    info = dict(name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["nvidia_smi"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
    except (OSError, subprocess.SubprocessError):
        info["nvidia_smi"] = None
    return info


def algorithmic_bytes(heads, dtype, masked):
    e = 2 if dtype == torch.bfloat16 else 4
    sk = sum(heads)
    return 2 * e * sk + 4 * len(heads) + (21 if e == 2 else 25) + (sk if masked else 0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "k4b_wide_logits.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device: nothing here is measured on the CPU")
    from srl_b200 import ops

    dev = torch.device("cuda")
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

    hp = ops.LossHyper(dual_clip=True, c_clip=3.0, value_loss="huber", value_loss_config=dict(delta=10.0),
                       value_loss_weight=1.0)
    popart = torch.tensor([0.5, 2.0], dtype=torch.float64, device=dev)
    gen = torch.Generator(device=dev).manual_seed(0)

    def inputs(heads, rows, dtype, p_avail):
        """[T, N] = [rows / 4096 or rows / 512, ...] minibatch of seeded device inputs."""
        N = 4096 if rows % 4096 == 0 else 512
        T = rows // N
        SK = sum(heads)
        logits = (torch.randn(T, N, SK, device=dev, generator=gen) * 2).to(dtype)
        actions = torch.stack([torch.randint(0, K, (T, N), device=dev, generator=gen) for K in heads], -1).to(torch.int32)
        avail = None
        if p_avail is not None:
            avail = (torch.rand(T, N, SK, device=dev, generator=gen) < p_avail).to(torch.uint8)
            off = 0
            for h, K in enumerate(heads):  # the chosen actions are available
                avail[..., off:off + K].scatter_(-1, actions[..., h:h + 1].long(), 1)
                off += K
        f = lambda *s: torch.randn(*s, device=dev, generator=gen)
        old_value, ret, adv = f(T + 1, N), f(T + 1, N), f(T + 1, N)
        on_reset = (torch.rand(T + 1, N, device=dev, generator=gen) < 0.01).to(torch.uint8)
        v_pred = (old_value[:T] + 0.1 * f(T, N)).to(dtype).contiguous()
        with torch.no_grad():
            z = logits.float() if avail is None else logits.float().masked_fill(avail == 0, -1e10)
            lp0 = torch.zeros(T, N, device=dev)
            off = 0
            for h, K in enumerate(heads):
                lp0 += torch.distributions.Categorical(logits=z[..., off:off + K]).log_prob(actions[..., h].long())
                off += K
            del z
        old_logp = (lp0 + 0.15 * f(T, N)).contiguous()
        mask = 1.0 - on_reset[1:].double()
        x = adv[:T].double() * mask
        stats = torch.tensor([mask.sum().item(), x.sum().item(), x.square().sum().item(), 0, 0, 0, 0, 0],
                             dtype=torch.float64, device=dev)
        smp = (old_logp, old_value[:T], ret[:T], adv[:T], on_reset[1:])
        return T, N, logits, actions, avail, v_pred, smp, stats

    def fused_fn(heads, logits, actions, avail, v_pred, smp, stats):
        return lambda: ops.ppo_loss_from_logits(logits, actions, heads, v_pred, *smp, stats, hp, popart_mean_std=popart,
                                                available=avail)

    def unfused_fn(heads, logits, actions, avail, v_pred, smp, stats):
        z_l = logits.detach().clone().requires_grad_(True)
        act_l = actions.long()
        vp32 = v_pred.float()

        def unfused():
            z_l.grad = None
            z = z_l.float()
            if avail is not None:
                z = z.masked_fill(avail == 0, -1e10)
            lps, ens, off = [], [], 0
            for h, k in enumerate(heads):
                dist = torch.distributions.Categorical(logits=z[..., off:off + k])
                lps.append(dist.log_prob(act_l[..., h]))
                ens.append(dist.entropy())
                off += k
            lp, en = torch.stack(lps, -1).sum(-1), torch.stack(ens, -1).sum(-1)
            g_lp, g_v, g_en, out, _ = ops.ppo_loss_fwd_bwd(lp.detach(), vp32, en.detach(), *smp, stats, hp,
                                                          popart_mean_std=popart)
            torch.autograd.backward([lp, en], [g_lp, g_en])
            return z_l.grad, g_v, out
        return unfused

    def entry(name, heads, dtype, masked, rows, med_list):
        nbytes = algorithmic_bytes(heads, dtype, masked) * rows
        med = statistics.median(t["median_us"] for t in med_list)
        return dict(median_us=med, rounds=med_list, algorithmic_bytes=nbytes, gbs=nbytes / (med * 1e3),
                    of_6550=nbytes / (med * 1e3) / PEAK_GBS)

    results = []
    for heads, rows, dtype, p_avail in SHAPES:
        T, N, logits, actions, avail, v_pred, smp, stats = inputs(heads, rows, dtype, p_avail)
        fused = fused_fn(heads, logits, actions, avail, v_pred, smp, stats)
        unfused = unfused_fn(heads, logits, actions, avail, v_pred, smp, stats)
        # the two paths agree (same inputs): loss, and the transitions whose d logits differ beyond 1e-5 on the g * sum(mask)
        # scale (bfloat16: beyond half a bfloat16 ulp of the float32 gradient as well)
        a, b = fused(), unfused()
        torch.cuda.synchronize()
        Ms = float(stats[0])
        ga, gb = a[0].double() * Ms, b[0].double() * Ms
        tol = 1e-5 * gb.abs().clamp(min=1.0) + (gb.abs() * 2.0 ** -8 if dtype == torch.bfloat16 else 0.0)
        agree = dict(loss_abs=abs(float(a[2][0]) - float(b[2][0])),
                     g_logits_transitions_off=int(((ga - gb).abs() > tol).any(-1).sum()))
        del ga, gb, tol, a, b
        sk = sum(heads)
        e = 2 if dtype == torch.bfloat16 else 4
        line = dict(T=T, N=N, heads=list(heads), sum_k=sk, dtype=str(dtype).replace("torch.", ""), masked=avail is not None,
                    available_fraction=None if avail is None else float(avail.float().mean()), agreement=agree)
        runs = {"wide": [], "unfused": []}
        for _ in range(2):  # alternate the paths twice: another tenant's load shows as a spread between the rounds
            for name, fn in (("wide", fused), ("unfused", unfused)):
                runs[name].append(timed(fn))
        for name, ts in runs.items():
            line[name] = entry(name, heads, dtype, avail is not None, T * N, ts)
        line["wide"]["second_read_bytes"] = e * sk * T * N
        line["unfused_over_wide"] = line["unfused"]["median_us"] / line["wide"]["median_us"]
        print(json.dumps(line), flush=True)
        results.append(line)
        del logits, actions, avail, v_pred, smp, fused, unfused
        torch.cuda.empty_cache()

    overlap = []
    for heads, p_avail in OVERLAP:
        T, N, logits, actions, avail, v_pred, smp, stats = inputs(heads, 128 * 4096, torch.float32, p_avail)
        k4b = fused_fn(heads, logits, actions, avail, v_pred, smp, stats)
        saved = ops.SRL_K4B_MAX_SUM_K, ops.SRL_K4B_MAX_SUM_K_MASKED

        def wide():
            ops.SRL_K4B_MAX_SUM_K = ops.SRL_K4B_MAX_SUM_K_MASKED = 0
            try:
                return k4b()
            finally:
                ops.SRL_K4B_MAX_SUM_K, ops.SRL_K4B_MAX_SUM_K_MASKED = saved
        a, b = wide(), k4b()
        torch.cuda.synchronize()
        line = dict(T=T, N=N, heads=list(heads), sum_k=sum(heads), masked=avail is not None,
                    agreement=dict(loss_abs=abs(float(a[2][0]) - float(b[2][0])),
                                   g_logits_max_abs=float((a[0] - b[0]).abs().max())))
        runs = {"wide": [], "k4b": []}
        for _ in range(2):
            for name, fn in (("wide", wide), ("k4b", k4b)):
                runs[name].append(timed(fn))
        for name, ts in runs.items():
            line[name] = entry(name, heads, torch.float32, avail is not None, T * N, ts)
        line["wide_over_k4b"] = line["wide"]["median_us"] / line["k4b"]["median_us"]
        print(json.dumps(line), flush=True)
        overlap.append(line)
        del logits, actions, avail, v_pred, smp
        torch.cuda.empty_cache()

    doc = dict(what="K4b-wide srl_ppo_loss_from_logits_wide vs unfused (eager masked_fill + Categorical + "
                    "srl_ppo_loss_fwd_bwd + autograd backward); overlap rows: K4b-wide vs K4b at widths both take",
               card=card(), reps=args.reps, warmup=args.warmup,
               timing="CUDA events per launch; L2 flushed (256 MiB write + 256 MiB read) and a device sleep queued before "
                      "each; median over reps, two alternating rounds per path, median of the two", roofline_gbs=PEAK_GBS,
               results=results, overlap=overlap)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(doc, fh, indent=1)
    print(json.dumps(dict(card=doc["card"])), flush=True)


if __name__ == "__main__":
    main()
