"""K4c microbenchmark: srl_ppo_loss_from_gaussian against the unfused path on the same inputs.

    python profiles/microbench/gaussian_loss_bench.py [--reps 300] [--warmup 20] [--out FILE.json]

Shapes: T = 128, N = 4096 (cfg2's minibatch), D in {6, 17}, log_std per transition and shared ([D]); huber value loss with
value clipping (the sample side reads old_value).  The unfused path is what a continuous-action policy runs without K4c:
torch.distributions.Normal log-prob and entropy summed over D (eager PyTorch), srl_ppo_loss_fwd_bwd on them, and the
autograd backward of the Normal ops to mean and log_std.

Timing: CUDA events around each launch (the fused call, or the whole unfused sequence), many launches after warm-up.  Before
each one the L2 is flushed (256 MiB device write, then 256 MiB device read, as bench.py does) and a ~0.5 ms device sleep is
queued, so the host has enqueued the timed work before the GPU reaches it: the events measure device time, not Python.
Algorithmic bytes per transition follow K4b's accounting: 20 D + 25 with a per-transition log_std (mean, log_std, action
in; d mean, d log_std out; v_pred, old_logp, old_value, ret, adv, on_reset_next in; d v_pred out), 12 D + 25 shared.  The
roofline denominator is 6550 GB/s, the measured copy bandwidth of DESIGN.md.  The card's name and power limit are read in
the same run.
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "k4c_gaussian_loss.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device: nothing here is measured on the CPU")
    from srl_b200 import ops

    dev = torch.device("cuda")
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
    hp = ops.LossHyper(clip_value=True, dual_clip=True, value_loss="huber", value_loss_config=dict(delta=10.0))
    smp = (old_value[:T], ret[:T], adv[:T], on_reset[1:])

    results = []
    for D in (6, 17):
        for shared in (False, True):
            mean = f(T, N, D)
            log_std = (0.3 * f(D) - 0.5) if shared else (0.3 * f(T, N, D) - 0.5)
            action = (mean + log_std.exp() * f(T, N, D)).contiguous()
            with torch.no_grad():
                lp0 = torch.distributions.Normal(mean, log_std.exp()).log_prob(action).sum(-1)
            old_logp = torch.cat([lp0 + 0.15 * f(T, N), torch.zeros(1, N, device=dev)]).contiguous()
            args_smp = (old_logp[:T], smp[0], smp[1], smp[2], smp[3])

            def fused():
                return ops.ppo_loss_from_gaussian(mean, log_std, action, v_pred, *args_smp, stats, hp)

            mean_l = mean.clone().requires_grad_(True)
            ls_l = log_std.clone().requires_grad_(True)

            def unfused():
                mean_l.grad = None
                ls_l.grad = None
                dist = torch.distributions.Normal(mean_l, ls_l.exp())
                lp = dist.log_prob(action).sum(-1)
                en = dist.entropy().sum(-1)
                g_lp, g_v, g_en, out, _ = ops.ppo_loss_fwd_bwd(lp.detach(), v_pred, en.detach(), *args_smp, stats, hp)
                torch.autograd.backward([lp, en], [g_lp, g_en])
                return mean_l.grad, ls_l.grad, g_v, out

            # the two paths agree (same inputs): a sanity line next to the times.  Per transition, outside 1e-5 on the
            # g * sum(mask) scale; a ratio within float32 noise of a clip edge (1 -/+ eps_clip) may land on either side of
            # it in two float32 evaluations of the log-prob, so those transitions are counted beside
            a, b = fused(), unfused()
            torch.cuda.synchronize()
            M = float(stats[0])
            off = lambda x, y: (((x.double() - y.double()).abs() * M) > 1e-5 * (y.double().abs() * M).clamp(min=1.0))
            with torch.no_grad():
                r = (lp0 - old_logp[:T]).exp()
                edge = ((r - (1 - hp.eps_clip)).abs() < 1e-5) | ((r - (1 + hp.eps_clip)).abs() < 1e-5)
            agree = dict(loss_abs=abs(float(a[3][0]) - float(b[3][0])),
                         g_mean_transitions_off=int(off(a[0], b[0]).any(-1).sum()),
                         g_log_std_off=int(off(a[1], b[1]).sum()),
                         g_value_off=int(off(a[2], b[2]).sum()), clip_edge_transitions=int(edge.sum()))
            bpt = (12 * D + 25) if shared else (20 * D + 25)
            nbytes = bpt * T * N
            tf, tu = timed(fused), timed(unfused)
            line = dict(T=T, N=N, D=D, log_std="shared [D]" if shared else "per transition [T, N, D]",
                        bytes_per_transition=bpt, algorithmic_bytes=nbytes,
                        fused=dict(**tf, gbs=nbytes / (tf["median_us"] * 1e3), of_6550=nbytes / (tf["median_us"] * 1e3) / PEAK_GBS),
                        unfused=tu, speedup_median=tu["median_us"] / tf["median_us"], agreement=agree)
            print(json.dumps(line), flush=True)
            results.append(line)
    doc = dict(what="K4c srl_ppo_loss_from_gaussian vs unfused (torch Normal + srl_ppo_loss_fwd_bwd + autograd backward)",
               card=card(), reps=args.reps, warmup=args.warmup,
               timing="CUDA events per launch; L2 flushed (256 MiB write + 256 MiB read) and a device sleep queued before "
                      "each; median over reps", roofline_gbs=PEAK_GBS, results=results)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(doc, fh, indent=1)
    print(json.dumps(dict(card=doc["card"])), flush=True)


if __name__ == "__main__":
    main()
