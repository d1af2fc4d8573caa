"""K4d microbenchmark: srl_ppo_loss_from_beta(_bf16) against the unfused path on the same inputs.

    python profiles/microbench/beta_loss_bench.py [--reps 300] [--warmup 20] [--out FILE.json]

Shapes: T = 128, N = 4096 (cfg2's minibatch), D in {2, 6, 17}, the policy side in float32 and in bfloat16; huber value
loss with value clipping (the sample side reads old_value). Concentrations log-uniform over [0.5, 20], actions drawn
from the Beta itself, old_logp the float64 log-prob of the values each dtype holds, perturbed and kept away from the
clip edges. The unfused path is what a Beta policy runs without K4d: torch.distributions.Beta log-prob and entropy
summed over D (eager PyTorch: xlogy, three lgamma, digamma, and polygamma(1, .) in the backward), then
srl_ppo_loss_fwd_bwd on them, then the autograd backward of the Beta ops to both concentrations. A bfloat16 policy on
that path has to widen its concentrations to float32 first (srl_ppo_loss_fwd_bwd reads float32 logp / entropy), so its
unfused line includes the two .float() casts and their backward.

Timing: CUDA events around each launch (the fused call, or the whole unfused sequence), many launches after warm-up.  Before
each one the L2 is flushed (256 MiB device write, then 256 MiB device read, as bench.py does) and a ~0.5 ms device sleep is
queued, so the host has enqueued the timed work before the GPU reaches it: the events measure device time, not Python.
Algorithmic bytes per transition in float32: 20 D + 25 (concentration1, concentration0, action in; both gradients out;
v_pred, old_logp, old_value, ret, adv, on_reset_next in; d v_pred out); in bfloat16 12 D + 21.  The roofline
denominator is 6550 GB/s, the measured copy bandwidth of DESIGN.md.  The card's name and power limit are read in the
same run.
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


def away_from_clip_edges(lp, old, hp, margin=1e-3):
    """old_logp whose ratios exp(lp - old_logp) stay `margin` away from every edge of the clipped surrogate (1 -/+ eps_clip
    and c_clip): the unfused path's float32 log-prob differs from the float64 one by up to ~1e-4 at these concentrations,
    and a ratio that close to an edge lands on either side of it in the two paths -- a zero or a full gradient for that
    transition, |adv| * |d logp / d c| ~ 14 |adv| on the g * sum(mask) scale at an action clamped to 1e-6."""
    for _ in range(8):
        r = torch.exp(lp.double() - old.double())
        near = torch.zeros_like(r, dtype=torch.bool)
        for e in (1 - hp.eps_clip, 1 + hp.eps_clip, hp.c_clip):
            near |= (r - e).abs() < margin
        if not bool(near.any()):
            break
        old = torch.where(near, old + 10 * margin, old)
    return old


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "k4d_beta_loss.json"))
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
    mask = 1.0 - on_reset[1:].double()
    x = adv[:T].double() * mask
    stats = torch.tensor([mask.sum().item(), x.sum().item(), x.square().sum().item(), 0, 0, 0, 0, 0], dtype=torch.float64,
                         device=dev)
    hp = ops.LossHyper(clip_value=True, dual_clip=True, value_loss="huber", value_loss_config=dict(delta=10.0))
    smp = (old_value[:T], ret[:T], adv[:T], on_reset[1:])
    M = float(stats[0])

    results = []
    for D in (2, 6, 17):
        log_unif = lambda: torch.from_numpy(np.exp(rng.uniform(np.log(0.5), np.log(20.0), (T, N, D))).astype(np.float32))
        c1_32, c0_32 = log_unif().to(dev), log_unif().to(dev)
        action = torch.distributions.Beta(c1_32, c0_32).sample().clamp(1e-6, 1 - 1e-6).contiguous()
        noise = 0.15 * f(T, N)
        v_32 = (old_value[:T] + 0.1 * f(T, N)).contiguous()
        for dtype in (torch.float32, torch.bfloat16):
            c1, c0 = c1_32.to(dtype), c0_32.to(dtype)
            v_pred = v_32.to(dtype)
            with torch.no_grad():
                lp0 = torch.distributions.Beta(c1.double(), c0.double()).log_prob(action.double()).sum(-1).float()
            old_logp = torch.cat([away_from_clip_edges(lp0, lp0 + noise, hp), torch.zeros(1, N, device=dev)])
            args_smp = (old_logp[:T], smp[0], smp[1], smp[2], smp[3])

            def fused():
                return ops.ppo_loss_from_beta(c1, c0, action, v_pred, *args_smp, stats, hp)

            c1_l = c1.clone().requires_grad_(True)
            c0_l = c0.clone().requires_grad_(True)
            v32 = v_pred.float()

            def unfused():
                c1_l.grad = None
                c0_l.grad = None
                dist = torch.distributions.Beta(c1_l.float(), c0_l.float())
                lp = dist.log_prob(action).sum(-1)
                en = dist.entropy().sum(-1)
                g_lp, g_v, g_en, out, _ = ops.ppo_loss_fwd_bwd(lp.detach(), v32, en.detach(), *args_smp, stats, hp)
                torch.autograd.backward([lp, en], [g_lp, g_en])
                return c1_l.grad, c0_l.grad, g_v, out

            # a sanity line next to the times: the largest difference between the two paths on the g * sum(mask) scale,
            # and the number of gradient elements outside 1e-4 * max(1, |unfused|) there.  The unfused path evaluates the
            # Beta's special functions in float32, so this is not a pass / fail; the tests compare against float64
            a, b = fused(), unfused()
            torch.cuda.synchronize()
            d = lambda x, y: float(((x.double() - y.double()).abs() * M).max())
            off = lambda x, y: int((((x.double() - y.double()).abs() * M) >
                                    1e-4 * (y.double().abs() * M).clamp(min=1.0)).sum())
            agree = dict(loss_abs=abs(float(a[3][0]) - float(b[3][0])), g_c1_max_abs=d(a[0], b[0]),
                         g_c0_max_abs=d(a[1], b[1]), g_value_max_abs=d(a[2], b[2]), g_c1_off_1e4=off(a[0], b[0]),
                         g_c0_off_1e4=off(a[1], b[1]))
            es = torch.empty((), dtype=dtype).element_size()
            bpt = 2 * D * es + 4 * D + 2 * D * es + 2 * es + 17
            nbytes = bpt * T * N
            tf, tu = timed(fused), timed(unfused)
            line = dict(T=T, N=N, D=D, dtype=str(dtype).replace("torch.", ""), bytes_per_transition=bpt,
                        algorithmic_bytes=nbytes,
                        fused=dict(**tf, gbs=nbytes / (tf["median_us"] * 1e3),
                                   of_6550=nbytes / (tf["median_us"] * 1e3) / PEAK_GBS),
                        unfused=tu, speedup_median=tu["median_us"] / tf["median_us"], agreement=agree)
            print(json.dumps(line), flush=True)
            results.append(line)
    doc = dict(what="K4d srl_ppo_loss_from_beta(_bf16) vs unfused (torch Beta + srl_ppo_loss_fwd_bwd + autograd backward)",
               card=card(), reps=args.reps, warmup=args.warmup,
               timing="CUDA events per launch; L2 flushed (256 MiB write + 256 MiB read) and a device sleep queued before "
                      "each; median over reps", roofline_gbs=PEAK_GBS, results=results)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(doc, fh, indent=1)
    print(json.dumps(dict(card=doc["card"])), flush=True)


if __name__ == "__main__":
    main()
