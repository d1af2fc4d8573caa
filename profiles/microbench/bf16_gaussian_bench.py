"""K4c with a bfloat16 policy side: srl_ppo_loss_from_gaussian_bf16 against the float32 entry and against the cast path a
bfloat16 Gaussian policy had without it, on the same values.

    python profiles/microbench/bf16_gaussian_bench.py [--reps 300] [--warmup 20] [--out FILE.json]

Shapes: T = 128, N = 4096 (cfg2's minibatch) with D in {6, 17} and log_std per transition and shared ([D], float32, as
autocast leaves an nn.Parameter); and cfg5's HBM-resident shape, T = 160, N = 65536 with D = 17 per transition, whose float32
mean, log_std and action blocks are ~0.7 GB each, far larger than the L2.  Huber value loss with value clipping (the sample
side reads old_value).  The mean, value and per-transition log_std are bfloat16 numbers, the action float32; the three
paths are
  bf16:  the bfloat16 entry on bfloat16 mean, value and per-transition log_std (what an autocast policy now runs);
  fp32:  the float32 entry on the same values held in float32 (what a float32 policy pays);
  cast:  .float() on mean, v_pred and a per-transition log_std, the float32 entry, then .bfloat16() on g_mean, g_value and
         a per-transition g_log_std (what a bfloat16 policy ran before the bfloat16 entry existed), timed as one sequence.

Timing: CUDA events around each launch or sequence, after warm-up.  Before each one the L2 is flushed (256 MiB device
write, then 256 MiB device read, as bench.py does) and a ~0.5 ms device sleep is queued, so the host has enqueued the timed
work before the GPU reaches it: the events measure device time, not Python.  The three paths alternate in two rounds of
`reps` launches each; the reported time is the median of the two rounds' medians.  Algorithmic bytes per transition follow
the K4c benchmark's accounting: float32 20 D + 25 per transition (mean, log_std, action in; d mean, d log_std out; v_pred,
old_logp, old_value, ret, adv, on_reset_next in; d v_pred out) and 12 D + 25 shared; with a bfloat16 policy side 12 D + 21
and 8 D + 21.  The cast path is charged the bfloat16 bytes, the work its caller needs done.  The roofline denominator is
6550 GB/s, the measured copy bandwidth of DESIGN.md.  The card's name and power limit are read in the same run.
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

import torch  # noqa: E402

PEAK_GBS = 6550.0
SHAPES = [(128, 4096, 6, False), (128, 4096, 6, True), (128, 4096, 17, False), (128, 4096, 17, True),
          (160, 65536, 17, False)]


def card():
    info = dict(name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["nvidia_smi"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
    except (OSError, subprocess.SubprocessError):
        info["nvidia_smi"] = None
    return info


def smem_per_cta(D, shared, elem):
    """ppo_loss_from_gaussian's dynamic shared memory (srl_b200/csrc/ppo_loss_gaussian.cu): the [256, D] mean block (and a
    per-row log_std block) of the element type, the float [256, D] action block, the mbarrier."""
    return (1 if shared else 2) * 256 * D * elem + 256 * D * 4 + 16


def make_inputs(T, N, D, shared, dev, seed):
    """bfloat16 mean, value and per-transition log_std (a shared log_std float32 [D]), a float32 action sampled from the
    head, the sample side with old_logp perturbed around the head's log-prob, and the statistics."""
    g = torch.Generator(device=dev).manual_seed(seed)
    f = lambda *s: torch.randn(*s, device=dev, generator=g)
    mean = f(T, N, D).bfloat16()
    log_std = (0.3 * f(D) - 0.5) if shared else (0.3 * f(T, N, D) - 0.5).bfloat16()
    action = (mean.float() + log_std.float().exp() * f(T, N, D)).contiguous()
    with torch.no_grad():
        lp0 = torch.distributions.Normal(mean.float(), log_std.float().exp()).log_prob(action).sum(-1)
    old_value, ret, adv = f(T + 1, N), f(T + 1, N), f(T + 1, N)
    on_reset = (torch.rand(T + 1, N, device=dev, generator=g) < 0.01).to(torch.uint8)
    v_pred = (old_value[:T] + 0.1 * f(T, N)).bfloat16()
    old_logp = (lp0 + 0.15 * f(T, N)).contiguous()
    del lp0
    mask = 1.0 - on_reset[1:].double()
    x = adv[:T].double() * mask
    stats = torch.tensor([mask.sum().item(), x.sum().item(), x.square().sum().item(), 0, 0, 0, 0, 0], dtype=torch.float64,
                         device=dev)
    smp = (old_logp, old_value[:T], ret[:T], adv[:T], on_reset[1:])
    return mean, log_std, action, v_pred, smp, stats


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "k4c_bf16_gaussian.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device: nothing here is measured on the CPU")
    from srl_b200 import ops

    dev = torch.device("cuda")
    props = torch.cuda.get_device_properties(0)
    sm_smem = getattr(props, "shared_memory_per_multiprocessor", None)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    flush_rd = torch.zeros(64 << 20, dtype=torch.int32, device=dev)
    hp = ops.LossHyper(clip_value=True, value_loss="huber", value_loss_config=dict(delta=10.0))

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

    results = []
    for si, (T, N, D, shared) in enumerate(SHAPES):
        mean, log_std, action, v_pred, smp, stats = make_inputs(T, N, D, shared, dev, seed=si)
        mean32, v_pred32 = mean.float(), v_pred.float()
        log_std32 = log_std if shared else log_std.float()

        def bf16(want=False):
            return ops.ppo_loss_from_gaussian(mean, log_std, action, v_pred, *smp, stats, hp, want_logp_entropy=want)

        def fp32():
            return ops.ppo_loss_from_gaussian(mean32, log_std32, action, v_pred32, *smp, stats, hp)

        def cast(want=False):
            g_mean, g_ls, g_v, out, out32, lp, en = ops.ppo_loss_from_gaussian(
                mean.float(), log_std if shared else log_std.float(), action, v_pred.float(), *smp, stats, hp,
                want_logp_entropy=want)
            return (g_mean.bfloat16(), g_ls if shared else g_ls.bfloat16(), g_v.bfloat16(), out, out32, lp, en)

        # the bfloat16 entry against the cast path on the same values: per-transition outputs (logp and entropy asked for
        # here only) and the shared [D] gradient, counted where not identical
        a, b = bf16(True), cast(True)
        torch.cuda.synchronize()
        agree = dict(g_mean_elements_differ=int((a[0] != b[0]).sum()), g_log_std_elements_differ=int((a[1] != b[1]).sum()),
                     g_value_differ=int((a[2] != b[2]).sum()), logp_differ=int((a[5] != b[5]).sum()),
                     entropy_differ=int((a[6] != b[6]).sum()), loss_abs=abs(float(a[3][0]) - float(b[3][0])))
        del a, b
        ls_kind = "shared [D] float32" if shared else "per transition [T, N, D]"
        print(json.dumps(dict(T=T, N=N, D=D, log_std=ls_kind, agreement_bf16_vs_cast=agree)), flush=True)
        bpt = {"bf16": (8 * D + 21) if shared else (12 * D + 21), "fp32": (12 * D + 25) if shared else (20 * D + 25)}
        bpt["cast"] = bpt["bf16"]
        line = dict(T=T, N=N, D=D, log_std=ls_kind, bytes_per_transition=bpt, agreement=agree)
        runs = {"bf16": [], "fp32": [], "cast": []}
        for _ in range(2):
            for name, fn in (("bf16", bf16), ("fp32", fp32), ("cast", cast)):
                runs[name].append(timed(fn))
        for name, ts in runs.items():
            nbytes = bpt[name] * T * N
            med = statistics.median(t["median_us"] for t in ts)
            entry = dict(median_us=med, rounds=ts, algorithmic_bytes=nbytes, gbs=nbytes / (med * 1e3),
                         of_6550=nbytes / (med * 1e3) / PEAK_GBS)
            if name != "cast":
                entry.update(dynamic_smem_per_cta=smem_per_cta(D, shared, 2 if name == "bf16" else 4))
            line[name] = entry
        line["fp32_over_bf16"] = line["fp32"]["median_us"] / line["bf16"]["median_us"]
        line["cast_over_bf16"] = line["cast"]["median_us"] / line["bf16"]["median_us"]
        print(json.dumps({k: v for k, v in line.items() if k not in ("bf16", "fp32", "cast")} |
                         {k: round(line[k]["median_us"], 1) for k in ("bf16", "fp32", "cast")}), flush=True)
        results.append(line)
        del mean, mean32, log_std, log_std32, action, v_pred, v_pred32, smp
        torch.cuda.empty_cache()
    doc = dict(what="K4c srl_ppo_loss_from_gaussian_bf16 vs the float32 entry on the same values vs the cast path "
                    "(.float() on mean, value and a per-transition log_std, the float32 entry, .bfloat16() on the "
                    "gradients)",
               card=card(), shared_memory_per_sm=sm_smem, reps=args.reps, warmup=args.warmup,
               loss="huber (delta 10) with value clipping",
               timing="CUDA events per launch; L2 flushed (256 MiB write + 256 MiB read) and a device sleep queued before "
                      "each; median over reps, two alternating rounds per path, median of the two", roofline_gbs=PEAK_GBS,
               results=results)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(doc, fh, indent=1)
    print(json.dumps(dict(card=doc["card"])), flush=True)


if __name__ == "__main__":
    main()
