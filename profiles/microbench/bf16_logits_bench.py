"""K4b with a bfloat16 policy side: srl_ppo_loss_from_logits(_masked)_bf16 against the float32 entry and against the cast
path a bfloat16 policy had without it, on the same values.

    python profiles/microbench/bf16_logits_bench.py [--reps 300] [--warmup 20] [--out FILE.json]

Shapes: T = 128, N = 4096 (cfg2's minibatch) with heads (18,) (Atari), (36,) with a mask (SMAC 27m, 30 % of the actions
unavailable, action 0 of every head always available) and (11, 11, 11, 2, 2) (hide-and-seek); and cfg5's HBM-resident
shape, T = 160, N = 65536 with heads (11, 11, 11, 2, 2), whose ~1.5 GB float32 logits block is far larger than the L2.
cfg3's loss (PopArt, dual clip, huber).  The logits and values are bfloat16 numbers; the three paths are
  bf16:  the bfloat16 entry on bfloat16 logits and value (what an autocast policy now runs);
  fp32:  the float32 entry on the same values held in float32 (what a float32 policy pays);
  cast:  logits.float(), v_pred.float(), the float32 entry, then g_logits.bfloat16() and g_value.bfloat16() (what a
         bfloat16 policy ran before the bfloat16 entry existed), timed as one sequence.

Timing: CUDA events around each launch or sequence, after warm-up.  Before each one the L2 is flushed (256 MiB device
write, then 256 MiB device read, as bench.py does) and a ~0.5 ms device sleep is queued, so the host has enqueued the timed
work before the GPU reaches it: the events measure device time, not Python.  The three paths alternate in two rounds of
`reps` launches each; the reported time is the median of the two rounds' medians.  Algorithmic bytes per transition are
bench.py's K4b accounting: 8 sum K + 4 heads + 25 in float32 (logits in, d logits out, actions, v_pred, old_logp,
old_value, ret, adv, on_reset_next in, d v_pred out), 4 sum K + 4 heads + 21 with a bfloat16 policy side, plus sum K for a
mask.  The cast path is charged the bfloat16 bytes, the work its caller needs done.  The roofline denominator is 6550 GB/s,
the measured copy bandwidth of DESIGN.md.  The card's name and power limit are read in the same run.
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
SHAPES = [(128, 4096, (18,), False), (128, 4096, (36,), True), (128, 4096, (11, 11, 11, 2, 2), False),
          (160, 65536, (11, 11, 11, 2, 2), False)]


def card():
    info = dict(name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["nvidia_smi"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
    except (OSError, subprocess.SubprocessError):
        info["nvidia_smi"] = None
    return info


def smem_per_cta(sk, masked, elem):
    """ppo_loss_from_logits' shared-memory layout (srl_b200/csrc/ppo_loss.cu): the [256, sum K] block of the element type,
    the float exponentials when they fit, the [256, sum K] mask bytes, the mbarrier."""
    row, e, mask = 256 * sk * elem, 256 * sk * 4, (256 * sk if masked else 0)
    cache_e = row + e + mask + 16 <= 200 * 1024
    return row + (e if cache_e else 0) + mask + 16, cache_e


def make_inputs(T, N, heads, masked, dev, seed):
    """bfloat16 logits (scale 2), actions sampled from the (masked) per-head distributions, a mask with 30 % of the
    actions unavailable and action 0 of every head available (or None), the sample side and the statistics."""
    g = torch.Generator(device=dev).manual_seed(seed)
    sk = sum(heads)
    logits = (2.0 * torch.randn(T, N, sk, device=dev, generator=g)).bfloat16()
    avail = None
    z = logits.float()
    if masked:
        avail = (torch.rand(T, N, sk, device=dev, generator=g) >= 0.3).to(torch.uint8)
        off = 0
        for k in heads:
            avail[..., off] = 1
            off += k
        z = z.masked_fill(avail == 0, -1e10)
    acts, lps, off = [], [], 0
    for k in heads:
        lsm = torch.log_softmax(z[..., off:off + k], -1)
        a = torch.multinomial(lsm.exp().view(-1, k), 1, generator=g).view(T, N)
        acts.append(a)
        lps.append(lsm.gather(-1, a.unsqueeze(-1))[..., 0])
        off += k
    actions = torch.stack(acts, -1).to(torch.int32).contiguous()
    lp0 = torch.stack(lps, -1).sum(-1)
    f = lambda *s: torch.randn(*s, device=dev, generator=g)
    old_value, ret, adv = f(T + 1, N), f(T + 1, N), f(T + 1, N)
    on_reset = (torch.rand(T + 1, N, device=dev, generator=g) < 0.01).to(torch.uint8)
    v_pred = (old_value[:T] + 0.1 * f(T, N)).bfloat16()
    old_logp = (lp0 + 0.15 * f(T, N)).contiguous()
    mask = 1.0 - on_reset[1:].double()
    x = adv[:T].double() * mask
    stats = torch.tensor([mask.sum().item(), x.sum().item(), x.square().sum().item(), 0, 0, 0, 0, 0], dtype=torch.float64,
                         device=dev)
    smp = (old_logp, old_value[:T], ret[:T], adv[:T], on_reset[1:])
    return logits, v_pred, actions, avail, smp, stats


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(tempfile.gettempdir(), "k4b_bf16_logits.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device: nothing here is measured on the CPU")
    from srl_b200 import ops

    dev = torch.device("cuda")
    props = torch.cuda.get_device_properties(0)
    sm_smem = getattr(props, "shared_memory_per_multiprocessor", None)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    flush_rd = torch.zeros(64 << 20, dtype=torch.int32, device=dev)
    popart = torch.tensor([0.5, 2.0], dtype=torch.float64, device=dev)
    hp = ops.LossHyper(dual_clip=True, c_clip=3.0, value_loss="huber", value_loss_config=dict(delta=10.0),
                       value_loss_weight=1.0)

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
    for si, (T, N, heads, masked) in enumerate(SHAPES):
        logits, v_pred, actions, avail, smp, stats = make_inputs(T, N, heads, masked, dev, seed=si)
        logits32, v_pred32 = logits.float(), v_pred.float()
        kw = dict(popart_mean_std=popart, available=avail)

        def bf16(want=False):
            return ops.ppo_loss_from_logits(logits, actions, heads, v_pred, *smp, stats, hp, want_logp_entropy=want, **kw)

        def fp32():
            return ops.ppo_loss_from_logits(logits32, actions, heads, v_pred32, *smp, stats, hp, **kw)

        def cast(want=False):
            g, gv, out, out32, lp, en = ops.ppo_loss_from_logits(logits.float(), actions, heads, v_pred.float(), *smp, stats,
                                                                  hp, want_logp_entropy=want, **kw)
            return g.bfloat16(), gv.bfloat16(), out, out32, lp, en

        # the bfloat16 entry against the cast path on the same values: per-transition outputs (logp and entropy asked for
        # here only), counted where not identical
        a, b = bf16(True), cast(True)
        torch.cuda.synchronize()
        agree = dict(g_logits_elements_differ=int((a[0] != b[0]).sum()), g_value_differ=int((a[1] != b[1]).sum()),
                     logp_differ=int((a[4] != b[4]).sum()), entropy_differ=int((a[5] != b[5]).sum()),
                     loss_abs=abs(float(a[2][0]) - float(b[2][0])))
        del a, b
        print(json.dumps(dict(heads=list(heads), masked=masked, T=T, N=N, agreement_bf16_vs_cast=agree)), flush=True)
        sk = sum(heads)
        mask_b = sk if masked else 0
        bpt = {"bf16": 4 * sk + 4 * len(heads) + 21 + mask_b, "fp32": 8 * sk + 4 * len(heads) + 25 + mask_b}
        bpt["cast"] = bpt["bf16"]
        line = dict(T=T, N=N, heads=list(heads), sum_k=sk, masked=masked, bytes_per_transition=bpt, agreement=agree)
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
                smem, cache_e = smem_per_cta(sk, masked, 2 if name == "bf16" else 4)
                entry.update(smem_per_cta=smem, cache_e=cache_e,
                             ctas_per_sm_by_smem=None if sm_smem is None else int(sm_smem // (smem + 1024)))
            line[name] = entry
        line["fp32_over_bf16"] = line["fp32"]["median_us"] / line["bf16"]["median_us"]
        line["cast_over_bf16"] = line["cast"]["median_us"] / line["bf16"]["median_us"]
        print(json.dumps({k: v for k, v in line.items() if k not in ("bf16", "fp32", "cast")} |
                         {k: round(line[k]["median_us"], 1) for k in ("bf16", "fp32", "cast")}), flush=True)
        results.append(line)
        del logits, logits32, v_pred, v_pred32, actions, avail, smp
        torch.cuda.empty_cache()
    doc = dict(what="K4b srl_ppo_loss_from_logits(_masked)_bf16 vs the float32 entry on the same values vs the cast path "
                    "(.float() on logits and value, the float32 entry, .bfloat16() on the gradients)",
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
