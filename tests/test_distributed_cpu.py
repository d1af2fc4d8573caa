"""World-size-2 gloo tests of the multi-rank contract (SURVEY.md §8e, F4), after the reference's own pattern
(legacy/tests/modules_test.py:273-299): every rank owns a slice of the environments; the ONLY data-path
collective is the SUM all-reduce of the float64 statistics table; normalising each shard with the reduced
table must reproduce the whole-batch normalisation, while the masked means stay rank-local."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _lane_part(adv, ret, done, trunc, on_reset, lo, hi):
    """numpy restatement of the per-lane table K2 emits (include/srl_b200.h, SRL_LANE_PART rows)."""
    mask = 1.0 - on_reset[lo + 1:hi + 1].astype(np.float64)
    x, y = adv[lo:hi].astype(np.float64) * mask, ret[lo:hi].astype(np.float64) * mask
    rows = [mask.sum(0), x.sum(0), np.square(x).sum(0), y.sum(0), np.square(y).sum(0),
            done[lo:hi].astype(np.float64).sum(0), trunc[lo:hi].astype(np.float64).sum(0), np.zeros(adv.shape[1])]
    return np.stack(rows)


def _worker(rank, world, port, tmp):
    sys.path.insert(0, ROOT)
    from oracle import ref_math as M
    from srl_b200 import synth
    from srl_b200.hotpath import exchange_stats
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    cfg = synth.PathConfig("dist", T=12, B=16, epochs=2, minibatches=2, p_end=0.1)
    s = synth.make_sample_scalars(cfg, seed=0)  # the same whole batch on every rank; each keeps its env slice
    t = {k: torch.from_numpy(v.reshape(cfg.L, cfg.N)).float() for k, v in s.items()}
    adv, ret = M.adv_and_value_target_ref(t["reward"], t["value"], t["truncated"], t["done"], t["on_reset"], 0.99, 0.97)
    adv, ret = M.pad_last_row(adv).numpy(), M.pad_last_row(ret).numpy()
    lo, hi = 0, cfg.T
    per = cfg.N // world
    mine = slice(rank * per, (rank + 1) * per)
    part = _lane_part(adv[:, mine], ret[:, mine], s["done"].reshape(cfg.L, -1)[:, mine],
                      s["truncated"].reshape(cfg.L, -1)[:, mine], s["on_reset"].reshape(cfg.L, -1)[:, mine], lo, hi)
    # statistics table: row 0 = this rank's whole slice, rows 1.. = its minibatches (local permutation of its envs)
    E, Mb = cfg.epochs, cfg.minibatches
    rows = [part.sum(1)]
    n = per // Mb
    for e in range(E):
        perm = M.philox_perm_ref(123, e, per)
        rows += [part[:, perm[j * n:(j + 1) * n]].sum(1) for j in range(Mb)]
    local = torch.from_numpy(np.stack(rows))
    glob = exchange_stats(local, torch.zeros_like(local))
    # (1) row 0 equals the whole-batch sums the reference would all-reduce (utils.py:58-61)
    mask_all = 1 - t["on_reset"][lo + 1:hi + 1]
    cnt, s1, s2 = M.masked_sums_ref(torch.from_numpy(adv[lo:hi]), mask_all)
    np.testing.assert_allclose(glob[0, :3].numpy(), [float(cnt), float(s1), float(s2)], rtol=1e-12)
    # (2) normalising the shard with the reduced sums == the shard of the whole-batch normalisation
    whole = M.masked_normalization_ref(torch.from_numpy(adv[lo:hi]), mask_all)
    shard = M.masked_normalization_ref(torch.from_numpy(adv[lo:hi, mine]), mask_all[:, mine],
                                       global_sums=tuple(glob[0, :3]))
    np.testing.assert_array_equal(shard.numpy(), whole[:, mine].numpy())
    # (3) the masked means stay local: sum(mask) of the shard is the LOCAL table entry, not the reduced one
    assert float(local[0, 0]) == float(mask_all[:, mine].sum()) and float(glob[0, 0]) == float(mask_all.sum())
    # (4) PopArt batch statistics (rows 3, 4) reduce to the whole-batch values as well (utils.py:121-124)
    y = torch.from_numpy(ret[lo:hi]).double() * mask_all.double()
    np.testing.assert_allclose(glob[0, 3:5].numpy(), [float(y.sum()), float(y.square().sum())], rtol=1e-12)
    with open(os.path.join(tmp, f"ok{rank}"), "w") as f:
        f.write("ok")
    dist.destroy_process_group()


def test_two_rank_stats_exchange_gloo(tmp_path):
    port = _free_port()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").exists() and (tmp_path / "ok1").exists()


def test_reference_arm_prints_one_line_for_rank0_only():
    """bench.py --impl reference under a 2-rank launch: rank 0 prints the JSON line, the others exit 0 silently."""
    import json
    import subprocess
    env = dict(os.environ, WORLD_SIZE="2", LOCAL_RANK="1", RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--config", "cfg1_atari_cpu", "--steps", "2", "--warmup", "1"], env=env, capture_output=True,
                         text=True, timeout=600)
    assert out.returncode == 0 and out.stdout.strip() == ""
    env.update(RANK="0", LOCAL_RANK="0")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--config", "cfg1_atari_cpu", "--steps", "2", "--warmup", "1"], env=env, capture_output=True,
                         text=True, timeout=600)
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "transitions/s" and line["value"] > 0
    assert line["steps"] == 2 and line["e2e"]["h2d_bytes_per_step"] == 0
    # "reference": the unmodified reference functions, where their files are staged (oracle/ref_loader.py); "port" (the
    # oracle restatement, no per-stage split) exactly when they are not
    from oracle import ref_loader
    if ref_loader.available():
        assert line["cpu_baseline"]["kind"] == "reference" and line["cpu_baseline"]["stages"]["gae_ms"] > 0
    else:
        assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["stages"] is None
