"""The statistics pass on real GPUs: kernel -> ONE NCCL all-reduce -> finalise, two ranks (needs >= 2 CUDA devices).

Reference: preprocess/compute_mel_stats.py:19-36 (single process).  Here every rank runs the fused kernel (peak normalisation +
log-mel + pad-to-4 + per-bin fp64 moments) over its shard of the clips, the shards are combined by exactly one all-reduce of
2 * 80 + 1 fp64 values over NCCL, and every rank must print the two lines the reference printed for the same files
(tests/golden/MANIFEST.json, minted from the unmodified reference)."""
import json
import os
import socket
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    import audio_calm_b200 as acb
    from audio_calm_b200 import sharding
    from oracle import logmel_oracle as o
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    device = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=device)
    fe = acb.LogMelFrontend(device)
    three = [o.hash_noise(16000, 1), o.hash_noise(40000, 2), o.hash_noise(100001, 3)]      # the files of MANIFEST["stats_three_files"]
    four = three + [o.synth_clip(24001, 12)]
    res = {}
    for tag, waves in (("three", three), ("four", four)):
        mine = sharding.balanced_shards([len(w) for w in waves], world)[rank]
        acc = acb.MelStatsAccumulator(80, device)
        if len(mine):
            batch = acb.pack_clips([torch.from_numpy(waves[i]) for i in mine], device)
            fe.forward_ragged(batch, pad_multiple=4, peak=fe.peak_abs_ragged(batch), moments=acc, stats_only=True)   # the KERNEL's moments
        calls = {"n": 0}
        real = dist.all_reduce

        def counting(*a, **k):
            calls["n"] += 1
            return real(*a, **k)
        dist.all_reduce = counting
        acc.all_reduce()
        dist.all_reduce = real
        st = acc.finalize()
        res[tag] = {"lines": st.lines(), "mean": st.bin_mean.tolist(), "std": st.bin_std.tolist(), "frames": st.frames,
                    "count": st.count, "calls": calls["n"], "mine": [int(i) for i in mine],
                    "backend": dist.get_backend(), "device": torch.cuda.get_device_name(device)}
    fe.check()
    with open(os.path.join(out_dir, f"r{rank}.json"), "w") as f:
        json.dump(res, f)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two CUDA devices")
def test_stats_pass_kernel_allreduce_finalise_two_ranks(tmp_path, manifest):
    import torch.multiprocessing as mp
    from oracle import logmel_oracle as o
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    r = [json.load(open(tmp_path / f"r{k}.json")) for k in range(world)]
    want = manifest["stats_three_files"]
    fe_tables = __import__("audio_calm_b200").tables.calm_tables()
    window, fb = fe_tables[0].numpy(), fe_tables[1].numpy()
    four = [o.hash_noise(16000, 1), o.hash_noise(40000, 2), o.hash_noise(100001, 3), o.synth_clip(24001, 12)]
    mels = [o.dataset_mel(w[None], window, fb) for w in four]
    s, s2, frames = o.stats_per_bin(mels)
    bm, bs = o.stats_per_bin_finalise(s, s2, frames)
    for x in r:
        assert x["three"]["backend"] == "nccl"
        assert x["three"]["calls"] == 1 and x["four"]["calls"] == 1                      # exactly one collective per pass
        assert x["three"]["lines"] == want["printed"]                                      # what the reference printed for these files
        assert x["three"]["count"] == want["total_count"]                                  # exact
        assert x["four"]["frames"] == frames
        assert np.max(np.abs(np.array(x["four"]["mean"]) - bm)) < 1e-5 and np.max(np.abs(np.array(x["four"]["std"]) - bs)) < 1e-5
    assert sorted(r[0]["four"]["mine"] + r[1]["four"]["mine"]) == [0, 1, 2, 3]             # disjoint cover of the utterances
    assert r[0]["three"]["mean"] == r[1]["three"]["mean"] and r[0]["four"]["std"] == r[1]["four"]["std"]   # identical on every rank
