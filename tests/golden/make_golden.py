"""Generates the golden vectors under tests/golden/ by running the LIVE reference hot path in this
container: torch 2.11.0+cu128, gloo backend, N local CPU processes wired per SetClusterSpec
(oracle/gloo_torchjob.replica_env).  The reference repo itself holds no test vectors (SURVEY.md §4),
so these runs are what pins oracle/allreduce_oracle.py.

    python tests/golden/make_golden.py        # rewrites the .npz / .json fixtures (seconds)

Fixtures
  allreduce_gloo_n{2,3,4,8}.npz  per world size: the seeded inputs of every rank (f32 and bf16 bit
      patterns), gloo's fp32 all_reduce of (x * 1/N) ["f32_prescaled"], of x ["f32_sum"], and gloo's
      native-dtype bf16 all_reduce of bf16(x)/N ["bf16_native"] (informational: gloo sums in bf16).
  sampler.json                    DistributedSampler indices for several (len, world, epoch, seed).
  mlp_torchjob_n2/                BASELINE config 0: 2-layer MLP, 1 master + 1 worker, gloo: losses,
      per-bucket pre/post tensors, argmax, final weights of rank 0 and 1 (the flat arrays as a
      seeded sample of their elements, indices in "sample_index").
"""
from __future__ import annotations

import json
import multiprocessing as mp
import os
import shutil
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

COUNT = 4099
SEED = 4242
MLP_SAMPLE = 1 << 12


def _rank(rank, world, port, q):
    import torch
    import torch.distributed as dist
    import harness
    from oracle.gloo_torchjob import replica_env
    os.environ.update(replica_env("golden", "master" if rank == 0 else "worker",
                                  0 if rank == 0 else rank - 1, world - 1, port))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    dist.init_process_group("gloo", init_method="env://")
    out = {}
    for pattern in ("randn", "wide"):
        x32 = harness.gen_input(SEED, rank, COUNT, "f32", pattern)
        xb = harness.gen_input(SEED, rank, COUNT, "bf16", pattern)
        t = torch.from_numpy(x32.copy())
        inv = torch.tensor(1.0 / world, dtype=torch.float32)
        a = t * inv
        dist.all_reduce(a)
        b = t.clone()
        dist.all_reduce(b)
        # bf16 inputs up-cast to fp32, pre-multiplied by fp32 1/N, gloo fp32 sum (SURVEY §8c-i)
        tb = harness.to_torch(xb, "bf16", "cpu")
        c = tb.float() * inv
        dist.all_reduce(c)
        # native bf16 wire, what the default hook does on a bf16 bucket: div_(N) then allreduce
        d = tb.clone().div_(world)
        dist.all_reduce(d)
        out[pattern] = dict(x32=x32, xb=xb, f32_prescaled=a.numpy(), f32_sum=b.numpy(),
                            bf16in_f32_prescaled=c.numpy(),
                            bf16_native=harness.from_torch(d, "bf16"))
    dist.destroy_process_group()
    q.put((rank, out))


def make_allreduce(world):
    from oracle.gloo_torchjob import free_port
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = free_port()
    ps = [ctx.Process(target=_rank, args=(r, world, port, q)) for r in range(world)]
    for p in ps:
        p.start()
    got = dict(q.get(timeout=300) for _ in range(world))
    for p in ps:
        p.join()
    arrays = {}
    for pattern in ("randn", "wide"):
        for r in range(world):
            arrays["%s_x32_r%d" % (pattern, r)] = got[r][pattern]["x32"]
            arrays["%s_xb_r%d" % (pattern, r)] = got[r][pattern]["xb"]
        for k in ("f32_prescaled", "f32_sum", "bf16in_f32_prescaled", "bf16_native"):
            for r in range(1, world):  # every rank must hold the same bits
                assert np.array_equal(got[0][pattern][k].view(np.uint8),
                                      got[r][pattern][k].view(np.uint8)), (k, r)
            arrays["%s_%s" % (pattern, k)] = got[0][pattern][k]
    np.savez_compressed(os.path.join(HERE, "allreduce_gloo_n%d.npz" % world), **arrays)


def make_sampler():
    import torch
    from torch.utils.data.distributed import DistributedSampler

    class DS(torch.utils.data.Dataset):
        def __init__(self, n):
            self.n = n

        def __len__(self):
            return self.n

        def __getitem__(self, i):
            return i

    out = []
    for n, world, epoch, seed, shuffle, drop_last in [
            (10, 2, 0, 0, True, False), (10, 3, 1, 0, True, False), (11, 4, 2, 7, True, False),
            (3, 8, 0, 0, True, False), (100, 8, 5, 1234, True, False), (17, 4, 0, 0, False, False),
            (17, 4, 3, 9, True, True), (64, 8, 0, 0, True, True)]:
        per_rank = []
        perm = None
        for r in range(world):
            s = DistributedSampler(DS(n), num_replicas=world, rank=r, shuffle=shuffle, seed=seed,
                                   drop_last=drop_last)
            s.set_epoch(epoch)
            per_rank.append(list(iter(s)))
        if shuffle:
            g = torch.Generator()
            g.manual_seed(seed + epoch)
            perm = torch.randperm(n, generator=g).tolist()
        else:
            perm = list(range(n))
        out.append(dict(n=n, world=world, epoch=epoch, seed=seed, shuffle=shuffle,
                        drop_last=drop_last, perm=perm, indices=per_rank))
    with open(os.path.join(HERE, "sampler.json"), "w") as f:
        json.dump(out, f)


def shrink_mlp_dump(d):
    """Keep the same fixed, seeded sample of MLP_SAMPLE elements of every flat per-parameter array
    (bucket tensors, final weights) so that each rank's fixture stays under 1 MB; the allreduce is
    element-wise, so the sampled elements are checked exactly as the full buckets would be."""
    for name in sorted(os.listdir(d)):
        if not name.endswith(".npz"):
            continue
        path = os.path.join(d, name)
        with np.load(path) as z:
            arrays = {k: z[k] for k in z.files}
        n = arrays["final_flat"].size
        idx = np.sort(np.random.RandomState(SEED).choice(n, MLP_SAMPLE, replace=False))
        for k, a in arrays.items():
            if a.shape == (n,):
                arrays[k] = a[idx]
        arrays["sample_index"] = idx.astype(np.int32)
        np.savez_compressed(path, **arrays)


def make_mlp():
    from oracle import gloo_torchjob
    d = os.path.join(HERE, "mlp_torchjob_n2")
    shutil.rmtree(d, ignore_errors=True)
    res = gloo_torchjob.run("mlp", world=2, steps=2, warmup=0, batch=64, threads=1, dtype="f32",
                            dump=d, job="golden-mlp")
    shrink_mlp_dump(d)
    with open(os.path.join(d, "run.json"), "w") as f:
        json.dump(dict(losses=res["losses"], steps=2, batch=64, lr=0.01, world=2), f)


if __name__ == "__main__":
    for w in (2, 3, 4, 8):
        make_allreduce(w)
    make_sampler()
    make_mlp()
    print("golden fixtures written to", HERE)
