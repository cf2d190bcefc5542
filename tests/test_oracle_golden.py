"""Pins oracle/allreduce_oracle.py against the golden vectors produced by the live reference hot
path (torch 2.11 gloo, tests/golden/make_golden.py).  CPU only."""
import json
import os

import numpy as np
import pytest

from oracle import allreduce_oracle as O

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(world):
    return np.load(os.path.join(GOLD, "allreduce_gloo_n%d.npz" % world))


@pytest.mark.parametrize("world", [2, 3, 4, 8])
@pytest.mark.parametrize("pattern", ["randn", "wide"])
def test_f32_prescaled_matches_gloo(world, pattern):
    g = load(world)
    ins = [g["%s_x32_r%d" % (pattern, r)] for r in range(world)]
    got = O.allreduce_oracle(ins, "f32", "f32", "f32", np.float32(1.0) / np.float32(world))
    want = g["%s_f32_prescaled" % pattern]
    if world == 2:  # a+b is order independent: bit-exact
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    # gloo's ring order differs from rank order for N>2: norm-wise tolerance stated by north_star
    err = np.abs(got.astype(np.float64) - want.astype(np.float64)).max()
    assert err / np.abs(want).max() <= 1e-5
    assert err / np.abs(want).max() <= 1e-6  # observed ~1e-7 (SURVEY §7.3-4)


@pytest.mark.parametrize("world", [2, 3, 4, 8])
def test_f32_post_scale_matches_sum_then_scale(world):
    g = load(world)
    ins = [g["randn_x32_r%d" % r] for r in range(world)]
    got = O.allreduce_oracle(ins, "f32", "f32", "f32", 1.0 / world, post=True)
    want = g["randn_f32_sum"].astype(np.float32) * np.float32(1.0 / world)
    assert np.abs(got - want).max() / np.abs(want).max() <= 1e-6


@pytest.mark.parametrize("world", [2, 3, 4, 8])
@pytest.mark.parametrize("pattern", ["randn", "wide"])
def test_bf16_wire_against_fp32_gloo_oracle(world, pattern):
    """bf16 bucket: inputs up-cast to fp32, pre-scaled, gloo fp32 sum, ONE rounding to bf16
    (SURVEY §8c-i) versus the oracle's bf16-wire path.  For power-of-two N the pre-scale is exact in
    bf16, so only the summation order can differ: at most one bf16 ulp on rare elements."""
    g = load(world)
    ins = [g["%s_xb_r%d" % (pattern, r)] for r in range(world)]
    got = O.allreduce_oracle(ins, "bf16", "bf16", "bf16", 1.0 / world)
    want = O.f32_to_bf16_bits(g["%s_bf16in_f32_prescaled" % pattern])
    ulp = O.ulp_distance(got, want, "bf16")
    if world == 2:
        assert ulp.max() == 0
    elif world in (4, 8):
        assert ulp.max() <= 1 and (ulp != 0).mean() < 0.01
    else:  # N=3: x*(1/3) is rounded to bf16 on the wire before the sum -> bf16-resolution error,
        # judged norm-wise (ulp distance is meaningless next to cancellations)
        a, b = O.to_f32(got, "bf16").astype(np.float64), O.to_f32(want, "bf16").astype(np.float64)
        assert np.abs(a - b).max() / np.abs(b).max() <= 2.0 ** -7


def test_native_bf16_gloo_is_not_the_target():
    """Informational golden: gloo sums a bf16 bucket IN bf16 (22-52% of elements differ from the
    fp32-accumulated sum for N>=3, SURVEY §7.3-4); the oracle is strictly more accurate."""
    g = load(8)
    ins = [g["randn_xb_r%d" % r] for r in range(8)]
    ours = O.to_f32(O.allreduce_oracle(ins, "bf16", "bf16", "bf16", 0.125), "bf16")
    native = O.to_f32(g["randn_bf16_native"], "bf16")
    exact = O.allreduce_f32_unrounded(ins, "bf16", "bf16", 0.125)
    assert np.abs(ours - exact).mean() <= np.abs(native - exact).mean()
    assert (ours != native).mean() > 0.05


def test_bf16_rounding_matches_torch():
    import torch
    rs = np.random.RandomState(0)
    x = (rs.standard_normal(200000) * np.exp(rs.uniform(-30, 30, 200000))).astype(np.float32)
    x[:4] = [0.0, -0.0, np.inf, -np.inf]
    want = torch.from_numpy(x).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)
    assert np.array_equal(O.f32_to_bf16_bits(x), want)
    back = torch.from_numpy(want.view(np.int16)).view(torch.bfloat16).float().numpy()
    assert np.array_equal(O.bf16_bits_to_f32(want).view(np.uint32), back.view(np.uint32))


def test_sampler_sharding_golden():
    cases = json.load(open(os.path.join(GOLD, "sampler.json")))
    assert len(cases) >= 8
    for c in cases:
        for r in range(c["world"]):
            got = O.shard_indices(c["perm"], r, c["world"], c["drop_last"])
            assert got == c["indices"][r], c


def test_mlp_bucket_golden():
    """BASELINE config 0 (MLP, 1 master + 1 worker, gloo): every recorded gradient bucket's
    post-allreduce tensor equals the oracle applied to the two replicas' pre tensors, bit for bit
    (N=2, fp32), on the fixture's seeded sample of bucket elements."""
    d = os.path.join(GOLD, "mlp_torchjob_n2")
    r0 = np.load(os.path.join(d, "rank0.npz"))
    r1 = np.load(os.path.join(d, "rank1.npz"))
    pres = sorted(k for k in r0.files if k.endswith("_pre"))
    assert pres
    for k in pres:
        want = r0[k.replace("_pre", "_post")]
        got = O.allreduce_oracle([r0[k], r1[k]], "f32", "f32", "f32", 0.5)
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), k
    assert np.array_equal(r0["final_flat"].view(np.uint32), r1["final_flat"].view(np.uint32))
