"""Parity tests proper: the CUDA hot path, called through the C ABI (Communicator -> libtok8s.so),
against oracle/allreduce_oracle.py on the same seeded inputs and against the committed gloo goldens.

Bars (stated per north_star): peer-memory algorithms (local / one-shot / two-shot) are BIT-EXACT
against the rank-ordered fp32-accumulation oracle for every dtype triple; NVLS (in-switch reduction,
unspecified order and rounding) is held to <= 1e-5 norm-wise for an fp32 wire and to <= 1 wire-ulp
for 16-bit wires.  Replicas run as processes (product shape) or threads; with a single visible GPU
they all share cuda:0, with several GPUs each replica gets its own.
"""
import os

import numpy as np
import pytest

import harness

pytestmark = pytest.mark.gpu

SHARED_ENV = {"TOK_MAX_CTAS": "16", "TOK_STAGING_MB": "32", "TOK_BARRIER_TIMEOUT_MS": "60000",
              "TOK_SYMM_POOL_MB": "160"}


def devices_for(world, n_gpus):
    if n_gpus >= world:
        return list(range(world)), {}
    return [0] * world, dict(SHARED_ENV)


def assert_all_exact(results, expect_cases, world):
    s = harness.summarize(results)
    assert s["total"] == expect_cases * world, s
    assert s["bad"] == 0, s["worst"]


def test_world1_local_kernel(tok_lib):
    """world 1 = the fused scale/cast alone: the LDG.128 wave for every dtype triple, and the
    cp.async.bulk (TMA) variant for the one-dtype cases (algo 7) incl. ragged tails and sizes that are
    not a whole number of 16 KiB tiles."""
    cases = harness.standard_cases(1, algos=(0,), quick=False)
    seed = 4000
    for dt in ("bf16", "f32", "f16"):
        for n in (1, 7, 8, 9, 4097, 8192, 65536 + 3, (1 << 20) + 5, 3 * (1 << 20) + 8):
            for post in (False, True):
                seed += 1
                cases.append(dict(count=n, **{"in": dt, "wire": dt, "out": dt}, algo=7, seed=seed,
                                  scale=1.0 / 3.0, post=post, pattern="wide",
                                  inplace=(seed % 2 == 0), expect_kernel="local_tma"))
    res = harness.launch(1, cases, devices=[0], mode="thread", timeout=300)
    assert_all_exact(res, len(cases), 1)


def test_world1_identity_bucket_is_elided(tok_lib):
    """in == out, one dtype, scale 1 at world 1 is already the answer: no launch, no HBM pass — unless
    the caller insists (TOK_FLAG_NO_ELIDE), in which case the kernel runs and changes nothing."""
    import tempfile
    import torch
    from torch_on_k8s_b200.comm import Communicator
    comm = Communicator("elide", 0, 1, 0, rendezvous_path=os.path.join(tempfile.mkdtemp(), "r"))
    try:
        x = torch.randn(1 << 20, device="cuda").to(torch.bfloat16)
        ref = x.clone()
        comm.allreduce_bucket(x, x, scale=1.0)
        st = comm.stats()
        assert (st.launches, st.elided) == (0, 1)
        comm.allreduce_bucket(x, x, scale=1.0, elide=False)
        torch.cuda.synchronize()
        st = comm.stats()
        assert (st.launches, st.elided) == (1, 1) and torch.equal(x, ref)
        comm.allreduce_bucket(x, x, scale=0.5)           # real work is never elided
        torch.cuda.synchronize()
        assert comm.stats().launches == 2 and torch.equal(x, (ref.float() * 0.5).to(torch.bfloat16))
    finally:
        comm.close()


@pytest.mark.parametrize("world", [2, 3, 4, 8])
def test_p2p_bit_exact_processes(tok_lib, n_gpus, world):
    """one-shot and two-shot over peer-mapped HBM, one process per replica."""
    devs, env = devices_for(world, n_gpus)
    cases = harness.standard_cases(world, algos=(2, 3), quick=(n_gpus < world))
    res = harness.launch(world, cases, devices=devs, mode="proc", timeout=600, env=env)
    assert_all_exact(res, len(cases), world)


@pytest.mark.parametrize("world", [2, 5, 8])
def test_p2p_bit_exact_threads(tok_lib, n_gpus, world):
    devs, env = devices_for(world, n_gpus)
    env = dict(env or SHARED_ENV)
    # AUTO is only bit-exact while it cannot pick NVLS (replicas sharing a GPU have no multicast)
    algos = (2, 3, 0) if n_gpus < world else (2, 3)
    cases = harness.standard_cases(world, algos=algos, quick=True)
    res = harness.launch(world, cases, devices=devs, mode="thread", timeout=600, env=env)
    assert_all_exact(res, len(cases), world)


def test_large_bucket_is_chunked(tok_lib, n_gpus):
    """Buckets larger than the staging buffer are split into several launches (ResNet-50's
    28.9 MB bucket against a 4 MiB staging buffer), ragged tail included."""
    world = 2
    devs, env = devices_for(world, n_gpus)
    env = dict(env or {}, TOK_STAGING_MB="4", TOK_MAX_CTAS="16")
    cases = [dict(count=28878848 // 2 + 3, **{"in": "bf16", "wire": "bf16", "out": "bf16"}, algo=a,
                  seed=77 + a, scale=0.5) for a in (2, 3)]
    cases.append(dict(count=(9 << 20) + 1, **{"in": "f32", "wire": "bf16", "out": "f32"}, algo=3,
                      seed=81, scale=0.5))
    res = harness.launch(world, cases, devices=devs, mode="proc", timeout=600, env=env)
    assert_all_exact(res, len(cases), world)
    launches = [r["launches"] for r in res[0] if "launches" in r][0]
    assert launches > len(cases)  # chunking happened


def test_exact_patterns_full_resnet_buckets(tok_lib, n_gpus):
    """BASELINE full sizes through size-independent properties: with small-integer data every sum is
    exact in every dtype, so out == sum of inputs element-wise (checked against the oracle), for the
    three ResNet-50 bf16 buckets at the largest world this box offers."""
    world = 8 if n_gpus >= 8 else (n_gpus if n_gpus >= 2 else 4)
    devs, env = devices_for(world, n_gpus)
    cases = [dict(count=n // 2, **{"in": "bf16", "wire": "bf16", "out": "bf16"}, algo=0,
                  seed=900 + i, scale=1.0, pattern="ints")
             for i, n in enumerate((4098000, 28878848, 18137216))]
    res = harness.launch(world, cases, devices=devs, mode="proc", timeout=900, env=env)
    s = harness.summarize(res)
    assert s["bad"] == 0, s["worst"]


def test_golden_gloo_vectors(tok_lib, n_gpus):
    """The committed gloo fixtures (tests/golden/allreduce_gloo_n*.npz): our CUDA result on the same
    inputs vs what the reference-style gloo job produced — through the staged kernels (replicas as
    threads) and through the zero-copy path DDP's buckets take (replicas as processes: the
    arrival + exchange pair needs one CUDA context per replica)."""
    import torch
    from oracle import allreduce_oracle as O
    from torch_on_k8s_b200.comm import Communicator
    gold_dir = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    import tempfile
    import threading
    for world in (2, 4, 8):
        gpath = os.path.join(gold_dir, "allreduce_gloo_n%d.npz" % world)
        with np.load(gpath) as z:
            g = {k: z[k] for k in z.files}  # NpzFile is not thread-safe: materialise first
        devs, env = devices_for(world, n_gpus)
        os.environ.update(env or SHARED_ENV)
        path = os.path.join(tempfile.mkdtemp(prefix="tok8s-gold-"), "r")
        outs, errs = {}, []

        def body(r):
            try:
                torch.cuda.set_device(devs[r])
                comm = Communicator("gold", r, world, devs[r], rendezvous_path=path)
                st = torch.cuda.Stream(device=devs[r])
                with torch.cuda.stream(st):
                    x = torch.from_numpy(g["randn_x32_r%d" % r].copy()).to("cuda:%d" % devs[r])
                    xb = harness.to_torch(g["randn_xb_r%d" % r], "bf16", "cuda:%d" % devs[r])
                    comm.allreduce_bucket(x, x, scale=1.0 / world, stream=st)
                    st.synchronize()   # threads share one CUDA context: nothing queued behind a
                    comm.allreduce_bucket(xb, xb, scale=1.0 / world, stream=st)   # waiting kernel
                    st.synchronize()
                comm.status()
                outs[r] = (x.cpu().numpy(), harness.from_torch(xb, "bf16"))
                comm.close()
            except Exception as e:  # noqa: BLE001
                errs.append(repr(e))

        ts = [threading.Thread(target=body, args=(r,)) for r in range(world)]
        [t.start() for t in ts]
        [t.join(300) for t in ts]
        assert not errs, errs
        want = g["randn_f32_prescaled"]
        for r in range(world):
            got32, gotb = outs[r]
            err = np.abs(got32.astype(np.float64) - want.astype(np.float64)).max()
            assert err / np.abs(want).max() <= 1e-5, (world, r)   # north_star tolerance
            if world == 2:
                assert np.array_equal(got32.view(np.uint32), want.view(np.uint32))
            wantb = O.f32_to_bf16_bits(g["randn_bf16in_f32_prescaled"])
            ulp = O.ulp_distance(gotb, wantb, "bf16")
            assert ulp.max() <= 1 and (ulp != 0).mean() < 0.01, (world, r)
            assert np.array_equal(outs[0][0].view(np.uint32), got32.view(np.uint32))
        # zero-copy: the same fixtures through pool buckets (P2P in place; NVLS in place when every
        # replica has its own GPU and the group has >= 2 of them)
        cases = [dict(golden=gpath, algo=3, count=0, **{"in": "f32", "wire": "f32", "out": "f32"})]
        if n_gpus >= world:
            cases.append(dict(golden=gpath, algo=4, count=0, **{"in": "f32", "wire": "f32", "out": "f32"}))
        res = harness.launch(world, cases, devices=devs, mode="proc", timeout=600, env=env)
        s = harness.summarize(res)
        assert s["bad"] == 0 and s["total"] == len(cases) * world, s


def test_long_rendezvous_path(tok_lib, tmp_path):
    """A rendezvous path longer than a Unix socket address holds (108 bytes, easily reached under a
    deep temporary or shared directory) still forms the group and exchanges buckets."""
    import threading
    import torch
    from torch_on_k8s_b200.comm import Communicator
    os.environ.update(SHARED_ENV)
    d = tmp_path / ("d" * 120)
    d.mkdir()
    path = str(d / "r")
    outs, errs = {}, []

    def body(r):
        try:
            torch.cuda.set_device(0)
            comm = Communicator("long", r, 2, 0, rendezvous_path=path)
            st = torch.cuda.Stream(device=0)
            with torch.cuda.stream(st):
                x = torch.full((4096,), float(r + 1), device="cuda:0")
                comm.allreduce_bucket(x, x, scale=0.5, stream=st)
                st.synchronize()
            comm.status()
            outs[r] = x.cpu()
            comm.close()
        except Exception as e:  # noqa: BLE001
            errs.append(repr(e))

    ts = [threading.Thread(target=body, args=(r,)) for r in range(2)]
    [t.start() for t in ts]
    [t.join(120) for t in ts]
    assert not errs, errs
    for r in range(2):
        assert torch.equal(outs[r], torch.full((4096,), 1.5)), r


@pytest.mark.parametrize("world", [2, 3, 4])
def test_zero_copy_symmetric_pool(tok_lib, n_gpus, world):
    """Buckets allocated in the symmetric pool (torch.cuda.MemPool over tok_pool_malloc) are
    exchanged in place: 1-warp arrival + the P2P in-place kernel (reduce own sub-slab from every
    replica's bucket, push the result into every replica's bucket).  PRE and POST scaling are
    bit-exact vs the oracle at every world size (1/3 is not a power of two); the split
    arrive-then-exchange form gives the same bits; AUTO never picks a kernel that would change the
    function; an asymmetric allocation is detected by the arrival instead of corrupting gradients."""
    devs, env = devices_for(world, n_gpus)
    cases = []
    seed = 700
    for dt in ("bf16", "f32", "f16"):
        for n in (8, 4096, 65536 + 8, (1 << 20) + 64, 5 * (1 << 20)):
            seed += 1
            cases.append(dict(count=n, **{"in": dt, "wire": dt, "out": dt}, algo=3, seed=seed,
                              scale=1.0 / world, symm=True, split=(seed % 2 == 0),
                              pattern="wide" if seed % 3 == 0 else "randn",
                              expect_kernel="two_shot_inplace"))
        seed += 1
        cases.append(dict(count=(1 << 18) + 8, **{"in": dt, "wire": dt, "out": dt}, algo=3, seed=seed,
                          scale=1.0 / 3.0, post=True, symm=True, pattern="wide",
                          expect_kernel="two_shot_inplace"))
        seed += 1   # AUTO + PRE with a factor that is not a power of two must stay on the exact kernel
        # (> 16 MiB: below that AUTO takes the one-shot kernel at N=2, pool bucket or not)
        cases.append(dict(count=9 << 20, **{"in": dt, "wire": dt, "out": dt}, algo=0, seed=seed,
                          scale=1.0 / 3.0, symm=True, split=True, expect_kernel="two_shot_inplace"))
    # not a whole number of 16-byte packs -> staged path, still correct
    cases.append(dict(count=65536 + 3, **{"in": "bf16", "wire": "bf16", "out": "bf16"}, algo=3,
                      seed=799, scale=1.0 / world, symm=True, expect_kernel="two_shot"))
    cases.append(dict(count=1 << 20, **{"in": "bf16", "wire": "bf16", "out": "bf16"}, algo=3,
                      seed=800, scale=1.0 / world, symm=True, skew=True))
    res = harness.launch(world, cases, devices=devs, mode="proc", timeout=600, env=env)
    s = harness.summarize(res)
    assert s["bad"] == 0, s["worst"]
    assert s["total"] == len(cases) * world, (s["total"], [len(v) for v in res.values()])


@pytest.mark.parametrize("world", [2, 4])
def test_broadcast_bit_exact(tok_lib, n_gpus, world):
    """tok_broadcast (row f2): the root's bytes on every replica, for buffers in the symmetric pool
    (multicast push when a multicast object is bound, else pulled from the root) and anywhere else
    (through the root's staging buffer, chunked when larger than it), any root, ragged byte counts."""
    devs, env = devices_for(world, n_gpus)
    env = dict(env or {}, TOK_STAGING_MB="4")
    cases = []
    for i, n in enumerate((1, 15, 16, 4097, (1 << 20) + 3, (9 << 20) + 5)):
        cases.append(dict(count=n, bcast=i % world, **{"in": "u8", "wire": "u8", "out": "u8"}))
    for i, n in enumerate((16, 4096, (1 << 20) + 16, 6 << 20)):
        cases.append(dict(count=n, bcast=(i + 1) % world, symm=True,
                          **{"in": "u8", "wire": "u8", "out": "u8"}))
    res = harness.launch(world, cases, devices=devs, mode="proc", timeout=600, env=env)
    s = harness.summarize(res)
    assert s["bad"] == 0, s["worst"]
    assert s["total"] == len(cases) * world
    kernels = {r["kernel"] for r in res[0] if "kernel" in r}
    assert "bcast_staged" in kernels and ({"bcast_pull", "bcast_mc_push"} & kernels), kernels


def test_symmetric_pool_recycles_released_segments(tok_lib):
    """tok_pool_free is a real free: a released segment is handed out again (first fit, neighbours
    merged, the top of the pool shrinks back) — DDP's bucket rebuild after iteration 1 and a re-wrap
    after an elastic re-form do not leak the pool."""
    import tempfile
    import torch
    from torch_on_k8s_b200 import _ffi
    from torch_on_k8s_b200.comm import Communicator
    os.environ["TOK_SYMM_POOL_MB"] = "64"
    comm = Communicator("pool", 0, 1, 0, rendezvous_path=os.path.join(tempfile.mkdtemp(), "r"))
    try:
        import ctypes as C
        L = _ffi.lib()

        def alloc(mb):
            p = C.c_void_p()
            _ffi.check(L.tok_comm_symm_alloc(comm._h, mb << 20, C.byref(p)))
            return p.value

        base, size, used = comm.symm_info()
        a, b, c = alloc(8), alloc(8), alloc(8)
        assert (a, b, c) == (base, base + (8 << 20), base + (16 << 20))
        _ffi.check(L.tok_comm_symm_free(comm._h, C.c_void_p(a), 8 << 20))
        _ffi.check(L.tok_comm_symm_free(comm._h, C.c_void_p(b), 8 << 20))   # merges with a
        assert comm.symm_info()[2] == 8 << 20
        assert alloc(12) == base                       # first fit in the merged 16 MiB hole
        assert alloc(4) == base + (12 << 20)
        _ffi.check(L.tok_comm_symm_free(comm._h, C.c_void_p(c), 8 << 20))   # top shrinks back
        assert alloc(2) == base + (16 << 20)
        assert L.tok_comm_symm_free(comm._h, C.c_void_p(base + (40 << 20)), 2 << 20) != 0
        # through torch: a MemPool tensor that is dropped gives its segment back
        for _ in range(40):                            # 40 x 8 MiB through a 64 MiB pool
            t = comm.symm_empty(8 << 20, torch.uint8)
            assert comm.in_symmetric_pool(t)
            del t
            comm.mem_pool()                            # keep the pool object alive
            torch.cuda.synchronize()
            torch.cuda.memory.empty_cache()
    finally:
        comm.close()
        os.environ["TOK_SYMM_POOL_MB"] = SHARED_ENV["TOK_SYMM_POOL_MB"]


def test_nvls_tolerance(tok_lib, n_gpus):
    """NVLS needs one GPU per replica and NVSwitch multicast; skipped on a single-GPU box."""
    if n_gpus < 2:
        pytest.skip("NVLS multicast needs >= 2 GPUs")
    world = n_gpus
    cases = []
    for (a, w, o) in harness.TRIPLES_CORE:
        for n in (9, 4097, (1 << 20) + 5):
            cases.append(dict(count=n, **{"in": a, "wire": w, "out": o}, algo=4, seed=500 + n % 97,
                              scale=1.0 / world))
    for n in (70001, (1 << 21) + 8):   # AUTO picks NVLS for these sizes once world >= 3
        cases.append(dict(count=n, **{"in": "bf16", "wire": "bf16", "out": "bf16"}, algo=0,
                          seed=650 + n % 7, scale=1.0 / world))
    for dt in ("bf16", "f32"):   # zero-copy NVLS: in-switch reduce straight on the pool buckets
        for n in (4096, (1 << 20) + 64, 5 * (1 << 20)):
            cases.append(dict(count=n, **{"in": dt, "wire": dt, "out": dt}, algo=4, seed=600 + n % 89,
                              scale=1.0 / world, symm=True, split=(n == 4096),
                              expect_kernel="nvls_inplace"))
    # what DDP's buckets take in bench.py: AUTO on pool buckets of the real ResNet-50 sizes, 1/N PRE
    pow2 = world & (world - 1) == 0
    auto_kernel = "nvls_inplace" if (world >= 5 and pow2) else "two_shot_inplace"   # 3-4: P2P past 12 MiB
    exact_ids = set()
    for i, nbytes in enumerate((28256208, 22857856)):
        cases.append(dict(count=nbytes // 2, **{"in": "bf16", "wire": "bf16", "out": "bf16"}, algo=0,
                          seed=660 + i, scale=1.0 / world, symm=True, split=True,
                          expect_kernel=auto_kernel))
        # exactly representable data: any summation order gives the same bits, NVLS included
        cases.append(dict(count=nbytes // 2, **{"in": "bf16", "wire": "bf16", "out": "bf16"}, algo=0,
                          seed=670 + i, scale=1.0 / world if pow2 else 1.0, symm=True, split=True,
                          pattern="ints", expect_kernel=auto_kernel if pow2 else None))
        exact_ids.add(670 + i)
    # f16 PRE buckets never take the in-switch sum (it could overflow before the 1/N)
    cases.append(dict(count=17 << 20, **{"in": "f16", "wire": "f16", "out": "f16"}, algo=0, seed=690,
                      scale=1.0 / world, symm=True, expect_kernel="two_shot_inplace"))
    res = harness.launch(world, cases, devices=list(range(world)), mode="proc", timeout=600)
    for rank, rs in res.items():
        for r in rs:
            if "case" not in r or "skipped" in r:
                continue
            assert "note" not in r, r
            if r["case"]["seed"] in exact_ids:
                assert r["exact"], r
            if r["exact"]:
                continue
            wire, out = r["case"]["wire"], r["case"]["out"]
            if wire == "f32":
                assert r["normwise"] <= 1e-5, r
            else:
                # one ulp of the 16-bit wire, expressed in ulps of the output dtype
                per = {"bf16": 1 << 16, "f16": 1 << 13}[wire] if out == "f32" else 1
                assert r["max_ulp"] <= per, r


@pytest.mark.parametrize("symm", [False, True])
def test_dead_peer_times_out_instead_of_hanging(tok_lib, symm):
    """A replica whose peer never shows up at the in-kernel barrier (staged bucket) or at the arrival
    (zero-copy bucket) gives up after TOK_BARRIER_TIMEOUT_MS, reports TOK_ERR_TIMEOUT, and leaves NaN
    in the bucket so that an optimizer cannot silently consume a half-exchanged gradient (a dead
    replica must not hang the GPU)."""
    import tempfile
    import threading
    import torch
    from torch_on_k8s_b200 import _ffi
    from torch_on_k8s_b200.comm import Communicator
    os.environ.update(SHARED_ENV)
    os.environ["TOK_BARRIER_TIMEOUT_MS"] = "300"
    path = os.path.join(tempfile.mkdtemp(prefix="tok8s-dead-"), "r")
    comms = {}

    def mk(r):
        comms[r] = Communicator("dead", r, 2, 0, rendezvous_path=path)

    ts = [threading.Thread(target=mk, args=(r,)) for r in range(2)]
    [t.start() for t in ts]
    [t.join(120) for t in ts]
    try:
        from torch_on_k8s_b200.elastic_dp import symm_tensor
        x = symm_tensor(comms[0], 4096, torch.float32).fill_(1.0) if symm else \
            torch.ones(4096, device="cuda")
        # (two-shot by name for the pool bucket: AUTO takes one-shot for 16 KiB)
        comms[0].allreduce_bucket(x, x, scale=0.5, algo=3 if symm else 0)   # rank 1 never calls
        torch.cuda.synchronize()
        with pytest.raises(_ffi.TokError) as e:
            comms[0].status()
        assert e.value.code == _ffi.TOK_ERR_TIMEOUT
        assert comms[0].last_algo() == ("two_shot_inplace" if symm else "one_shot")
        assert bool(torch.isnan(x).all())
    finally:
        os.environ["TOK_BARRIER_TIMEOUT_MS"] = "60000"
        for c in comms.values():
            c.close()


def test_elastic_reform_in_place(tok_lib, n_gpus):
    """Elastic add/drop (BASELINE config 2's 4 -> 8 -> 4): survivors keep their heaps, new replicas
    join at the new epoch, results stay bit-exact at every size."""
    import tempfile
    import threading
    import torch
    from oracle import allreduce_oracle as O
    from torch_on_k8s_b200.comm import Communicator
    os.environ.update(SHARED_ENV)
    path = os.path.join(tempfile.mkdtemp(prefix="tok8s-el-"), "r")
    devs = list(range(8)) if n_gpus >= 8 else [0] * 8
    comms, errs = {}, []

    def run_all(fn, ids):
        ts = [threading.Thread(target=fn, args=(i,)) for i in ids]
        [t.start() for t in ts]
        [t.join(300) for t in ts]
        assert not errs, errs

    def guarded(fn):
        def w(i):
            try:
                fn(i)
            except Exception as e:  # noqa: BLE001
                errs.append("%d: %r" % (i, e))
        return w

    def check(ids, world, seed):
        ins = {i: harness.gen_input(seed, ids.index(i), 70001, "bf16") for i in ids}
        want = O.allreduce_oracle([ins[i] for i in ids], "bf16", "bf16", "bf16", 1.0 / world)
        outs = {}

        def body(i):
            d = devs[i]
            torch.cuda.set_device(d)
            st = torch.cuda.Stream(device=d)
            with torch.cuda.stream(st):
                x = harness.to_torch(ins[i], "bf16", "cuda:%d" % d)
                comms[i].allreduce_bucket(x, x, scale=1.0 / world, stream=st, algo=3)  # exact path
                st.synchronize()
            comms[i].status()
            outs[i] = harness.from_torch(x, "bf16")
        run_all(guarded(body), ids)
        for i in ids:
            assert np.array_equal(outs[i], want), (world, i)

    # epoch 0: 4 replicas
    run_all(guarded(lambda i: comms.__setitem__(
        i, Communicator("el", i, 4, devs[i], rendezvous_path=path, max_world=8))), [0, 1, 2, 3])
    check([0, 1, 2, 3], 4, 1)
    # epoch 1: scale out to 8 — survivors re-form, 4 new replicas join
    def grow(i):
        if i < 4:
            comms[i].reform(8, i, 0xF, 1)
        else:
            comms[i] = Communicator("el", i, 8, devs[i], rendezvous_path=path, max_world=8, epoch=1)
    run_all(guarded(grow), list(range(8)))
    check(list(range(8)), 8, 2)
    # epoch 2: scale in to 4 — replicas 1,3,5,7 leave, the rest are renumbered
    keep = [0, 2, 4, 6]
    for i in (1, 3, 5, 7):
        comms.pop(i).close()
    run_all(guarded(lambda i: comms[i].reform(4, keep.index(i), 0x55, 2)), keep)
    check(keep, 4, 3)
    assert comms[0].caps().epoch == 2
    for c in comms.values():
        c.close()


def test_elastic_training_without_torch_distributed(tok_lib, n_gpus, monkeypatch):
    """BASELINE config 2 in miniature (rescale 2 -> 4 -> 2 mid-run): ElasticDataParallel keeps its
    gradient buckets in the symmetric pool, averages them with the zero-copy kernel, and survives
    peer-group re-forms without restarting any process.  Every averaged bucket is checked bit-for-bit
    against the oracle; replicas stay bit-identical; a joiner receives the parameters in place."""
    import tempfile
    import threading
    import torch
    from oracle import allreduce_oracle as O
    from torch_on_k8s_b200.comm import Communicator
    from torch_on_k8s_b200.elastic_dp import ElasticDataParallel
    from workloads.mlp import batch, mlp
    os.environ.update(SHARED_ENV)
    # Replicas are THREADS of this process here.  The zero-copy exchange is a pair of kernels per
    # bucket (1-warp arrival, then the exchange): inside ONE CUDA context the exchange kernel queued
    # behind a waiting arrival blocks the context's work queue, a peer's arrival enqueued later is
    # never dispatched, and both time out (tools/thread_arrival_diag.py).  One context per replica —
    # processes, the product shape — is what tests/test_controller_gpu.py runs the zero-copy + re-form
    # combination in; this test keeps the pool buckets but exchanges them with the staged kernels.
    monkeypatch.setenv("TOK_DISABLE_ZERO_COPY", "1")
    # For the same reason nothing at all may be queued behind a kernel that waits for a peer's kernel
    # (a hand-over is several collectives with copies in between): in this test every collective is
    # followed by a synchronize of the stream it was launched on.
    real_bcast, real_ar = Communicator.broadcast, Communicator.allreduce_bucket

    def bcast_sync(self, buf, root=0, stream=None):
        out = real_bcast(self, buf, root, stream=stream)
        (stream or torch.cuda.current_stream(buf.device)).synchronize()
        return out

    def ar_sync(self, inp, out=None, **kw):
        res = real_ar(self, inp, out, **kw)
        (kw.get("stream") or torch.cuda.current_stream(inp.device)).synchronize()
        return res
    monkeypatch.setattr(Communicator, "broadcast", bcast_sync)
    monkeypatch.setattr(Communicator, "allreduce_bucket", ar_sync)
    path = os.path.join(tempfile.mkdtemp(prefix="tok8s-edp-"), "r")
    devs = list(range(4)) if n_gpus >= 4 else [0] * 4
    state, errs = {}, []
    pre, post = {}, {}
    init_lock = threading.Lock()   # workloads.mlp seeds the process-global CPU generator

    def guarded(fn):
        def w(i):
            try:
                with torch.cuda.stream(state[i]["stream"]) if i in state and "stream" in state[i] \
                        else torch.cuda.device(devs[i]):
                    fn(i)
            except Exception:  # noqa: BLE001
                import traceback
                errs.append("%d: %s" % (i, traceback.format_exc()))
        return w

    def run_all(fn, ids):
        ts = [threading.Thread(target=guarded(fn), args=(i,)) for i in ids]
        [t.start() for t in ts]
        [t.join(300) for t in ts]
        assert not errs, "\n=====\n".join(errs)

    def make(i, rank, world, epoch):
        torch.cuda.set_device(devs[i])
        st = torch.cuda.Stream(device=devs[i])
        comm = Communicator("edp", rank, world, devs[i], rendezvous_path=path, max_world=4, epoch=epoch)
        with torch.cuda.stream(st):
            with init_lock:
                model = mlp(seed=0 if epoch == 0 else 100 + i)   # joiners start "wrong"
            model = model.cuda(devs[i])
            edp = ElasticDataParallel(model, comm, algo=3, pool_broadcast=False)
            x, y = batch(i, 64)
            state[i] = dict(comm=comm, edp=edp, x=x.cuda(devs[i]), y=y.cuda(devs[i]), stream=st,
                            opt=torch.optim.SGD(model.parameters(), lr=0.05, momentum=0.9))
            st.synchronize()

    def step(ids, tag):
        def body(i):
            s = state[i]
            s["edp"].zero_grad()
            torch.nn.functional.cross_entropy(s["edp"](s["x"]), s["y"]).backward()
            s["stream"].synchronize()
            pre[(tag, i)] = [b.detach().cpu().numpy().copy() for b in s["edp"].buckets]
            s["edp"].reduce_grads(stream=s["stream"])
            s["stream"].synchronize()
            s["comm"].status()
            post[(tag, i)] = [b.detach().cpu().numpy().copy() for b in s["edp"].buckets]
            s["opt"].step()
            s["stream"].synchronize()
        run_all(body, ids)
        world = len(ids)
        for k in range(len(post[(tag, ids[0])])):
            want = O.allreduce_oracle([pre[(tag, i)][k] for i in ids], "f32", "f32", "f32",
                                      1.0 / world)
            for i in ids:
                assert np.array_equal(post[(tag, i)][k].view(np.uint32), want.view(np.uint32)), (tag, i, k)
        flat = {i: torch.cat([p.detach().flatten() for p in state[i]["edp"].module.parameters()]).cpu()
                for i in ids}
        for i in ids[1:]:
            assert torch.equal(flat[ids[0]], flat[i]), (tag, i)   # replicas stay bit-identical

    run_all(lambda i: make(i, i, 2, 0), [0, 1])
    assert len(state[0]["edp"].buckets) >= 1 and state[0]["comm"].in_symmetric_pool(state[0]["edp"].buckets[0])
    step([0, 1], "w2a")
    step([0, 1], "w2b")

    def grow(i):
        if i < 2:
            state[i]["edp"].reform(4, i, 0b11, 1)
        else:
            make(i, i, 4, 1)
    run_all(grow, [0, 1, 2, 3])
    # joiners receive parameters, buffers AND the optimizer's momentum: without the latter the
    # replicas would apply the same averaged gradients with different momentum and drift apart
    run_all(lambda i: (state[i]["edp"].sync_params(root=0),
                       state[i]["edp"].sync_optimizer_state(state[i]["opt"], root=0),
                       state[i]["stream"].synchronize()), [0, 1, 2, 3])
    mom = {i: torch.cat([state[i]["opt"].state[p]["momentum_buffer"].flatten()
                         for p in state[i]["edp"].module.parameters()]).cpu() for i in range(4)}
    assert all(torch.equal(mom[0], mom[i]) for i in (1, 2, 3)) and float(mom[0].abs().sum()) > 0
    step([0, 1, 2, 3], "w4a")
    step([0, 1, 2, 3], "w4b")
    step([0, 1, 2, 3], "w4c")   # still bit-identical three momentum steps after the join

    keep = [0, 2]
    for i in (1, 3):
        state.pop(i)["comm"].close()
    run_all(lambda i: state[i]["edp"].reform(2, keep.index(i), 0b0101, 2), keep)
    step(keep, "w2c")
    assert state[0]["comm"].caps().epoch == 2
    for s in state.values():
        s["comm"].close()
