"""LDA class statistics on the device (vbgpu_lda_*, host.LdaEstimateGpu) and the device form of the feature pipeline
(vbgpu_feat_run_dev) that feeds them in the LDA+MLLT recipe.

The truth is a float64 restatement of LdaEstimate::Accumulate over the same float32 rows widened to float64.  Only the
order of the FP64 additions may differ, so every element must lie within 1e-11 of the sum of the absolute values of its
terms; zero (the summed weights) must be exact when the weights are integers."""
import ctypes as C
import os
import tempfile

import numpy as np
import pytest

from tests.common import STATS_RTOL, recipe_opts
from voicebridge_b200 import capi, host, synth

TOL = 1e-11


def truth(X, ids, w, num_classes):
    """(zero, first, second packed) and the matching sums of |terms|, over frames with a valid class and weight != 0."""
    X = np.asarray(X, np.float32).astype(np.float64)
    ids = np.asarray(ids, np.int64)
    w = np.ones(len(ids)) if w is None else np.asarray(w, np.float32).astype(np.float64)
    keep = (ids >= 0) & (ids < num_classes) & (w != 0)
    X, ids, w = X[keep], ids[keep], w[keep]
    D = X.shape[1]
    zero, szero = np.zeros(num_classes), np.zeros(num_classes)
    first, sfirst = np.zeros((num_classes, D)), np.zeros((num_classes, D))
    np.add.at(zero, ids, w)
    np.add.at(szero, ids, np.abs(w))
    np.add.at(first, ids, w[:, None] * X)
    np.add.at(sfirst, ids, np.abs(w[:, None] * X))
    ii, jj = np.tril_indices(D)  # row-major lower triangle = SpMatrix packing
    second = (X.T @ (w[:, None] * X))[ii, jj]
    ssecond = (np.abs(X).T @ (np.abs(w)[:, None] * np.abs(X)))[ii, jj]
    return (zero, first, second), (szero, sfirst, ssecond)


def assert_matches(got, want, scale, exact_zero=False):
    for name, g, t, s in zip(("zero", "first", "second"), got, want, scale):
        assert g.shape == t.shape, (name, g.shape, t.shape)
        assert np.isfinite(g).all(), name
        err = np.abs(g - t) - TOL * s
        assert (err <= 0).all(), "%s: worst |got - want| %.3g over %.3g of sum |terms|" % (
            name, np.abs(g - t).max(), TOL)
    if exact_zero:
        assert np.array_equal(got[0], want[0])


def make_batch(T, D, C, stride, weights, seed):
    """Rows with a per-dimension offset (so that the second-order sums do not cancel to nothing), classes drawn from a
    few of the C (most classes never seen)."""
    rng = np.random.default_rng(seed)
    X = np.zeros((T, stride), np.float32)
    X[:, :D] = (rng.standard_normal((T, D)) * 3.0 + rng.uniform(-5, 5, D)).astype(np.float32)
    X[:, D:] = np.nan  # padding past D is never read
    used = rng.choice(C, size=min(C, 17), replace=False)
    ids = used[rng.integers(0, len(used), T)].astype(np.int32)
    if weights == "none":
        w = None
    elif weights == "uniform":
        w = rng.uniform(0.1, 2.0, T).astype(np.float32)
    else:  # zeros and negatives among them
        w = rng.uniform(-1.0, 2.0, T).astype(np.float32)
        w[rng.random(T) < 0.3] = 0.0
    return X, ids, w


def gpu_or_skip():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


# ---- argument checks: no device needed ---------------------------------------------------------------------------------
def test_argument_errors_need_no_gpu():
    lib = capi.lib()
    h = C.c_void_p()
    assert lib.vbgpu_lda_create(0, 13, 0, C.byref(h)) == capi.ERR_INVALID
    assert lib.vbgpu_lda_create(-3, 13, 0, C.byref(h)) == capi.ERR_INVALID
    assert lib.vbgpu_lda_create(10, 0, 0, C.byref(h)) == capi.ERR_INVALID
    assert lib.vbgpu_lda_create(10, 257, 0, C.byref(h)) == capi.ERR_INVALID
    assert b"dim" in lib.vbgpu_last_error()
    assert lib.vbgpu_lda_create(10, 13, 0, None) == capi.ERR_INVALID
    x = np.zeros((4, 13), np.float32)
    ids = np.zeros(4, np.int32)
    assert lib.vbgpu_lda_accumulate(None, x.ctypes.data, 4, 13, ids.ctypes.data, None) == capi.ERR_INVALID
    assert lib.vbgpu_lda_accumulate_dev(None, None, 4, 13, None, None, None) == capi.ERR_INVALID
    assert lib.vbgpu_lda_zero(None) == capi.ERR_INVALID
    assert lib.vbgpu_lda_download(None, None, None, None) == capi.ERR_INVALID
    assert lib.vbgpu_feat_run_dev(None, None, 13, None, 0, None, 0, None, None, 0, None, 91, None) == capi.ERR_INVALID


def test_no_cpu_fallback():
    lib = capi.lib()
    n = C.c_int(0)
    if lib.vbgpu_device_count(C.byref(n)) == 0 and n.value > 0:
        pytest.skip("a GPU is present")
    h = C.c_void_p()
    assert lib.vbgpu_lda_create(10, 13, 0, C.byref(h)) == capi.ERR_CUDA
    with pytest.raises(capi.VbgpuError):
        host.LdaEstimateGpu(10, 13)


# ---- statistics against the restatement --------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("weights", ["none", "uniform", "mixed"])
@pytest.mark.parametrize("T", [0, 1, 3000])
@pytest.mark.parametrize("D", [1, 13, 91, 117, 256])
def test_matches_restatement(D, T, weights):
    C_ = 500
    X, ids, w = make_batch(T, D, C_, D + 3, weights, 10 * D + T)
    est = host.LdaEstimateGpu(C_, D)
    assert (est.NumClasses(), est.Dim()) == (C_, D)
    est.Accumulate(X, ids, w)
    want, scale = truth(X[:, :D], ids, w, C_)
    assert_matches(est.stats(), want, scale, exact_zero=weights == "none")
    # the same through the device entry point
    torch = gpu_or_skip()
    est.ZeroAccumulators()
    if T:
        est.accumulate_dev(torch.from_numpy(X).cuda(), T, D + 3, torch.from_numpy(ids).cuda(),
                           None if w is None else torch.from_numpy(w).cuda())
    torch.cuda.synchronize()
    assert_matches(est.stats(), want, scale, exact_zero=weights == "none")
    assert est.bad_count() == 0


@pytest.mark.gpu
def test_argument_errors_with_a_handle():
    est = host.LdaEstimateGpu(10, 13)
    x = np.zeros((4, 16), np.float32)
    ids = np.zeros(4, np.int32)
    lib = capi.lib()
    assert lib.vbgpu_lda_accumulate(est.h, x.ctypes.data, 4, 12, ids.ctypes.data, None) == capi.ERR_INVALID  # stride < D
    assert lib.vbgpu_lda_accumulate(est.h, None, 4, 16, ids.ctypes.data, None) == capi.ERR_INVALID
    assert lib.vbgpu_lda_accumulate(est.h, x.ctypes.data, 4, 16, None, None) == capi.ERR_INVALID
    assert lib.vbgpu_lda_accumulate(est.h, None, 0, 16, None, None) == 0  # nothing to read
    assert lib.vbgpu_lda_accumulate(est.h, x.ctypes.data, -1, 16, ids.ctypes.data, None) == capi.ERR_INVALID


@pytest.mark.gpu
def test_zero_weight_frames_with_nonfinite_features_are_skipped():
    D, C_, T = 91, 50, 2000
    X, ids, w = make_batch(T, D, C_, 92, "uniform", 3)
    bad = np.arange(5, T, 97)
    X[bad[::3], :D] = np.nan
    X[bad[1::3], :D] = np.inf
    X[bad[2::3], 7] = -np.inf
    w[bad] = 0.0
    est = host.LdaEstimateGpu(C_, D)
    est.Accumulate(X, ids, w)
    got = est.stats()
    keep = np.setdiff1d(np.arange(T), bad)
    want, scale = truth(X[keep, :D], ids[keep], w[keep], C_)
    assert_matches(got, want, scale)


@pytest.mark.gpu
def test_invalid_class_ids():
    torch = gpu_or_skip()
    D, C_, T = 13, 40, 1000
    X, ids, w = make_batch(T, D, C_, 16, "uniform", 4)
    ids[[3, 500]] = -1
    ids[[10, 999]] = C_
    X[[3, 10], :D] = np.nan  # an invalid frame adds nothing, whatever it holds
    keep = ids >= 0
    keep &= ids < C_
    want, scale = truth(X[keep, :D], ids[keep], w[keep], C_)
    est = host.LdaEstimateGpu(C_, D)
    with pytest.raises(capi.VbgpuError) as e:
        est.Accumulate(X, ids, w)
    assert e.value.code == capi.ERR_NUMERIC
    assert_matches(est.stats(), want, scale)
    assert est.bad_count() == 0  # the host form reports through its return code only

    est.ZeroAccumulators()
    est.accumulate_dev(torch.from_numpy(X).cuda(), T, 16, torch.from_numpy(ids).cuda(), torch.from_numpy(w).cuda())
    assert est.bad_count() == 4
    assert est.bad_count() == 0
    assert_matches(est.stats(), want, scale)


@pytest.mark.gpu
def test_calls_add_up_zero_clears_handles_are_independent():
    torch = gpu_or_skip()
    D, C_, T = 91, 300, 4000
    X, ids, w = make_batch(T, D, C_, 96, "mixed", 5)
    want, scale = truth(X[:, :D], ids, w, C_)
    a, b = host.LdaEstimateGpu(C_, D), host.LdaEstimateGpu(C_, D)
    b.Accumulate(X[:100], ids[:100], w[:100])  # another handle's statistics must not show in a
    for cut in (7, 128, 2048):  # 128: a work unit of the class sums; 2048: a multiple of every chunk of the triangle
        a.ZeroAccumulators()
        a.Accumulate(X[:cut], ids[:cut], w[:cut])
        a.Accumulate(X[cut:], ids[cut:], w[cut:])
        assert_matches(a.stats(), want, scale)
    a.ZeroAccumulators()
    assert all((s == 0).all() for s in a.stats())
    assert a.TotCount() == 0.0
    wb, sb = truth(X[:100, :D], ids[:100], w[:100], C_)
    assert_matches(b.stats(), wb, sb)

    # the device form on a non-default stream equals the host form
    a.Accumulate(X, ids, w)
    host_stats = a.stats()
    a.ZeroAccumulators()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        dx, di, dw = torch.from_numpy(X).cuda(), torch.from_numpy(ids).cuda(), torch.from_numpy(w).cuda()
        a.accumulate_dev(dx[:1000], 1000, 96, di[:1000], dw[:1000], stream=s)
        a.accumulate_dev(dx[1000:], T - 1000, 96, di[1000:], dw[1000:], stream=s)
    s.synchronize()
    assert_matches(a.stats(), want, scale)
    for g, h_ in zip(a.stats(), host_stats):
        np.testing.assert_allclose(g, h_, rtol=0, atol=TOL * np.abs(h_).max() + 1e-300)


# ---- end to end, the way train_lda_mllt feeds acc-lda ------------------------------------------------------------------
def splice_numpy(x, fo, left, right):
    out = []
    for u in range(len(fo) - 1):
        y = x[fo[u]:fo[u + 1]]
        n = len(y)
        idx = np.clip(np.arange(n)[:, None] + np.arange(-left, right + 1)[None, :], 0, n - 1)
        out.append(y[idx].reshape(n, -1))
    return np.concatenate(out)


@pytest.mark.gpu
def test_end_to_end_mfcc_cmvn_splice_stats(orc):
    torch = gpu_or_skip()
    from tests.gpu_common import oracle_feats, oracle_mfcc_batch, oracle_stats
    n_spk, C_ = 3, 120
    pcm, so, u2s = synth.make_corpus(n_spk, 3, 1.0, 2.5, 21)
    mo = recipe_opts(capi)
    mfcc = host.Mfcc(mo)
    fo = mfcc.frame_offsets(so)
    T, K = int(fo[-1]), 13 * 7
    d_pcm = torch.from_numpy(np.asarray(pcm, np.int16)).cuda()
    d_mf = torch.zeros((T, 16), dtype=torch.float32, device="cuda")
    s = torch.cuda.current_stream()
    mfcc.compute_dev(d_pcm, so, d_mf, 16, stream=s)
    torch.cuda.synchronize()
    mf = d_mf[:, :13].cpu().numpy()
    fopts = capi.default_feat_opts(mode=1)
    eye = np.eye(K, dtype=np.float32)
    fp = host.FeaturePipeline(fopts, 13, transform=eye)
    st = fp.cmvn_stats(mf, fo, u2s, n_spk)  # vbgpu_cmvn_stats
    d_sp = torch.zeros((T, 92), dtype=torch.float32, device="cuda")
    fp.run_dev(d_mf, 16, fo, d_sp, 92, u2s, n_spk, cmvn_stats=st, stream=s)
    torch.cuda.synchronize()
    spliced = d_sp[:, :K].cpu().numpy()
    assert np.array_equal(spliced, fp.run(mf, fo, u2s, n_spk, cmvn_stats=st)), "run_dev differs from vbgpu_feat_run"

    # CMVN off: the identity transform is a splice, bit for bit
    fp0 = host.FeaturePipeline(capi.default_feat_opts(mode=1, norm_means=0), 13, transform=eye)
    d_sp0 = torch.zeros((T, 92), dtype=torch.float32, device="cuda")
    fp0.run_dev(d_mf, 16, fo, d_sp0, 92, u2s, n_spk, stream=s)
    torch.cuda.synchronize()
    assert np.array_equal(d_sp0[:, :K].cpu().numpy(), splice_numpy(mf, fo, 3, 3))

    # pdfs from an alignment, silence classes weighted 0 (weight-silence-post 0.0)
    ids = synth.make_alignment(C_, T, 22).astype(np.int32)
    w = np.where(ids < 5, 0.0, 1.0).astype(np.float32)
    est = host.LdaEstimateGpu(C_, K)
    est.accumulate_dev(d_sp, T, 92, torch.from_numpy(ids).cuda(), torch.from_numpy(w).cuda(), stream=s)
    got = est.stats()
    assert est.bad_count() == 0
    want, scale = truth(spliced, ids, w, C_)
    assert_matches(got, want, scale, exact_zero=True)

    # the oracle chain: its own MFCC, CMVN and splice (identity transform), restated the same way
    mf_o, fo_o = oracle_mfcc_batch(orc, mo, pcm, so)
    assert np.array_equal(fo_o, fo)
    st_o = oracle_stats(orc, mf_o, fo_o, u2s, n_spk)
    feats_o = oracle_feats(orc, mf_o, fo_o, u2s, st_o, fopts, eye)
    want_o, scale_o = truth(feats_o, ids, w, C_)
    assert np.array_equal(got[0], want_o[0])
    for g, t, sc, name in zip(got[1:], want_o[1:], scale_o[1:], ("first", "second")):
        # relative to the magnitude accumulated (as for the fMLLR statistics): CMVN'd features cancel in these sums
        err = np.abs(g - t) / np.maximum(sc, 1e-300)
        assert err.max() <= STATS_RTOL, "LDA %s vs oracle chain: %.3g of sum |terms|" % (name, err.max())


# ---- bench-sized -------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_bench_sized_properties():
    torch = gpu_or_skip()
    T, C_, D = 200_000, 2500, 91
    rng = np.random.default_rng(8)
    X = torch.from_numpy((rng.standard_normal((T, D)) * 4.0).astype(np.float32)).cuda()
    ids = torch.from_numpy(synth.make_alignment(C_, T, 9).astype(np.int32)).cuda()
    w_np = np.where(rng.random(T) < 0.2, 0.0, rng.uniform(0.5, 1.5, T)).astype(np.float32)
    est = host.LdaEstimateGpu(C_, D)
    est.accumulate_dev(X, T, D, ids, torch.from_numpy(w_np).cuda())
    zero, first, second = est.stats()
    assert np.isfinite(zero).all() and np.isfinite(first).all() and np.isfinite(second).all()
    assert abs(est.TotCount() - w_np.astype(np.float64).sum()) <= 1e-9 * w_np.sum()
    diag = second[np.arange(1, D + 1) * np.arange(2, D + 2) // 2 - 1]  # (i, i) at i(i+1)/2 + i
    assert (diag >= 0).all()
    assert est.bad_count() == 0


# ---- two GPUs: shard, accumulate, all-reduce ---------------------------------------------------------------------------
def nccl_comm(rank, world, device):
    """A raw ncclComm_t: the unique id is made on rank 0 and shared through torch.distributed (a copy of the helper in
    tools/em_multi_gpu.py, with the id sent over the CPU group)."""
    import glob
    import torch
    import torch.distributed as dist
    cands = glob.glob(os.path.join(os.path.dirname(torch.__file__), "..", "nvidia", "nccl", "lib", "libnccl.so.2"))
    lib = C.CDLL(cands[0] if cands else "libnccl.so.2", mode=C.RTLD_GLOBAL)

    class UniqueId(C.Structure):
        _fields_ = [("internal", C.c_byte * 128)]
    uid = UniqueId()
    if rank == 0:
        assert lib.ncclGetUniqueId(C.byref(uid)) == 0
    t = torch.frombuffer(bytearray(bytes(uid.internal)), dtype=torch.uint8).clone()
    dist.broadcast(t, 0)
    C.memmove(C.byref(uid), bytes(t.numpy().tobytes()), 128)
    comm = C.c_void_p()
    lib.ncclCommInitRank.argtypes = [C.POINTER(C.c_void_p), C.c_int, UniqueId, C.c_int]
    with torch.cuda.device(device):
        assert lib.ncclCommInitRank(C.byref(comm), world, uid, rank) == 0
    return lib, comm


def _rank_main(rank, world, init_file, out_dir):
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("gloo", init_method="file://" + init_file, rank=rank, world_size=world)
    lib, comm = nccl_comm(rank, world, rank)
    T, C_, D = 50_000, 400, 91
    X, ids, w = make_batch(T, D, C_, D, "mixed", 77)
    lo, hi = rank * T // world, (rank + 1) * T // world
    est = host.LdaEstimateGpu(C_, D, device=rank)
    s = torch.cuda.current_stream()
    est.accumulate_dev(torch.from_numpy(X[lo:hi]).cuda(), hi - lo, D, torch.from_numpy(ids[lo:hi]).cuda(),
                       torch.from_numpy(w[lo:hi]).cuda(), stream=s)
    est.allreduce(comm, stream=s)
    s.synchronize()
    merged = np.concatenate([v.ravel() for v in est.stats()])
    one = host.LdaEstimateGpu(C_, D, device=rank)
    one.Accumulate(X, ids, w)
    single = np.concatenate([v.ravel() for v in one.stats()])
    np.save(os.path.join(out_dir, "rank%d.npy" % rank), np.stack([merged, single]))
    lib.ncclCommDestroy(comm)
    dist.destroy_process_group()


@pytest.mark.gpu
def test_two_gpus_allreduce():
    torch = gpu_or_skip()
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    with tempfile.TemporaryDirectory() as d:
        mp.spawn(_rank_main, args=(2, os.path.join(d, "init"), d), nprocs=2, join=True)
        for r in range(2):
            merged, single = np.load(os.path.join(d, "rank%d.npy" % r))
            assert np.abs(merged - single).max() <= 1e-12 * np.abs(single).max(), r
