"""Handle lifetime: every handle gives back all the device and pinned memory it took, on destroy and on a failed create.

vbgpu_debug_live_bytes counts the library's own cudaMalloc / cudaMallocHost bytes, so the checks are exact and do not see
torch's allocations or other processes on the same GPU.  Each cycle builds the handles it uses (models included), grows
their scratch with one call, and closes them all; the counts must come back to what they were before the cycle."""
import ctypes as C
import gc

import numpy as np
import pytest

from tests.common import recipe_opts
from voicebridge_b200 import capi, host, synth


def live():
    gc.collect()
    d, p = C.c_int64(0), C.c_int64(0)
    capi.check(capi.lib().vbgpu_debug_live_bytes(C.byref(d), C.byref(p)))
    return d.value, p.value


def test_live_bytes_need_no_gpu():
    lib = capi.lib()
    d, p = C.c_int64(-1), C.c_int64(-1)
    assert lib.vbgpu_debug_live_bytes(C.byref(d), C.byref(p)) == 0
    assert d.value >= 0 and p.value >= 0
    assert lib.vbgpu_debug_live_bytes(None, C.byref(p)) == capi.ERR_INVALID


def gpu_or_skip():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def corpus():
    pcm, so, u2s = synth.make_corpus(2, 2, 0.5, 1.0, 7)
    return np.asarray(pcm, np.int16), so, u2s


def model(D, seed=3):
    return host.AmDiagGmmGpu.from_model(synth.make_model(40, 200, D, seed))


def use_downsample():
    ds = host.Downsampler(16000, 8000)
    ds(synth.make_wave(4000, 1).astype(np.float32))
    return [ds]


def use_front_end(cls):
    def use():
        pcm, so, _ = corpus()
        fe = cls(recipe_opts(capi))
        fe.compute_batch(pcm, so)
        return [fe]
    return use


def use_pitch():
    p = host.Pitch()
    w = synth.make_pitch_wave(8000, 2)
    p.compute_batch(w, np.array([0, len(w)], np.int64))
    return [p]


def use_feat(mode):
    def use():
        rng = np.random.default_rng(4)
        x = rng.standard_normal((120, 13)).astype(np.float32)
        fo = np.array([0, 50, 120], np.int64)
        if mode == "delta":
            fp = host.FeaturePipeline(capi.default_feat_opts(), 13)
        else:
            fp = host.FeaturePipeline(capi.default_feat_opts(mode=1), 13, synth.make_lda(40, 91, 2))
        fp.run(x, fo, cmvn_stats=fp.cmvn_stats(x, fo))
        return [fp]
    return use


def use_gmm(D):
    def use():
        m = synth.make_model(40, 200, D, 3)
        am = host.AmDiagGmmGpu.from_model(m)
        assert (am.plan_note() == "") == (D <= 47), am.plan_note()
        X = synth.make_feats(m, 300, 4)
        am.score(X)
        am.score_subset(X, np.array([0, 100, 300], np.int64), [[0, 5, 7], [1, 2]])  # the lazy copy stream and events
        return [am]
    return use


def use_acc():
    m = synth.make_model(40, 200, 39, 3)
    am = host.AmDiagGmmGpu.from_model(m)
    acc = host.AccumAmDiagGmmGpu(am, num_tids=60)
    X = synth.make_feats(m, 300, 4)
    acc.AccumulateForUtterance(X, synth.make_alignment(40, 300, 5))
    acc.AccumulateTransitions(np.arange(300, dtype=np.int32) % 60 + 1)
    return [acc, am]


def use_fmllr():
    m = synth.make_model(40, 200, 39, 3)
    am = host.AmDiagGmmGpu.from_model(m)
    f = host.FmllrDiagGmmAccsGpu(am)
    f.AccumulateForUtterances(synth.make_feats(m, 300, 4), synth.make_alignment(40, 300, 5))
    return [f, am]


def use_lda():
    lda = host.LdaEstimateGpu(10, 39)
    x = np.random.default_rng(6).standard_normal((300, 39)).astype(np.float32)
    lda.Accumulate(x, np.arange(300, dtype=np.int32) % 10)
    return [lda]


def use_tree():
    fo = np.array([0, 60, 150], np.int64)
    topo, tids, _ = synth.make_phone_alignment(12, fo, 8)
    ts = host.TreeStatsGpu(topo, 39, 1 << 12, 3, 1, (1,))
    x = np.random.default_rng(9).standard_normal((150, 39)).astype(np.float32)
    ts.AccumulateTreeStats(x, tids, fo)
    return [ts]


def use_pipeline():
    pcm, so, u2s = corpus()
    mf, fp, am = host.Mfcc(recipe_opts(capi)), host.FeaturePipeline(in_dim=13), model(39)
    pipe = host.ScoringPipeline(mf, fp, am)
    pipe.score(pcm, so, u2s)  # pageable numpy buffers: staged through the pipeline's pinned buffers
    return [pipe, am, fp, mf]


KINDS = {
    "downsample": use_downsample,
    "mfcc": use_front_end(host.Mfcc),
    "fbank": use_front_end(host.Fbank),
    "plp": use_front_end(host.Plp),
    "pitch": use_pitch,
    "feat_delta": use_feat("delta"),
    "feat_lda": use_feat("lda"),
    "gmm_tc": use_gmm(39),
    "gmm_simt": use_gmm(52),
    "acc": use_acc,
    "fmllr": use_fmllr,
    "lda": use_lda,
    "tree": use_tree,
    "pipeline": use_pipeline,
}


@pytest.mark.gpu
@pytest.mark.parametrize("kind", sorted(KINDS))
def test_handle_returns_everything(kind):
    """create -> one call that grows the scratch -> close, three times: the counts rise, then come back exactly."""
    gpu_or_skip()
    for _ in range(3):
        before = live()
        handles = KINDS[kind]()
        during = live()
        assert during[0] > before[0]
        if kind == "pipeline":
            assert during[1] > before[1]
        for h in handles:
            h.close()
        del handles
        assert live() == before


@pytest.mark.gpu
def test_one_shot_calls_free_their_buffers():
    """MlltAccsGpu.AccumulateForUtterance (an internal fMLLR handle) and ComponentPosteriors (local buffers) keep
    nothing once they return."""
    gpu_or_skip()
    m = synth.make_model(40, 200, 39, 3)
    am = host.AmDiagGmmGpu.from_model(m)
    X, ali = synth.make_feats(m, 300, 4), synth.make_alignment(40, 300, 5)
    before = live()
    host.MlltAccsGpu(am).AccumulateForUtterance(X, ali)
    assert live() == before
    am.ComponentPosteriors(X, ali, m.pdf_offsets, np.ones(300, np.float32))
    assert live() == before
    am.close()


@pytest.mark.gpu
def test_failed_creates_free_what_they_took():
    """Requests beyond the 180 GB of a B200: cudaMalloc refuses them (an ordinary allocation error) and the create
    frees the stream and the buffers it already had."""
    gpu_or_skip()
    before = live()
    topo = synth.phone_topology(5)
    with pytest.raises(capi.VbgpuError) as e:
        host.TreeStatsGpu(topo, 256, 1 << 26)  # statistics alone: 2^26 keys x 513 doubles, about 275 GB
    assert e.value.code == capi.ERR_NOMEM
    assert live() == before
    with pytest.raises(capi.VbgpuError) as e:
        host.LdaEstimateGpu(1 << 30, 256)
    assert e.value.code == capi.ERR_NOMEM
    assert live() == before
    lda = host.LdaEstimateGpu(4, 3)  # the refused allocations do not surface in later calls
    lda.Accumulate(np.ones((5, 3), np.float32), np.arange(5, dtype=np.int32) % 4)
    assert lda.TotCount() == 5.0
    lda.close()


@pytest.mark.gpu
def test_downsample_checks_the_device():
    gpu_or_skip()
    lib = capi.lib()
    n = C.c_int(0)
    assert lib.vbgpu_device_count(C.byref(n)) == 0
    h = C.c_void_p()
    assert lib.vbgpu_downsample_create(16000.0, 8000.0, n.value, C.byref(h)) == capi.ERR_INVALID
    assert b"out of range" in lib.vbgpu_last_error()
    assert not h.value
