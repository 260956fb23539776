"""Parity of the CUDA path (through the C ABI) with the CPU oracle, the compiled reference (when its prebuilt
library is present) and the committed golden vectors.  Tolerances are BASELINE.json's: features 1e-4 relative,
log-likelihoods 1e-3 absolute, statistics 1e-4 relative."""
import numpy as np
import pytest

from oracle import pyoracle as po
from tests.common import assert_acc_close, assert_feats_close, assert_ll_close, assert_stats_close
from tests.golden.make_golden import HTK_CASES, HTK_VTLN
from tests.gpu_common import oracle_feats, oracle_mfcc_batch, oracle_stats, to_orc_opts
from voicebridge_b200 import capi, host, synth

pytestmark = pytest.mark.gpu


def gopts(**kw):
    base = dict(dither=0.0, use_energy=0)
    base.update(kw)
    return capi.default_mfcc_opts(**base)


# ======================================================================================================= front end
MFCC_VARIANTS = [
    dict(), dict(use_energy=1), dict(use_energy=1, raw_energy=0), dict(use_energy=1, energy_floor=1e9),
    dict(snip_edges=0), dict(samp_freq=8000.0), dict(htk_compat=1), dict(htk_compat=1, use_energy=1),
    dict(window_type=1), dict(window_type=4), dict(remove_dc_offset=0), dict(preemph_coeff=0.0),
    dict(cepstral_lifter=0.0), dict(num_bins=30, num_ceps=20), dict(low_freq=100.0, high_freq=-400.0),
    dict(htk_mode=1), dict(frame_length_ms=20.0, frame_shift_ms=5.0), dict(samp_freq=44100.0),
    dict(samp_freq=4000.0), dict(window_type=2), dict(window_type=3), dict(window_type=3, preemph_coeff=0.0, remove_dc_offset=0),
]


@pytest.mark.parametrize("kw", MFCC_VARIANTS, ids=lambda d: ",".join("%s=%s" % kv for kv in d.items()) or "default")
def test_mfcc_single_utterance(orc, kw):
    o = gopts(**kw)
    w = synth.make_wave(int(o.samp_freq * 1.3), 5, o.samp_freq)
    m = host.Mfcc(o)
    got = m.ComputeFeatures(w, o.samp_freq)
    want = orc.mfcc(to_orc_opts(o), w.astype(np.float32))
    assert got.shape == want.shape and got.shape[0] == m.NumFrames(len(w))
    assert_feats_close(got, want)
    got_f = m.ComputeFeatures(w.astype(np.float32))  # Kaldi's float-wave form
    assert np.array_equal(got, got_f)


@pytest.mark.parametrize("case", sorted(HTK_CASES))
def test_mfcc_htk_known_answers(golden, case):
    """The reference's own KAT (feature-mfcc-test.cc:112-650): |MFCC+deltas - HTK| <= 1.0 away from the edges."""
    htk, _ = golden
    o = capi.default_mfcc_opts(dither=0.0, **HTK_CASES[case])
    m = host.Mfcc(o)
    raw = m.ComputeFeatures(htk["pcm"], 16000.0, HTK_VTLN.get(case, 1.0))
    fp = host.FeaturePipeline(capi.default_feat_opts(norm_means=0), in_dim=13)
    feats = fp.run(raw, [0, len(raw)])
    want = htk["htk%d" % case]
    assert feats.shape == want.shape
    assert np.abs(feats[10:-10] - want[10:-10]).max() <= 1.0


def test_mfcc_against_reference_dumps(golden):
    htk, g = golden
    pcm = htk["pcm"]
    assert_feats_close(host.Mfcc(gopts()).ComputeFeatures(pcm), g["mfcc16"])
    assert_feats_close(host.Mfcc(capi.default_mfcc_opts(dither=0.0)).ComputeFeatures(pcm), g["mfcc16_energy"])
    assert_feats_close(host.Mfcc(gopts(snip_edges=0)).ComputeFeatures(pcm), g["mfcc16_nosnip"])
    assert_feats_close(host.Mfcc(gopts()).ComputeFeatures(pcm, vtln_warp=0.9), g["mfcc16_vtln09"])
    assert_feats_close(host.Mfcc(gopts(samp_freq=8000.0)).ComputeFeatures(g["wave8"]), g["mfcc8"])


@pytest.mark.parametrize("snip", [1, 0])
def test_mfcc_ragged_batch(orc, snip):
    """Empty, shorter-than-a-window, odd-length and long utterances in one packed batch, with per-utterance VTLN."""
    o = gopts(snip_edges=snip)
    lens = [0, 100, 399, 400, 401, 1, 559, 560, 4801, 16000, 33333, 81, 7777]
    so = np.zeros(len(lens) + 1, np.int64)
    so[1:] = np.cumsum(lens)
    pcm = synth.make_wave(int(so[-1]), 3)
    vtln = np.array([1.0, 0.9, 1.1, 1.0, 1.0, 1.0, 0.9, 1.2, 1.0, 0.85, 1.0, 1.0, 1.1], np.float32)
    m = host.Mfcc(o)
    for vt in (None, vtln):
        got, fo = m.compute_batch(pcm, so, vt)
        want, fo_want = oracle_mfcc_batch(orc, o, pcm, so, vt)
        assert np.array_equal(fo, fo_want)
        assert_feats_close(got, want)
    if not snip:  # frames shorter than the window are reflected repeatedly (feature-window.cc:199-211)
        assert fo[2] - fo[1] == 1 and fo[6] - fo[5] == 0


def test_mfcc_batch_equals_single_at_scale():
    """Size-independent property at bench scale: batching is invisible — every utterance of a large packed batch
    is bit-identical to the same utterance computed alone."""
    o = gopts()
    pcm, so, _ = synth.make_corpus(8, 16, 5.0, 20.0, 21, fast=True)
    m = host.Mfcc(o)
    got, fo = m.compute_batch(pcm, so)
    assert fo[-1] > 100000 and np.isfinite(got).all()
    for u in (0, 17, 63, 127):
        one = m.ComputeFeatures(pcm[so[u]:so[u + 1]])
        assert np.array_equal(one, got[fo[u]:fo[u + 1]])


def test_mfcc_dither_is_noise_of_the_right_size():
    o0, o1 = gopts(), gopts(dither=1.0)
    w = synth.make_wave(16000 * 4, 9)
    a, b = host.Mfcc(o0).ComputeFeatures(w), host.Mfcc(o1).ComputeFeatures(w)
    d = np.abs(a - b)
    assert d.max() > 0 and np.median(d) < 0.5      # +-1 LSB noise on +-2^14 audio barely moves cepstra
    z = host.Mfcc(o1).ComputeFeatures(np.zeros(16000, np.int16))
    assert np.isfinite(z).all() and z.std(axis=0).max() > 0  # silence + dither: no log(0), frames differ


def test_mfcc_errors():
    m = host.Mfcc(gopts())
    with pytest.raises(capi.VbgpuError):
        m.ComputeFeatures(np.zeros(1000, np.int16), sample_freq=8000.0)  # feature-common-inl.h:37-54
    with pytest.raises(capi.VbgpuError):
        m.compute_batch(np.zeros(10, np.int16), [0, 20, 10])
    assert m.ComputeFeatures(np.zeros(10, np.int16)).shape == (0, 13)


# ================================================================================================ feature pipeline
def _mfcc_batch(n_spk=3, upspk=3, seed=4):
    o = gopts()
    pcm, so, u2s = synth.make_corpus(n_spk, upspk, 0.3, 1.2, seed)
    mf, fo = host.Mfcc(o).compute_batch(pcm, so)
    return mf, fo, u2s


@pytest.mark.parametrize("per_utt", [False, True])
def test_cmvn_stats(orc, per_utt):
    mf, fo, u2s = _mfcc_batch()
    fp = host.FeaturePipeline(in_dim=13)
    u = None if per_utt else u2s
    n_spk = len(fo) - 1 if per_utt else 3
    got = fp.cmvn_stats(mf, fo, u, n_spk)
    want = oracle_stats(orc, mf, fo, u, n_spk)
    assert np.array_equal(got[:, 0, 13], want[:, 0, 13])  # counts exact
    assert_stats_close(got, want, 1e-12)
    got2 = fp.cmvn_stats(mf, fo, u, n_spk, stats=got.copy())  # adds to existing stats
    assert_stats_close(got2, 2 * want, 1e-12)


FEAT_CASES = [
    dict(), dict(norm_vars=1), dict(norm_means=0), dict(delta_order=1, delta_window=3), dict(delta_order=3, delta_window=1),
    dict(delta_order=0), dict(mode=1), dict(mode=1, splice_left=4, splice_right=4), dict(mode=1, splice_left=0, splice_right=2),
]


@pytest.mark.parametrize("kw", FEAT_CASES, ids=lambda d: ",".join("%s=%s" % kv for kv in d.items()) or "default")
@pytest.mark.parametrize("fmllr_cols", [0, 1, 2])  # none, D+1 (affine), D (linear)
def test_feature_pipeline(orc, kw, fmllr_cols):
    mf, fo, u2s = _mfcc_batch()
    fopts = capi.default_feat_opts(**kw)
    lda = None
    if fopts.mode == 1:
        K = 13 * (fopts.splice_left + fopts.splice_right + 1)
        lda = synth.make_lda(40, K + (1 if fopts.splice_left == 4 else 0), 3)
    fp = host.FeaturePipeline(fopts, 13, lda)
    OD = fp.out_dim()
    fm = None
    if fmllr_cols:
        fm = synth.make_fmllr(3, OD, 8)
        if fmllr_cols == 2:
            fm = np.ascontiguousarray(fm[:, :, :OD])
    stats = oracle_stats(orc, mf, fo, u2s, 3)
    got = fp.run(mf, fo, u2s, 3, stats, fm)
    want = oracle_feats(orc, mf, fo, u2s, stats, fopts, lda, fm)
    assert_feats_close(got, want, what=str(kw))


def test_feature_pipeline_short_utterances_and_tiles(orc):
    """1- and 2-frame utterances (every tap clamped), empty ones, and utterance boundaries inside a 64-frame tile."""
    rng = np.random.default_rng(0)
    lens = [1, 2, 0, 5, 63, 64, 65, 1, 130, 0, 9]
    fo = np.zeros(len(lens) + 1, np.int64)
    fo[1:] = np.cumsum(lens)
    mf = rng.standard_normal((int(fo[-1]), 13)).astype(np.float32) * 5
    stats = oracle_stats(orc, mf, fo, None, len(lens))
    stats[[2, 9], 0, 13] = 1.0  # empty utterances never get applied; keep their count valid
    for fopts, lda in ((capi.default_feat_opts(), None), (capi.default_feat_opts(mode=1), synth.make_lda(40, 91, 1))):
        fp = host.FeaturePipeline(fopts, 13, lda)
        got = fp.run(mf, fo, None, None, stats)
        want = oracle_feats(orc, mf, fo, None, stats, fopts, lda)
        assert_feats_close(got, want)


def test_feature_pipeline_against_reference_dumps(golden):
    _, g = golden
    x, st = g["mfcc16"], g["cmvn_stats"][None]
    fo = [0, len(x)]
    assert_feats_close(host.FeaturePipeline(in_dim=13).run(x, fo, cmvn_stats=st), g["delta"])
    assert_feats_close(host.FeaturePipeline(capi.default_feat_opts(delta_order=1, delta_window=3), 13)
                       .run(x, fo, cmvn_stats=st), g["delta_o1_w3"])
    assert_feats_close(host.FeaturePipeline(capi.default_feat_opts(mode=1), 13, g["lda_mat"]).run(x, fo, cmvn_stats=st),
                       g["lda"])
    assert_feats_close(host.FeaturePipeline(capi.default_feat_opts(mode=1), 13, g["lda_aff_mat"])
                       .run(x, fo, cmvn_stats=st), g["lda_aff"])
    assert_feats_close(host.FeaturePipeline(in_dim=13).run(x, fo, cmvn_stats=st, fmllr=g["fmllr_mat"][None]), g["fmllr"])
    fpv = host.FeaturePipeline(capi.default_feat_opts(norm_vars=1, delta_order=0), 13)
    assert_feats_close(fpv.run(x, fo, cmvn_stats=st), g["cmvn_meanvar"])


def test_feature_pipeline_errors():
    fp = host.FeaturePipeline(in_dim=13)
    x = np.ones((10, 13), np.float32)
    with pytest.raises(capi.VbgpuError) as e:  # count < 1 (cmvn.cc:80-82)
        fp.run(x, [0, 10], cmvn_stats=np.zeros((1, 2, 14)))
    assert e.value.code == capi.ERR_NUMERIC
    st = np.zeros((1, 2, 14))
    st[0, 0, 13] = 10
    with pytest.raises(capi.VbgpuError):       # transform-feats.cpp:108-114: bad transform dimension
        fp.run(x, [0, 10], cmvn_stats=st, fmllr=np.zeros((1, 39, 42), np.float32))
    with pytest.raises(capi.VbgpuError):
        host.FeaturePipeline(capi.default_feat_opts(mode=1), 13, np.zeros((40, 90), np.float32))


# ========================================================================================================== scoring
def _pinned_model(chk, m):
    gc, miv, iv = chk.model_params(m.pdf_offsets, m.weights, m.means, m.iv)
    return synth.GmmModel(m.pdf_offsets, m.weights, m.means, iv, miv, gc)


@pytest.mark.parametrize("kernel", [1, 0])
@pytest.mark.parametrize("P,N,D,T,seed", [(11, 60, 39, 100, 1), (50, 400, 39, 333, 2), (30, 200, 40, 257, 3),
                                          (7, 7, 13, 64, 4), (130, 2000, 39, 1000, 5), (3, 700, 39, 50, 6)])
def test_scoring_vs_oracle(orc, kernel, P, N, D, T, seed):
    m = _pinned_model(orc, synth.make_model(P, N, D, seed))
    X = synth.make_feats(m, T, seed + 10)
    am = host.AmDiagGmmGpu.from_model(m)
    am.set_kernel(kernel)
    assert (am.NumPdfs(), am.NumGauss(), am.Dim()) == (P, m.num_gauss, D)
    got = am.score(X)
    rc, want = orc.gmm_loglikes(m, X)
    assert rc == 0
    assert_ll_close(got, want)


@pytest.mark.parametrize("kernel", [1, 0])
def test_scoring_against_reference_dumps(golden, kernel):
    _, g = golden
    am = host.AmDiagGmmGpu(g["pdf_offsets"], g["gconsts"], g["miv"], g["iv"])
    am.set_kernel(kernel)
    assert_ll_close(am.score(g["delta"]), g["loglikes"])


def test_scoring_vs_compiled_reference(ref):
    m = _pinned_model(ref, synth.make_model(40, 300, 39, 9))
    X = synth.make_feats(m, 200, 19)
    rc, want = ref.gmm_loglikes(m, X)
    assert rc == 0
    assert_ll_close(host.AmDiagGmmGpu.from_model(m).score(X), want)


@pytest.mark.parametrize("kernel", [1, 0])
def test_scoring_full_size_properties(orc, kernel):
    """BASELINE cfg 3 shape (P=4000, N=40000, D=39): spot-check random pdf columns against the oracle, then
    size-independent properties: a gconst shift c moves every loglike by c; LSE >= best single Gaussian is
    implied by the oracle check; duplicated frames give duplicated rows."""
    m = synth.make_model(4000, 40000, 39, 11)
    T = 1500
    X = synth.make_feats(m, T, 12)
    X[T // 2:] = X[: T - T // 2]  # duplicated frames
    am = host.AmDiagGmmGpu.from_model(m)
    am.set_kernel(kernel)
    got = am.score(X)
    assert got.shape == (T, 4000) and np.isfinite(got).all()
    assert np.array_equal(got[T // 2:], got[: T - T // 2])
    rng = np.random.default_rng(0)
    pdfs = np.sort(rng.choice(4000, 40, replace=False))
    sub_off = np.zeros(41, np.int32)
    idx = []
    for i, p in enumerate(pdfs):
        g0, g1 = m.pdf_offsets[p], m.pdf_offsets[p + 1]
        idx.extend(range(g0, g1))
        sub_off[i + 1] = sub_off[i] + (g1 - g0)
    idx = np.array(idx)
    sub = synth.GmmModel(sub_off, m.weights[idx], m.means[idx], m.iv[idx], m.miv[idx], m.gconsts[idx])
    rc, want = orc.gmm_loglikes(sub, X[:300])
    assert rc == 0
    assert_ll_close(got[:300][:, pdfs], want)
    am.set_gconsts(m.gconsts + np.float32(2.5))
    shifted = am.score(X[:256])
    assert np.abs((shifted - got[:256]) - 2.5).max() <= 1e-3


def _custom_model(sizes, D, seed, tight=()):
    """A model with the given Gaussians per pdf; pdfs listed in `tight` get a very narrow first Gaussian at the origin
    (largest gconst of its pdf) next to broad ones elsewhere."""
    rng = np.random.default_rng(seed)
    sizes = np.asarray(sizes, np.int32)
    offs = np.zeros(len(sizes) + 1, np.int32)
    offs[1:] = np.cumsum(sizes)
    n = int(offs[-1])
    means = rng.standard_normal((n, D)).astype(np.float32)
    var = (np.exp(0.3 * rng.standard_normal((n, D))) * 0.8).astype(np.float32)
    w = np.exp(rng.standard_normal(n)).astype(np.float32)
    for p in tight:
        g = offs[p]
        means[g] = 0.0
        var[g] = 0.01
        w[g] = 20.0
    for p in range(len(sizes)):
        sl = slice(offs[p], offs[p + 1])
        w[sl] = w[sl] / w[sl].sum()
    iv = (1.0 / var).astype(np.float32)
    miv = (means * iv).astype(np.float32)
    return synth.GmmModel(offs, w, means, iv, miv, synth.compute_gconsts(w, miv, iv))


def test_scoring_column_layout_edge_cases(orc):
    """Tensor-core column layout: runs of single-Gaussian pdfs, pdfs of 63/64/65 Gaussians (parts of 16 + a remainder),
    pdfs cut by a panel edge, more pdfs in a panel than one owner class serves, a trailing incomplete output group."""
    sizes = [1, 1, 1, 2, 1, 3, 1, 1, 64, 1, 63, 2, 1, 5, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 7, 33, 32, 31, 1, 30] + [1] * 70
    for extra in ([], [65]):
        m = _pinned_model(orc, _custom_model(sizes + extra, 39, 31))
        X = (np.random.default_rng(5).standard_normal((300, 39)) * 1.2).astype(np.float32)
        am = host.AmDiagGmmGpu.from_model(m)
        am.set_kernel(2)
        rc, want = orc.gmm_loglikes(m, X)
        assert rc == 0
        assert_ll_close(am.score(X), want)


def test_scoring_widely_separated_gaussians(orc):
    """Gaussians of one pdf thousands of nats apart for the same frame (a very narrow component with the largest
    gconst next to broad ones): the log-sum-exp must stay anchored on the true maximum, not on any fixed column."""
    sizes = [4, 6, 2, 9, 3, 5, 12, 2, 2, 7] * 3
    m = _pinned_model(orc, _custom_model(sizes, 39, 41, tight=(1, 2, 7, 13, 29)))
    X = (np.random.default_rng(6).standard_normal((200, 39)) * 1.5 + 1.0).astype(np.float32)
    X[::7] *= 0.01  # a few frames sit on the narrow Gaussians instead
    rc, want = orc.gmm_loglikes(m, X)
    assert rc == 0
    g = m.pdf_offsets[1]
    ll_first = m.gconsts[g] + X @ m.miv[g] - 0.5 * (X * X) @ m.iv[g]
    assert (want[:, 1] - ll_first).max() > 400.0  # the scenario really is the overflow one
    am = host.AmDiagGmmGpu.from_model(m)
    am.set_kernel(2)
    assert_ll_close(am.score(X), want)


def test_scoring_reports_nonfinite(orc):
    m = synth.make_model(3, 6, 5, 1)
    gc = m.gconsts.copy()
    gc[m.pdf_offsets[1]:m.pdf_offsets[2]] = -np.inf  # zero-weight Gaussians (diag-gmm.cc:141-146)
    am = host.AmDiagGmmGpu(m.pdf_offsets, gc, m.miv, m.iv)
    with pytest.raises(capi.VbgpuError) as e:  # decodable-am-diag-gmm.cc:65-66 raises KALDI_ERR
        am.score(synth.make_feats(m, 8, 2))
    assert e.value.code == capi.ERR_NUMERIC
    # a single -inf component inside a healthy pdf is fine and ignored
    gc = m.gconsts.copy()
    gc[m.pdf_offsets[1]] = -np.inf
    m2 = synth.GmmModel(m.pdf_offsets, m.weights, m.means, m.iv, m.miv, gc)
    X = synth.make_feats(m, 8, 2)
    rc, want = orc.gmm_loglikes(m2, X)
    if m.pdf_offsets[2] - m.pdf_offsets[1] > 1:
        assert rc == 0
        assert_ll_close(host.AmDiagGmmGpu.from_model(m2).score(X), want)
    with pytest.raises(capi.VbgpuError):
        host.AmDiagGmmGpu(m.pdf_offsets, np.full_like(gc, np.nan), m.miv, m.iv)


def test_decodable_interface(orc):
    m = _pinned_model(orc, synth.make_model(11, 40, 39, 3))
    X = synth.make_feats(m, 30, 4)
    tid2pdf = np.array([0] + [i // 2 for i in range(22)], np.int32)  # 1-based transition ids
    dec = host.DecodableAmDiagGmmGpu(host.AmDiagGmmGpu.from_model(m), tid2pdf, X, scale=0.0833333)
    _, ll = orc.gmm_loglikes(m, X)
    assert dec.NumFramesReady() == 30 and dec.NumIndices() == 22
    assert dec.IsLastFrame(29) and not dec.IsLastFrame(0)
    for f, tid in ((0, 1), (7, 22), (29, 13)):
        assert abs(dec.LogLikelihood(f, tid) - 0.0833333 * ll[f, tid2pdf[tid]]) <= 1e-3 * 0.0833333


# ======================================================================================================= statistics
@pytest.mark.parametrize("P,N,D,T,seed", [(11, 60, 39, 200, 1), (50, 400, 40, 500, 2), (5, 300, 13, 300, 3)])
@pytest.mark.parametrize("mode", ["plain", "weighted", "twofeats"])
def test_accumulate_vs_oracle(orc, P, N, D, T, seed, mode):
    m = _pinned_model(orc, synth.make_model(P, N, D, seed))
    X = synth.make_feats(m, T, seed + 10)
    ali = synth.make_alignment(P, T, seed)
    w = np.random.default_rng(seed).uniform(0.1, 1.0, T).astype(np.float32) if mode != "plain" else None
    X2 = synth.make_feats(m, T, seed + 20) if mode == "twofeats" else None
    acc = host.AccumAmDiagGmmGpu(host.AmDiagGmmGpu.from_model(m))
    tl = acc.AccumulateForUtterance(X, ali, w, X2)
    occ, mean, var, tot_like, tot_frames = acc.download()
    rc, o2, m2, v2, tl2, tf2 = orc.acc_ali(m, X, ali, w, X2)
    assert rc == 0
    assert_acc_close((occ, mean, var), (o2, m2, v2))
    assert abs(tot_like - tl2) <= 1e-5 * abs(tl2) and abs(tl - tl2) <= 1e-5 * abs(tl2)
    assert abs(tot_frames - tf2) <= 1e-6 * tf2
    # Add / SetZero (AccumAmDiagGmm::Add, mle-am-diag-gmm.cc:279-287)
    acc2 = host.AccumAmDiagGmmGpu(acc.am)
    acc2.Add(0.5, acc)
    acc2.Add(0.5, acc)
    o3, m3, v3, tl3, tf3 = acc2.download()
    assert np.allclose(o3, occ, rtol=1e-14) and np.allclose(m3, mean, rtol=1e-14) and abs(tf3 - tot_frames) < 1e-9
    acc.SetZero()
    assert acc.download()[0].sum() == 0 and acc.TotCount() == 0


def test_accumulate_against_reference_dumps(golden):
    _, g = golden
    am = host.AmDiagGmmGpu(g["pdf_offsets"], g["gconsts"], g["miv"], g["iv"])
    acc = host.AccumAmDiagGmmGpu(am)
    acc.AccumulateForUtterance(g["delta"], g["ali"])
    occ, mean, var, tl, tf = acc.download()
    assert_acc_close((occ, mean, var), (g["acc_occ"], g["acc_mean"], g["acc_var"]))
    assert abs(tl - g["acc_tot"][0]) <= 1e-5 * abs(g["acc_tot"][0]) and tf == g["acc_tot"][1]
    acc.SetZero()
    acc.AccumulateForUtterance(g["delta"], g["ali"], g["ali_w"], g["fmllr"])
    occ, mean, var, tl, tf = acc.download()
    assert_acc_close((occ, mean, var), (g["acc2_occ"], g["acc2_mean"], g["acc2_var"]))


def test_accumulate_full_size_properties():
    """cfg 5 shape (N=40000): sum of occupancies == number of frames (posteriors sum to 1), per-pdf occupancy ==
    frames aligned to it, variance stats non-negative; an invalid pdf-id is reported."""
    m = synth.make_model(4000, 40000, 39, 11)
    T = 50000
    X = synth.make_feats(m, T, 12)
    ali = synth.make_alignment(4000, T, 5)
    acc = host.AccumAmDiagGmmGpu(host.AmDiagGmmGpu.from_model(m))
    acc.AccumulateForUtterance(X, ali)
    occ, mean, var, tl, tf = acc.download()
    assert tf == T and abs(occ.sum() - T) <= 1e-5 * T and (var >= 0).all() and np.isfinite(mean).all()
    per_pdf = np.add.reduceat(occ, m.pdf_offsets[:-1])
    assert np.abs(per_pdf - np.bincount(ali, minlength=4000)).max() <= 1e-3
    bad = ali.copy()
    bad[7] = 4000
    with pytest.raises(capi.VbgpuError):
        acc.AccumulateForUtterance(X[:100], bad[:100])


# ============================================================================================== the fused pipeline
@pytest.mark.parametrize("cfg", ["delta", "delta_sat", "lda"])
def test_pipeline_pcm_to_loglikes(orc, cfg):
    """The measured path end to end: PCM -> MFCC -> CMVN(per speaker) -> deltas|LDA -> [fMLLR] -> loglikes, host
    buffers through the C ABI, against the oracle chain."""
    import torch
    o = gopts()
    n_spk = 3
    pcm, so, u2s = synth.make_corpus(n_spk, 3, 0.4, 1.1, 31)
    fopts = capi.default_feat_opts(mode=1 if cfg == "lda" else 0)
    lda = synth.make_lda(40, 91, 2) if cfg == "lda" else None
    D = 40 if cfg == "lda" else 39
    fm = synth.make_fmllr(n_spk, D, 6) if cfg == "delta_sat" else None
    mf_want, fo = oracle_mfcc_batch(orc, o, pcm, so)
    st = oracle_stats(orc, mf_want, fo, u2s, n_spk)
    feats_want = oracle_feats(orc, mf_want, fo, u2s, st, fopts, lda, fm)
    model = _pinned_model(orc, synth.make_model_from_feats(feats_want, 60, 500, 3))
    rc, ll_want = orc.gmm_loglikes(model, feats_want)
    assert rc == 0

    mf, fp, am = host.Mfcc(o), host.FeaturePipeline(fopts, 13, lda), host.AmDiagGmmGpu.from_model(model)
    pipe = host.ScoringPipeline(mf, fp, am)
    ll, feats = pipe.score(pcm, so, u2s, n_spk, fmllr=fm, return_feats=True)
    assert_feats_close(feats, feats_want)
    assert_ll_close(ll, ll_want)
    # pinned buffers take the direct-DMA path and give the same bits
    pin_pcm = torch.from_numpy(pcm).pin_memory()
    pin_out = torch.empty((ll.shape[0], am.NumPdfs()), dtype=torch.float32).pin_memory()
    ll2 = pipe.score(pin_pcm, so, u2s, n_spk, fmllr=fm, out=pin_out)
    assert np.array_equal(ll2.numpy(), ll)
    # device-resident form == host form
    d_pcm = torch.from_numpy(pcm).cuda()
    d_ll = torch.empty((ll.shape[0], am.NumPdfs()), dtype=torch.float32, device="cuda")
    d_fm = torch.from_numpy(fm).cuda() if fm is not None else None
    pipe.score_dev(d_pcm, so, u2s, n_spk, d_fm, (D + 1) if fm is not None else 0, d_ll, am.NumPdfs())
    torch.cuda.synchronize()
    assert np.array_equal(d_ll.cpu().numpy(), ll)
    assert am.bad_count() == 0
    # training form: PCM + alignment -> statistics
    ali = synth.make_alignment(60, ll.shape[0], 8)
    acc = host.AccumAmDiagGmmGpu(am)
    pipe.accumulate_dev(acc, d_pcm, so, u2s, n_spk, d_fm, (D + 1) if fm is not None else 0,
                        torch.from_numpy(ali).cuda())
    torch.cuda.synchronize()
    occ, mean, var, tl, tf = acc.download()
    # statistics are judged on identical features (feature parity is asserted above; posteriors amplify the
    # 1e-5-level feature noise of two FP32 front ends beyond the statistics tolerance on a batch this small)
    rc, o2, m2, v2, tl2, tf2 = orc.acc_ali(model, feats, ali)
    assert_acc_close((occ, mean, var), (o2, m2, v2))
    assert tf == tf2 and abs(tl - tl2) <= 1e-5 * abs(tl2)


def test_pipeline_many_slabs(orc):
    """A batch large enough that the host form streams several output slabs (overlapped D2H); results must equal the
    single-call scorer on the same features."""
    o = gopts()
    pcm, so, u2s = synth.make_corpus(8, 8, 3.0, 6.0, 41, fast=True)
    model = synth.make_model(3000, 9000, 39, 4)
    mf, fp, am = host.Mfcc(o), host.FeaturePipeline(in_dim=13), host.AmDiagGmmGpu.from_model(model)
    pipe = host.ScoringPipeline(mf, fp, am)
    ll, feats = pipe.score(pcm, so, u2s, 8, return_feats=True)
    assert ll.shape[0] * 3000 * 4 > 600e6 / 2  # > 1 slab of 256 MiB
    direct = am.score(feats)
    assert np.array_equal(direct, ll)


# ================================================================================== filterbank front end (§8f n4)
FBANK_VARIANTS = [
    dict(), dict(use_energy=1), dict(use_energy=1, htk_compat=1), dict(use_energy=1, raw_energy=0, energy_floor=1e9),
    dict(samp_freq=8000.0), dict(num_bins=30), dict(htk_mode=1), dict(snip_edges=0), dict(low_freq=100.0, high_freq=-400.0),
]


@pytest.mark.parametrize("use_log,use_power", [(1, 1), (0, 1), (1, 0)])
@pytest.mark.parametrize("kw", FBANK_VARIANTS, ids=lambda d: ",".join("%s=%s" % kv for kv in d.items()) or "default")
def test_fbank_single_utterance(orc, kw, use_log, use_power):
    o = gopts(**kw)
    w = synth.make_wave(int(o.samp_freq * 1.3), 5, o.samp_freq)
    fb = host.Fbank(o, use_log, use_power)
    got = fb.ComputeFeatures(w, o.samp_freq)
    want = orc.fbank(to_orc_opts(o), w.astype(np.float32), 1.0, use_log, use_power)
    assert got.shape == want.shape == (fb.NumFrames(len(w)), fb.Dim())
    assert fb.Dim() == o.num_bins + (1 if o.use_energy else 0)
    assert_feats_close(got, want, what="fbank")
    assert np.array_equal(got, fb.ComputeFeatures(w.astype(np.float32)))


# per-utterance VTLN warps of one ragged batch: 0.9 and 1.1 come back after other warps, 1.0 (no warp) sits between them
BATCH_VTLN_LENS = [0, 399, 400, 4801, 16000, 7777, 3000, 5000, 2500]
BATCH_VTLN_WARPS = [1.0, 0.9, 1.1, 1.0, 0.85, 1.2, 0.9, 1.1, 1.0]


def _batch_vtln_wave():
    so = np.zeros(len(BATCH_VTLN_LENS) + 1, np.int64)
    so[1:] = np.cumsum(BATCH_VTLN_LENS)
    return synth.make_wave(int(so[-1]), 3), so, np.array(BATCH_VTLN_WARPS, np.float32)


@pytest.mark.parametrize("use_log,use_power", [(1, 1), (0, 1), (1, 0)])
def test_fbank_batch_vtln(orc, use_log, use_power):
    """A ragged batch with a VTLN warp per utterance (per-warp mel banks on the device): every utterance equals the oracle
    run on it alone with its warp, and the reference's own code where it is built."""
    o = gopts(use_energy=1)
    pcm, so, vtln = _batch_vtln_wave()
    fb = host.Fbank(o, use_log, use_power)
    got, fo = fb.compute_batch(pcm, so, vtln)
    oo = to_orc_opts(o)
    ref = po.load("ref") if po.have_ref() else None
    for u in range(len(so) - 1):
        w = pcm[so[u]:so[u + 1]].astype(np.float32)
        want = orc.fbank(oo, w, float(vtln[u]), use_log, use_power)
        assert_feats_close(got[fo[u]:fo[u + 1]], want, what="fbank utt %d (warp %g)" % (u, vtln[u]))
        if ref is not None:
            assert_feats_close(got[fo[u]:fo[u + 1]], ref.fbank(oo, w, float(vtln[u]), use_log, use_power),
                               what="fbank utt %d vs reference" % u)


# ================================================================================== host threads (nj jobs of the recipes)
def test_concurrent_job_threads(orc):
    """The recipes run nj job threads, each with its own Mfcc / model objects (decode_gmm.cpp:300-324).  Four host threads
    with their own handles (one model shared read-only through separate handles) must reproduce the serial results."""
    import threading
    o = gopts()
    fopts = capi.default_feat_opts()
    m = _pinned_model(orc, synth.make_model(60, 600, 39, 81))
    jobs = []
    for j in range(4):
        pcm, so, u2s = synth.make_corpus(2, 3, 0.4, 0.9, 200 + j)
        jobs.append((pcm, so, u2s))

    def run(j, out):
        pcm, so, u2s = jobs[j]
        pipe = host.ScoringPipeline(host.Mfcc(o), host.FeaturePipeline(fopts, 13), host.AmDiagGmmGpu.from_model(m))
        for _ in range(3):
            out[j] = pipe.score(pcm, so, u2s, 2)

    serial, par = {}, {}
    for j in range(4):
        run(j, serial)
    th = [threading.Thread(target=run, args=(j, par)) for j in range(4)]
    [t.start() for t in th]
    [t.join() for t in th]
    for j in range(4):
        assert par[j].shape == serial[j].shape and np.array_equal(par[j], serial[j])


# ============================================================================================ PLP front end (§8f n4)
PLP_VARIANTS = [
    dict(), dict(use_energy=1), dict(use_energy=1, htk_compat=1), dict(samp_freq=8000.0, num_bins=15), dict(cepstral_lifter=0.0),
    dict(htk_mode=1), dict(snip_edges=0), dict(num_ceps=9), dict(use_energy=1, raw_energy=0, energy_floor=1e9),
]


@pytest.mark.parametrize("kw", PLP_VARIANTS, ids=lambda d: ",".join("%s=%s" % kv for kv in d.items()) or "default")
def test_plp_single_utterance(orc, kw):
    o = gopts(**kw)
    w = synth.make_wave(int(o.samp_freq * 1.3), 5, o.samp_freq)
    for extra in (dict(), dict(lpc_order=14, compress_factor=0.5, cepstral_scale=10.0)):
        plp = host.Plp(o, **extra)
        got = plp.ComputeFeatures(w, o.samp_freq)
        want = orc.plp(to_orc_opts(o), w.astype(np.float32), 1.0, **extra)
        assert got.shape == want.shape == (plp.NumFrames(len(w)), o.num_ceps)
        assert_feats_close(got, want, what="plp")
        assert np.array_equal(got, plp.ComputeFeatures(w.astype(np.float32)))


def test_plp_batch_vtln(orc):
    """PLP of the same ragged VTLN batch (per-warp mel banks and equal-loudness tables): every utterance equals the oracle
    with its warp, and the reference's own code where it is built."""
    o = gopts(use_energy=1)
    pcm, so, vtln = _batch_vtln_wave()
    got, fo = host.Plp(o).compute_batch(pcm, so, vtln)
    oo = to_orc_opts(o)
    ref = po.load("ref") if po.have_ref() else None
    for u in range(len(so) - 1):
        w = pcm[so[u]:so[u + 1]].astype(np.float32)
        assert_feats_close(got[fo[u]:fo[u + 1]], orc.plp(oo, w, float(vtln[u])), what="plp utt %d (warp %g)" % (u, vtln[u]))
        if ref is not None:
            assert_feats_close(got[fo[u]:fo[u + 1]], ref.plp(oo, w, float(vtln[u])), what="plp utt %d vs reference" % u)
    with pytest.raises(capi.VbgpuError):  # num_ceps > lpc_order + 1 (feature-plp.cc:126)
        host.Plp(gopts(num_ceps=13), lpc_order=8)


def test_scoring_tail_wave_is_split(orc):
    """More frame tiles than four waves of CTAs, with a remainder: the tiles of the last, partial wave are cut into panel
    ranges (score_tc_launch).  Same results as the FP32 SIMT kernel on every frame, and as the oracle on the frames of
    the whole-tile region, of the cut tiles and of the ragged last tile."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    m = _pinned_model(orc, synth.make_model(300, 3000, 39, 91))
    T = 256 * (4 * sms + 30) + 17
    X = synth.make_feats(m, T, 92)
    am = host.AmDiagGmmGpu.from_model(m)
    am.set_kernel(2)
    got = am.score(X)
    am.set_kernel(1)
    simt = am.score(X)
    assert got.shape == (T, 300) and np.isfinite(got).all()
    assert np.abs(got - simt).max() <= 5e-4
    rows = np.r_[0:40, 256 * 4 * sms - 20:256 * 4 * sms + 40, 256 * (4 * sms + 29) + 200:T]
    rc, want = orc.gmm_loglikes(m, X[rows])
    assert rc == 0
    assert_ll_close(got[rows], want)


# ================================================================================ round 2: parity where the numbers are taken
def _sub_model(m, pdfs):
    sub_off = np.zeros(len(pdfs) + 1, np.int32)
    idx = []
    for i, p in enumerate(pdfs):
        g0, g1 = m.pdf_offsets[p], m.pdf_offsets[p + 1]
        idx.extend(range(g0, g1))
        sub_off[i + 1] = sub_off[i] + (g1 - g0)
    idx = np.array(idx)
    return synth.GmmModel(sub_off, m.weights[idx], m.means[idx], m.iv[idx], m.miv[idx], m.gconsts[idx])


@pytest.mark.parametrize("P,N,D,name", [(2000, 10000, 39, "cfg 2 tri-delta"), (2500, 15000, 40, "cfg 4 LDA+MLLT (K = 96 instantiation)")])
def test_scoring_full_size_other_configs(orc, P, N, D, name):
    """BASELINE configs[1] and [3] at FULL model size on the tensor-core handle: random pdf columns of 1500 frames against
    the oracle; every column against the FP32 SIMT kernel."""
    m = synth.make_model(P, N, D, 31)
    X = synth.make_feats(m, 1500, 32)
    am = host.AmDiagGmmGpu.from_model(m)
    assert am.plan_note() == "", am.plan_note()
    am.set_kernel(2)
    got = am.score(X)
    am.set_kernel(1)
    simt = am.score(X[:400])
    assert np.abs(got[:400] - simt).max() <= 5e-4
    pdfs = np.sort(np.random.default_rng(3).choice(P, 60, replace=False))
    rc, want = orc.gmm_loglikes(_sub_model(m, pdfs), X)
    assert rc == 0
    assert_ll_close(got[:, pdfs], want, what=name)


def test_scoring_error_vs_magnitude(orc):
    """Where does 1e-3 absolute stop being meaningful?  The same frames are pushed away from the model (x -> c + k (x - c)),
    which moves |loglike| from ~100 to several thousand.  The reference computes in FP32 (ulp 6e-5 at 500, 4.9e-4 at 5000).
    The split-fp16 error of a frame scales with the size of the terms that are summed (x^2 / var), i.e. with the frame's
    largest |loglike|, not with the one pdf looked at, so the bound is per frame: 1e-3 for frames whose scores all stay
    within |ll| <= 1000, and 16 ulp of the frame's largest FP32 |ll| beyond (measured on B200: 4.4e-4 within 1000, 1.2e-3
    around 2500, 2.4e-3 = 10 ulp of that frame's largest score around 5800 — the decoder's beam discards such frames, and two BLAS libraries differ by as
    much there).  The table is printed with pytest -s."""
    m = _pinned_model(orc, synth.make_model(120, 1000, 39, 51))
    X0 = synth.make_feats(m, 256, 52)
    c = (m.means * 1.0).mean(axis=0)
    am = host.AmDiagGmmGpu.from_model(m)
    am.set_kernel(2)
    rows = []
    for k in (1.0, 1.5, 2.0, 3.0, 4.0, 6.0, 8.0):
        X = (c + k * (X0 - c)).astype(np.float32)
        rc, want = orc.gmm_loglikes(m, X)
        assert rc == 0
        got = am.score(X)
        err, mag = np.abs(got - want), np.abs(want)
        rows.append((k, float(np.median(mag)), float(mag.max()), float(err.max())))
        frame_mag = mag.max(axis=1)
        small = frame_mag <= 1000.0
        if small.any():
            assert err[small].max() <= 1e-3, "k = %g: %.3g on frames within |ll| <= 1000" % (k, err[small].max())
        tol = np.maximum(1e-3, 16.0 * np.spacing(frame_mag.astype(np.float32)).astype(np.float64))
        worst = (err.max(axis=1) / tol).max()
        assert worst <= 1.0, "k = %g: max err %.3g at |ll| up to %.0f (%.2f of the per-frame bound)" % (k, err.max(), mag.max(), worst)
    print("\\n  stretch  median|ll|   max|ll|   max abs err")
    for r in rows:
        print("  %6.1f  %10.0f  %8.0f   %.2e" % r)
    assert rows[0][3] <= 3e-4            # at the model's own scale the scheme sits well inside the budget


def test_scoring_outlier_frames_and_large_pdfs_stay_on_the_tensor_cores(orc):
    """A frame 100 sigma away from every Gaussian (outside the fp16 scaling plan: re-scored by the FP32 fix-up kernel, the
    reference returns a finite, very negative score) and a pdf of 600 Gaussians (cut into virtual pdfs + merge kernel): both on
    the tcgen05 handle, no error, oracle values."""
    sizes = [5, 600, 3, 41, 9, 81, 12] + [4] * 20
    m = _pinned_model(orc, _custom_model(sizes, 39, 77))
    am = host.AmDiagGmmGpu.from_model(m)
    assert am.plan_note() == "", am.plan_note()
    am.set_kernel(2)
    X = (np.random.default_rng(8).standard_normal((300, 39)) * 1.1).astype(np.float32)
    X[17] = 100.0 * np.sign(X[17])       # ~100 sigma out in every dimension
    X[255] *= 60.0
    X[299, 5] = -3000.0                  # one wild coordinate
    rc, want = orc.gmm_loglikes(m, X)
    assert rc == 0 and np.isfinite(want).all()
    got = am.score(X)
    ok = np.ones(300, bool)
    ok[[17, 255, 299]] = False
    assert_ll_close(got[ok], want[ok], what="regular frames next to outliers")
    # the outlier rows come from the FP32 kernel: FP32 accuracy at their magnitude (|ll| up to 1e7)
    for t in (17, 255, 299):
        rel = np.abs(got[t] - want[t]) / np.abs(want[t])
        assert rel.max() <= 2e-6, (t, rel.max(), np.abs(want[t]).max())


@pytest.mark.gpu
def test_scoring_long_run_of_sunk_frames_is_rescored_in_parallel(orc):
    """An utterance that went wrong: 3000 consecutive frames far from the model (scores below the padding level).  All of
    them are re-scored by the FP32 kernel, the count is reported, the frames around them keep the tensor-core values, and the
    launch stays fast (the flagged frames are spread over the whole grid, not walked by the warp that owns their position)."""
    import time
    m = _pinned_model(orc, synth.make_model(300, 3000, 39, 61))
    X = synth.make_feats(m, 6000, 62)
    X[1500:4500] *= 40.0
    rc, want = orc.gmm_loglikes(m, X)
    assert rc == 0 and np.isfinite(want).all()
    am = host.AmDiagGmmGpu.from_model(m)
    am.set_kernel(2)
    got = am.score(X)
    n = am.rescored_frames()
    assert n >= 2900, n
    ok = np.ones(6000, bool)
    ok[1500:4500] = False
    assert_ll_close(got[ok], want[ok], what="frames around the broken run")
    rel = np.abs(got[~ok] - want[~ok]) / np.abs(want[~ok])
    assert rel.max() <= 2e-6, rel.max()
    t0 = time.perf_counter()
    am.score(X)
    assert time.perf_counter() - t0 < 0.5      # was seconds when one warp walked a run of flagged frames


@pytest.mark.gpu
@pytest.mark.parametrize("orig,new,n", [(16000, 8000, 16000), (44100, 16000, 30001), (48000, 16000, 5000), (22050, 16000, 12345),
                                        (16000, 8000, 7), (11025, 8000, 3000), (16000, 8000, 0)])
def test_downsample_waveform_vs_oracle_and_reference(orc, orig, new, n):
    """DownsampleWaveForm (feat/resample.cc:368-376) on the device: length and samples.  The oracle port is pinned against the
    compiled reference in tests/test_oracle_vs_ref.py; 2e-6 of the largest sample (FP32 dot products in a different order).
    The comparison with the compiled reference itself runs only where oracle/_ref is built; in every checkout the same rate
    pairs are checked against stored reference outputs by test_downsample_golden_dumps_of_the_reference."""
    w = (np.random.default_rng(n + orig).standard_normal(n) * 3000).astype(np.float32)
    want = orc.downsample_waveform(orig, new, w)
    d = host.Downsampler(orig, new)
    assert d.NumOut(n) == len(want)
    got = d(w)
    assert got.shape == want.shape
    if len(want):
        assert np.abs(got - want).max() <= 2e-6 * np.abs(want).max()
    if po.have_ref() and n:
        ref = po.load("ref").downsample_waveform(orig, new, w)
        assert len(ref) == len(got) and np.abs(got - ref).max() <= 2e-6 * np.abs(ref).max()


@pytest.mark.gpu
def test_mfcc_compute_features_allow_downsample(orc):
    """OfflineFeatureTpl::ComputeFeatures (feature-common-inl.h:29-55): a wave above the configured rate is down-sampled when
    allow_downsample is set, refused otherwise; a wave below it is always refused."""
    opts = capi.default_mfcc_opts(dither=0.0, samp_freq=8000.0)
    w16 = synth.make_wave(16000 * 2, 5, 16000).astype(np.float32)
    want = orc.mfcc(to_orc_opts(opts), orc.downsample_waveform(16000, 8000, w16))
    got = host.Mfcc(opts, allow_downsample=True).ComputeFeatures(w16, 16000)
    assert_feats_close(got, want, what="MFCC of a down-sampled wave")
    with pytest.raises(capi.VbgpuError, match="allow_downsample"):
        host.Mfcc(opts).ComputeFeatures(w16, 16000)
    with pytest.raises(capi.VbgpuError, match="larger than waveform"):
        host.Mfcc(opts, allow_downsample=True).ComputeFeatures(w16, 4000)
    with pytest.raises(capi.VbgpuError):
        host.Downsampler(8000, 16000)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(24))
def test_scoring_tensor_core_vs_fp32_kernel_random_layouts(seed):
    """Random model shapes through both scorers of the library: pdf sizes from several distributions (all ones, uniform small,
    heavy tail up to 300 Gaussians, everything at the 10 / 20 / 40 slot boundaries), D from 13 to 47 (both K instantiations),
    ragged frame counts (partial tiles, panel splits), features stretched up to 3x away from the model.  The FP32 SIMT kernel
    is the parity anchor (itself checked against the oracle above); the bound is the one of test_scoring_error_vs_magnitude."""
    rng = np.random.default_rng(1000 + seed)
    P = int(rng.choice([1, 3, 17, 64, 150, 333, 600]))
    kind = seed % 6
    if kind == 0:
        sizes = np.ones(P, np.int64)
    elif kind == 1:
        sizes = rng.integers(1, 13, P)
    elif kind == 2:
        sizes = np.minimum(300, np.maximum(1, (rng.pareto(1.2, P) * 4).astype(np.int64)))
    elif kind == 3:
        sizes = rng.choice([10, 11, 20, 21, 40, 41], P)
    elif kind == 4:
        sizes = rng.integers(30, 90, P)
    else:
        sizes = rng.integers(1, 41, P)
    D = int(rng.choice([13, 20, 39, 40, 47]))
    T = int(rng.choice([1, 31, 129, 257, 1000, 2500]))
    m = _custom_model([int(v) for v in sizes], D, 2000 + seed)
    X = (np.random.default_rng(3000 + seed).standard_normal((T, D)) * rng.uniform(0.5, 3.0)).astype(np.float32)
    am = host.AmDiagGmmGpu.from_model(m)
    assert am.plan_note() == "", am.plan_note()
    am.set_kernel(1)
    want = am.score(X)
    am.set_kernel(2)
    got = am.score(X)
    assert np.isfinite(want).all() and got.shape == want.shape
    err, mag = np.abs(got - want), np.abs(want)
    frame_mag = mag.max(axis=1)
    tol = np.maximum(1e-3, 16.0 * np.spacing(frame_mag.astype(np.float32)).astype(np.float64))
    worst = (err.max(axis=1) / tol).max()
    assert worst <= 1.0, "P=%d D=%d T=%d kind=%d: max err %.3g at |ll| up to %.0f (%.2f of the bound)" % (P, D, T, kind, err.max(), mag.max(), worst)


@pytest.mark.gpu
def test_downsample_golden_dumps_of_the_reference():
    """The device DownsampleWaveForm and ComputeFeatures(allow_downsample) against dumps of the compiled reference
    (tests/golden/downsample_golden.npz; no oracle in between)."""
    import os
    from tests.golden.make_downsample_golden import PAIRS, noise
    d = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    g = dict(np.load(os.path.join(d, "downsample_golden.npz")))
    pcm = np.load(os.path.join(d, "htk_golden.npz"))["pcm"].astype(np.float32)
    cases = [(16000, 8000, pcm, "speech_16k_to_8k"), (16000, 11025, pcm, "speech_16k_to_11025")]
    cases += [(o, n_, noise(n, n), "noise_%d_to_%d_%d" % (o, n_, n)) for o, n_, n in PAIRS]
    for orig, new, w, key in cases:
        got, want = host.Downsampler(orig, new)(w), g[key]
        assert got.shape == want.shape, key
        assert np.abs(got - want).max() <= 2e-6 * np.abs(want).max(), key
    opts = capi.default_mfcc_opts(dither=0.0, samp_freq=8000.0)
    got = host.Mfcc(opts, allow_downsample=True).ComputeFeatures(pcm, 16000)
    assert_feats_close(got, g["mfcc_of_speech_8k"], what="MFCC of the down-sampled test.wav")
