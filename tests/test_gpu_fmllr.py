"""fMLLR and MLLT sufficient statistics on the device (SURVEY.md §8f n1) against the float64 restatements and the plain-C
oracle; where the reference is built (oracle/_ref), its solvers must also land on the same transform from the device's
statistics as from its own."""
import numpy as np
import pytest

from tests.common import assert_fmllr_close, fmllr_truth
from voicebridge_b200 import capi, host, synth

pytestmark = pytest.mark.gpu


def _model(chk, P, N, D, seed):
    m = synth.make_model(P, N, D, seed)
    gc, miv, iv = chk.model_params(m.pdf_offsets, m.weights, m.means, m.iv)
    return synth.GmmModel(m.pdf_offsets, m.weights, m.means, iv, miv, gc)


@pytest.mark.parametrize("D,weighted,T", [(39, False, 1200), (40, True, 1500), (13, True, 700), (39, True, 1)])
def test_fmllr_stats_single_speaker(orc, D, weighted, T):
    m = _model(orc, 25, 180, D, 51)
    X = synth.make_feats(m, T, 52)
    ali = synth.make_alignment(25, T, 53)
    w = np.random.default_rng(54).uniform(0.2, 1.0, T).astype(np.float32) if weighted else None
    acc = host.FmllrDiagGmmAccsGpu(host.AmDiagGmmGpu.from_model(m))
    tl = acc.AccumulateForUtterances(X, ali, weights=w)
    rc, ob, oK, oG, ol = orc.fmllr_acc(m, X, ali, w)
    assert rc == 0 and abs(tl - ol) <= 1e-4 * abs(ol)
    assert_fmllr_close(acc.stats(0), fmllr_truth(m, X, ali, w), what="GPU")
    # a second call adds; SetZero clears
    acc.AccumulateForUtterances(X, ali, weights=w)
    b2, K2, G2 = acc.stats(0)
    assert abs(b2 - 2 * ob) <= 1e-4 * max(ob, 1.0) and np.abs(G2 - 2 * oG).max() <= 2e-4 * np.abs(oG).max()
    acc.SetZero()
    b0, K0, G0 = acc.stats(0)
    assert b0 == 0.0 and not K0.any() and not G0.any()


# A packed batch of (frames, speaker): speakers whose utterances are not adjacent, empty and one-frame utterances inside a
# speaker's run, runs of 2600 (three 1024-frame work units), exactly 1024 and 1025 frames, and speakers without data.
MANY_SPEAKERS = [
    (300, 0),                                     # speaker 0 at the start ...
    (257, 2), (0, 2), (1, 2), (130, 2),           # 0- and 1-frame utterances inside one run of speaker 2
    (90, 1), (60, 4), (75, 1), (40, 5), (120, 1),  # speaker 1 interleaved with speakers 4 and 5
    (1000, 6), (900, 6), (700, 6),                # one run of 2600 frames
    (1024, 7),                                    # one run of exactly one work unit
    (600, 8), (425, 8),                           # 1025 frames: a full unit and a one-frame unit
    (0, 9),                                       # speaker 9: only an empty utterance
    (100, 4), (0, 1), (50, 4),                    # an empty utterance of speaker 1 inside a run of speaker 4
    (400, 0),                                     # ... and at the end
]
MANY_SPEAKERS_N = 11                              # speakers 3 and 10: no utterance at all


@pytest.mark.parametrize("P,N,D,seed", [(5, 300, 13, 3), (40, 900, 39, 61), (12, 700, 40, 5)])
def test_fmllr_stats_many_speakers(orc, monkeypatch, P, N, D, seed):
    """Every speaker's statistics of one packed, weighted call equal the float64 restatement over that speaker's frames
    alone, and the call's log-likelihood the oracle's.  The models hold pdfs of more than 64 Gaussians next to smaller
    ones, so some frames take the bucketed posterior kernel and the rest fmllr_ab_kernel; VBGPU_ACC_FRAMEWISE sends every
    frame through fmllr_ab_kernel; the device form reads strided features on a caller's stream.  All three agree with
    the restatement.  Where the reference is built, FmllrDiagGmmAccs::Update also gives the same transform from the
    device statistics as from the reference's own."""
    import torch
    from oracle import pyoracle as po
    m = _model(orc, P, N, D, seed)
    lens = np.array([n for n, _ in MANY_SPEAKERS])
    u2s = np.array([s for _, s in MANY_SPEAKERS], np.int32)
    fo = np.zeros(len(lens) + 1, np.int64)
    fo[1:] = np.cumsum(lens)
    T, n_spk = int(fo[-1]), MANY_SPEAKERS_N
    X = synth.make_feats(m, T, seed + 1)
    ali = synth.make_alignment(P, T, seed + 2)
    rng = np.random.default_rng(seed + 3)
    w = rng.uniform(0.2, 1.0, T).astype(np.float32)
    w[rng.random(T) < 0.1] = 0.0
    sizes = np.diff(m.pdf_offsets)
    big = sizes[ali] > 64  # frames of fmllr_ab_kernel; the rest take the bucketed kernel
    assert (sizes > 64).any() and (sizes <= 64).any() and big.any() and (~big).any()
    assert (big & (w == 0)).any() and (big & (w > 0)).any()
    spk_rows = [np.concatenate([np.arange(fo[u], fo[u + 1]) for u in range(len(lens)) if u2s[u] == s] or [np.zeros(0, int)])
                for s in range(n_spk)]
    truth, want_like = {}, 0.0
    for s, rows in enumerate(spk_rows):
        if len(rows):
            truth[s] = fmllr_truth(m, X[rows], ali[rows], w[rows])
            rc, _, _, _, ol = orc.fmllr_acc(m, X[rows], ali[rows], w[rows])
            assert rc == 0
            want_like += ol
    assert sorted(truth) == [0, 1, 2, 4, 5, 6, 7, 8]

    def check(acc, what):
        for s in range(n_spk):
            b, K, G = acc.stats(s)
            if s not in truth:
                assert b == 0.0 and not K.any() and not G.any(), "%s: speaker %d has no data" % (what, s)
            else:
                assert_fmllr_close((b, K, G), truth[s], what="%s, speaker %d" % (what, s))

    am = host.AmDiagGmmGpu.from_model(m)
    acc = host.FmllrDiagGmmAccsGpu(am, n_spk=n_spk)
    tl = acc.AccumulateForUtterances(X, ali, frame_offsets=fo, utt2spk=u2s, weights=w)
    assert abs(tl - want_like) <= 1e-4 * abs(want_like)
    check(acc, "GPU")
    with monkeypatch.context() as mp:
        mp.setenv("VBGPU_ACC_FRAMEWISE", "1")
        fw = host.FmllrDiagGmmAccsGpu(am, n_spk=n_spk)
        tl_fw = fw.AccumulateForUtterances(X, ali, frame_offsets=fo, utt2spk=u2s, weights=w)
    assert abs(tl_fw - want_like) <= 1e-4 * abs(want_like)
    check(fw, "GPU frame-wise")
    # device form: rows D + 5 floats apart (the padding holds values no feature has), on a non-default stream
    d_x = torch.full((T, D + 5), 1e3, dtype=torch.float32, device="cuda")
    d_x[:, :D] = torch.from_numpy(X).cuda()
    d_ids, d_w = torch.from_numpy(ali).cuda(), torch.from_numpy(w).cuda()
    torch.cuda.synchronize()
    stream = torch.cuda.Stream()
    dev = host.FmllrDiagGmmAccsGpu(am, n_spk=n_spk)
    dev.accumulate_dev(d_x, T, D + 5, d_ids, fo, u2s, d_w, stream=stream)
    stream.synchronize()
    check(dev, "GPU device form")
    for s in truth:  # the same statistics as the host form (FP64 atomics: equal up to the order of the additions)
        assert_fmllr_close(dev.stats(s), (*acc.stats(s), *truth[s][3:]), what="device form vs host form, speaker %d" % s)
    if not po.have_ref():
        return
    ref = po.load("ref")
    for s, rows in enumerate(spk_rows):
        if s not in truth:
            continue
        b, K, G = acc.stats(s)
        rc, rb, rK, rG, _ = ref.fmllr_acc(m, X[rows], ali[rows], w[rows])
        assert rc == 0
        r1, x_gpu, i1, c1 = ref.fmllr_update(b, K, G)
        r2, x_ref, i2, c2 = ref.fmllr_update(rb, rK, rG)
        assert r1 == 0 and r2 == 0 and abs(c1 - c2) <= 1e-3 * c2
        assert np.abs(x_gpu - x_ref).max() <= 1e-3
        if c2 > 500:
            assert np.abs(x_ref - np.eye(D, D + 1)).max() > 1e-3 and abs(i1 - i2) <= 1e-3 * max(abs(i2), 1.0)


def test_fmllr_stats_errors(orc):
    m = _model(orc, 5, 20, 39, 71)
    am = host.AmDiagGmmGpu.from_model(m)
    acc = host.FmllrDiagGmmAccsGpu(am, n_spk=2)
    X = synth.make_feats(m, 50, 72)
    ali = synth.make_alignment(5, 50, 73)
    bad = ali.copy()
    bad[7] = 99  # invalid pdf id: reported, the frame adds nothing
    with pytest.raises(capi.VbgpuError) as e:
        acc.AccumulateForUtterances(X, bad)
    assert e.value.code == capi.ERR_NUMERIC
    with pytest.raises(capi.VbgpuError):  # speaker outside [0, n_spk)
        acc.AccumulateForUtterances(X, ali, frame_offsets=[0, 50], utt2spk=[2])
    with pytest.raises(capi.VbgpuError):  # frame_offsets beyond T
        acc.AccumulateForUtterances(X, ali, frame_offsets=[0, 60], utt2spk=[0])
    big = synth.make_model(3, 6, 41, 74)
    with pytest.raises(capi.VbgpuError):  # D > 40
        host.FmllrDiagGmmAccsGpu(host.AmDiagGmmGpu.from_model(big))


def test_fmllr_stats_full_size_properties():
    """BASELINE cfg 3 model (P=4000, N=40000, D=39), 200 000 frames, 16 speakers: size-independent properties.
    beta_s = frames of speaker s (posteriors sum to one); the statistics of two calls over disjoint speaker sets equal
    those of one call over everything; G[i](D, D) = sum_t b_t[i] is a sum of positive inverse variances."""
    D, P, n_spk = 39, 4000, 16
    m = synth.make_model(P, 40000, D, 11)
    rng = np.random.default_rng(5)
    lens = rng.integers(900, 1600, size=160)
    fo = np.zeros(len(lens) + 1, np.int64)
    fo[1:] = np.cumsum(lens)
    T = int(fo[-1])
    u2s = np.repeat(np.arange(n_spk, dtype=np.int32), len(lens) // n_spk)
    X = synth.make_feats(m, T, 12)
    ali = synth.make_alignment(P, T, 13)
    am = host.AmDiagGmmGpu.from_model(m)
    one = host.FmllrDiagGmmAccsGpu(am, n_spk=n_spk)
    one.AccumulateForUtterances(X, ali, frame_offsets=fo, utt2spk=u2s)
    two = host.FmllrDiagGmmAccsGpu(am, n_spk=n_spk)
    half = len(lens) // 2  # a speaker boundary: 80 utterances = 8 speakers
    two.AccumulateForUtterances(X[:fo[half]], ali[:fo[half]], frame_offsets=fo[:half + 1], utt2spk=u2s[:half])
    two.AccumulateForUtterances(X[fo[half]:], ali[fo[half]:], frame_offsets=fo[half:] - fo[half], utt2spk=u2s[half:])
    jj, kk = np.tril_indices(D + 1)
    last = np.flatnonzero((jj == D) & (kk == D))[0]
    for s in range(n_spk):
        b1, K1, G1 = one.stats(s)
        b2, K2, G2 = two.stats(s)
        frames = int(lens[u2s == s].sum())
        assert abs(b1 - frames) <= 1e-5 * frames
        assert abs(b1 - b2) <= 1e-9 * b1
        assert np.abs(K1 - K2).max() <= 1e-9 * np.abs(K1).max() and np.abs(G1 - G2).max() <= 1e-9 * np.abs(G1).max()
        assert (G1[:, last] > 0).all()  # sum_t b_t[i] of positive inverse variances
        assert np.isfinite(G1).all() and np.isfinite(K1).all()


# ------------------------------------------------------------------------------------------ MLLT statistics (gmm-acc-mllt)
@pytest.mark.parametrize("D,weighted,T,model", [
    pytest.param(40, False, 900, (20, 150, 3), id="40-False-900"),
    pytest.param(13, True, 700, (20, 150, 3), id="13-True-700"),
    pytest.param(39, True, 1, (20, 150, 3), id="39-True-1"),
    # pdfs of up to 123 Gaussians: several 32-Gaussian passes of mllt_rows_kernel, and more than 64 per pdf
    pytest.param(39, True, 900, (12, 700, 5), id="39-True-900-large-pdfs"),
    pytest.param(40, True, 900, (12, 700, 5), id="40-True-900-large-pdfs"),
])
def test_mllt_stats(orc, D, weighted, T, model):
    """MlltAccs on the device (the fMLLR G contraction over one pseudo-frame per (frame, Gaussian)) against the float64
    restatement and the oracle; where the reference is built, also through its own MlltAccs::Update."""
    from oracle import pyoracle as po
    from tests.common import mllt_truth
    P, N, seed = model
    m = _model(orc, P, N, D, seed)
    if model[0] == 12:
        sizes = np.diff(m.pdf_offsets)
        assert (sizes > 64).any() and ((sizes > 32) & (sizes <= 64)).any() and (sizes <= 32).any()
    X = synth.make_feats(m, T, 4)
    ali = synth.make_alignment(P, T, 5)
    w = np.random.default_rng(1).uniform(0.2, 1.0, T).astype(np.float32) if weighted else None
    acc = host.MlltAccsGpu(host.AmDiagGmmGpu.from_model(m))
    tl = acc.AccumulateForUtterance(X, ali, w)
    rc, ob, oG, ol = orc.mllt_acc(m, X, ali, w)
    assert rc == 0 and abs(tl - ol) <= 1e-4 * abs(ol)
    tb, tG, SG = mllt_truth(m, X, ali, w)
    assert abs(acc.beta - tb) <= 1e-4 * max(tb, 1.0)
    assert (np.abs(acc.G - tG) / np.maximum(SG, 1e-30)).max() <= 1e-4
    if T >= 700 and po.have_ref():
        ref = po.load("ref")
        r1, M1, i1, c1 = ref.mllt_update(acc.beta, acc.G)
        r2, M2, i2, c2 = ref.mllt_update(ob, oG)
        assert r1 == 0 and r2 == 0 and np.abs(M1 - M2).max() <= 1e-3 and abs(i1 - i2) <= 1e-3 * max(abs(i2), 1.0)
    acc.AccumulateForUtterance(X, ali, w)  # a second call adds
    assert abs(acc.beta - 2 * tb) <= 2e-4 * max(tb, 1.0)


def _mllt_truth_by_pdf(model, X, ali, chunk=256):
    """tests.common.mllt_truth (unweighted) with the frames of each pdf taken a chunk at a time: the same sums, fast
    enough for tens of thousands of frames."""
    X = np.asarray(X, np.float64)
    D = X.shape[1]
    gc, miv, iv = (np.asarray(v, np.float64) for v in (model.gconsts, model.miv, model.iv))
    rr, cc = np.tril_indices(D)
    G, SG = np.zeros((D, len(rr))), np.zeros((D, len(rr)))
    beta = 0.0
    for p in np.unique(ali):
        g0, g1 = model.pdf_offsets[p], model.pdf_offsets[p + 1]
        idx = np.flatnonzero(ali == p)
        for c0 in range(0, len(idx), chunk):
            x = X[idx[c0:c0 + chunk]]                                               # [n, D]
            ll = gc[g0:g1] + x @ miv[g0:g1].T - 0.5 * ((x * x) @ iv[g0:g1].T)       # [n, M]
            post = np.exp(ll - ll.max(axis=1, keepdims=True))
            post /= post.sum(axis=1, keepdims=True)
            off = (miv[g0:g1] / iv[g0:g1])[None] - x[:, None, :]                    # [n, M, D]
            z = (off[:, :, rr] * off[:, :, cc]).reshape(-1, len(rr))               # [n M, pairs]
            a = (iv[g0:g1][None] * post[:, :, None]).reshape(-1, D)               # [n M, D]
            G += a.T @ z
            SG += a.T @ np.abs(z)
            beta += post.sum()
    return beta, G, SG


def test_mllt_stats_many_slabs_and_bad_ids(orc):
    from tests.common import mllt_truth
    m = _model(orc, 30, 900, 39, 8)  # ~30 Gaussians per pdf: 60 000 frames make several row slabs
    T = 60000
    X = synth.make_feats(m, T, 9)
    ali = synth.make_alignment(30, T, 10)
    assert np.diff(m.pdf_offsets)[ali].sum() > 1500000  # (frame, Gaussian) rows beyond one slab (kMaxRows)
    am = host.AmDiagGmmGpu.from_model(m)
    whole = host.MlltAccsGpu(am)
    whole.AccumulateForUtterance(X, ali)
    # the grouped restatement is the per-frame one, and the device result of many slabs matches it
    b1, G1, _ = _mllt_truth_by_pdf(m, X[:300], ali[:300])
    b2, G2, S2 = mllt_truth(m, X[:300], ali[:300])
    assert abs(b1 - b2) <= 1e-12 * b2 and (np.abs(G1 - G2) / np.maximum(S2, 1e-30)).max() <= 1e-12
    tb, tG, SG = _mllt_truth_by_pdf(m, X, ali)
    assert abs(whole.beta - tb) <= 1e-4 * tb
    assert (np.abs(whole.G - tG) / np.maximum(SG, 1e-30)).max() <= 1e-4
    parts = host.MlltAccsGpu(am)
    for a, b in ((0, 7), (7, 25000), (25000, T)):
        parts.AccumulateForUtterance(X[a:b], ali[a:b])
    assert abs(whole.beta - T) <= 1e-5 * T and abs(whole.beta - parts.beta) <= 1e-9 * T
    assert np.abs(whole.G - parts.G).max() <= 1e-6 * np.abs(whole.G).max()
    bad = ali[:100].copy()
    bad[3] = -1
    with pytest.raises(capi.VbgpuError) as e:
        host.MlltAccsGpu(am).AccumulateForUtterance(X[:100], bad)
    assert e.value.code == capi.ERR_NUMERIC


def test_component_posteriors(orc):
    """gmm-post-to-gpost: Gaussian-level posteriors of every frame's aligned pdf, pdfs of 1 .. 100 Gaussians."""
    m = _model(orc, 40, 900, 39, 61)
    T = 500
    X = synth.make_feats(m, T, 62)
    ali = synth.make_alignment(40, T, 63)
    w = np.random.default_rng(64).uniform(0.2, 1.0, T).astype(np.float32)
    am = host.AmDiagGmmGpu.from_model(m)
    for weights in (None, w):
        post, offs, ll = am.ComponentPosteriors(X, ali, m.pdf_offsets, weights)
        rc, po_, oo, lo = orc.component_posteriors(m, X, ali, weights)
        assert rc == 0 and np.array_equal(offs, oo)
        assert np.abs(post - po_).max() <= 1e-5 and np.abs(ll - lo).max() <= 1e-3
        sums = np.add.reduceat(post, offs[:-1])
        assert np.abs(sums - (1.0 if weights is None else weights)).max() <= 1e-5
