"""The shapes the kernels are compiled for, beyond the 13-coefficient MFCC recipe (D = 39 / 40) that most parity tests run:
every K-step instantiation of the tensor-core scorer in both CTA shapes, every SIMT width, output and feature layouts the
library otherwise never sees, the feature pipeline and EM statistics at wider inputs, and Kaldi's MFCC + pitch system
(16 pasted columns, 48 after deltas) end to end.  Everything is checked against the CPU oracle at BASELINE.json's
tolerances (tests/common.py)."""
import numpy as np
import pytest

from tests.common import assert_acc_close, assert_feats_close, assert_ll_close, assert_stats_close
from tests.gpu_common import oracle_feats, oracle_mfcc_batch, oracle_stats
from tests.test_gpu_parity import _custom_model, _pinned_model, gopts
from tests.test_tc_layout import tc_layout
from voicebridge_b200 import capi, host, synth

pytestmark = pytest.mark.gpu

NAN = float("nan")


@pytest.fixture
def tc_shape(monkeypatch):
    """Selects the CTA shape of the tensor-core handles created afterwards in the test (score_tc_prepare reads
    VBGPU_TC_SINGLE when the model is created); the variable is restored when the test ends."""
    def select(shape):
        if shape == "single":
            monkeypatch.setenv("VBGPU_TC_SINGLE", "1")
        else:
            monkeypatch.delenv("VBGPU_TC_SINGLE", raising=False)
    return select


def _mixed_sizes(seed):
    """150 pdfs: single Gaussians, pdfs that fill W = 1, 2 and 4 groups (<= 10, 11..20, 21..40 Gaussians) and one of 57
    that is cut into virtual pdfs and merged."""
    rng = np.random.default_rng(seed)
    s = [1] * 50 + list(rng.integers(2, 11, 40)) + list(rng.integers(11, 21, 30)) + list(rng.integers(21, 41, 29)) + [57]
    rng.shuffle(s)
    return [int(v) for v in s]


def _cols_dev(am, X):
    """score_cols_dev into a NaN-prefilled device buffer, mapped back to pdf order: a row or column the kernel never
    wrote stays NaN."""
    import torch
    T, nc = X.shape[0], am.NumCols()
    d_x = torch.from_numpy(np.ascontiguousarray(X, np.float32)).cuda()
    d_ll = torch.full((T, nc), NAN, dtype=torch.float32, device="cuda")
    am.score_cols_dev(d_x, T, X.shape[1], d_ll, nc)
    torch.cuda.synchronize()
    return d_ll.cpu().numpy()[:, am.col_of_pdf()]


def _fp32_bound_ok(got, want):
    """The bound of test_scoring_tensor_core_vs_fp32_kernel_random_layouts: 1e-3, or 16 ulp of the frame's largest |ll|."""
    err, mag = np.abs(got - want), np.abs(want)
    frame_mag = mag.max(axis=1)
    tol = np.maximum(1e-3, 16.0 * np.spacing(frame_mag.astype(np.float32)).astype(np.float64))
    return (err.max(axis=1) / tol).max()


# ========================================================================================= tensor-core scorer: every KS
@pytest.mark.parametrize("shape", ["pair", "single"])
@pytest.mark.parametrize("D", [15, 16, 23, 24, 31, 32, 39, 40, 47])
def test_tc_scorer_every_k_step_vs_oracle(orc, tc_shape, D, shape):
    """Both sides of every K-step boundary (KS = ceil((2D + 2) / 16): 2 .. 6) in the CTA-pair and the single-CTA shape, for
    ragged frame counts, through the host call (scratch + gather) and natively into a NaN-prefilled device buffer.  In the
    single shape a CTA owns two 128-frame tiles of a unit: rows 128..255 must be written too."""
    tc_shape(shape)
    m = _pinned_model(orc, _custom_model(_mixed_sizes(D), D, 100 + D))
    pair_lay, single_lay = tc_layout(m, True)[0], tc_layout(m, False)[0]
    assert pair_lay["KS"] == single_lay["KS"] == (2 * D + 2 + 15) // 16
    # the two shapes lay the model out differently, so the column map tells which plan the handle is on
    assert not np.array_equal(pair_lay["col_of_pdf"], single_lay["col_of_pdf"])
    am = host.AmDiagGmmGpu.from_model(m)
    assert am.plan_note() == "", am.plan_note()
    assert np.array_equal(am.col_of_pdf(), (pair_lay if shape == "pair" else single_lay)["col_of_pdf"])
    X = synth.make_feats(m, 1003, 200 + D)
    rc, want = orc.gmm_loglikes(m, X)
    assert rc == 0
    for T in (1, 255, 257, 1003):
        got = am.score(X[:T])
        assert_ll_close(got, want[:T], what="D=%d %s T=%d" % (D, shape, T))
        assert np.array_equal(_cols_dev(am, X[:T]), got), "D=%d %s T=%d: native columns differ" % (D, shape, T)


def test_tc_single_shape_tail_split(orc, tc_shape):
    """Single-CTA shape with more than four waves of 256-frame units and a remainder: the last, partial wave is cut into panel
    ranges.  Every frame against the FP32 SIMT kernel of the same handle, the whole-tile start and the cut tail against the
    oracle."""
    import torch
    tc_shape("single")
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    m = _pinned_model(orc, synth.make_model(40, 300, 13, 7))
    lay = tc_layout(m, False)[0]
    assert len(lay["hdr"]) >= 2        # at least two panels: the tail tiles really are cut
    T = 256 * (4 * sms + 30) + 17
    n_mtiles = (T + 255) // 256
    assert n_mtiles >= 4 * sms and n_mtiles % sms and min(len(lay["hdr"]), 16, sms // (n_mtiles % sms)) >= 2
    X = synth.make_feats(m, T, 71)
    am = host.AmDiagGmmGpu.from_model(m)
    assert am.plan_note() == "" and np.array_equal(am.col_of_pdf(), lay["col_of_pdf"])
    am.set_kernel(2)
    got = am.score(X)
    assert np.array_equal(_cols_dev(am, X), got)
    am.set_kernel(1)
    simt = am.score(X)
    assert np.isfinite(simt).all() and got.shape == simt.shape
    worst = _fp32_bound_ok(got, simt)
    assert worst <= 1.0, "%.2f of the bound" % worst
    tail = 256 * (n_mtiles % sms + 2)
    rows = np.r_[0:2048, T - tail:T]
    rc, want = orc.gmm_loglikes(m, X[rows])
    assert rc == 0
    assert_ll_close(got[rows], want, what="whole tiles and the cut tail")


# ============================================================================================== SIMT scorer: every width
@pytest.mark.parametrize("D", [16, 17, 24, 25, 32, 33, 41, 48, 49, 64])
def test_simt_scorer_every_width_vs_oracle(orc, D):
    """Padded widths DP = 16, 24, 32, 40, 48, 64 on both sides of each boundary, with a pdf above 64 Gaussians and one -inf
    gconst (a zero-weight Gaussian) inside a healthy pdf.  Beyond D = 47 the automatic choice is the SIMT kernel and the
    plan note says why."""
    rng = np.random.default_rng(D)
    sizes = [3, 1, 70, 2, 5, 9, 1, 17, 33, 4, 64, 65, 2, 1, 12] + [int(v) for v in rng.integers(1, 12, 55)]
    m = _pinned_model(orc, _custom_model(sizes, D, 300 + D))
    gc = m.gconsts.copy()
    gc[m.pdf_offsets[4] + 2] = -np.inf
    m = synth.GmmModel(m.pdf_offsets, m.weights, m.means, m.iv, m.miv, gc)
    X = synth.make_feats(m, 301, 400 + D)
    rc, want = orc.gmm_loglikes(m, X)
    assert rc == 0 and np.isfinite(want).all()
    am = host.AmDiagGmmGpu.from_model(m)
    kinds = [1]
    if D >= 48:
        assert "dimension" in am.plan_note(), am.plan_note()
        kinds.append(0)
    for k in kinds:
        am.set_kernel(k)
        assert_ll_close(am.score(X), want, what="D=%d kernel %d" % (D, k))


# ========================================================================= layouts of the tensor-core scorer's operands
def test_tc_scorer_unaligned_features_and_outputs(orc, tc_shape):
    """D = 40 on the CTA-pair shape: features at stride 41 and one float into a buffer (scalar A-panel loads), results at
    ll_stride = NumCols() + 1 and one float into a buffer (scalar epilogue stores).  Same bits as the aligned run, oracle
    values, and padding around the results left as it was."""
    import torch
    tc_shape("pair")
    D, T = 40, 300
    m = _pinned_model(orc, _custom_model(_mixed_sizes(D), D, 140))
    am = host.AmDiagGmmGpu.from_model(m)
    assert am.plan_note() == "", am.plan_note()
    col, nc = am.col_of_pdf(), am.NumCols()
    X = synth.make_feats(m, T, 41)
    rc, want = orc.gmm_loglikes(m, X)
    assert rc == 0
    x_aligned = torch.from_numpy(X).cuda()
    x_wide = torch.full((T, D + 1), NAN, dtype=torch.float32, device="cuda")   # stride 41, NaN in the unused column
    x_wide[:, :D] = x_aligned
    x_buf = torch.full((T * D + 4,), NAN, dtype=torch.float32, device="cuda")
    x_off = x_buf[1:1 + T * D]                                                 # 4 bytes past a 16-byte boundary
    x_off.copy_(x_aligned.reshape(-1))

    def run(d_x, stride, out_stride, out_off):
        buf = torch.full((out_off + T * out_stride + 4,), NAN, dtype=torch.float32, device="cuda")
        am.score_cols_dev(d_x, T, stride, buf[out_off:], out_stride)
        torch.cuda.synchronize()
        b = buf.cpu().numpy()
        res = b[out_off:out_off + T * out_stride].reshape(T, out_stride)
        pad = np.concatenate([b[:out_off], res[:, nc:].ravel(), b[out_off + T * out_stride:]])
        assert np.isnan(pad).all(), "padding around the results was written"
        return res[:, col]

    ref = run(x_aligned, D, nc, 0)
    assert_ll_close(ref, want, what="aligned")
    for name, d_x, stride, out_stride, out_off in (("features at stride 41", x_wide, D + 1, nc, 0),
                                                   ("features one float in", x_off, D, nc, 0),
                                                   ("ll_stride NumCols() + 1", x_aligned, D, nc + 1, 0),
                                                   ("results one float in", x_aligned, D, nc, 1)):
        got = run(d_x, stride, out_stride, out_off)
        assert np.array_equal(got, ref), name
        assert_ll_close(got, want, what=name)


def test_tc_scorer_pdf_gather_beyond_shared_memory(orc, tc_shape):
    """26 000 pdfs of 1..3 Gaussians: a row of the device-order matrix no longer fits the staged gather's 100 KiB, so the host
    call takes the per-pdf gather kernel."""
    tc_shape("pair")
    rng = np.random.default_rng(5)
    m = _pinned_model(orc, _custom_model([int(v) for v in rng.integers(1, 4, 26000)], 13, 6))
    am = host.AmDiagGmmGpu.from_model(m)
    assert am.plan_note() == "", am.plan_note()
    assert am.NumCols() * 4 > 100 * 1024
    col = am.col_of_pdf()
    assert not np.array_equal(col, np.arange(m.num_pdfs))   # the gather really permutes
    X = synth.make_feats(m, 200, 61)
    got = am.score(X)
    rc, want = orc.gmm_loglikes(m, X)
    assert rc == 0
    assert_ll_close(got, want)
    assert np.array_equal(_cols_dev(am, X), got)


# ================================================================================== feature pipeline at wider inputs
# 1- and 2-frame utterances, empty ones, utterance and speaker changes inside 64-frame tiles, a speaker that comes back
LENS = [1, 2, 0, 5, 63, 64, 65, 1, 130, 0, 9, 300, 257]
U2S = [0, 0, 1, 1, 1, 2, 2, 0, 3, 3, 3, 1, 2]
N_SPK = 4


def _wide_batch(in_dim, seed):
    rng = np.random.default_rng(seed)
    fo = np.zeros(len(LENS) + 1, np.int64)
    fo[1:] = np.cumsum(LENS)
    mf = (rng.standard_normal((int(fo[-1]), in_dim)) * 3.0 + rng.uniform(-5.0, 5.0, in_dim)).astype(np.float32)
    return mf, fo


@pytest.mark.parametrize("per_utt", [False, True])
@pytest.mark.parametrize("in_dim", [1, 15, 16, 17, 20, 23, 32, 40])
def test_cmvn_stats_wide(orc, in_dim, per_utt):
    """Statistics of D + 1 > 16 columns take several passes of the 16-lane groups; at D = 16 and 32 the last pass holds
    the count alone."""
    mf, fo = _wide_batch(in_dim, in_dim)
    fp = host.FeaturePipeline(in_dim=in_dim)
    u = None if per_utt else U2S
    n_spk = len(LENS) if per_utt else N_SPK
    got = fp.cmvn_stats(mf, fo, u, n_spk)
    want = oracle_stats(orc, mf, fo, u, n_spk)
    assert np.array_equal(got[:, 0, in_dim], want[:, 0, in_dim])  # counts exact
    assert_stats_close(got, want, 1e-12)


FEAT_WIDE = [
    (16, dict(), None, 48),
    (16, dict(mode=1, splice_left=3, splice_right=3), (40, 112), 40),
    (20, dict(), None, 60),
    (23, dict(), None, 69),
    (23, dict(delta_order=1), None, 46),
    (40, dict(mode=1, splice_left=4, splice_right=4), (40, 361), 40),   # > 48 KB of dynamic shared memory
]


@pytest.mark.parametrize("fmllr_cols", [0, 1, 2], ids=["none", "affine", "linear"])
@pytest.mark.parametrize("in_dim,kw,lda_shape,od", FEAT_WIDE,
                         ids=["%d-%s" % (c[0], ",".join("%s=%s" % kv for kv in c[1].items()) or "deltas") for c in FEAT_WIDE])
def test_feature_pipeline_wide(orc, in_dim, kw, lda_shape, od, fmllr_cols):
    import torch
    mf, fo = _wide_batch(in_dim, 50 + in_dim)
    fopts = capi.default_feat_opts(**kw)
    lda = synth.make_lda(*lda_shape, in_dim) if lda_shape else None
    fp = host.FeaturePipeline(fopts, in_dim, lda)
    assert fp.out_dim() == od
    fm = None
    if fmllr_cols:
        fm = synth.make_fmllr(N_SPK, od, 8)
        if fmllr_cols == 2:
            fm = np.ascontiguousarray(fm[:, :, :od])
    stats = oracle_stats(orc, mf, fo, U2S, N_SPK)
    got = fp.run(mf, fo, U2S, N_SPK, stats, fm)
    want = oracle_feats(orc, mf, fo, U2S, stats, fopts, lda, fm)
    assert_feats_close(got, want, what="in_dim %d %s" % (in_dim, kw))
    if in_dim == 16:  # the device-resident form gives the same bits
        T, ost = got.shape[0], host.kaldi_stride(od)
        d_out = torch.full((T, ost), NAN, dtype=torch.float32, device="cuda")
        d_in = torch.from_numpy(mf).cuda()
        d_fm = torch.from_numpy(fm).cuda() if fm is not None else None
        fp.run_dev(d_in, in_dim, fo, d_out, ost, U2S, N_SPK, stats, d_fm, fm.shape[-1] if fm is not None else 0)
        torch.cuda.synchronize()
        assert np.array_equal(d_out[:, :od].cpu().numpy(), got)


def test_feature_pipeline_refuses_beyond_shared_memory(orc):
    """in_dim 128 spliced 4/4 with a 40 x 1153 transform needs more than 200 KB of shared memory: both forms refuse with
    ERR_INVALID and leave the output as it was."""
    import torch
    fopts = capi.default_feat_opts(mode=1, splice_left=4, splice_right=4)
    fp = host.FeaturePipeline(fopts, 128, synth.make_lda(40, 1153, 3))
    mf = np.random.default_rng(1).standard_normal((75, 128)).astype(np.float32)
    fo = np.array([0, 70, 75], np.int64)
    st = oracle_stats(orc, mf, fo, None, 2)
    out = np.full((75, 40), 7.0, np.float32)
    lib = capi.lib()
    rc = lib.vbgpu_feat_run(fp.h, mf.ctypes.data, 128, fo.ctypes.data, 2, None, 2, st.ctypes.data, None, 0, out.ctypes.data, 40)
    assert rc == capi.ERR_INVALID and "shared memory" in lib.vbgpu_last_error().decode()
    assert (out == 7.0).all()
    d_in = torch.from_numpy(mf).cuda()
    d_out = torch.full((75, 40), 7.0, dtype=torch.float32, device="cuda")
    with pytest.raises(capi.VbgpuError, match="shared memory") as e:
        fp.run_dev(d_in, 128, fo, d_out, 40, None, 2, st)
    assert e.value.code == capi.ERR_INVALID
    torch.cuda.synchronize()
    assert (d_out == 7.0).all().item()


# ================================================================================= EM statistics at D = 48 and D = 64
@pytest.mark.parametrize("mode", ["plain", "weighted", "twofeats"])
@pytest.mark.parametrize("D", [48, 64])
def test_accumulate_wide_vs_oracle(orc, D, mode):
    """test_accumulate_vs_oracle at D = 48 and 64, on pdfs of at most and of more than 64 Gaussians (bucketed kernel and
    acc_kernel in one call), through the host call and through accumulate_dev at a feature stride of D + 1."""
    import torch
    sizes = [1, 3, 64, 65, 7, 12, 100, 2, 30, 5, 1, 9]
    P, T = len(sizes), 400
    m = _pinned_model(orc, _custom_model(sizes, D, 400 + D))
    X = synth.make_feats(m, T, D + 10)
    rng = np.random.default_rng(D)
    segs = np.tile(np.arange(P, dtype=np.int32), T // (7 * P) + 1)
    rng.shuffle(segs)
    ali = np.repeat(segs, 7)[:T]
    assert set(ali.tolist()) == set(range(P))   # every pdf is aligned, those above 64 Gaussians included
    w = rng.uniform(0.1, 1.0, T).astype(np.float32) if mode != "plain" else None
    X2 = synth.make_feats(m, T, D + 20) if mode == "twofeats" else None
    am = host.AmDiagGmmGpu.from_model(m)
    acc = host.AccumAmDiagGmmGpu(am)
    tl = acc.AccumulateForUtterance(X, ali, w, X2)
    occ, mean, var, tot_like, tot_frames = acc.download()
    rc, o2, m2, v2, tl2, tf2 = orc.acc_ali(m, X, ali, w, X2)
    assert rc == 0
    assert_acc_close((occ, mean, var), (o2, m2, v2), what="D=%d %s" % (D, mode))
    assert abs(tot_like - tl2) <= 1e-5 * abs(tl2) and abs(tl - tl2) <= 1e-5 * abs(tl2)
    assert abs(tot_frames - tf2) <= 1e-6 * tf2

    def odd_stride(A):  # rows at stride D + 1 (not a multiple of 4), NaN in the column that is not a feature
        d = torch.full((T, D + 1), NAN, dtype=torch.float32, device="cuda")
        d[:, :D] = torch.from_numpy(A).cuda()
        return d
    d_x, d_ali = odd_stride(X), torch.from_numpy(ali).cuda()
    d_w = torch.from_numpy(w).cuda() if w is not None else None
    d_x2 = odd_stride(X2) if X2 is not None else None
    acc.SetZero()
    acc.accumulate_dev(d_x, T, D + 1, d_ali, d_w, d_x2)
    torch.cuda.synchronize()
    occ, mean, var, tot_like, tot_frames = acc.download()
    assert_acc_close((occ, mean, var), (o2, m2, v2), what="D=%d %s, stride %d" % (D, mode, D + 1))
    assert abs(tot_like - tl2) <= 1e-5 * abs(tl2) and abs(tot_frames - tf2) <= 1e-6 * tf2


# ================================================================================ MFCC + pitch, and the limits at D = 48
def test_mfcc_pitch_system_end_to_end(orc):
    """make_mfcc_pitch (13 + 3 pasted columns) -> CMVN + deltas (48) -> a model at D = 48 (SIMT) -> loglikes and EM
    statistics, each step against the oracle fed the same device features."""
    mo = gopts()
    pp = capi.default_process_pitch_opts(delta_pitch_noise_stddev=0.0)
    lens = [16000 * 2, 5000, 16000, 12000, 7000, 20000]
    u2s = np.array([0, 0, 1, 1, 2, 2], np.int32)
    so = np.zeros(len(lens) + 1, np.int64)
    so[1:] = np.cumsum(lens)
    pcm = np.concatenate([synth.make_pitch_wave(n, 60 + i) for i, n in enumerate(lens)])
    pasted = host.make_mfcc_pitch(host.Mfcc(mo), host.Pitch(), pcm, so, pp)
    assert all(x is not None and x.shape[1] == 16 for x in pasted)
    fo = np.zeros(len(lens) + 1, np.int64)
    fo[1:] = np.cumsum([len(x) for x in pasted])
    mf = np.concatenate(pasted)
    fopts = capi.default_feat_opts()
    fp = host.FeaturePipeline(fopts, in_dim=16)
    st = oracle_stats(orc, mf, fo, u2s, 3)
    got_st = fp.cmvn_stats(mf, fo, u2s, 3)
    assert np.array_equal(got_st[:, 0, 16], st[:, 0, 16])
    assert_stats_close(got_st, st, 1e-12)
    feats = fp.run(mf, fo, u2s, 3, st)
    assert feats.shape == (int(fo[-1]), 48)
    assert_feats_close(feats, oracle_feats(orc, mf, fo, u2s, st, fopts))
    model = _pinned_model(orc, synth.make_model_from_feats(feats, 60, 500, 5))
    am = host.AmDiagGmmGpu.from_model(model)
    assert "dimension" in am.plan_note(), am.plan_note()
    rc, ll = orc.gmm_loglikes(model, feats)
    assert rc == 0
    assert_ll_close(am.score(feats), ll)
    ali = synth.make_alignment(60, feats.shape[0], 9)
    acc = host.AccumAmDiagGmmGpu(am)
    tl = acc.AccumulateForUtterance(feats, ali)
    occ, mean, var, _, tf = acc.download()
    rc, o2, m2, v2, tl2, tf2 = orc.acc_ali(model, feats, ali)
    assert rc == 0
    assert_acc_close((occ, mean, var), (o2, m2, v2))
    assert tf == tf2 and abs(tl - tl2) <= 1e-5 * abs(tl2)


@pytest.mark.parametrize("num_ceps", [16, 20])
def test_pipeline_wide_pcm_to_loglikes(orc, num_ceps):
    """test_pipeline_pcm_to_loglikes with 16 and 20 cepstra (D = 48 / 60 after deltas, scored on SIMT) and a per-speaker
    fMLLR matrix of D rows: features against the oracle chain, loglikes and statistics against the oracle on the
    pipeline's own features."""
    import torch
    o = gopts(num_ceps=num_ceps)
    n_spk, D = 3, 3 * num_ceps
    pcm, so, u2s = synth.make_corpus(n_spk, 3, 0.4, 1.1, 31 + num_ceps)
    fopts = capi.default_feat_opts()
    fm = synth.make_fmllr(n_spk, D, 6)
    mf_want, fo = oracle_mfcc_batch(orc, o, pcm, so)
    st = oracle_stats(orc, mf_want, fo, u2s, n_spk)
    feats_want = oracle_feats(orc, mf_want, fo, u2s, st, fopts, None, fm)
    model = _pinned_model(orc, synth.make_model_from_feats(feats_want, 60, 500, 3))

    mf, fp, am = host.Mfcc(o), host.FeaturePipeline(fopts, num_ceps), host.AmDiagGmmGpu.from_model(model)
    assert "dimension" in am.plan_note(), am.plan_note()
    pipe = host.ScoringPipeline(mf, fp, am)
    ll, feats = pipe.score(pcm, so, u2s, n_spk, fmllr=fm, return_feats=True)
    assert_feats_close(feats, feats_want)
    # the scores are judged on identical features, as the statistics below: at D = 48 / 60 a feature difference of a
    # fifth of the 1e-4 feature budget already moves these loglikes by ~2e-3, beyond the 1e-3 loglike budget
    rc, ll_want = orc.gmm_loglikes(model, feats)
    assert rc == 0
    assert_ll_close(ll, ll_want)
    d_pcm = torch.from_numpy(pcm).cuda()
    d_ll = torch.full((ll.shape[0], am.NumPdfs()), NAN, dtype=torch.float32, device="cuda")
    d_fm = torch.from_numpy(fm).cuda()
    pipe.score_dev(d_pcm, so, u2s, n_spk, d_fm, D + 1, d_ll, am.NumPdfs())
    torch.cuda.synchronize()
    assert np.array_equal(d_ll.cpu().numpy(), ll)
    assert am.bad_count() == 0
    ali = synth.make_alignment(60, ll.shape[0], 8)
    acc = host.AccumAmDiagGmmGpu(am)
    pipe.accumulate_dev(acc, d_pcm, so, u2s, n_spk, d_fm, D + 1, torch.from_numpy(ali).cuda())
    torch.cuda.synchronize()
    occ, mean, var, tl, tf = acc.download()
    rc, o2, m2, v2, tl2, tf2 = orc.acc_ali(model, feats, ali)
    assert rc == 0
    assert_acc_close((occ, mean, var), (o2, m2, v2))
    assert tf == tf2 and abs(tl - tl2) <= 1e-5 * abs(tl2)


def test_transform_statistics_refuse_beyond_d40(orc):
    """fMLLR, MLLT and component-posterior statistics serve D <= 40 (fmllr.cu kMaxD).  At D = 48 each refuses with
    ERR_INVALID and a message naming the limit, writes nothing, and the model handle keeps scoring.  MLLT has no check of
    its own: it fails in the fMLLR handle it creates."""
    m = _pinned_model(orc, synth.make_model(10, 60, 48, 3))
    am = host.AmDiagGmmGpu.from_model(m)
    X = synth.make_feats(m, 50, 4)
    ali = synth.make_alignment(10, 50, 5)
    with pytest.raises(capi.VbgpuError, match=r"\b40\b") as e:
        host.FmllrDiagGmmAccsGpu(am)
    assert e.value.code == capi.ERR_INVALID
    mllt = host.MlltAccsGpu(am)
    with pytest.raises(capi.VbgpuError, match=r"\b40\b") as e:
        mllt.AccumulateForUtterance(X, ali)
    assert e.value.code == capi.ERR_INVALID
    assert mllt.beta == 0.0 and not mllt.G.any()
    with pytest.raises(capi.VbgpuError, match=r"\b40\b") as e:
        am.ComponentPosteriors(X, ali, m.pdf_offsets)
    assert e.value.code == capi.ERR_INVALID
    rc, want = orc.gmm_loglikes(m, X)
    assert rc == 0
    assert_ll_close(am.score(X), want)
