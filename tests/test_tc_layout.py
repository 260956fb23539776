"""The tensor-core scorer's model layout, checked WITHOUT a GPU: the host code that sorts the pdfs into groups / panels and
writes the fp16 hi/lo B image (voicebridge_b200/csrc/score_tc.cu: build_layout) is decoded here and pushed through a
numpy restatement of the kernel's arithmetic (3 fp16 products, slot-interleaved log-sum-exp per group entry, merge list, column map), for the CTA-pair image (each CTA
holds half of a panel's columns) and the single-CTA image; the
result must match the oracle's DiagGmm::LogLikelihoods + LogSumExp (gmm/diag-gmm.cc:528-562)."""
import ctypes as C

import numpy as np
import pytest

from voicebridge_b200 import capi, synth


def tc_layout(model, pair=True):
    lib = capi.lib()
    P, D = model.num_pdfs, model.dim
    po = np.ascontiguousarray(model.pdf_offsets, np.int32)
    gc = np.ascontiguousarray(model.gconsts, np.float32)
    miv = np.ascontiguousarray(model.miv, np.float32)
    iv = np.ascontiguousarray(model.iv, np.float32)
    info = np.zeros(8, np.int32)
    args = (P, D, po.ctypes.data, gc.ctypes.data, miv.ctypes.data, iv.ctypes.data, D, int(pair))
    rc = lib.vbgpu_debug_tc_layout(*args, info.ctypes.data, None, 0, None, 0, None, 0, None, None, 0, None, None, None, None)
    if rc < 0:
        return None, lib.vbgpu_last_error().decode()
    KS, n_panels, n_cols, n_merge, img16, n_groups = [int(v) for v in info[:6]]
    image = np.zeros(img16 * 16, np.uint8)
    hdr = np.zeros((n_panels, 4), np.int32)
    grp = np.zeros((n_groups, 2), np.int32)
    col = np.zeros(P, np.int32)
    merge = np.zeros((max(n_merge, 1), 2), np.int32)
    centre, s1, s2 = (np.zeros(D, np.float32) for _ in range(3))
    capi.check(lib.vbgpu_debug_tc_layout(*args, info.ctypes.data, image.ctypes.data, image.size, hdr.ctypes.data, hdr.size,
                                         grp.ctypes.data, grp.size, col.ctypes.data, merge.ctypes.data, merge.size,
                                         centre.ctypes.data, s1.ctypes.data, s2.ctypes.data, None))
    return dict(KS=KS, n_cols=n_cols, image=image, hdr=hdr, grp=grp, col_of_pdf=col, merge=merge[:n_merge], centre=centre,
                s1=s1, s2=s2, pair=bool(pair)), ""


def decode_block(image, off, nb, KS):
    """[K, nb] hi and lo halves of one block: chunk kc of 8 K-values, column group n/8, 8 columns x 16 bytes."""
    half = np.frombuffer(image[off:off + 4 * KS * 16 * nb].tobytes(), np.float16).reshape(4 * KS, nb // 8, 8, 8)
    # [chunk, col group, col in group, k in chunk] -> [chunk, k, col group, col]
    m = half.transpose(0, 3, 1, 2).reshape(4 * KS * 8, nb)
    return m[:2 * KS * 8].astype(np.float64), m[2 * KS * 8:].astype(np.float64)


def decode_panel(image, off, N, KS, pair):
    """What the tensor cores see as the panel's B operand: in a CTA pair each CTA holds N/2 columns."""
    if not pair:
        return decode_block(image, off, N, KS)
    h0, l0 = decode_block(image, off, N // 2, KS)
    h1, l1 = decode_block(image, off + 4 * KS * 16 * (N // 2), N // 2, KS)
    return np.concatenate([h0, h1], axis=1), np.concatenate([l0, l1], axis=1)


def emulate(lay, feats, D):
    """The kernel's arithmetic in numpy: returns the score matrix in device column order."""
    KS = lay["KS"]
    K = 16 * KS
    T = feats.shape[0]
    A = np.zeros((T, K), np.float32)
    xc = feats.astype(np.float32) - lay["centre"]
    A[:, 0:2 * D:2] = xc * lay["s1"]
    A[:, 1:2 * D:2] = (xc * xc) * lay["s2"]
    A[:, 2 * D] = 1.0
    A[:, 2 * D + 1] = 1.0
    assert np.abs(A).max() <= 65504
    a_hi = A.astype(np.float16)
    a_lo = (A - a_hi.astype(np.float32)).astype(np.float16)
    a_hi, a_lo = a_hi.astype(np.float64), a_lo.astype(np.float64)
    out = np.full((T, lay["n_cols"]), np.nan, np.float32)
    nmax = 256 if lay["pair"] else 160
    for off16, y, g0, _ in lay["hdr"]:
        N, ng = y & 0xffff, (y >> 16) & 0xffff
        assert N % 16 == 0 and 16 <= N <= nmax and ng >= 1
        b_hi, b_lo = decode_panel(lay["image"], int(off16) * 16, N, KS, lay["pair"])
        Y = (a_lo @ b_hi + a_hi @ b_lo + a_hi @ b_hi).astype(np.float32)   # log2 units
        used = 0
        for gx, out_col in lay["grp"][g0:g0 + ng]:
            S, W, col0 = gx & 0xff, (gx >> 8) & 0xff, (gx >> 16) & 0xffff
            assert W in (1, 2, 4) and 1 <= S <= 10 and col0 == used
            used += 16 * S
            grp = Y[:, col0:col0 + 16 * S].reshape(T, S, 16 // W, W).transpose(0, 2, 1, 3).reshape(T, 16 // W, S * W)
            mx = grp.max(axis=2, keepdims=True)
            lse = (mx[:, :, 0] + np.log2(np.exp2(grp - mx).sum(axis=2))) * np.float32(0.6931471805599453)
            assert out_col % (16 // W if W < 4 else 4) == 0
            out[:, out_col:out_col + 16 // W] = lse
        assert used == N
    i = 0
    mg = lay["merge"]
    while i < len(mg):
        main = mg[i, 0]
        cols = [main]
        while i < len(mg) and mg[i, 0] == main:
            cols.append(mg[i, 1])
            i += 1
        v = out[:, cols].astype(np.float64)
        m = v.max(axis=1)
        out[:, main] = (m + np.log(np.exp(v - m[:, None]).sum(axis=1))).astype(np.float32)
    return out


def sized_model(sizes, D, seed):
    """A model with the given numbers of Gaussians per pdf, matched to features drawn near it."""
    rng = np.random.default_rng(seed)
    P, N = len(sizes), int(np.sum(sizes))
    m = synth.make_model(P, max(N, P + 1), D, seed)
    offs = np.zeros(P + 1, np.int32)
    offs[1:] = np.cumsum(sizes)
    scale = (1.0 / (1.0 + 0.1 * np.arange(D))).astype(np.float32)
    centers = rng.standard_normal((P, D)).astype(np.float32)
    means = ((np.repeat(centers, sizes, axis=0) + 0.5 * rng.standard_normal((N, D)).astype(np.float32)) * scale).astype(np.float32)
    var = (np.exp(0.5 * rng.standard_normal((N, D))) * 0.6 + 0.01).astype(np.float32) * scale * scale
    iv = (1.0 / var).astype(np.float32)
    w = np.exp(rng.standard_normal(N)).astype(np.float32)
    for p in range(P):
        s = slice(offs[p], offs[p + 1])
        w[s] /= w[s].sum()
    miv = (means * iv).astype(np.float32)
    return synth.GmmModel(offs, w, means, iv, miv, synth.compute_gconsts(w, miv, iv))


CASES = [
    ("power-law sizes, D=39", lambda: synth.make_model(300, 3000, 39, 1)),
    ("D=40 (K=96)", lambda: synth.make_model(120, 700, 40, 2)),
    ("D=13", lambda: synth.make_model(40, 200, 13, 3)),
    ("one Gaussian per pdf", lambda: synth.make_model(50, 50, 39, 4)),
    ("large pdfs: 41, 100, 600 Gaussians", lambda: sized_model([3, 41, 100, 7, 600, 12, 20, 21, 40, 10, 11], 39, 5)),
    ("single pdf", lambda: sized_model([9], 20, 6)),
    ("D=24 (KS=4)", lambda: sized_model([1, 1, 2, 5, 9, 10, 11, 14, 20, 21, 33, 40, 57, 3, 1, 7], 24, 7)),
    ("D=31 (KS=4)", lambda: synth.make_model(90, 600, 31, 8)),
    ("D=47 (KS=6)", lambda: sized_model([1, 4, 12, 25, 41, 2, 1, 18, 39, 6, 1, 1, 30], 47, 9)),
]


@pytest.mark.parametrize("pair", [True, False], ids=["pair", "single"])
@pytest.mark.parametrize("name,make", CASES, ids=[c[0] for c in CASES])
def test_layout_reproduces_oracle_loglikes(orc, name, make, pair):
    model = make()
    feats = synth.make_feats(model, 96, 11)
    lay, why = tc_layout(model, pair)
    assert lay is not None, why
    assert lay["KS"] == (2 * model.dim + 2 + 15) // 16   # the K-step instantiation the device would launch
    P = model.num_pdfs
    col = lay["col_of_pdf"]
    assert len(set(col.tolist())) == P and col.min() >= 0 and col.max() < lay["n_cols"]
    got = emulate(lay, feats, model.dim)[:, col]
    rc, want = orc.gmm_loglikes(model, feats)
    assert rc == 0
    err = np.abs(got - want).max()
    print("%s: max |dLL| = %.2e at max |LL| = %.0f" % (name, err, np.abs(want).max()))
    assert err < 1e-3


def test_zero_weight_gaussians_keep_the_dummy_score(orc):
    model = synth.make_model(30, 200, 39, 8)
    gc = model.gconsts.copy()
    gc[model.pdf_offsets[3]] = -np.inf     # one Gaussian of pdf 3 (the pdf keeps others)
    if model.pdf_offsets[4] - model.pdf_offsets[3] < 2:
        pytest.skip("pdf 3 has a single Gaussian in this draw")
    model = synth.GmmModel(model.pdf_offsets, model.weights, model.means, model.iv, model.miv, gc)
    feats = synth.make_feats(model, 64, 12)
    lay, why = tc_layout(model)
    assert lay is not None, why
    got = emulate(lay, feats, model.dim)[:, lay["col_of_pdf"]]
    rc, want = orc.gmm_loglikes(model, feats)
    assert np.abs(got - want).max() < 1e-3


def test_models_off_the_plan_are_reported():
    model = synth.make_model(10, 40, 48, 9)       # D = 48 > 47
    lay, why = tc_layout(model)
    assert lay is None and "dimension" in why
    model = synth.make_model(10, 40, 39, 9)
    gc = model.gconsts.copy()
    gc[model.pdf_offsets[2]:model.pdf_offsets[3]] = -np.inf   # a pdf with no finite gconst
    lay, why = tc_layout(synth.GmmModel(model.pdf_offsets, model.weights, model.means, model.iv, model.miv, gc))
    assert lay is None and "finite gconst" in why


@pytest.mark.parametrize("pair", [True, False], ids=["pair", "single"])
def test_idle_slots_score_zero_and_real_pdfs_stay_above_the_sunk_level(pair):
    """The epilogue hands a frame to the FP32 kernel when any result falls below -27000 nats (within reach of the padding
    columns' dummy score, -40000 ln 2).  That test runs over every column of a group, so columns without a pdf must not look
    sunk: they score exactly 0, and in-model frames stay far above the level."""
    model = sized_model([3, 41, 100, 7, 600, 12, 20, 21, 40, 10, 11], 39, 5)
    lay, why = tc_layout(model, pair)
    assert lay is not None, why
    out = emulate(lay, synth.make_feats(model, 64, 3), model.dim)
    mg = lay["merge"]
    used = set(lay["col_of_pdf"].tolist()) | set(mg[:, 1].tolist())
    written = np.isfinite(out[0])
    idle = [c for c in range(lay["n_cols"]) if written[c] and c not in used]
    assert idle, "this model leaves slots without a pdf"
    assert np.all(out[:, idle] == 0.0)
    assert out[:, sorted(used)].min() > -27000.0
