"""Wire / disk formats (SURVEY.md §8f n2): vbgpu_io_* against the reference's own writers and readers (compiled from
/root/reference into oracle/_ref/libvbref.so) — bit-exact in both directions."""
import numpy as np
import pytest

from voicebridge_b200 import capi, kaldi_io as kio, synth


def _feats(rows, cols, seed):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((rows, cols)) * np.linspace(20.0, 0.5, cols) + rng.standard_normal(cols) * 3).astype(np.float32)


@pytest.mark.parametrize("kind,name", [(0, "FM"), (1, "DM"), (2, "CM"), (3, "CM2"), (4, "CM3")])
@pytest.mark.parametrize("rows,cols", [(141, 13), (3, 39), (1000, 40), (1, 1), (5, 7)])
def test_read_matrix_objects_written_by_the_reference(ref, kind, name, rows, cols):
    m = _feats(rows, cols, 100 * kind + rows)
    b = ref.io_write_matrix(m, kind)
    info = kio.object_info(b)
    # the automatic method keeps matrices of 8 rows or fewer in the 2-byte format (compressed-matrix.cc:88-103)
    assert (info.rows, info.cols) == (rows, cols) and info.total_bytes == len(b)
    assert kio.KINDS[info.kind] == name or (kind == 2 and kio.KINDS[info.kind] in ("CM", "CM2"))
    got = kio.read_matrix(b)
    want = ref.io_read_matrix(b)  # Matrix<BaseFloat>::Read, which expands CompressedMatrix objects itself
    assert got.dtype == np.float32 and np.array_equal(got, want)
    if kind == 0:
        assert np.array_equal(got, m) and kio.write_matrix(m) == b  # and our writer emits the same bytes


def test_empty_and_truncated_objects(ref):
    e = ref.io_write_matrix(np.zeros((0, 0), np.float32), 0)
    assert kio.read_matrix(e).shape == (0, 0) and kio.write_matrix(np.zeros((0, 0), np.float32)) == e
    b = ref.io_write_matrix(_feats(20, 13, 1), 2)
    for cut in (1, 3, 10, len(b) - 1):
        with pytest.raises(capi.VbgpuError):
            kio.read_matrix(b[:cut])
    with pytest.raises(capi.VbgpuError):
        kio.read_matrix(b"\0BXX 123")


def test_int32_vectors_both_ways(ref):
    for n in (0, 1, 7, 1234):
        v = np.random.default_rng(n).integers(-5, 50000, n).astype(np.int32)
        b = ref.io_write_int32_vector(v)
        assert np.array_equal(kio.read_int32_vector(b), v)
        mine = kio.write_int32_vector(v)
        assert mine == b and np.array_equal(ref.io_read_int32_vector(mine), v)


def test_archive_of_mixed_objects(ref):
    """A binary archive as copy-feats / ali-to-pdf write it: keys, compressed and plain matrices, alignments."""
    mats = {"spk1_utt1": (_feats(50, 13, 1), 2), "spk1_utt2": (_feats(9, 13, 2), 0), "s2-u1": (_feats(300, 40, 3), 4)}
    ali = np.arange(77, dtype=np.int32)
    ark = b"".join(kio.write_ark_entry(k, ref.io_write_matrix(m, kind)) for k, (m, kind) in mats.items())
    ark += kio.write_ark_entry("ali1", ref.io_write_int32_vector(ali))
    seen = []
    for key, info, off in kio.read_ark(ark):
        seen.append(key)
        if key in mats:
            assert np.array_equal(kio.read_matrix(ark, off), ref.io_read_matrix(ref.io_write_matrix(*mats[key])))
        else:
            assert kio.KINDS[info.kind] == "IV" and np.array_equal(kio.read_int32_vector(ark, off), ali)
    assert seen == list(mats) + ["ali1"]
    with pytest.raises(capi.VbgpuError):
        list(kio.read_ark(ark[:-5]))


def test_model_file(ref):
    n_phones, D = 4, 13
    m = synth.make_model(3 * n_phones, 40, D, 5)
    b = ref.io_write_mdl(m, n_phones)
    got = kio.read_mdl(b)
    want = ref.io_read_mdl(b, D)
    assert got["dim"] == D and len(got["pdf_offsets"]) == want["num_pdfs"] + 1
    assert np.array_equal(got["pdf_offsets"], m.pdf_offsets)
    assert len(got["tid2pdf"]) == len(want["tid2pdf"]) and len(got["tid2pdf"]) > 1
    assert np.array_equal(got["tid2pdf"][1:], want["tid2pdf"][1:])
    assert np.array_equal(got["trans_log_probs"][1:], want["trans_log_probs"][1:])
    for k in ("gconsts", "weights", "means_invvars", "inv_vars"):  # gconsts: recomputed on read, on both sides
        assert np.array_equal(got[k], want[k]), k
    # a bare AmDiagGmm (no transition model) is accepted too: cut the file at <DIMENSION>
    bare = b[b.index(b"<DIMENSION>"):]
    g2 = kio.read_mdl(bare)
    assert len(g2["tid2pdf"]) == 0 and np.array_equal(g2["gconsts"], got["gconsts"])
    with pytest.raises(capi.VbgpuError):
        kio.read_mdl(b[: len(b) // 2])


def test_statistics_file_read_back_by_the_reference(ref):
    m = synth.make_model(6, 30, 13, 9)
    N, D = len(m.gconsts), 13
    rng = np.random.default_rng(3)
    occ, mean, var = rng.uniform(0, 50, N), rng.standard_normal((N, D)) * 100, rng.uniform(0, 1e4, (N, D))
    trans = rng.uniform(0, 9, 25)
    b = kio.write_acc(m.pdf_offsets, occ, mean, var, -12345.678, 4321.0, trans_accs=trans)
    tr, o2, m2, v2, tl, tf = ref.io_read_acc(m, b, len(trans))
    # (TotLogLike() / TotCount() hand the stored doubles back as BaseFloat, mle-am-diag-gmm.h:81-83)
    assert np.array_equal(tr, trans) and tl == float(np.float32(-12345.678)) and tf == 4321.0
    # AccumDiagGmm::Write narrows to float (mle-diag-gmm.cc:86-101)
    assert np.array_equal(o2, occ.astype(np.float32).astype(np.float64))
    assert np.array_equal(m2, mean.astype(np.float32).astype(np.float64))
    assert np.array_equal(v2, var.astype(np.float32).astype(np.float64))
    b0 = kio.write_acc(m.pdf_offsets, occ, mean, var, 1.0, 2.0)  # without transition accs
    assert ref.io_read_acc(m, b0, 0)[4:] == (1.0, 2.0)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1, 2, 3, 4])
def test_matrix_to_device_is_bit_exact(ref, kind):
    import torch
    for rows, cols, stride in ((1237, 13, 16), (50, 40, 40), (33, 65, 68)):
        b = ref.io_write_matrix(_feats(rows, cols, 7 + kind), kind)
        want = ref.io_read_matrix(b)
        d_out = torch.full((rows, stride), -7.0, dtype=torch.float32, device="cuda")
        scratch = torch.empty(len(b) + 16, dtype=torch.uint8, device="cuda")
        kio.matrix_to_device(b, d_out, stride, scratch)
        torch.cuda.synchronize()
        got = d_out.cpu().numpy()
        assert np.array_equal(got[:, :cols], want)
        assert (got[:, cols:] == -7.0).all()  # the stride padding is left alone


@pytest.mark.gpu
def test_scorer_from_model_file(ref):
    """final.mdl bytes -> device scorer + tid2pdf: the DecodableInterface view agrees with the reference's own reading
    of the same file."""
    from voicebridge_b200 import host
    from tests.common import assert_ll_close
    n_phones, D = 5, 13
    m = synth.make_model(3 * n_phones, 60, D, 15)
    b = ref.io_write_mdl(m, n_phones)
    am, tid2pdf = host.AmDiagGmmGpu.from_mdl(b)
    want = ref.io_read_mdl(b, D)
    assert np.array_equal(tid2pdf[1:], want["tid2pdf"][1:])
    X = synth.make_feats(m, 64, 16)
    gc, miv, iv = ref.model_params(m.pdf_offsets, m.weights, m.means, m.iv)
    rc, ll = ref.gmm_loglikes(synth.GmmModel(m.pdf_offsets, m.weights, m.means, iv, miv, gc), X)
    assert rc == 0
    assert_ll_close(am.score(X), ll)


def test_parsers_survive_corrupt_input(ref):
    """Truncations and byte flips of real objects must end in a VbgpuError (or a clean parse), never in a crash or an
    out-of-bounds read: the parsers run on files a job did not write itself."""
    rng = np.random.default_rng(11)
    m = synth.make_model(6, 20, 13, 5)
    blobs = {
        "mdl": ref.io_write_mdl(m, 2),
        "cm": ref.io_write_matrix(_feats(40, 13, 1), 2),
        "fm": ref.io_write_matrix(_feats(7, 5, 2), 0),
        "iv": ref.io_write_int32_vector(np.arange(50, dtype=np.int32)),
    }
    ark = b"".join(kio.write_ark_entry("k%d" % i, blobs[k]) for i, k in enumerate(("cm", "fm", "iv")))

    def attempt(fn, b):
        try:
            fn(b)
        except capi.VbgpuError:
            pass

    for name, b in blobs.items():
        fn = {"mdl": kio.read_mdl, "cm": kio.read_matrix, "fm": kio.read_matrix, "iv": kio.read_int32_vector}[name]
        for cut in sorted(set(rng.integers(0, len(b), 60).tolist() + [0, 1, 2, 3, len(b) - 1])):
            with pytest.raises(capi.VbgpuError):
                fn(b[:cut])
        for _ in range(150):
            c = bytearray(b)
            for pos in rng.integers(0, min(len(c), 400), rng.integers(1, 4)):
                c[pos] = rng.integers(0, 256)
            attempt(fn, bytes(c))
    for _ in range(150):
        c = bytearray(ark)
        for pos in rng.integers(0, len(c), rng.integers(1, 4)):
            c[pos] = rng.integers(0, 256)
        attempt(lambda x: [kio.read_matrix(x, off) if info.kind <= 5 else None for _, info, off in kio.read_ark(x)], bytes(c))


@pytest.mark.gpu
def test_wav_files_to_feature_archive_like_make_mfcc(ref):
    """compute-mfcc-feats at file level: RIFF images in, a binary feature archive out, read back by the reference's
    own matrix reader and compared with the reference's own MFCCs of the same waveforms."""
    from oracle import pyoracle as po
    from tests.common import assert_feats_close
    from tests.test_wave import riff
    from voicebridge_b200 import host
    o = capi.default_mfcc_opts(dither=0.0, use_energy=0)
    mfcc = host.Mfcc(o)
    waves = {"utt%d" % i: synth.make_wave(6000 + 3211 * i, 40 + i) for i in range(4)}
    ark = b""
    for key, w in waves.items():
        wd = host.WaveData(riff(w))                      # WaveData::Read
        assert wd.SampFreq() == 16000.0
        feats = mfcc.ComputeFeatures(wd.Data()[0], wd.SampFreq())
        ark += kio.write_ark_entry(key, kio.write_matrix(feats))
    oo = po.default_opts(dither=0.0, use_energy=0)
    seen = 0
    for key, info, off in kio.read_ark(ark):
        back = ref.io_read_matrix(ark[off:off + info.total_bytes])   # the reference parses what we wrote
        assert_feats_close(back, ref.mfcc(oo, waves[key].astype(np.float32)))
        seen += 1
    assert seen == len(waves)


# ---------------------------------------------------------------------- matrix objects built here, without the reference
# The bytes of FM / DM / CM / CM2 / CM3 objects as Matrix::Write and CompressedMatrix::Write lay them out
# (kaldi-matrix.cc, compressed-matrix.cc:568-600), and CompressedMatrix::CopyToMat restated in NumPy with every float32 and
# float64 step explicit.  The library must expand them to the same bits on the host and on the device.
def _int32(v):
    return b"\x04" + np.int32(v).tobytes()  # WriteBasicType: a size byte, then the value


def _plain_obj(m, token):
    with np.errstate(over="ignore"):
        m = np.asarray(m, np.float32 if token == "FM" else np.float64)
    return b"\0B" + token.encode() + b" " + _int32(m.shape[0]) + _int32(m.shape[1]) + m.tobytes()


def _packed_obj(token, min_value, range_, rows, cols, payload):
    head = np.array([min_value, range_], np.float32).tobytes() + np.array([rows, cols], np.int32).tobytes()
    return b"\0B" + token.encode() + b" " + head + payload


def _u16_to_float(mn, rg, q):  # min_value + range * 1.52590218966964e-05F * value, all in float
    return (rg * np.float32(1.52590218966964e-05)) * np.asarray(q).astype(np.float32) + mn


def _char_to_float(p0, p25, p75, p100, v):
    """CharToFloat: p + (q - p) * k * (1/c.0), the float product (q - p) * k widened to double, scaled and added to p
    there, then narrowed."""
    v = np.asarray(v).astype(np.int32)
    lo, mid = v <= 64, v <= 192
    base = np.where(lo, p0, np.where(mid, p25, p75))
    diff = np.where(lo, p25 - p0, np.where(mid, p75 - p25, p100 - p75))
    k = np.where(lo, v, np.where(mid, v - 64, v - 192)).astype(np.float32)
    scale = np.where(lo, 1 / 64.0, np.where(mid, 1 / 128.0, 1 / 63.0))
    with np.errstate(over="ignore"):
        prod = diff * k  # float32 [rows, cols]
    return (base.astype(np.float64) + prod.astype(np.float64) * scale).astype(np.float32)


def _copy_to_mat(token, min_value, range_, rows, cols, payload):
    mn, rg = np.float32(min_value), np.float32(range_)
    with np.errstate(over="ignore"):
        if token == "CM":
            hdr = np.frombuffer(payload, np.uint16, 4 * cols).reshape(cols, 4)
            v = np.frombuffer(payload, np.uint8, rows * cols, 8 * cols).reshape(cols, rows).T
            p = _u16_to_float(mn, rg, hdr)  # [cols, 4]
            return _char_to_float(p[:, 0], p[:, 1], p[:, 2], p[:, 3], v)
        dt, n = (np.uint16, 65535.0) if token == "CM2" else (np.uint8, 255.0)
        inc = np.float32(np.float64(rg) * (1.0 / n))  # increment = range * (1.0 / 65535.0), narrowed to float
        return np.frombuffer(payload, dt, rows * cols).reshape(rows, cols).astype(np.float32) * inc + mn


# (p0, p25, p75, p100) quantiles of special columns: equal, descending, at the ends of the uint16 range
_SPECIAL_HEADERS = [(0, 0, 0, 0), (65535, 65535, 65535, 65535), (30000, 30000, 30000, 30000), (65535, 40000, 1000, 0),
                    (0, 0, 65535, 65535), (0, 65535, 0, 65535), (12345, 12346, 54321, 54322), (1, 32768, 32767, 65534),
                    (11486, 53298, 60000, 65535), (0, 11486, 53298, 65535)]  # (the last two: see the boundary test)
_RANGES = [(-3.5, 0.0), (0.0, 0.0), (-123.456, 250.75), (1.5, 1e-3), (-1e38, 2e38)]
_SHAPES = [(1, 1), (3, 1), (31, 33), (256, 70), (300, 13)]


def _cm_case(token, mn, rg, rows, cols, seed):
    rng = np.random.default_rng(seed)
    if token == "CM":
        hdr = np.sort(rng.integers(0, 65536, (cols, 4)), axis=1).astype(np.uint16)
        for j, h in enumerate(_SPECIAL_HEADERS[:cols]):
            hdr[(j * 5) % cols] = h
        # every byte value in every column (when rows >= 256), at a different row per column
        v = ((np.arange(rows)[:, None] * 7 + np.arange(cols)[None, :] * 3) % 256).astype(np.uint8)
        payload = hdr.tobytes() + np.ascontiguousarray(v.T).tobytes()
    elif token == "CM2":
        v = rng.integers(0, 65536, (rows, cols)).astype(np.uint16)
        v.flat[:2] = (0, 65535)[:v.size]
        payload = v.tobytes()
    else:
        v = ((np.arange(rows * cols) * 13 + seed) % 256).astype(np.uint8).reshape(rows, cols)
        payload = v.tobytes()
    return _packed_obj(token, mn, rg, rows, cols, payload), _copy_to_mat(token, mn, rg, rows, cols, payload)


def _plain_case(token, rows, cols, seed):
    m = np.random.default_rng(seed).standard_normal((rows, cols)) * 1e3
    special = [np.nan, np.inf, -np.inf, -0.0, 1e39, -1e39, 1e-40, 1e-50, 1 + 2.0 ** -24, 1 + 3 * 2.0 ** -24,
               -(1 + 2.0 ** -24), 3.4028235677973366e38]
    m.flat[:len(special)] = special[:m.size]
    with np.errstate(over="ignore"):  # Matrix<float>::Read of a DM object: element-wise (float) narrowing, to nearest
        want = m.astype(np.float32)
    return _plain_obj(m, token), want


def _matrix_cases():
    cases = []
    for token in ("CM", "CM2", "CM3"):
        for i, (mn, rg) in enumerate(_RANGES):
            for j, (r, c) in enumerate(_SHAPES):
                cases.append(("%s-min%g-range%g-%dx%d" % (token, mn, rg, r, c), token, r, c, 31 * i + j))
    for token in ("FM", "DM"):
        for j, (r, c) in enumerate(_SHAPES):
            cases.append(("%s-%dx%d" % (token, r, c), token, r, c, j))
    return cases


def _build(token, rows, cols, seed):
    if token in ("FM", "DM"):
        return _plain_case(token, rows, cols, seed)
    i = seed // 31
    return _cm_case(token, *_RANGES[i], rows, cols, seed)


MATRIX_CASES = _matrix_cases()


def assert_same_bits(got, want, what=""):
    """Bit for bit (the sign of zero included), with any NaN matching any NaN: a NaN's payload after narrowing is the
    hardware's choice."""
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan), what + ": NaN pattern differs"
    bad = np.flatnonzero(got.view(np.uint32)[~nan] != want.view(np.uint32)[~nan])
    assert bad.size == 0, "%s: %d elements differ, first %r vs %r" % (what, bad.size, got[~nan][bad[0]], want[~nan][bad[0]])


def test_copy_to_mat_restatement_sees_the_quantile_boundaries():
    """The cases above must tell CharToFloat's three ranges apart at 64 | 65 and 192 | 193: for some column, the value
    of byte 64 (first range) differs in its bits from p25 (where the second range starts), and likewise byte 192 from
    p75.  Otherwise moving a boundary by one would go unseen."""
    mn, rg = _RANGES[2]
    cols = 70
    b, want = _cm_case("CM", mn, rg, 256, cols, 7)
    hdr = np.frombuffer(b[2 + 3 + 16:2 + 3 + 16 + 8 * cols], np.uint16).reshape(cols, 4)
    p = _u16_to_float(np.float32(mn), np.float32(rg), hdr)
    at = lambda v: _char_to_float(p[:, 0], p[:, 1], p[:, 2], p[:, 3], np.full(cols, v))
    assert (at(64) != p[:, 1]).any() and (at(192) != p[:, 2]).any()
    assert np.array_equal(at(0), p[:, 0]) and np.array_equal(at(65), _char_to_float(p[:, 0], p[:, 1], p[:, 2], p[:, 3],
                                                                                       np.full(cols, 65)))


@pytest.mark.parametrize("name,token,rows,cols,seed", MATRIX_CASES, ids=[c[0] for c in MATRIX_CASES])
def test_read_matrix_matches_copy_to_mat(name, token, rows, cols, seed):
    """Host expansion (vbgpu_io_read_matrix) of objects built here: bit-identical to the restatement, into a row
    stride wider than cols with the padding untouched, and from inside an archive at an odd byte offset."""
    b, want = _build(token, rows, cols, seed)
    info = kio.object_info(b)
    assert kio.KINDS[info.kind] == token and (info.rows, info.cols) == (rows, cols) and info.total_bytes == len(b)
    assert_same_bits(kio.read_matrix(b), want, name)
    stride = cols + 5
    out = np.full((rows, stride), -7.0, np.float32)
    a = np.frombuffer(b, np.uint8)
    capi.check(capi.lib().vbgpu_io_read_matrix(a.ctypes.data, len(a), out.ctypes.data, stride))
    assert_same_bits(out[:, :cols], want, name + " strided")
    assert (out[:, cols:] == -7.0).all()
    ark = kio.write_ark_entry("k1", kio.write_matrix(np.ones((2, 3), np.float32))) + kio.write_ark_entry("u7", b)
    (_, _, o1), (k2, i2, o2) = list(kio.read_ark(ark))
    assert k2 == "u7" and o2 % 2 == 1 and i2.total_bytes == len(b)
    assert_same_bits(kio.read_matrix(ark, o2), want, name + " in an archive")


@pytest.mark.gpu
@pytest.mark.parametrize("name,token,rows,cols,seed", MATRIX_CASES, ids=[c[0] for c in MATRIX_CASES])
def test_matrix_to_device_matches_copy_to_mat(name, token, rows, cols, seed):
    """Device expansion (expand_cm_kernel / expand_linear_kernel / narrow_kernel / the strided copy) of the same objects:
    bit-identical to the restatement, the stride padding untouched, also from an odd offset inside an archive."""
    import torch
    b, want = _build(token, rows, cols, seed)
    ark = kio.write_ark_entry("k", b"") + kio.write_ark_entry("u7", b)
    off = ark.index(b"\0B")
    assert off % 2 == 1
    for buf, at in ((b, 0), (ark, off)):
        stride = cols + 3
        d_out = torch.full((rows, stride), -7.0, dtype=torch.float32, device="cuda")
        scratch = torch.empty(len(b) + 16, dtype=torch.uint8, device="cuda")
        kio.matrix_to_device(buf, d_out, stride, scratch, offset=at)
        torch.cuda.synchronize()
        got = d_out.cpu().numpy()
        assert_same_bits(got[:, :cols], want, "%s at offset %d" % (name, at))
        assert (got[:, cols:] == -7.0).all()
