"""One-best decoding on the device (vbgpu_decoder_*, gmm-decode-faster), through the C ABI: agreement with the float64
restatement tests/decode_ref.py fed with the device's own log-likelihoods (identical alignments, words and status,
costs to 1e-12 relative) over beams, max_active, both scorers and graphs with negative epsilon weights, epsilon olabels,
three epsilon levels and ties; equality with vbgpu_align at beam = +inf; recovery of a sampled path's words; the End
table's cases; call checks; the feature, log-likelihood and host forms, groups and streams; the PCM chain; error
counts and leaks."""
import ctypes as C

import numpy as np
import pytest

from tests.decode_ref import beam_decode_ref, loglikes_in_pdf_order
from voicebridge_b200 import capi, host, synth

INF_ACTIVE = 2**31 - 1
pytestmark = pytest.mark.gpu


def torch_dev():
    import torch
    return torch, torch.device("cuda", 0)


def batch(n_utts, lo, hi, seed):
    lens = np.random.default_rng(seed).integers(lo, hi + 1, n_utts)
    return np.r_[0, np.cumsum(lens)].astype(np.int64)


@pytest.fixture(scope="module")
def setup():
    topo = synth.phone_topology(40)
    g = synth.make_decoding_graph(topo, 300, 600, 7)
    m = synth.make_model(600, 2400, 39, 8)
    fo = batch(6, 20, 60, 9)
    X = synth.make_feats(m, int(fo[-1]), 10)
    return topo, g, m, X, fo


def device_loglikes(am, X):
    """The device's own log-likelihoods: (torch [T x NumCols] in column order, numpy [T x P] in pdf order)."""
    torch, dev = torch_dev()
    T = X.shape[0]
    d_x = torch.from_numpy(X).to(dev)
    d_ll = torch.zeros((max(T, 1), am.NumCols()), dtype=torch.float32, device=dev)
    am.score_cols_dev(d_x, T, X.shape[1], d_ll, am.NumCols(), stream=torch.cuda.current_stream())
    torch.cuda.synchronize()
    return d_ll, loglikes_in_pdf_order(d_ll.cpu().numpy()[:T], am.col_of_pdf())


def outputs(n, T, max_words):
    torch, dev = torch_dev()
    z = lambda k, t=torch.int32: torch.zeros(max(k, 1), dtype=t, device=dev)  # noqa: E731
    return dict(d_ali=z(T), d_pdf_ids=z(T), d_words=z(n * max_words), d_num_words=z(n),
                d_tot_cost=z(n, torch.float64), d_status=z(n))


def host_view(o, fo, max_words):
    n, T = len(fo) - 1, int(fo[-1])
    nw = o["d_num_words"].cpu().numpy()[:n]
    w = o["d_words"].cpu().numpy()
    return (o["d_ali"].cpu().numpy()[:T], o["d_pdf_ids"].cpu().numpy()[:T],
            [w[u * max_words:u * max_words + min(int(nw[u]), max_words)].tolist() for u in range(n)], nw,
            o["d_tot_cost"].cpu().numpy()[:n], o["d_status"].cpu().numpy()[:n])


def decode_ll(dec, am, d_ll, fo, max_words=64, scale=0.1, stream=None):
    torch, _ = torch_dev()
    o = outputs(len(fo) - 1, int(fo[-1]), max_words)
    dec.decode_loglikes_dev(am, d_ll, d_ll.shape[1], fo, max_words=max_words, acoustic_scale=scale,
                            stream=stream or torch.cuda.current_stream(), **o)
    torch.cuda.synchronize()
    return host_view(o, fo, max_words)


def check_against_ref(g, tid2pdf, ll, fo, got, beam, max_active, max_tokens=65536, scale=0.1, max_words=64):
    ali, pdf, words, nw, tot, st = got
    for u in range(len(fo) - 1):
        rows = slice(int(fo[u]), int(fo[u + 1]))
        r_st, r_cost, r_ali, r_pdf, r_words, r_nw = beam_decode_ref(g, ll[rows], tid2pdf, scale, beam, max_active,
                                                                    max_tokens)
        assert st[u] == r_st, (u, st[u], r_st)
        assert np.array_equal(ali[rows], r_ali) and np.array_equal(pdf[rows], r_pdf), u
        assert nw[u] == r_nw and words[u] == r_words[:max_words], u
        if np.isfinite(r_cost):
            assert abs(tot[u] - r_cost) <= 1e-12 * max(abs(r_cost), 1.0), (u, tot[u], r_cost)
        else:
            assert tot[u] == np.inf


@pytest.mark.parametrize("kernel", [1, 2])
@pytest.mark.parametrize("beam,max_active", [(np.inf, INF_ACTIVE), (16.0, 1000), (8.0, 50), (2.0, 1), (16.0, INF_ACTIVE),
                                             (8.0, INF_ACTIVE)])
def test_agreement_with_restatement(setup, kernel, beam, max_active):
    topo, g, m, X, fo = setup
    am = host.AmDiagGmmGpu.from_model(m)
    try:
        am.set_kernel(kernel)
    except capi.VbgpuError:
        pytest.skip("scorer %d unavailable for this model" % kernel)
    d_ll, ll = device_loglikes(am, X)
    dec = host.GmmDecodeFasterGpu(g, g["tid2pdf"], beam=beam, max_active=max_active)
    got = decode_ll(dec, am, d_ll, fo)
    check_against_ref(g, g["tid2pdf"], ll, fo, got, beam, max_active)
    if beam == np.inf:  # (narrow beams may end partial or, at one token per frame, empty: checked above)
        assert (got[5] == 0).all()


def tie_graph(seed, S=40):
    """A graph built to tie: transition-ids 1-3 and 4-6 read one pdf each, weights from {0, 0.5} (-0.5 on some epsilon
    arcs), parallel arcs of equal weight, zero-weight epsilon arcs into states that emitting arcs also reach, and final
    costs from {0, 0.5} on many states; sums of these are exact, so equal-cost candidates and tokens are common."""
    rng = np.random.default_rng(seed)
    arcs = []
    for s in range(S):
        for _ in range(int(rng.integers(2, 5))):
            d, w = int(rng.integers(0, S)), float(rng.choice([0.0, 0.5]))
            arcs.append((s, d, int(rng.integers(1, 7)), int(rng.integers(0, 4)), w))
            if rng.random() < 0.3:  # a parallel arc of the same weight
                arcs.append((s, d, int(rng.integers(1, 7)), int(rng.integers(0, 4)), w))
        for _ in range(int(rng.integers(0, 3))):
            if s + 1 < S:
                arcs.append((s, int(rng.integers(s + 1, min(S, s + 8))), 0, int(rng.integers(0, 4)),
                             float(rng.choice([0.0, 0.0, 0.5, -0.5]))))
    a = np.array(arcs, np.float64)
    return dict(num_states=S, start=0, final_cost=rng.choice([np.inf, 0.0, 0.5], S).astype(np.float32),
                arc_src=a[:, 0].astype(np.int32), arc_dst=a[:, 1].astype(np.int32), arc_ilabel=a[:, 2].astype(np.int32),
                arc_olabel=a[:, 3].astype(np.int32), arc_weight=a[:, 4].astype(np.float32))


@pytest.mark.parametrize("kernel", [1, 2])
def test_ties_agree_with_restatement(setup, kernel):
    """Graphs built to tie, on both scorers: identical to the restatement, and the restatement's tie counters show
    that every tie rule decided something (equal candidates into a state, an emitting back-pointer keeping an equal
    epsilon candidate, equal epsilon candidates, tied best tokens, equal costs at c_(max_active+1), tied finals)."""
    from collections import Counter
    topo, g0, m, X, fo = setup
    am = host.AmDiagGmmGpu.from_model(m)
    try:
        am.set_kernel(kernel)
    except capi.VbgpuError:
        pytest.skip("scorer %d unavailable for this model" % kernel)
    d_ll, ll = device_loglikes(am, X)
    t2p = np.array([0, 17, 17, 17, 230, 230, 230], np.int32)
    ties, statuses = Counter(), Counter()
    for seed in range(4):
        g = tie_graph(100 + seed)
        for beam, max_active in ((np.inf, INF_ACTIVE), (1.0, INF_ACTIVE), (0.5, 3), (2.0, 5), (1.0, 1)):
            dec = host.GmmDecodeFasterGpu(g, t2p, beam=beam, max_active=max_active)
            got = decode_ll(dec, am, d_ll, fo)
            check_against_ref(g, t2p, ll, fo, got, beam, max_active)
            statuses.update(got[5].tolist())
            for u in range(len(fo) - 1):
                beam_decode_ref(g, ll[int(fo[u]):int(fo[u + 1])], t2p, 0.1, beam, max_active, ties=ties)
            dec.close()
    assert all(ties[k] > 0 for k in ("arcs", "emit_kept", "eps_equal", "best", "boundary", "final")), ties
    assert statuses[0] > 0, statuses


def test_exact_search_equals_align(setup):
    """beam = +inf, unlimited max_active: every utterance that reaches a final state has vbgpu_align's alignment and,
    bit for bit, its cost (the same graph given to the align handle once per utterance)."""
    topo, g0, m, X, fo = setup
    g = synth.make_decoding_graph(topo, 60, 600, 17)
    assert g["num_states"] <= 4096
    am = host.AmDiagGmmGpu.from_model(m)
    d_ll, ll = device_loglikes(am, X)
    dec = host.GmmDecodeFasterGpu(g, g["tid2pdf"], beam=np.inf)
    ali, pdf, words, nw, tot, st = decode_ll(dec, am, d_ll, fo)
    n, S, A = len(fo) - 1, int(g["num_states"]), len(g["arc_src"])
    graphs = dict(state_offsets=np.arange(n + 1, dtype=np.int32) * S, start=np.full(n, g["start"], np.int32),
                  final_cost=np.tile(g["final_cost"], n), arc_offsets=np.arange(n + 1, dtype=np.int64) * A,
                  **{k: np.tile(g[k], n) for k in ("arc_src", "arc_dst", "arc_ilabel", "arc_weight")})
    a_ali, a_pdf, a_cost = host.GmmAlignCompiledGpu(graphs, g["tid2pdf"]).Align(am, X, fo)
    assert (st == 0).all()
    assert np.array_equal(ali, a_ali) and np.array_equal(pdf, a_pdf)
    assert np.array_equal(tot, a_cost)


def test_recovers_sampled_words():
    """Features drawn along a sampled path from a well-separated model decode back to its words at beam 16."""
    topo = synth.phone_topology(30)
    g = synth.make_decoding_graph(topo, 150, 200, 21, phones_per_word=(2, 2))
    m = synth.make_model(200, 200, 39, 22, spread=3.0)
    rng = np.random.default_rng(23)
    paths = [synth.sample_decoding_path(g, 30 + k, 80) for k in range(6)]
    tids = np.concatenate([p[1] for p in paths])
    fo = np.r_[0, np.cumsum([len(p[1]) for p in paths])].astype(np.int64)
    pt = g["tid2pdf"][tids]
    X = (m.means[pt] + np.sqrt(1.0 / m.iv[pt]) * rng.standard_normal((len(tids), 39))).astype(np.float32)
    am = host.AmDiagGmmGpu.from_model(m)
    dec = host.GmmDecodeFasterGpu(g, g["tid2pdf"], beam=16.0)
    ali, pdf, words, nw, tot, st = dec.Decode(am, X, fo)
    assert (st == 0).all()
    for u, p in enumerate(paths):
        assert words[u] == p[0], (u, words[u], p[0])


def tiny_decoder(arcs, finals, S, tid2pdf, **kw):
    a = np.array(arcs, np.float64).reshape(-1, 5)
    g = dict(num_states=S, start=0, final_cost=np.array(finals, np.float32), arc_src=a[:, 0].astype(np.int32),
             arc_dst=a[:, 1].astype(np.int32), arc_ilabel=a[:, 2].astype(np.int32), arc_olabel=a[:, 3].astype(np.int32),
             arc_weight=a[:, 4].astype(np.float32))
    return g, host.GmmDecodeFasterGpu(g, tid2pdf, **kw)


def test_end_cases(setup):
    """T = 0, status 1 (partial path equal to the restatement's), status 2, status 3 (small max_tokens), and
    num_words > max_words with nothing written beyond the cap."""
    torch, dev = torch_dev()
    topo, g, m, X, fo = setup
    am = host.AmDiagGmmGpu.from_model(m)
    d_ll, ll = device_loglikes(am, X)
    t2p = g["tid2pdf"]
    # T = 0 between two utterances: the start closure's best final
    fo0 = np.array([0, 30, 30, 60], np.int64)
    dec = host.GmmDecodeFasterGpu(g, t2p)
    got = decode_ll(dec, am, d_ll, fo0)
    check_against_ref(g, t2p, ll, fo0, got, 16.0, INF_ACTIVE)
    assert got[5][1] == 0 and got[4][1] == float(g["final_cost"][g["start"]])
    # status 1: no final state
    g1 = dict(g, final_cost=np.full(g["num_states"], np.inf, np.float32))
    got = decode_ll(host.GmmDecodeFasterGpu(g1, t2p), am, d_ll, fo)
    assert (got[5] == 1).all()
    check_against_ref(g1, t2p, ll, fo, got, 16.0, INF_ACTIVE)
    # status 2: a dead end after one frame (utterance 0), neighbours unaffected
    tiny_t2p = np.array([0, 1, 2], np.int32)
    gt, dt = tiny_decoder([(0, 1, 1, 3, 0.0), (1, 1, 2, 4, 0.0)], [np.inf, 0.0, np.inf], 3, tiny_t2p)
    gt2, dt2 = tiny_decoder([(0, 1, 1, 3, 0.0), (0, 2, 2, 0, 0.0)], [np.inf, 0.0, 0.0], 3, tiny_t2p)
    fo_t = np.array([0, 3], np.int64)
    got = decode_ll(dt, am, d_ll, fo_t)
    assert got[5][0] == 0 and got[3][0] == 3 and got[2][0] == [3, 4, 4]
    got = decode_ll(dt2, am, d_ll, fo_t)
    assert got[5][0] == 2 and got[4][0] == np.inf and not got[0].any() and (got[1] == -1).all() and got[3][0] == 0
    # status 3: max_tokens below a frame's set
    for mt in (1, 5, 40):
        dec3 = host.GmmDecodeFasterGpu(g, t2p, max_tokens=mt)
        got = decode_ll(dec3, am, d_ll, fo)
        assert (got[5] == 3).all(), mt
        assert np.isinf(got[4]).all() and not got[0].any() and (got[1] == -1).all() and not got[3].any()
        check_against_ref(g, t2p, ll, fo, got, 16.0, INF_ACTIVE, max_tokens=mt)
    # num_words > max_words: the true count, the first max_words words, and a sentinel past the cap untouched
    full = decode_ll(dec, am, d_ll, fo)
    assert full[3].max() > 2
    o = outputs(len(fo) - 1, int(fo[-1]), 3)
    o["d_words"].fill_(-7)
    dec.decode_loglikes_dev(am, d_ll, d_ll.shape[1], fo, max_words=2, stream=torch.cuda.current_stream(), **o)
    torch.cuda.synchronize()
    w = o["d_words"].cpu().numpy()
    n = len(fo) - 1
    assert np.array_equal(o["d_num_words"].cpu().numpy(), full[3])
    for u in range(n):
        k = min(2, int(full[3][u]))
        assert w[2 * u:2 * u + k].tolist() == full[2][u][:2]
    assert (w[2 * n:] == -7).all()


def test_call_checks(setup):
    torch, dev = torch_dev()
    topo, g, m, X, fo = setup
    am = host.AmDiagGmmGpu.from_model(m)
    d_ll, ll = device_loglikes(am, X)
    dec = host.GmmDecodeFasterGpu(g, g["tid2pdf"])
    for field, bad in (("beam", 0.0), ("beam", -1.0), ("beam", float("nan")), ("max_active", 0), ("max_tokens", 0)):
        good = getattr(dec.opts, field)
        setattr(dec.opts, field, bad)
        with pytest.raises(capi.VbgpuError) as e:
            decode_ll(dec, am, d_ll, fo)
        assert e.value.code == capi.ERR_INVALID and field in str(e.value)
        setattr(dec.opts, field, good)
    o = outputs(len(fo) - 1, int(fo[-1]), 4)
    with pytest.raises(capi.VbgpuError, match="ll_stride"):
        dec.decode_loglikes_dev(am, d_ll, am.NumCols() - 1, fo, max_words=4, **o)
    small = host.AmDiagGmmGpu.from_model(synth.make_model(10, 20, 39, 1))
    with pytest.raises(capi.VbgpuError, match="tid2pdf names pdf"):
        dec.Decode(small, X, fo)
    with pytest.raises(capi.VbgpuError, match="max_words"):
        dec.decode_loglikes_dev(am, d_ll, d_ll.shape[1], fo, max_words=-1, **o)


def test_forms_groups_and_streams(setup):
    """Feature form = log-likelihood form on score_cols_dev output (bit for bit); host form = _dev form; one utterance
    per group; two streams on one handle."""
    torch, dev = torch_dev()
    topo, g, m, X, fo = setup
    for kernel in (1, 2):
        am = host.AmDiagGmmGpu.from_model(m)
        try:
            am.set_kernel(kernel)
        except capi.VbgpuError:
            continue
        d_ll, ll = device_loglikes(am, X)
        dec = host.GmmDecodeFasterGpu(g, g["tid2pdf"], beam=12.0, max_active=200)
        want = decode_ll(dec, am, d_ll, fo)
        o = outputs(len(fo) - 1, int(fo[-1]), 64)
        dec.decode_dev(am, torch.from_numpy(X).to(dev), 39, fo, max_words=64, stream=torch.cuda.current_stream(), **o)
        torch.cuda.synchronize()
        got = host_view(o, fo, 64)
        hostf = dec.Decode(am, X, fo)
        for a, b, c in zip(want, got, hostf):
            if isinstance(a, list):
                assert a == b == c
            else:
                assert np.array_equal(a, b) and np.array_equal(a, c)
        dec.set_workspace(1)
        assert all(np.array_equal(a, b) if not isinstance(a, list) else a == b
                   for a, b in zip(want, dec.Decode(am, X, fo)))
        dec.set_workspace(0)
        sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
        outs = [outputs(len(fo) - 1, int(fo[-1]), 64) for _ in range(2)]
        torch.cuda.synchronize()
        dec.decode_loglikes_dev(am, d_ll, d_ll.shape[1], fo, max_words=64, stream=sa, **outs[0])
        dec.decode_loglikes_dev(am, d_ll, d_ll.shape[1], fo, max_words=64, stream=sb, **outs[1])
        torch.cuda.synchronize()
        for o in outs:
            for a, b in zip(want, host_view(o, fo, 64)):
                assert np.array_equal(a, b) if not isinstance(a, list) else a == b


def test_pcm_chain_on_device():
    """PCM -> vbgpu_pipeline_score_cols_dev -> vbgpu_decode_loglikes_dev with everything on the device; equal to the
    restatement on the pipeline's log-likelihoods."""
    torch, dev = torch_dev()
    pcm, so, u2s = synth.make_corpus(2, 2, 0.5, 1.0, 31)
    mf = host.Mfcc(capi.default_mfcc_opts(dither=0.0, use_energy=0))
    fp = host.FeaturePipeline(capi.default_feat_opts(), 13)
    m = synth.make_model(600, 2400, 39, 32)
    am = host.AmDiagGmmGpu.from_model(m)
    pipe = host.ScoringPipeline(mf, fp, am)
    fo = np.r_[0, np.cumsum([mf.NumFrames(int(so[u + 1] - so[u])) for u in range(len(so) - 1)])].astype(np.int64)
    T = int(fo[-1])
    d_pcm = torch.from_numpy(np.asarray(pcm, np.int16)).to(dev)
    d_ll = torch.zeros((T, am.NumCols()), dtype=torch.float32, device=dev)
    pipe.score_cols_dev(d_pcm, so, u2s, int(u2s.max()) + 1, None, 0, d_ll, am.NumCols(),
                        stream=torch.cuda.current_stream())
    g = synth.make_decoding_graph(synth.phone_topology(40), 300, 600, 33)
    dec = host.GmmDecodeFasterGpu(g, g["tid2pdf"], beam=13.0, max_active=7000)
    got = decode_ll(dec, am, d_ll, fo)
    ll = loglikes_in_pdf_order(d_ll.cpu().numpy(), am.col_of_pdf())
    check_against_ref(g, g["tid2pdf"], ll, fo, got, 13.0, 7000)


def test_error_counts_and_leaks(setup):
    torch, dev = torch_dev()
    topo, g, m, X, fo = setup
    before = C.c_int64(), C.c_int64()
    capi.lib().vbgpu_debug_live_bytes(C.byref(before[0]), C.byref(before[1]))
    am = host.AmDiagGmmGpu.from_model(m)
    for _ in range(3):
        dec = host.GmmDecodeFasterGpu(g, g["tid2pdf"], beam=10.0)
        dec.Decode(am, X, fo)
        dec.close()
    Xbad = X.copy()
    Xbad[7] = np.nan
    dec = host.GmmDecodeFasterGpu(g, g["tid2pdf"], beam=10.0)
    with pytest.raises(capi.VbgpuError) as e:
        dec.Decode(am, Xbad, fo)
    assert e.value.code == capi.ERR_NUMERIC
    assert am.bad_count() == 0
    o = outputs(len(fo) - 1, int(fo[-1]), 8)
    dec.decode_dev(am, torch.from_numpy(Xbad).to(dev), 39, fo, max_words=8, stream=torch.cuda.current_stream(), **o)
    torch.cuda.synchronize()
    assert am.bad_count() > 0
    d_ll, _ = device_loglikes(am, X)
    am.bad_count()
    d_ll[3, int(am.col_of_pdf()[0])] = float("inf")
    dec.decode_loglikes_dev(am, d_ll, d_ll.shape[1], fo, max_words=8, stream=torch.cuda.current_stream(), **o)
    torch.cuda.synchronize()
    assert am.bad_count() == 1
    del o, d_ll
    dec.close()
    am.close()
    after = C.c_int64(), C.c_int64()
    capi.lib().vbgpu_debug_live_bytes(C.byref(after[0]), C.byref(after[1]))
    assert (after[0].value, after[1].value) == (before[0].value, before[1].value)
