"""Lattice generation on the device (vbgpu_decode_lattice*, gmm-latgen-faster up to the raw lattice), through the C ABI:
the lattice equals the float64 restatement tests/latgen_ref.py array for array, bit for bit, over beams, max_active,
lattice beams and both scorers, on the synthetic graph and on graphs built to tie; the one-best outputs equal
vbgpu_decode_loglikes_dev's; acoustic costs equal -(scale * ll); tokens kept only for an epsilon path into an expanded
token; decoder statuses 0-3 and both lattice-store and output-capacity statuses; T = 0; groups, streams, the
feature / log-likelihood / host forms; the PCM chain; call checks, error counts and leaks."""
import ctypes as C

import numpy as np
import pytest

from tests.decode_ref import loglikes_in_pdf_order
from tests.latgen_ref import LATTICE_KEYS, latgen_ref
from tests.test_gpu_decode import batch, device_loglikes, host_view, outputs, tie_graph, torch_dev
from voicebridge_b200 import capi, host, synth

INF_ACTIVE = 2**31 - 1
pytestmark = pytest.mark.gpu
SMALL = dict(max_states=4096, max_arcs=16384, arena_tokens=512, arena_links=2048)


@pytest.fixture(scope="module")
def setup():
    topo = synth.phone_topology(40)
    g = synth.make_decoding_graph(topo, 300, 600, 7)
    m = synth.make_model(600, 2400, 39, 8)
    fo = batch(6, 20, 60, 9)
    X = synth.make_feats(m, int(fo[-1]), 10)
    return topo, g, m, X, fo


def lattice_buffers(n, lo):
    torch, dev = torch_dev()
    d = {}
    for k, t, per_state in host.GmmDecodeFasterGpu.LATTICE_ARRAYS:
        d[k] = torch.zeros(max(n * (lo.max_states if per_state else lo.max_arcs), 1),
                           dtype=torch.float32 if t == np.float32 else torch.int32, device=dev)
    for k in ("num_states", "num_arcs", "lattice_status"):
        d[k] = torch.full((max(n, 1),), -5, dtype=torch.int32, device=dev)
    d["arena_peak"] = torch.zeros(max(2 * n, 2), dtype=torch.int32, device=dev)
    return d


def lattice_host(d, n, lo):
    arr = {k: v.cpu().numpy() for k, v in d.items()}
    return host.GmmDecodeFasterGpu.split_lattices(arr, n, lo.max_states, lo.max_arcs)


def latgen_ll(dec, am, d_ll, fo, lo, max_words=64, scale=0.1, stream=None):
    torch, _ = torch_dev()
    n = len(fo) - 1
    o, lat = outputs(n, int(fo[-1]), max_words), lattice_buffers(n, lo)
    dec.decode_lattice_loglikes_dev(am, d_ll, d_ll.shape[1], fo, max_words=max_words, lattice=lat, lattice_opts=lo,
                                    acoustic_scale=scale, stream=stream or torch.cuda.current_stream(), **o)
    torch.cuda.synchronize()
    return host_view(o, fo, max_words), lattice_host(lat, n, lo)


def decode_plain(dec, am, d_ll, fo, max_words=64):
    torch, _ = torch_dev()
    o = outputs(len(fo) - 1, int(fo[-1]), max_words)
    dec.decode_loglikes_dev(am, d_ll, d_ll.shape[1], fo, max_words=max_words, stream=torch.cuda.current_stream(), **o)
    torch.cuda.synchronize()
    return host_view(o, fo, max_words)


def same_one_best(a, b):
    for x, y in zip(a, b):
        assert (x == y) if isinstance(x, list) else np.array_equal(x, y)


def check_lattices(g, t2p, ll, fo, one, lats, beam, max_active, lattice_beam, max_tokens=65536, scale=0.1):
    """Every utterance's lattice equals the restatement's bit for bit, and its acoustic costs are -(scale * ll)."""
    n_states = 0
    for u in range(len(fo) - 1):
        rows = slice(int(fo[u]), int(fo[u + 1]))
        r_one, r_lat = latgen_ref(g, ll[rows], t2p, scale, beam, max_active, max_tokens, lattice_beam)
        assert one[5][u] == r_one[0], u
        got = lats[u]
        assert got["lattice_status"] == 0, (u, got["lattice_status"])
        for k in LATTICE_KEYS:
            assert got[k].dtype == r_lat[k].dtype and np.array_equal(got[k].view(np.int32), r_lat[k].view(np.int32)), \
                (u, k)
        em = got["arc_ilabel"] > 0
        fr = got["state_frame"][got["arc_src"][em]]
        want_ac = (-(np.float32(scale) * ll[rows][fr, t2p[got["arc_ilabel"][em]]])).astype(np.float32)
        assert np.array_equal(got["arc_ac_cost"][em], want_ac)
        assert (got["arc_ac_cost"][~em] == 0).all()
        assert got["num_states"] == len(got["state_frame"]) and got["num_arcs"] == len(got["arc_src"])
        n_states += got["num_states"]
    return n_states


def model_with(m, kernel):
    am = host.AmDiagGmmGpu.from_model(m)
    try:
        am.set_kernel(kernel)
    except capi.VbgpuError:
        pytest.skip("scorer %d unavailable for this model" % kernel)
    return am


@pytest.mark.parametrize("kernel", [1, 2])
@pytest.mark.parametrize("beam,max_active", [(np.inf, INF_ACTIVE), (16.0, 1000), (8.0, 50), (2.0, 1)])
def test_agreement_with_restatement(setup, kernel, beam, max_active):
    topo, g, m, X, fo = setup
    am = model_with(m, kernel)
    d_ll, ll = device_loglikes(am, X)
    dec = host.GmmDecodeFasterGpu(g, g["tid2pdf"], beam=beam, max_active=max_active)
    want = decode_plain(dec, am, d_ll, fo)
    for lattice_beam in (0.0, 4.0, 10.0):
        lo = capi.default_lattice_opts(lattice_beam=lattice_beam, max_states=1 << 15, max_arcs=1 << 17,
                                       arena_tokens=4096, arena_links=12288)
        one, lats = latgen_ll(dec, am, d_ll, fo, lo)
        same_one_best(want, one)
        n_states = check_lattices(g, g["tid2pdf"], ll, fo, one, lats, beam, max_active, lattice_beam)
        assert n_states > 0 or (one[5] >= 2).all()  # (a narrow beam at one token per frame may empty the set)
    dec.close()


@pytest.mark.parametrize("kernel", [1, 2])
def test_ties_agree_with_restatement(setup, kernel):
    topo, g0, m, X, fo = setup
    am = model_with(m, kernel)
    d_ll, ll = device_loglikes(am, X)
    t2p = np.array([0, 17, 17, 17, 230, 230, 230], np.int32)
    for seed in range(3):
        g = tie_graph(100 + seed)
        for beam, max_active, lb in ((np.inf, INF_ACTIVE, 1.0), (1.0, INF_ACTIVE, 0.0), (2.0, 5, 2.0), (1.0, 1, 0.5)):
            dec = host.GmmDecodeFasterGpu(g, t2p, beam=beam, max_active=max_active)
            lo = capi.default_lattice_opts(lattice_beam=lb, **SMALL)
            one, lats = latgen_ll(dec, am, d_ll, fo, lo)
            same_one_best(decode_plain(dec, am, d_ll, fo), one)
            check_lattices(g, t2p, ll, fo, one, lats, beam, max_active, lb)
            dec.close()


def eps_into_survivor_graph():
    """State 1 is reached by an emitting arc; its epsilon arc into state 2 has weight -4, so with max_active = 1 the
    prune expands only state 2, and state 1 stays in the lattice only for its epsilon path into it."""
    arcs = [(0, 1, 1, 0, 0.0), (0, 3, 2, 0, 0.5), (1, 2, 0, 5, -4.0), (2, 1, 1, 0, 0.0), (2, 3, 2, 0, 0.0),
            (3, 1, 1, 0, 0.0), (3, 3, 2, 0, 0.0)]
    a = np.array(arcs, np.float64)
    return dict(num_states=4, start=0, final_cost=np.array([np.inf, 0.0, 0.0, 0.5], np.float32),
                arc_src=a[:, 0].astype(np.int32), arc_dst=a[:, 1].astype(np.int32), arc_ilabel=a[:, 2].astype(np.int32),
                arc_olabel=a[:, 3].astype(np.int32), arc_weight=a[:, 4].astype(np.float32))


def test_epsilon_path_into_expanded_token(setup):
    topo, g0, m, X, fo = setup
    am = host.AmDiagGmmGpu.from_model(m)
    d_ll, ll = device_loglikes(am, X)
    g, t2p = eps_into_survivor_graph(), np.array([0, 3, 9], np.int32)
    dec = host.GmmDecodeFasterGpu(g, t2p, beam=np.inf, max_active=1)
    lo = capi.default_lattice_opts(lattice_beam=np.inf, **SMALL)
    one, lats = latgen_ll(dec, am, d_ll, fo, lo)
    check_lattices(g, t2p, ll, fo, one, lats, np.inf, 1, np.inf)
    found = 0
    for lat in lats:  # a non-final-frame state 1 whose only way on is its epsilon arc into state 2
        last = lat["state_frame"].max()
        for i in np.flatnonzero((lat["state_graph"] == 1) & (lat["state_frame"] < last)):
            outs = np.flatnonzero(lat["arc_src"] == i)
            found += len(outs) > 0 and (lat["arc_ilabel"][outs] == 0).all()
    assert found > 0


def test_statuses_capacities_and_t0(setup):
    topo, g, m, X, fo = setup
    am = host.AmDiagGmmGpu.from_model(m)
    d_ll, ll = device_loglikes(am, X)
    t2p = g["tid2pdf"]
    lo = capi.default_lattice_opts(lattice_beam=6.0, **SMALL)
    # T = 0 between two utterances; status 0 elsewhere
    fo0 = np.array([0, 30, 30, 60], np.int64)
    dec = host.GmmDecodeFasterGpu(g, t2p, beam=10.0, max_active=100)
    one, lats = latgen_ll(dec, am, d_ll, fo0, lo)
    same_one_best(decode_plain(dec, am, d_ll, fo0), one)
    check_lattices(g, t2p, ll, fo0, one, lats, 10.0, 100, 6.0)
    assert one[5][1] == 0 and (lats[1]["state_frame"] == 0).all() and lats[1]["num_states"] >= 1
    # status 1: no final state
    g1 = dict(g, final_cost=np.full(g["num_states"], np.inf, np.float32))
    d1 = host.GmmDecodeFasterGpu(g1, t2p, beam=10.0, max_active=100)
    one, lats = latgen_ll(d1, am, d_ll, fo, lo)
    assert (one[5] == 1).all()
    check_lattices(g1, t2p, ll, fo, one, lats, 10.0, 100, 6.0)
    assert all((lat["state_final"][lat["state_frame"] == lat["state_frame"].max()] == 0).all() for lat in lats)
    # status 2: a dead end; status 3: max_tokens below a frame's set: empty lattices
    tiny = [(0, 1, 1, 3, 0.0), (0, 2, 2, 0, 0.0)]
    a = np.array(tiny, np.float64)
    g2 = dict(num_states=3, start=0, final_cost=np.array([np.inf, 0.0, 0.0], np.float32),
              arc_src=a[:, 0].astype(np.int32), arc_dst=a[:, 1].astype(np.int32), arc_ilabel=a[:, 2].astype(np.int32),
              arc_olabel=a[:, 3].astype(np.int32), arc_weight=a[:, 4].astype(np.float32))
    one, lats = latgen_ll(host.GmmDecodeFasterGpu(g2, np.array([0, 1, 2], np.int32)), am, d_ll,
                          np.array([0, 3], np.int64), lo)
    assert one[5][0] == 2 and lats[0]["num_states"] == 0 and lats[0]["lattice_status"] == 0
    one, lats = latgen_ll(host.GmmDecodeFasterGpu(g, t2p, max_tokens=5), am, d_ll, fo, lo)
    assert (one[5] == 3).all() and all(lt["num_states"] == lt["num_arcs"] == lt["lattice_status"] == 0 for lt in lats)
    # lattice status 1: a store too small; the one-best outputs stay valid
    want = decode_plain(dec, am, d_ll, fo)
    lo1 = capi.default_lattice_opts(lattice_beam=6.0, max_states=4096, max_arcs=16384, arena_tokens=2, arena_links=4)
    one, lats = latgen_ll(dec, am, d_ll, fo, lo1)
    same_one_best(want, one)
    assert all(lt["lattice_status"] == 1 and lt["num_states"] == 0 for lt in lats)
    # lattice status 2: over the output capacity, with the true counts; a retry at those counts writes the lattice
    one, full = latgen_ll(dec, am, d_ll, fo, lo)
    ms, ma = max(lt["num_states"] for lt in full), max(lt["num_arcs"] for lt in full)
    lo2 = capi.default_lattice_opts(lattice_beam=6.0, max_states=ms - 1, max_arcs=ma, arena_tokens=512,
                                    arena_links=2048)
    one2, lats2 = latgen_ll(dec, am, d_ll, fo, lo2)
    same_one_best(want, one2)
    for a, b in zip(full, lats2):
        assert (a["num_states"], a["num_arcs"]) == (b["num_states"], b["num_arcs"])
        assert b["lattice_status"] == (2 if a["num_states"] > ms - 1 else 0)
    lo3 = capi.default_lattice_opts(lattice_beam=6.0, max_states=ms, max_arcs=ma - 1, arena_tokens=512,
                                    arena_links=2048)
    _, lats3 = latgen_ll(dec, am, d_ll, fo, lo3)
    assert any(b["lattice_status"] == 2 for b in lats3)
    assert all(b["lattice_status"] == (2 if a["num_arcs"] > ma - 1 else 0) for a, b in zip(full, lats3))


def test_forms_groups_and_streams(setup):
    """Feature form = log-likelihood form = host form, bit for bit; one utterance per group; two streams."""
    torch, dev = torch_dev()
    topo, g, m, X, fo = setup
    am = host.AmDiagGmmGpu.from_model(m)
    d_ll, ll = device_loglikes(am, X)
    dec = host.GmmDecodeFasterGpu(g, g["tid2pdf"], beam=12.0, max_active=200)
    lo = capi.default_lattice_opts(lattice_beam=5.0, **SMALL)
    n = len(fo) - 1
    want_one, want = latgen_ll(dec, am, d_ll, fo, lo)
    check_lattices(g, g["tid2pdf"], ll, fo, want_one, want, 12.0, 200, 5.0)

    def same(one, lats):
        same_one_best(want_one, one)
        for a, b in zip(want, lats):
            for k in LATTICE_KEYS + ("num_states", "num_arcs", "lattice_status"):
                assert np.array_equal(np.asarray(a[k]).view(np.int32) if k in LATTICE_KEYS else a[k],
                                      np.asarray(b[k]).view(np.int32) if k in LATTICE_KEYS else b[k]), k

    o, lat = outputs(n, int(fo[-1]), 64), lattice_buffers(n, lo)
    dec.decode_lattice_dev(am, torch.from_numpy(X).to(dev), 39, fo, max_words=64, lattice=lat, lattice_opts=lo,
                           stream=torch.cuda.current_stream(), **o)
    torch.cuda.synchronize()
    same(host_view(o, fo, 64), lattice_host(lat, n, lo))
    r = dec.DecodeLattice(am, X, fo, lattice_beam=5.0, **SMALL)
    same(r[:6], r[6])
    dec.set_workspace(1)
    r = dec.DecodeLattice(am, X, fo, lattice_beam=5.0, **SMALL)
    same(r[:6], r[6])
    dec.set_workspace(0)
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    bufs = [(outputs(n, int(fo[-1]), 64), lattice_buffers(n, lo)) for _ in range(2)]
    torch.cuda.synchronize()
    for (o, lat), st in zip(bufs, (sa, sb)):
        dec.decode_lattice_loglikes_dev(am, d_ll, d_ll.shape[1], fo, max_words=64, lattice=lat, lattice_opts=lo,
                                        stream=st, **o)
    torch.cuda.synchronize()
    for o, lat in bufs:
        same(host_view(o, fo, 64), lattice_host(lat, n, lo))


def test_pcm_chain_on_device():
    """PCM -> vbgpu_pipeline_score_cols_dev -> vbgpu_decode_lattice_loglikes_dev on the device; equal to the
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
    lo = capi.default_lattice_opts(lattice_beam=6.0, max_states=1 << 15, max_arcs=1 << 17, arena_tokens=4096,
                                   arena_links=16384)
    one, lats = latgen_ll(dec, am, d_ll, fo, lo)
    ll = loglikes_in_pdf_order(d_ll.cpu().numpy(), am.col_of_pdf())
    check_lattices(g, g["tid2pdf"], ll, fo, one, lats, 13.0, 7000, 6.0)


def test_call_checks_error_counts_and_leaks(setup):
    torch, dev = torch_dev()
    topo, g, m, X, fo = setup
    before = C.c_int64(), C.c_int64()
    capi.lib().vbgpu_debug_live_bytes(C.byref(before[0]), C.byref(before[1]))
    am = host.AmDiagGmmGpu.from_model(m)
    d_ll, _ = device_loglikes(am, X)
    dec = host.GmmDecodeFasterGpu(g, g["tid2pdf"], beam=10.0)
    for field, bad in (("lattice_beam", -1.0), ("lattice_beam", float("nan")), ("max_states", -1), ("max_arcs", -1),
                       ("arena_tokens", 0), ("arena_links", 0), ("arena_links", 1 << 30)):
        lo = capi.default_lattice_opts(**SMALL)
        setattr(lo, field, bad)
        with pytest.raises(capi.VbgpuError) as e:
            latgen_ll(dec, am, d_ll, fo, lo)
        assert e.value.code == capi.ERR_INVALID
    for _ in range(2):
        dec.DecodeLattice(am, X, fo, **SMALL)
    Xbad = X.copy()
    Xbad[7] = np.nan
    with pytest.raises(capi.VbgpuError) as e:
        dec.DecodeLattice(am, Xbad, fo, **SMALL)
    assert e.value.code == capi.ERR_NUMERIC
    assert am.bad_count() == 0
    n, lo = len(fo) - 1, capi.default_lattice_opts(**SMALL)
    o, lat = outputs(n, int(fo[-1]), 8), lattice_buffers(n, lo)
    dec.decode_lattice_dev(am, torch.from_numpy(Xbad).to(dev), 39, fo, max_words=8, lattice=lat, lattice_opts=lo,
                           stream=torch.cuda.current_stream(), **o)
    torch.cuda.synchronize()
    assert am.bad_count() > 0
    d_ll[3, int(am.col_of_pdf()[0])] = float("inf")
    latgen_ll(dec, am, d_ll, fo, lo, max_words=8)
    assert am.bad_count() == 1
    del o, lat, d_ll
    dec.close()
    am.close()
    after = C.c_int64(), C.c_int64()
    capi.lib().vbgpu_debug_live_bytes(C.byref(after[0]), C.byref(after[1]))
    assert (after[0].value, after[1].value) == (before[0].value, before[1].value)
