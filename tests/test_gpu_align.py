"""Forced alignment on the device (vbgpu_align_*, gmm-align-compiled): the float64 restatement tests/align_ref.py
viterbi_align_ref checked against brute-force path enumeration, create-time rejection of bad graphs (no GPU needed), and
on the GPU, through the C ABI, the device alignment against the restatement fed with the device's own subset
log-likelihoods (identical alignments), against the oracle's log-likelihoods, batching, streams, the host form, the
statistics chain and the error counts."""
import ctypes as C

import numpy as np
import pytest

from tests.align_ref import align_subsets, viterbi_align_ref
from tests.common import assert_acc_close
from voicebridge_b200 import capi, host, synth


def pack(utts):
    """Graphs dict from [(S, start, finals, [(src, dst, ilabel, weight), ...]), ...]."""
    so, ao, st, fin, arcs = [0], [0], [], [], []
    for S, start, finals, a in utts:
        so.append(so[-1] + S)
        st.append(start)
        fin += list(finals)
        arcs += list(a)
        ao.append(len(arcs))
    a = np.array(arcs, np.float64).reshape(-1, 4)
    return dict(state_offsets=np.array(so, np.int32), start=np.array(st, np.int32), final_cost=np.array(fin, np.float32),
                arc_offsets=np.array(ao, np.int64), arc_src=a[:, 0].astype(np.int32), arc_dst=a[:, 1].astype(np.int32),
                arc_ilabel=a[:, 2].astype(np.int32), arc_weight=a[:, 3].astype(np.float32))


def brute_force(g, u, ll, pdfs, tid2pdf, acoustic_scale):
    """Every path of utterance u, costed in the order of the semantics: (min cost, set of alignments reaching it)."""
    so, ao = g["state_offsets"], g["arc_offsets"]
    a0, a1 = int(ao[u]), int(ao[u + 1])
    final = g["final_cost"][so[u]:so[u + 1]].astype(np.float64)
    col = {int(p): i for i, p in enumerate(pdfs)}
    ac = (-(np.float32(acoustic_scale) * np.asarray(ll, np.float32))).astype(np.float32).astype(np.float64)
    T = ac.shape[0]
    out = []

    def walk(s, r, cost, ali):
        if r == T:
            out.append((cost + final[s], tuple(ali)))
        for a in range(a0, a1):
            if g["arc_src"][a] != s:
                continue
            d, lab, w = int(g["arc_dst"][a]), int(g["arc_ilabel"][a]), float(g["arc_weight"][a])
            if lab == 0:
                walk(d, r, cost + w, ali)
            elif r < T:
                walk(d, r + 1, (cost + w) + ac[r, col[int(tid2pdf[lab])]], ali + [lab])

    walk(int(g["start"][u]), 0, 0.0, [])
    best = min([c for c, _ in out], default=np.inf)
    return best, {a for c, a in out if c == best and best < np.inf}


def random_tiny_graph(rng, n_tids):
    S = int(rng.integers(2, 6))
    arcs = []
    for s in range(S):
        for _ in range(int(rng.integers(0, 3))):
            arcs.append((s, int(rng.integers(0, S)), int(rng.integers(1, n_tids + 1)), float(rng.choice([0.0, 0.5, 1.0]))))
        if s + 1 < S and rng.random() < 0.5:  # epsilon arcs go forward: no cycle
            arcs.append((s, int(rng.integers(s + 1, S)), 0, float(rng.choice([0.0, 0.5]))))
    finals = [float(rng.choice([np.inf, np.inf, 0.0, 0.5])) for _ in range(S)]
    return S, 0, finals, arcs


def test_restatement_equals_brute_force():
    """T <= 6, epsilon arcs, branches, ties (weights and log-likelihoods from tiny sets), unreachable finals, T = 0."""
    rng = np.random.default_rng(3)
    n_tids = 4
    tid2pdf = np.array([0, 0, 1, 2, 1], np.int32)  # tids 2 and 4 share pdf 1
    seen_inf = seen_tie = seen_t0 = 0
    for trial in range(150):
        g = pack([random_tiny_graph(rng, n_tids)])
        pdfs = align_subsets(g, tid2pdf)[0]
        T = int(rng.integers(0, 7))
        ll = rng.choice([-1.0, -2.0, -3.5], size=(T, len(pdfs))).astype(np.float32)
        for scale in (0.1, 1.0):
            cost, ali, pdf = viterbi_align_ref(g, 0, ll, pdfs, tid2pdf, acoustic_scale=scale)
            want, best_alis = brute_force(g, 0, ll, pdfs, tid2pdf, scale)
            assert cost == want, (trial, cost, want)
            if want == np.inf:
                seen_inf += 1
                assert not ali.any() and (pdf == -1).all()
            else:
                assert tuple(ali) in best_alis
                assert np.array_equal(pdf, tid2pdf[ali])
                seen_tie += len(best_alis) > 1
            seen_t0 += T == 0
    assert seen_inf and seen_tie and seen_t0


def test_restatement_tie_rules():
    """Equal-cost predecessors: the first arc in arc order; an epsilon arc only when strictly lower."""
    tid2pdf = np.array([0, 0, 0], np.int32)  # both tids read pdf 0: equal acoustic cost
    g = pack([(2, 0, [np.inf, 0.0], [(0, 1, 2, 0.0), (0, 1, 1, 0.0)])])
    assert viterbi_align_ref(g, 0, np.full((1, 1), -1.0, np.float32), [0], tid2pdf)[1].tolist() == [2]
    # state 1 reached by emission (tid 1) at cost 0.1 and by emission (tid 2) into 2, then epsilon 2 -> 1 at the same cost
    g = pack([(3, 0, [np.inf, 0.0, np.inf], [(0, 2, 2, 0.0), (2, 1, 0, 0.1), (0, 1, 1, 0.1)])])
    assert viterbi_align_ref(g, 0, np.full((1, 1), -1.0, np.float32), [0], tid2pdf)[1].tolist() == [1]


def create(g, tid2pdf):
    h = C.c_void_p()
    keys = ("state_offsets", "start", "final_cost", "arc_offsets", "arc_src", "arc_dst", "arc_ilabel", "arc_weight")
    rc = capi.lib().vbgpu_align_create(len(g["start"]), *(g[k].ctypes.data for k in keys), tid2pdf.ctypes.data,
                                       len(tid2pdf) - 1, 0, C.byref(h))
    if rc == 0:
        capi.lib().vbgpu_align_destroy(h)
    return rc, capi.lib().vbgpu_last_error().decode()


@pytest.mark.parametrize("case", ["dst", "ilabel", "eps_cycle", "states", "tid2pdf"])
def test_create_rejects_bad_graphs(case):
    """Invalid graphs are rejected on the host before any device work (so with or without a GPU)."""
    tid2pdf = np.array([0, 0, 1], np.int32)
    ok = [(0, 1, 1, 0.0), (1, 2, 0, 0.0), (2, 2, 2, 0.0)]
    g = pack([(3, 0, [np.inf, np.inf, 0.0], ok)])
    assert create(g, tid2pdf)[0] in (0, capi.ERR_CUDA)  # the valid graph passes the checks
    want = {"dst": "outside the utterance", "ilabel": "ilabel 3 outside", "eps_cycle": "cycle", "states": "more than the 4096",
            "tid2pdf": "negative"}[case]
    if case == "dst":
        g = pack([(3, 0, [np.inf, np.inf, 0.0], ok + [(2, 3, 1, 0.0)])])
    elif case == "ilabel":
        g = pack([(3, 0, [np.inf, np.inf, 0.0], ok + [(2, 0, 3, 0.0)])])
    elif case == "eps_cycle":
        g = pack([(3, 0, [np.inf, np.inf, 0.0], ok + [(2, 1, 0, 0.0)])])
    elif case == "states":
        g = pack([(3, 0, [np.inf, np.inf, 0.0], ok), (4097, 0, [0.0] * 4097, [(0, 1, 1, 0.0)])])
    else:
        tid2pdf = np.array([0, 0, -1], np.int32)
    rc, msg = create(g, tid2pdf)
    assert rc == capi.ERR_INVALID, (rc, msg)
    assert want in msg, msg


# ---------------------------------------------------------------------------------------------------------------------
# on the device
# ---------------------------------------------------------------------------------------------------------------------
def corpus(n_utts, lo_s, hi_s, seed, n_phones=200):
    rng = np.random.default_rng(seed)
    lens = (rng.uniform(lo_s, hi_s, n_utts) * 100).astype(np.int64)
    fo = np.zeros(n_utts + 1, np.int64)
    fo[1:] = np.cumsum(lens)
    topo, tids, seqs = synth.make_phone_alignment(n_phones, fo, seed + 1)
    return fo, topo, tids, seqs


def ref_all(g, tid2pdf, blocks, subs, tid_cost=None, scale=0.1):
    res = [viterbi_align_ref(g, u, blocks[u], subs[u], tid2pdf, tid_cost, scale) for u in range(len(subs))]
    return (np.array([r[0] for r in res]), np.concatenate([r[1] for r in res]), np.concatenate([r[2] for r in res]))


def tid_costs(num_tids, seed):
    return np.random.default_rng(seed).uniform(0.0, 3.0, num_tids + 1).astype(np.float32)


@pytest.fixture(scope="module")
def cfg3():
    """64 utterances of 5-20 s, the cfg 3 model (P = 4000, N = 40000, D = 39), graphs over 200 phones."""
    fo, topo, tids, seqs = corpus(64, 5.0, 20.0, 41)
    g = synth.make_training_graphs(topo, seqs, 4000, 42)
    m = synth.make_model(4000, 40000, 39, 43)
    X = synth.make_feats(m, int(fo[-1]), 44)
    return fo, g, m, X


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,with_tc,scale", [(0, False, 0.1), (0, True, 1.0), (1, True, 0.1), (1, False, 1.0)])
def test_exact_agreement_with_restatement(cfg3, kernel, with_tc, scale):
    """The restatement on the device's own subset log-likelihoods: identical alignments, tot_cost to 1e-12 relative."""
    fo, g, m, X = cfg3
    tid2pdf = g["tid2pdf"]
    am = host.AmDiagGmmGpu.from_model(m)
    am.set_kernel(kernel)
    subs = align_subsets(g, tid2pdf)
    blocks = am.score_subset(X, fo, subs)
    tc = tid_costs(g["num_tids"], 5) if with_tc else None
    want_cost, want_ali, want_pdf = ref_all(g, tid2pdf, blocks, subs, tc, scale)
    al = host.GmmAlignCompiledGpu(g, tid2pdf)
    ali, pdf, cost = al.Align(am, X, fo, tid_cost=tc, acoustic_scale=scale)
    assert np.isfinite(cost).all()
    assert np.array_equal(ali, want_ali)
    assert np.array_equal(pdf, want_pdf)
    assert np.abs(cost - want_cost).max() <= 1e-12 * np.abs(want_cost).max()


@pytest.mark.gpu
def test_against_oracle(orc):
    """The device path re-costed with the oracle's log-likelihoods is within acoustic_scale * 1e-3 * T_u of the optimum
    the restatement finds on those log-likelihoods (the log-likelihood tolerance carried along the path)."""
    fo, topo, tids, seqs = corpus(12, 1.0, 4.0, 51, n_phones=60)
    g = synth.make_training_graphs(topo, seqs, 1000, 52)
    tid2pdf = g["tid2pdf"]
    m = synth.make_model(1000, 8000, 39, 53)
    X = synth.make_feats(m, int(fo[-1]), 54)
    rc, dense = orc.gmm_loglikes(m, X)
    assert rc == 0
    am = host.AmDiagGmmGpu.from_model(m)
    subs = align_subsets(g, tid2pdf)
    dev_blocks = am.score_subset(X, fo, subs)
    for scale in (0.1, 1.0):
        ali, pdf, cost = host.GmmAlignCompiledGpu(g, tid2pdf).Align(am, X, fo, acoustic_scale=scale)
        for u in range(len(subs)):
            rows = slice(int(fo[u]), int(fo[u + 1]))
            T = int(fo[u + 1] - fo[u])
            col = {int(p): i for i, p in enumerate(subs[u])}
            c = [col[int(p)] for p in pdf[rows]]

            def ac(blk):
                return float(np.sum((-(np.float32(scale) * blk[np.arange(T), c])).astype(np.float32), dtype=np.float64))
            recost = cost[u] - ac(dev_blocks[u]) + ac(dense[rows][:, subs[u]].astype(np.float32))
            best = viterbi_align_ref(g, u, dense[rows][:, subs[u]], subs[u], tid2pdf, acoustic_scale=scale)[0]
            assert recost >= best - 1e-6 * abs(best)
            assert recost - best <= scale * 1e-3 * T, (u, recost, best)


@pytest.mark.gpu
def test_recovers_generating_alignment():
    """Features drawn along a known alignment from a well-separated model: the device alignment is the generating one on
    at least 99 % of the frames."""
    fo, topo, tids, seqs = corpus(16, 2.0, 6.0, 61, n_phones=50)
    g = synth.make_training_graphs(topo, seqs, 200, 62)
    tid2pdf = g["tid2pdf"]
    m = synth.make_model(200, 200, 39, 63, spread=3.0)
    pdf_true = tid2pdf[tids]
    rng = np.random.default_rng(64)
    X = (m.means[pdf_true] + np.sqrt(1.0 / m.iv[pdf_true]) * rng.standard_normal((len(tids), 39))).astype(np.float32)
    am = host.AmDiagGmmGpu.from_model(m)
    ali, pdf, cost = host.GmmAlignCompiledGpu(g, tid2pdf).Align(am, X, fo)
    assert np.isfinite(cost).all()
    assert (ali == tids).mean() >= 0.99, (ali == tids).mean()


def small_case(seed, n_utts=6, lo=0.5, hi=3.0, n_phones=40, P=300):
    fo, topo, tids, seqs = corpus(n_utts, lo, hi, seed, n_phones)
    g = synth.make_training_graphs(topo, seqs, P, seed + 1)
    m = synth.make_model(P, 4 * P, 39, seed + 2)
    X = synth.make_feats(m, int(fo[-1]), seed + 3)
    return fo, g, m, X, tids, seqs, topo


@pytest.mark.gpu
def test_graph_cases():
    """An unreachable final state (+inf, zero / -1 rows, neighbours unaffected), a T = 0 utterance, an exact tie."""
    fo, g, m, X, tids, seqs, topo = small_case(71)
    # utterance 2 loses its final states; an empty utterance (T = 0, empty transcript) is appended
    g2 = synth.make_training_graphs(topo, seqs + [[]], 300, 72)
    g2["final_cost"][g2["state_offsets"][2]:g2["state_offsets"][3]] = np.inf
    fo2 = np.r_[fo, fo[-1]]
    tid2pdf = g2["tid2pdf"]
    am = host.AmDiagGmmGpu.from_model(m)
    subs = align_subsets(g2, tid2pdf)
    blocks = am.score_subset(X, fo2, subs)
    ali, pdf, cost = host.GmmAlignCompiledGpu(g2, tid2pdf).Align(am, X, fo2)
    want_cost, want_ali, want_pdf = ref_all(g2, tid2pdf, blocks, subs)
    assert cost[2] == np.inf and np.isfinite(np.delete(cost, 2)).all()
    rows = slice(int(fo2[2]), int(fo2[3]))
    assert not ali[rows].any() and (pdf[rows] == -1).all()
    assert np.array_equal(ali, want_ali) and np.array_equal(pdf, want_pdf)
    assert np.array_equal(cost == np.inf, want_cost == np.inf)
    fin = np.isfinite(want_cost)
    assert np.abs(cost[fin] - want_cost[fin]).max() <= 1e-12 * np.abs(want_cost[fin]).max()
    # T = 0: start -eps-> J -eps(-log 0.5)-> pre (final 0.5) -eps-> end (final 0)
    assert cost[-1] == float(np.float32(-np.log(0.5)))
    # exact tie: two arcs of equal cost into one state, tids reading the same pdf; the first in arc order wins
    tie_t2p = np.array([0, 5, 5], np.int32)
    gt = pack([(2, 0, [np.inf, 0.0], [(0, 1, 2, 0.0), (0, 1, 1, 0.0)]), (2, 0, [np.inf, 0.0], [(0, 1, 1, 0.0), (0, 1, 2, 0.0)])])
    ali, pdf, cost = host.GmmAlignCompiledGpu(gt, tie_t2p).Align(am, X[[0, 0]], [0, 1, 2])
    assert ali.tolist() == [2, 1] and pdf.tolist() == [5, 5] and cost[0] == cost[1]


@pytest.mark.gpu
def test_batching_groups_streams_and_host_form():
    import torch
    fo, g, m, X, tids, seqs, topo = small_case(81, n_utts=10)
    tid2pdf = g["tid2pdf"]
    am = host.AmDiagGmmGpu.from_model(m)
    tc = tid_costs(g["num_tids"], 8)
    al = host.GmmAlignCompiledGpu(g, tid2pdf)
    ali, pdf, cost = al.Align(am, X, fo, tid_cost=tc)
    # the batch equals the concatenation of single-utterance calls
    for u in range(len(fo) - 1):
        one = {k: v for k, v in g.items()}
        so, ao = g["state_offsets"], g["arc_offsets"]
        one.update(state_offsets=np.array([0, so[u + 1] - so[u]], np.int32), start=g["start"][u:u + 1],
                   final_cost=g["final_cost"][so[u]:so[u + 1]], arc_offsets=np.array([0, ao[u + 1] - ao[u]], np.int64),
                   **{k: g[k][ao[u]:ao[u + 1]] for k in ("arc_src", "arc_dst", "arc_ilabel", "arc_weight")})
        rows = slice(int(fo[u]), int(fo[u + 1]))
        a1, p1, c1 = host.GmmAlignCompiledGpu(one, tid2pdf).Align(am, X[rows], [0, fo[u + 1] - fo[u]], tid_cost=tc)
        assert np.array_equal(a1, ali[rows]) and np.array_equal(p1, pdf[rows]) and c1[0] == cost[u]
    # a cap that forces several groups (one utterance each at 1 byte) gives the same results as one group
    for cap in (1, 200_000):
        al.set_workspace(cap)
        a2, p2, c2 = al.Align(am, X, fo, tid_cost=tc)
        assert np.array_equal(a2, ali) and np.array_equal(p2, pdf) and np.array_equal(c2, cost)
    al.set_workspace(0)
    # two streams on one handle, back to back, equal the host form
    dev = torch.device("cuda", 0)
    d_x = torch.from_numpy(X).to(dev)
    T, n = int(fo[-1]), len(fo) - 1
    outs = [(torch.zeros(T, dtype=torch.int32, device=dev), torch.zeros(T, dtype=torch.int32, device=dev),
             torch.zeros(n, dtype=torch.float64, device=dev)) for _ in range(2)]
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    al.align_dev(am, d_x, 39, fo, *outs[0], tid_cost=tc, stream=sa)
    al.align_dev(am, d_x, 39, fo, *outs[1], tid_cost=tc, stream=sb)
    torch.cuda.synchronize()
    for a, p, c in outs:
        assert np.array_equal(a.cpu().numpy(), ali) and np.array_equal(p.cpu().numpy(), pdf)
        assert np.array_equal(c.cpu().numpy(), cost)


@pytest.mark.gpu
def test_chain_into_accumulation():
    """d_pdf_ids / d_ali of vbgpu_align_dev feed vbgpu_acc_accumulate_dev / _transitions_dev: the statistics equal those
    of the restatement's alignment."""
    import torch
    fo, g, m, X, tids, seqs, topo = small_case(91, n_utts=8)
    tid2pdf = g["tid2pdf"]
    am = host.AmDiagGmmGpu.from_model(m)
    subs = align_subsets(g, tid2pdf)
    want_cost, want_ali, want_pdf = ref_all(g, tid2pdf, am.score_subset(X, fo, subs), subs)
    dev = torch.device("cuda", 0)
    d_x = torch.from_numpy(X).to(dev)
    T = int(fo[-1])
    d_ali, d_pdf = torch.zeros(T, dtype=torch.int32, device=dev), torch.zeros(T, dtype=torch.int32, device=dev)
    d_cost = torch.zeros(len(fo) - 1, dtype=torch.float64, device=dev)
    s = torch.cuda.current_stream()
    host.GmmAlignCompiledGpu(g, tid2pdf).align_dev(am, d_x, 39, fo, d_ali, d_pdf, d_cost, stream=s)
    a = host.AccumAmDiagGmmGpu(am, num_tids=g["num_tids"])
    a.accumulate_dev(d_x, T, 39, d_pdf, stream=s)
    a.accumulate_transitions_dev(d_ali, T, stream=s)
    b = host.AccumAmDiagGmmGpu(am, num_tids=g["num_tids"])
    b.AccumulateForUtterance(X, want_pdf)
    b.AccumulateTransitions(want_ali)
    torch.cuda.synchronize()
    assert np.array_equal(a.transition_accs(), b.transition_accs())
    da, db = a.download(), b.download()
    assert_acc_close(da[:3], db[:3])
    assert da[4] == db[4] == T
    assert am.bad_count() == 0


@pytest.mark.gpu
def test_no_leaks_and_error_counts():
    import torch
    before = C.c_int64(), C.c_int64()
    capi.lib().vbgpu_debug_live_bytes(C.byref(before[0]), C.byref(before[1]))
    fo, g, m, X, tids, seqs, topo = small_case(101, n_utts=4)
    am = host.AmDiagGmmGpu.from_model(m)
    al = host.GmmAlignCompiledGpu(g, g["tid2pdf"])
    al.Align(am, X, fo)
    Xbad = X.copy()
    Xbad[5] = np.nan
    with pytest.raises(capi.VbgpuError) as e:
        al.Align(am, Xbad, fo)
    assert e.value.code == capi.ERR_NUMERIC
    assert am.bad_count() == 0  # the host form counts in a slot of its own
    dev = torch.device("cuda", 0)
    T = int(fo[-1])
    outs = (torch.zeros(T, dtype=torch.int32, device=dev), None, torch.zeros(len(fo) - 1, dtype=torch.float64, device=dev))
    al.align_dev(am, torch.from_numpy(Xbad).to(dev), 39, fo, *outs)
    assert am.bad_count() > 0
    with pytest.raises(capi.VbgpuError):  # frame offsets of another batch size
        al.Align(am, X, fo[:-1])
    small = host.AmDiagGmmGpu.from_model(synth.make_model(10, 20, 39, 1))
    with pytest.raises(capi.VbgpuError):  # tid2pdf beyond the model's pdfs
        al.Align(small, X, fo)
    del outs
    for h in (al, am, small):
        h.close()
    after = C.c_int64(), C.c_int64()
    capi.lib().vbgpu_debug_live_bytes(C.byref(after[0]), C.byref(after[1]))
    assert (after[0].value, after[1].value) == (before[0].value, before[1].value)
