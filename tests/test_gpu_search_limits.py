"""Alignment, decoding and lattice generation at the limits include/vbgpu.h states, each device result checked against
its float64 restatement (tests/align_ref.py, decode_ref.py, latgen_ref.py):
  * alignment: int16 / int32 traceback entries at 32 767 / 32 768 / 32 769 arcs and in a handle that mixes widths; the
    full 128 KiB of shared memory (4 096 states, 8 192 subset pdfs); 48 epsilon levels with negative weights and an
    epsilon tie; the create-time subset limit;
  * decoding: bench-like token counts on a 57 057-state graph; a token set of exactly max_tokens (and one more) on an
    86 130-state graph; more utterances in one call than a B200 keeps CTAs resident; padded log-likelihood rows with
    NaN in every column that holds no pdf;
  * lattices: the 57 057-state graph; the lattice store at its exact token and link capacities.
Every case also asserts, from the restatement's own outputs, that it reaches the edge it is named for; where that needs
no device the check is a test of its own."""
import numpy as np
import pytest

from tests.align_ref import _levels, align_subsets, viterbi_align_ref
from tests.decode_ref import beam_decode_ref
from tests.latgen_ref import LATTICE_KEYS, raw_lattice
from tests.test_gpu_align import create, pack, random_tiny_graph, ref_all, small_case, tid_costs
from tests.test_gpu_decode import batch, check_against_ref, decode_ll, device_loglikes, torch_dev
from tests.test_gpu_latgen import check_lattices, latgen_ll, same_one_best
from voicebridge_b200 import capi, host, synth

INF_ACTIVE = 2**31 - 1
RESIDENT_CTAS = 148 * 8  # a B200 keeps at most 8 CTAs of 256 threads on each of its 148 SMs


# ---------------------------------------------------------------------------------------------------------------------
# alignment
# ---------------------------------------------------------------------------------------------------------------------
def unpack(g):
    """The [(S, start, finals, arcs), ...] form of pack() from a packed graphs dict."""
    so, ao = g["state_offsets"], g["arc_offsets"]
    out = []
    for u in range(len(so) - 1):
        a = slice(int(ao[u]), int(ao[u + 1]))
        arcs = list(zip(g["arc_src"][a].tolist(), g["arc_dst"][a].tolist(), g["arc_ilabel"][a].tolist(),
                        g["arc_weight"][a].tolist()))
        out.append((int(so[u + 1] - so[u]), int(g["start"][u]), g["final_cost"][so[u]:so[u + 1]].tolist(), arcs))
    return out


def dense_utt(seed, A, num_tids, S=400, T=300):
    """A utterance of A arcs over S states whose best path is planned: first A - T filler arcs between random states
    with random transition-ids, of weight 10^6 (more than any acoustic or transition cost a path of T frames could
    save); then the chain 0 -> 1 -> ... -> T of weight-0 emitting arcs, the only way into the only final state T, so
    the path of T frames ends on the last arc, index A - 1."""
    rng = np.random.default_rng(seed)
    n = A - T
    fill = list(zip(rng.integers(0, S, n).tolist(), rng.integers(0, S, n).tolist(),
                    rng.integers(1, num_tids + 1, n).tolist(), [1e6] * n))
    chain = [(s, s + 1, int(rng.integers(1, num_tids + 1)), 0.0) for s in range(T)]
    finals = [np.inf] * S
    finals[T] = 0.0
    return (S, 0, finals, fill + chain), T


def deep_eps_utt(topo, n_lvls=48):
    """H (start, final) emits into A or B by two transition-ids of one pdf at one weight; B -> X and A -> X are epsilon
    arcs of equal weight, B -> X first in arc order although B is the higher state and its transition-id the higher one;
    X -> e_1 -> ... -> e_k -> H is an epsilon chain over n_lvls levels with weights alternating -0.5 / +1.0, every link
    doubled by a parallel arc of the same weight and every other link bypassed by an arc of the cost it skips.  Every
    frame goes H -> B -> X -> ... -> H, so ali is the B transition-id throughout.  Returns (utterance, A tid, B tid)."""
    ta, tb = sorted((topo["tid"][(2, 0, True)], topo["tid"][(2, 0, False)]))  # (one pdf: the state's loop and exit)
    H, A, B, X = 0, 1, 2, 3
    k = n_lvls - 2  # X is level 1, e_1 ... e_k levels 2 ... k + 1, H level k + 2 = n_lvls
    e = list(range(4, 4 + k))
    arcs = [(H, A, ta, 0.0), (H, B, tb, 0.0), (B, X, 0, 0.25), (A, X, 0, 0.25)]
    chain = [X] + e + [H]
    for i in range(len(chain) - 1):
        w = -0.5 if i % 2 == 0 else 1.0
        if i % 2 == 1 and i + 2 < len(chain):
            arcs.append((chain[i], chain[i + 2], 0, 0.5))  # a bypass before the two links it skips
        arcs += [(chain[i], chain[i + 1], 0, w), (chain[i], chain[i + 1], 0, w)]
    S = 4 + k
    return (S, H, [0.0] + [np.inf] * (S - 1), arcs), ta, tb


def chain_utt(n_states=4096):
    """A n_states-state chain: per state s a self-loop (tid 2s + 1) and a forward arc into s + 1 (tid 2s + 2; the last
    state's is a second loop); tid t reads pdf t - 1, except that the forward arc into the last state reads the largest
    pdf (subset column 2 n_states - 1).  Only the last state is final."""
    arcs = []
    for s in range(n_states):
        arcs.append((s, s, 2 * s + 1, 0.1))
        arcs.append((s, min(s + 1, n_states - 1), 2 * s + 2, 0.2))
    t2p = np.arange(-1, 2 * n_states, dtype=np.int32)
    t2p[0] = 0
    t2p[2 * n_states - 2], t2p[2 * n_states] = t2p[2 * n_states], t2p[2 * n_states - 2]
    finals = [np.inf] * n_states
    finals[-1] = 0.0
    return (n_states, 0, finals, arcs), t2p


def with_tids(utt, offset):
    S, start, finals, arcs = utt
    return S, start, finals, [(a, b, lab + offset if lab else 0, w) for a, b, lab, w in arcs]


def random_ll(rng, T, n):
    return rng.uniform(-80.0, -40.0, (T, n)).astype(np.float32)


def test_restatement_path_is_the_best_path():
    """viterbi_align_ref's path: a walk from the start state to a final state whose emitting arcs are ali and whose
    cost, summed in the search's operation order, is tot_cost (random tiny graphs, ties and epsilon arcs included)."""
    rng = np.random.default_rng(11)
    tid2pdf = np.array([0, 0, 1, 2, 1], np.int32)
    seen = 0
    for _ in range(150):
        g = pack([random_tiny_graph(rng, 4)])
        pdfs = align_subsets(g, tid2pdf)[0]
        ll = rng.choice([-1.0, -2.0, -3.5], size=(int(rng.integers(0, 7)), len(pdfs))).astype(np.float32)
        path = []
        cost, ali, _ = viterbi_align_ref(g, 0, ll, pdfs, tid2pdf, path=path)
        if cost == np.inf:
            assert path == []
            continue
        col = {int(p): i for i, p in enumerate(pdfs)}
        s, t, c = int(g["start"][0]), 0, 0.0
        for a in path:
            assert g["arc_src"][a] == s
            w, lab = float(g["arc_weight"][a]), int(g["arc_ilabel"][a])
            if lab:
                c = (c + w) + float(np.float32(-(np.float32(0.1) * ll[t, col[int(tid2pdf[lab])]])))
                assert ali[t] == lab
                t += 1
            else:
                c = c + w
            s = int(g["arc_dst"][a])
        assert t == len(ali) and c + float(g["final_cost"][s]) == cost
        seen += len(path) > 0
    assert seen > 50


@pytest.mark.parametrize("A", [32767, 32768, 32769])
def test_dense_path_ends_on_the_last_arc(A):
    """The planned path of dense_utt is the restatement's, on any log-likelihoods, and uses arc A - 1."""
    t2p = np.arange(0, 101, dtype=np.int32)
    utt, T = dense_utt(A, A, 100)
    g = pack([utt])
    assert int(g["arc_offsets"][-1]) == A
    pdfs = align_subsets(g, t2p)[0]
    for seed in range(2):
        path = []
        cost, ali, _ = viterbi_align_ref(g, 0, random_ll(np.random.default_rng(seed), T, len(pdfs)), pdfs, t2p,
                                         tid_cost=tid_costs(100, seed), path=path)
        assert np.isfinite(cost) and max(path) == path[-1] == A - 1
        assert ali.tolist() == [a[2] for a in utt[3][-T:]]


def test_deep_epsilon_levels_and_tie():
    topo = synth.phone_topology(40)
    utt, ta, tb = deep_eps_utt(topo)
    g = pack([utt])
    lab = g["arc_ilabel"]
    assert int(_levels(utt[0], g["arc_src"][lab == 0], g["arc_dst"][lab == 0]).max()) == 48
    t2p = np.zeros(len(topo["phone"]), np.int32)
    t2p[[ta, tb]] = 7
    ll = random_ll(np.random.default_rng(1), 30, 1)
    path = []
    cost, ali, _ = viterbi_align_ref(g, 0, ll, [7], t2p, path=path)
    assert np.isfinite(cost) and (ali == tb).all()  # the first arc in arc order, not the lower state or label
    assert sum(lab[a] == 0 for a in path) >= 30 * 24  # every frame runs the epsilon chain (bypasses skip <= half)


def test_chain_reaches_the_last_subset_column():
    utt, t2p = chain_utt()
    g = pack([utt])
    pdfs = align_subsets(g, t2p)[0]
    assert utt[0] == 4096 and len(pdfs) == 8192
    path = []
    cost, ali, pdf = viterbi_align_ref(g, 0, random_ll(np.random.default_rng(2), 4100, 8192), pdfs, t2p, path=path)
    assert np.isfinite(cost) and pdfs[8191] in pdf.tolist()
    assert g["arc_dst"][path[-1]] == 4095


def test_create_refuses_8193_subset_pdfs():
    """The subset limit is checked on the host before any device work; 8 192 pdfs and 4 096 states pass the checks."""
    utt, t2p = chain_utt()
    S, start, finals, arcs = utt
    g = pack([(S, start, finals, arcs + [(0, 0, len(t2p), 0.0)])])
    rc, msg = create(g, np.r_[t2p, 8192].astype(np.int32))
    assert rc == capi.ERR_INVALID and "reads 8193 distinct pdfs, more than the 8192" in msg, (rc, msg)
    rc, msg = create(pack([utt]), t2p)  # (the last error is only fresh when create fails: no device here)
    assert rc == 0 or (rc == capi.ERR_CUDA and "more than the" not in msg), (rc, msg)


@pytest.mark.gpu
def test_create_accepts_the_limits():
    utt, t2p = chain_utt()
    rc, msg = create(pack([utt]), t2p)
    assert rc == 0, msg


def check_align(g, t2p, am, X, fo, tc, scale):
    subs = align_subsets(g, t2p)
    want_cost, want_ali, want_pdf = ref_all(g, t2p, am.score_subset(X, fo, subs), subs, tc, scale)
    ali, pdf, cost = host.GmmAlignCompiledGpu(g, t2p).Align(am, X, fo, tid_cost=tc, acoustic_scale=scale)
    assert np.isfinite(cost).all()
    assert np.array_equal(ali, want_ali) and np.array_equal(pdf, want_pdf)
    assert np.abs(cost - want_cost).max() <= 1e-12 * np.abs(want_cost).max()
    return ali


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["A32767", "A32768", "A32769", "mixed"])
def test_traceback_width(case):
    """32 767 arcs: int16 entries; 32 768 and 32 769: int32 entries, the path on arc 32 767 / 32 768 (the first an int16
    entry would wrap to a negative 'no arc'); mixed: training graphs around a 32 769-arc utterance, all through the
    int32 kernels.  Both scorers, with and without transition costs."""
    fo0, g0, m, X0, _, _, _ = small_case(201, n_utts=6)
    t2p = g0["tid2pdf"]
    A = 32769 if case == "mixed" else int(case[1:])
    utt, T = dense_utt(A, A, len(t2p) - 1)
    rng = np.random.default_rng(A)
    if case == "mixed":
        train = unpack(g0)
        g = pack(train[:3] + [utt] + train[3:])
        lens = np.diff(fo0).tolist()
        fo = np.r_[0, np.cumsum(lens[:3] + [T] + lens[3:])].astype(np.int64)
        Xd = synth.make_feats(m, T, 202)
        X = np.concatenate([X0[:fo0[3]], Xd, X0[fo0[3]:]])
        wide = 3
    else:
        g, fo, X, wide = pack([utt]), np.array([0, T], np.int64), synth.make_feats(m, T, 203), 0
    assert int(g["arc_offsets"][wide + 1] - g["arc_offsets"][wide]) == A
    am = host.AmDiagGmmGpu.from_model(m)
    for kernel, with_tc, scale in ((0, False, 0.1), (0, True, 1.0), (1, True, 0.1), (1, False, 1.0)):
        am.set_kernel(kernel)
        tc = tid_costs(len(t2p) - 1, int(rng.integers(1000))) if with_tc else None
        ali = check_align(g, t2p, am, X, fo, tc, scale)
        subs = align_subsets(g, t2p)
        rows = slice(int(fo[wide]), int(fo[wide + 1]))
        path = []
        viterbi_align_ref(g, wide, am.score_subset(X[rows], [0, T], subs[wide:wide + 1])[0], subs[wide], t2p, tc, scale,
                          path=path)
        assert path[-1] == A - 1
        assert ali[rows].tolist() == [a[2] for a in utt[3][-T:]]


@pytest.mark.gpu
def test_shared_memory_at_the_maximum():
    """4 096 states and 8 192 subset pdfs (128 KiB of dynamic shared memory) next to a small training graph, in one
    group and then one utterance per group: identical results, equal to the restatement."""
    chain, t2p = chain_utt()
    fo0, g0, _, _, _, _, _ = small_case(211, n_utts=1)
    off = len(t2p) - 1
    g = pack([with_tids(unpack(g0)[0], off), chain])
    t2p = np.r_[t2p, g0["tid2pdf"][1:]].astype(np.int32)
    subs = align_subsets(g, t2p)
    assert g["state_offsets"][2] - g["state_offsets"][1] == 4096 and len(subs[1]) == 8192
    m = synth.make_model(9000, 18000, 39, 212)
    T0, T1 = int(fo0[1]), 4100
    fo = np.array([0, T0, T0 + T1], np.int64)
    X = synth.make_feats(m, int(fo[-1]), 213)
    am = host.AmDiagGmmGpu.from_model(m)
    blocks = am.score_subset(X, fo, subs)
    want_cost, want_ali, want_pdf = ref_all(g, t2p, blocks, subs)
    assert subs[1][8191] in want_pdf[T0:].tolist()  # the path reads the last subset column
    al = host.GmmAlignCompiledGpu(g, t2p)
    got = al.Align(am, X, fo)
    al.set_workspace(1)
    one = al.Align(am, X, fo)
    for a, b in zip(got, one):
        assert np.array_equal(a, b)
    ali, pdf, cost = got
    assert np.isfinite(cost).all()
    assert np.array_equal(ali, want_ali) and np.array_equal(pdf, want_pdf)
    assert np.abs(cost - want_cost).max() <= 1e-12 * np.abs(want_cost).max()


@pytest.mark.gpu
def test_deep_epsilon_levels():
    """48 epsilon levels with negative weights, parallel arcs and an equal-cost epsilon tie, between training graphs."""
    fo0, g0, m, X0, _, _, topo = small_case(221, n_utts=4)
    utt, ta, tb = deep_eps_utt(topo)
    train = unpack(g0)
    g = pack(train[:2] + [utt] + train[2:])
    t2p = g0["tid2pdf"]
    assert t2p[ta] == t2p[tb]
    T = 40
    lens = np.diff(fo0).tolist()
    fo = np.r_[0, np.cumsum(lens[:2] + [T] + lens[2:])].astype(np.int64)
    X = np.concatenate([X0[:fo0[2]], synth.make_feats(m, T, 222), X0[fo0[2]:]])
    am = host.AmDiagGmmGpu.from_model(m)
    for scale in (0.1, 1.0):
        ali = check_align(g, t2p, am, X, fo, None, scale)
        assert (ali[fo[2]:fo[3]] == tb).all()


# ---------------------------------------------------------------------------------------------------------------------
# decoding
# ---------------------------------------------------------------------------------------------------------------------
def model_for(m, kernel):
    am = host.AmDiagGmmGpu.from_model(m)
    try:
        am.set_kernel(kernel)
    except capi.VbgpuError:
        pytest.skip("scorer %d unavailable for this model" % kernel)
    return am


@pytest.fixture(scope="module")
def graph57k():
    """make_decoding_graph over 120 phones and 6 000 words: 57 057 states, 126 112 arcs."""
    g = synth.make_decoding_graph(synth.phone_topology(120), 6000, 2000, 5)
    return g, synth.make_model(2000, 8000, 39, 6)


def ref_with_stats(g, t2p, ll, fo, got, beam, max_active, max_tokens=65536):
    """check_against_ref's comparison, one utterance at a time, returning the restatement's set sizes per frame."""
    stats = []
    for u in range(len(fo) - 1):
        rows = slice(int(fo[u]), int(fo[u + 1]))
        st = []
        r = beam_decode_ref(g, ll[rows], t2p, 0.1, beam, max_active, max_tokens, stats=st)
        stats.append(np.array(st))
        ali, pdf, words, nw, tot, status = got
        assert status[u] == r[0] and np.array_equal(ali[rows], r[2]) and np.array_equal(pdf[rows], r[3]), u
        assert nw[u] == r[5] and words[u] == r[4][:64], u
        assert abs(tot[u] - r[1]) <= 1e-12 * max(abs(r[1]), 1.0) if np.isfinite(r[1]) else tot[u] == np.inf
    return stats


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", [1, 2])
def test_decode_at_bench_token_counts(graph57k, kernel):
    """Two utterances of 150 / 160 frames on the 57 057-state graph at beam 13 / max_active 7 000 and beam 16 /
    max_active 20 000: identical to the restatement, whose sets pass max_active on many frames (the radix select
    runs over thousands of keys)."""
    g, m = graph57k
    assert g["num_states"] == 57057 and len(g["arc_src"]) == 126112
    am = model_for(m, kernel)
    fo = np.array([0, 150, 310], np.int64)
    d_ll, ll = device_loglikes(am, synth.make_feats(m, int(fo[-1]), 7))
    for beam, max_active, min_over in ((13.0, 7000, 20), (16.0, 20000, 1)):
        dec = host.GmmDecodeFasterGpu(g, g["tid2pdf"], beam=beam, max_active=max_active)
        got = decode_ll(dec, am, d_ll, fo)
        st = np.concatenate(ref_with_stats(g, g["tid2pdf"], ll, fo, got, beam, max_active))
        assert (st > max_active).sum() >= min_over and st.max() > max_active, (beam, st.max())
        dec.close()


@pytest.fixture(scope="module")
def graph86k():
    """make_decoding_graph over 120 phones and 9 000 words: 86 130 states, more than the default 65 536 tokens."""
    g = synth.make_decoding_graph(synth.phone_topology(120), 9000, 2000, 5)
    return g, synth.make_model(2000, 8000, 39, 6)


CAP_FO = np.array([0, 6, 8, 10], np.int64)  # six frames, then two of two frames


def peak_sets(g, ll, fo):
    """Per utterance, the largest token set of the restatement at beam = +inf, the set after the last frame included
    (the stats of one frame more end with it)."""
    out = []
    for u in range(len(fo) - 1):
        rows = ll[int(fo[u]):int(fo[u + 1])]
        st = []
        beam_decode_ref(g, np.concatenate([rows, rows[-1:]]), g["tid2pdf"], 0.1, np.inf, INF_ACTIVE, 10**6, stats=st)
        out.append(max(st))
    return out


def test_capacity_case_passes_the_default():
    """At beam = +inf the sets do not depend on the log-likelihoods: the first utterance peaks between 65 536 and the
    state count, the others below its peak minus one."""
    g = synth.make_decoding_graph(synth.phone_topology(120), 9000, 2000, 5)
    ll = random_ll(np.random.default_rng(3), int(CAP_FO[-1]), 2000)
    M = peak_sets(g, ll, CAP_FO)
    assert 65536 < M[0] < g["num_states"] == 86130 and max(M[1:]) < M[0] - 1, M


@pytest.mark.gpu
def test_exact_token_capacity(graph86k):
    """max_tokens = M (the restatement's peak set) equals max_tokens >= S (the state-count capacity) and the
    restatement; M - 1 gives status 3 for that utterance only; so does the default 65 536 < M."""
    g, m = graph86k
    am = host.AmDiagGmmGpu.from_model(m)
    fo = CAP_FO
    d_ll, ll = device_loglikes(am, synth.make_feats(m, int(fo[-1]), 8))
    M = peak_sets(g, ll, fo)
    S = int(g["num_states"])
    assert 65536 < M[0] < S and max(M[1:]) < M[0] - 1, M

    def run(max_tokens):
        dec = host.GmmDecodeFasterGpu(g, g["tid2pdf"], beam=np.inf, max_tokens=max_tokens)
        out = decode_ll(dec, am, d_ll, fo)
        dec.close()
        return out

    full = run(S)
    assert (full[5] == 0).all()
    check_against_ref(g, g["tid2pdf"], ll, fo, full, np.inf, INF_ACTIVE, max_tokens=10**6)
    same_one_best(full, run(M[0]))
    for mt in (M[0] - 1, 65536):
        got = run(mt)
        assert got[5].tolist() == [3, 0, 0], mt
        assert np.isinf(got[4][0]) and got[3][0] == 0 and not got[0][:6].any() and (got[1][:6] == -1).all()
        rest = slice(int(fo[1]), int(fo[-1]))
        assert np.array_equal(got[0][rest], full[0][rest]) and np.array_equal(got[1][rest], full[1][rest])
        assert got[2][1:] == full[2][1:] and np.array_equal(got[3][1:], full[3][1:])
        assert np.array_equal(got[4][1:], full[4][1:])


@pytest.mark.gpu
def test_more_utterances_than_resident_ctas():
    """1 300 utterances of 0.5-1 s in one call and one group on the 2 667-state graph: a seeded 50 equal
    single-utterance calls, a seeded 10 equal the restatement."""
    g = synth.make_decoding_graph(synth.phone_topology(40), 300, 600, 7)
    m = synth.make_model(600, 2400, 39, 8)
    fo = batch(1300, 50, 100, 301)
    n = len(fo) - 1
    assert n > RESIDENT_CTAS
    am = host.AmDiagGmmGpu.from_model(m)
    d_ll, ll = device_loglikes(am, synth.make_feats(m, int(fo[-1]), 302))
    dec = host.GmmDecodeFasterGpu(g, g["tid2pdf"], beam=13.0, max_active=1000)
    dec.set_workspace(1 << 40)  # one group
    got = decode_ll(dec, am, d_ll, fo)
    ali, pdf, words, nw, tot, st = got
    rng = np.random.default_rng(303)

    def view(u):
        rows = slice(int(fo[u]), int(fo[u + 1]))
        return ali[rows], pdf[rows], [words[u]], nw[u:u + 1], tot[u:u + 1], st[u:u + 1]

    for u in rng.choice(n, 50, replace=False):
        one = decode_ll(dec, am, d_ll[int(fo[u]):int(fo[u + 1])], np.array([0, fo[u + 1] - fo[u]], np.int64))
        same_one_best(view(u), one)
    for u in rng.choice(n, 10, replace=False):
        rows = slice(int(fo[u]), int(fo[u + 1]))
        check_against_ref(g, g["tid2pdf"], ll[rows], np.array([0, fo[u + 1] - fo[u]]), view(u), 13.0, 1000)


def test_tensor_core_plan_has_columns_without_a_pdf():
    """The decode model's tensor-core layout has device-order columns that hold no pdf (what the padded test
    poisons inside NumCols)."""
    from tests.test_tc_layout import tc_layout
    lay, why = tc_layout(synth.make_model(600, 2400, 39, 8))
    assert lay is not None, why
    assert lay["n_cols"] > 600 and len(set(lay["col_of_pdf"].tolist())) == 600


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", [1, 2])
def test_padded_loglike_rows(kernel):
    """ll_stride = NumCols + 13 with NaN in every column that is no pdf's (device-order padding inside NumCols and the
    stride padding): outputs and lattices equal the clean call's, and no log-likelihood counts as bad."""
    torch, dev = torch_dev()
    g = synth.make_decoding_graph(synth.phone_topology(40), 300, 600, 7)
    m = synth.make_model(600, 2400, 39, 8)
    fo = batch(6, 20, 60, 9)
    am = model_for(m, kernel)
    d_ll, _ = device_loglikes(am, synth.make_feats(m, int(fo[-1]), 10))
    nc, P = am.NumCols(), am.NumPdfs()
    cols = torch.from_numpy(am.col_of_pdf().astype(np.int64)).to(dev)
    if kernel == 2:
        assert nc > P  # the tensor-core plan has non-pdf columns inside NumCols
    d_pad = torch.full((d_ll.shape[0], nc + 13), float("nan"), dtype=torch.float32, device=dev)
    d_pad[:, cols] = d_ll[:, cols]
    assert int(torch.isnan(d_pad).sum(1)[0]) == nc + 13 - P
    dec = host.GmmDecodeFasterGpu(g, g["tid2pdf"], beam=13.0, max_active=1000)
    lo = capi.default_lattice_opts(lattice_beam=6.0, max_states=1 << 15, max_arcs=1 << 17, arena_tokens=4096,
                                   arena_links=16384)
    want, want_lat = decode_ll(dec, am, d_ll, fo), latgen_ll(dec, am, d_ll, fo, lo)
    am.bad_count()
    same_one_best(want, decode_ll(dec, am, d_pad, fo))
    one, lats = latgen_ll(dec, am, d_pad, fo, lo)
    assert am.bad_count() == 0
    same_one_best(want, one)
    same_one_best(want_lat[0], one)
    for a, b in zip(want_lat[1], lats):
        assert a["lattice_status"] == b["lattice_status"] == 0 and a["num_states"] > 0
        for k in LATTICE_KEYS:
            assert np.array_equal(a[k].view(np.int32), b[k].view(np.int32)), k


# ---------------------------------------------------------------------------------------------------------------------
# lattices
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_lattice_at_bench_token_counts(graph57k):
    """One 150-frame utterance on the 57 057-state graph, beam 13 / max_active 7 000 / lattice beam 6: the lattice
    equals the restatement's array for array, and it has the bench's size (over a thousand states)."""
    g, m = graph57k
    am = host.AmDiagGmmGpu.from_model(m)
    fo = np.array([0, 150], np.int64)
    d_ll, ll = device_loglikes(am, synth.make_feats(m, 150, 9))
    dec = host.GmmDecodeFasterGpu(g, g["tid2pdf"], beam=13.0, max_active=7000)
    lo = capi.default_lattice_opts(lattice_beam=6.0, max_states=1 << 15, max_arcs=1 << 17)
    one, lats = latgen_ll(dec, am, d_ll, fo, lo)
    check_lattices(g, g["tid2pdf"], ll, fo, one, lats, 13.0, 7000, 6.0)
    assert one[5][0] == 0 and lats[0]["num_states"] > 1000 and lats[0]["num_arcs"] > 1000


def store_opts(tokens, links):
    return capi.default_lattice_opts(lattice_beam=6.0, max_states=1 << 15, max_arcs=1 << 17, arena_tokens=tokens,
                                     arena_links=links)


def start_closure_store(g):
    """Tokens and links of the start closure (a T = 0 utterance's whole store), from the restatement."""
    one, frames, links = raw_lattice(g, np.zeros((0, 600), np.float32), g["tid2pdf"], 0.1, 13.0, 7000)
    assert one[0] == 0 and len(frames) == 1
    return len(frames[0]), len(links)


def test_start_closure_store():
    g = synth.make_decoding_graph(synth.phone_topology(40), 300, 600, 7)
    K, KL = start_closure_store(g)
    assert K == 302 and KL == 301  # G, its 300 word entries and the silence entry; one link into each but G


@pytest.mark.gpu
def test_lattice_store_boundary():
    """arena_peak is the store's use: per utterance, arena_tokens = ceil(peak tokens / (T + 1)) writes the same
    lattice, one less ends it in lattice status 1 with the one-best outputs unchanged; likewise for links.  A T = 0
    utterance (NT = arena_tokens, NL = arena_links) meets both capacities with equality."""
    g = synth.make_decoding_graph(synth.phone_topology(40), 300, 600, 7)
    m = synth.make_model(600, 2400, 39, 8)
    fo = batch(6, 20, 60, 9)
    am = host.AmDiagGmmGpu.from_model(m)
    d_ll, ll = device_loglikes(am, synth.make_feats(m, int(fo[-1]), 10))
    dec = host.GmmDecodeFasterGpu(g, g["tid2pdf"], beam=13.0, max_active=7000)
    big = (4096, 16384)
    T1 = np.diff(fo) + 1
    one, lats = latgen_ll(dec, am, d_ll, fo, store_opts(*big))
    check_lattices(g, g["tid2pdf"], ll, fo, one, lats, 13.0, 7000, 6.0)
    peak = np.array([lt["arena_peak"] for lt in lats])
    assert (peak[:, 0] <= T1 * big[0]).all() and (peak[:, 1] <= T1 * big[1]).all()
    for which in (0, 1):
        need = -(-peak[:, which] // T1)  # per utterance, the least per-frame size that holds its store
        assert (need > 1).all()
        for a in sorted(set(need.tolist()) | set((need - 1).tolist())):
            sizes = list(big)
            sizes[which] = a
            o, lt = latgen_ll(dec, am, d_ll, fo, store_opts(*sizes))
            same_one_best(one, o)
            for u in range(len(fo) - 1):
                assert lt[u]["lattice_status"] == int(need[u] > a), (which, a, u)
                if need[u] <= a:
                    assert lt[u]["arena_peak"] == lats[u]["arena_peak"]
                    for k in LATTICE_KEYS:
                        assert np.array_equal(lt[u][k].view(np.int32), lats[u][k].view(np.int32)), (which, a, u, k)
                else:
                    assert lt[u]["num_states"] == 0
    # T = 0: the store holds the start closure's K tokens and KL links exactly
    K, KL = start_closure_store(g)
    fo0 = np.array([0, 0], np.int64)
    one0, l0 = latgen_ll(dec, am, d_ll, fo0, store_opts(*big))
    assert one0[5][0] == 0 and l0[0]["arena_peak"] == (K, KL)
    for tokens, links, status in ((K, KL, 0), (K - 1, KL, 1), (K, KL - 1, 1)):
        o, lt = latgen_ll(dec, am, d_ll, fo0, store_opts(tokens, links))
        same_one_best(one0, o)
        assert lt[0]["lattice_status"] == status, (tokens, links)
        if status == 0:
            for k in LATTICE_KEYS:
                assert np.array_equal(lt[0][k].view(np.int32), l0[0][k].view(np.int32)), k
