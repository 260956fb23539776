"""The float64 restatement of one-best decoding (tests/decode_ref.py beam_decode_ref) without a GPU: against brute-force
path enumeration and viterbi_align_ref at beam = +inf, against a plain pull-form token-passing loop written from the
header text at finite beams, the synthetic decoding graph and its path sampler, and the create-time checks."""
import ctypes as C

import numpy as np
import pytest

from tests.align_ref import _levels, viterbi_align_ref
from tests.decode_ref import beam_decode_ref
from voicebridge_b200 import capi, synth

INF_ACTIVE = 2**31 - 1


def tiny_graph(rng, n_tids, neg=False):
    S = int(rng.integers(2, 7))
    arcs = []
    for s in range(S):
        for _ in range(int(rng.integers(0, 3))):
            arcs.append((s, int(rng.integers(0, S)), int(rng.integers(1, n_tids + 1)), int(rng.integers(0, 3)),
                         float(rng.choice([0.0, 0.5, 1.0]))))
        for _ in range(int(rng.integers(0, 2))):
            if s + 1 < S:  # epsilon arcs go forward: no cycle
                arcs.append((s, int(rng.integers(s + 1, S)), 0, int(rng.integers(0, 3)),
                             float(rng.choice([-0.5, 0.0, 0.5] if neg else [0.0, 0.5]))))
    a = np.array(arcs, np.float64).reshape(-1, 5)
    return dict(num_states=S, start=0, final_cost=np.array([rng.choice([np.inf, np.inf, 0.0, 0.5]) for _ in range(S)],
                                                           np.float32),
                arc_src=a[:, 0].astype(np.int32), arc_dst=a[:, 1].astype(np.int32), arc_ilabel=a[:, 2].astype(np.int32),
                arc_olabel=a[:, 3].astype(np.int32), arc_weight=a[:, 4].astype(np.float32))


def brute_force(g, ll, tid2pdf, scale):
    """Every path, costed in the order of the semantics: (min cost + final, {(ali, words) reaching it})."""
    ac = (-(np.float32(scale) * np.asarray(ll, np.float32))).astype(np.float32).astype(np.float64)
    T = ac.shape[0]
    out = []

    def walk(s, r, cost, ali, words):
        if r == T and g["final_cost"][s] < np.inf:
            out.append((cost + float(g["final_cost"][s]), tuple(ali), tuple(words)))
        for a in range(len(g["arc_src"])):
            if g["arc_src"][a] != s:
                continue
            d, lab, w = int(g["arc_dst"][a]), int(g["arc_ilabel"][a]), float(g["arc_weight"][a])
            o = [int(g["arc_olabel"][a])] if g["arc_olabel"][a] else []
            if lab == 0:
                walk(d, r, cost + w, ali, words + o)
            elif r < T:
                walk(d, r + 1, (cost + w) + ac[r, tid2pdf[lab]], ali + [lab], words + o)

    walk(int(g["start"]), 0, 0.0, [], [])
    best = min([c for c, _, _ in out], default=np.inf)
    return best, {(a, w) for c, a, w in out if c == best and best < np.inf}


def as_align_graphs(g):
    S = int(g["num_states"])
    return dict(state_offsets=np.array([0, S], np.int32), start=np.array([g["start"]], np.int32),
                final_cost=g["final_cost"], arc_offsets=np.array([0, len(g["arc_src"])], np.int64),
                arc_src=g["arc_src"], arc_dst=g["arc_dst"], arc_ilabel=g["arc_ilabel"], arc_weight=g["arc_weight"])


def test_exact_search_equals_brute_force_and_align():
    """beam = +inf, unlimited max_active: the cost of brute force, one of its best (alignment, words), and the result of
    viterbi_align_ref on the same graph (cost and alignment)."""
    rng = np.random.default_rng(11)
    tid2pdf = np.array([0, 0, 1, 2, 1], np.int32)
    seen = dict(final=0, partial=0, tie=0, t0=0)
    for trial in range(200):
        g = tiny_graph(rng, 4, neg=trial % 2 == 1)
        T = int(rng.integers(0, 6))
        ll = rng.choice([-1.0, -2.0, -3.5], size=(T, 3)).astype(np.float32)
        st, cost, ali, pdf, words, nw = beam_decode_ref(g, ll, tid2pdf, 1.0, np.inf)
        want, best = brute_force(g, ll, tid2pdf, 1.0)
        if st == 0:
            seen["final"] += 1
            assert cost == want, (trial, cost, want)
            assert (tuple(ali), tuple(words)) in best
            assert np.array_equal(pdf, tid2pdf[ali]) and nw == len(words)
            seen["tie"] += len(best) > 1
            a_cost, a_ali, _ = viterbi_align_ref(as_align_graphs(g), 0, ll, [0, 1, 2], tid2pdf, acoustic_scale=1.0)
            assert a_cost == cost and np.array_equal(a_ali, ali)
        else:
            assert want == np.inf
            seen["partial"] += st == 1
            if st == 2:
                assert not ali.any() and (pdf == -1).all() and nw == 0
        seen["t0"] += T == 0
    assert all(seen.values()), seen


def token_passing(g, ll, tid2pdf, scale, beam, max_active, max_tokens):
    """The header's steps 1-6 as a pull-form loop over states and arcs in arc order (strict <), independent of
    beam_decode_ref's push form: returns (status, cost, ali, words)."""
    S = int(g["num_states"])
    src, dst, lab, ol = g["arc_src"], g["arc_dst"], g["arc_ilabel"], g["arc_olabel"]
    w = g["arc_weight"].astype(np.float64)
    emit = lab > 0
    level = _levels(S, src[~emit], dst[~emit])
    beam = float(np.float32(beam))

    def close(tok, cut):
        for lv in range(1, int(level.max(initial=0)) + 1):
            for s in range(S):
                if level[s] != lv:
                    continue
                best = tok.get(s)
                for a in range(len(src)):
                    if dst[a] != s or emit[a] or src[a] not in tok or not tok[src[a]][0] < cut:
                        continue
                    v = tok[src[a]][0] + w[a]
                    if v < np.inf and (best is None or v < best[0]):
                        best = (v, tok[src[a]][1] + [a])
                if best is not None:
                    tok[s] = best
            if len(tok) > max_tokens:
                return False
        return True

    tok = {int(g["start"]): (0.0, [])}
    ok = close(tok, np.inf)
    T = ll.shape[0]
    for t in range(T if ok else 0):
        cs = sorted(c for c, _ in tok.values())
        cut = cs[0] + beam
        if len(cs) > max_active:
            cut = min(cut, cs[max_active])
        keep = {s: v for s, v in tok.items() if v[0] < cut or v[0] == cs[0]}
        if len(keep) > max_active:
            return 3, np.inf, None, None
        ac = (-(np.float32(scale) * ll[t])).astype(np.float32).astype(np.float64)
        new = {}
        for s in range(S):
            for a in range(len(src)):
                if dst[a] == s and emit[a] and src[a] in keep:
                    v = (keep[src[a]][0] + w[a]) + ac[tid2pdf[lab[a]]]
                    if v < np.inf and (s not in new or v < new[s][0]):
                        new[s] = (v, keep[src[a]][1] + [a])
        if len(new) > max_tokens:
            return 3, np.inf, None, None
        if not new:
            return 2, np.inf, None, None
        tok = new
        if not close(tok, min(c for c, _ in tok.values()) + beam):
            return 3, np.inf, None, None
    if not ok:
        return 3, np.inf, None, None
    fin = [(c + float(g["final_cost"][s]), s) for s, (c, _) in tok.items() if g["final_cost"][s] < np.inf]
    st = 0 if fin else 1
    cost, s = min(fin) if fin else min((c, s) for s, (c, _) in tok.items())
    path = np.array(tok[s][1], np.int64)
    return st, cost, lab[path][emit[path]], [int(o) for o in ol[path] if o]


@pytest.mark.parametrize("beam,max_active", [(np.inf, INF_ACTIVE), (2.0, INF_ACTIVE), (1.0, 3), (0.5, 2), (8.0, 1),
                                             (1.5, 1)])
def test_beam_search_equals_token_passing(beam, max_active):
    """Finite beams and max_active, tied best tokens, ties at the max_active boundary, negative epsilon weights,
    epsilon olabels, small max_tokens."""
    rng = np.random.default_rng(int(min(beam, 99.0) * 10) + max_active % 97)
    tid2pdf = np.array([0, 0, 1, 2, 1], np.int32)
    statuses = set()
    for trial in range(150):
        g = tiny_graph(rng, 4, neg=True)
        T = int(rng.integers(0, 6))
        ll = rng.choice([-1.0, -2.0], size=(T, 3)).astype(np.float32)  # few distinct values: many ties
        max_tokens = int(rng.choice([2, 3, 100]))
        st, cost, ali, pdf, words, nw = beam_decode_ref(g, ll, tid2pdf, 1.0, beam, max_active, max_tokens)
        st2, cost2, ali2, words2 = token_passing(g, ll, tid2pdf, 1.0, beam, max_active, max_tokens)
        statuses.add(st)
        assert (st, cost) == (st2, cost2), trial
        if st <= 1:
            assert np.array_equal(ali, ali2) and words == words2, trial
    assert {0, 3} <= statuses, statuses


def test_tie_rules():
    """Equal emitting costs: the lowest arc; an epsilon arc only when strictly lower; equal epsilon candidates: the
    lowest arc; tied final costs: the lowest state."""
    t2p = np.array([0, 0, 0], np.int32)
    base = dict(num_states=3, start=0)
    g = dict(base, final_cost=np.array([np.inf, 0.0, 0.0], np.float32), arc_src=np.array([0, 0, 0], np.int32),
             arc_dst=np.array([2, 1, 1], np.int32), arc_ilabel=np.array([1, 2, 1], np.int32),
             arc_olabel=np.array([7, 8, 9], np.int32), arc_weight=np.zeros(3, np.float32))
    st, cost, ali, pdf, words, nw = beam_decode_ref(g, np.full((1, 1), -1.0, np.float32), t2p, 1.0)
    assert (st, ali.tolist(), words) == (0, [2], [8])  # states 1 and 2 tie on cost + final: state 1; into 1: arc 1
    g = dict(base, final_cost=np.array([np.inf, 0.0, np.inf], np.float32), arc_src=np.array([0, 2, 2, 0], np.int32),
             arc_dst=np.array([2, 1, 1, 1], np.int32), arc_ilabel=np.array([1, 0, 0, 2], np.int32),
             arc_olabel=np.array([0, 5, 6, 7], np.int32), arc_weight=np.array([0.0, 0.0, 0.0, 0.0], np.float32))
    assert beam_decode_ref(g, np.full((1, 1), -1.0, np.float32), t2p, 1.0)[4] == [7]  # emitting keeps an equal cost
    g["arc_weight"] = np.array([0.0, 0.0, 0.0, 0.5], np.float32)
    assert beam_decode_ref(g, np.full((1, 1), -1.0, np.float32), t2p, 1.0)[4] == [5]  # lower epsilon arc wins the tie


def test_synthetic_graph_and_sampled_paths():
    topo = synth.phone_topology(30)
    g = synth.make_decoding_graph(topo, 200, 500, 5)
    S = g["num_states"]
    emit = g["arc_ilabel"] > 0
    level = _levels(S, g["arc_src"][~emit], g["arc_dst"][~emit])
    assert level is not None and level.max() >= 3
    assert (g["arc_weight"][~emit] < 0).any()
    assert (g["arc_olabel"][~emit] > 0).any() and (g["arc_olabel"][emit] > 0).any()
    assert (g["final_cost"] < np.inf).sum() >= 2
    for seed in range(20):
        words, tids, arcs = synth.sample_decoding_path(g, seed, 50)
        s = int(g["start"])
        for a in arcs:
            assert g["arc_src"][a] == s
            s = int(g["arc_dst"][a])
        assert g["final_cost"][s] < np.inf and len(tids) >= 50
        assert np.array_equal(tids, g["arc_ilabel"][arcs][g["arc_ilabel"][arcs] > 0])
        assert words == [int(o) for o in g["arc_olabel"][arcs] if o]


def create(g, tid2pdf):
    h = C.c_void_p()
    keys = ("arc_src", "arc_dst", "arc_ilabel", "arc_olabel", "arc_weight")
    rc = capi.lib().vbgpu_decoder_create(int(g["num_states"]), int(g["start"]), g["final_cost"].ctypes.data,
                                         len(g["arc_src"]), *(g[k].ctypes.data for k in keys), tid2pdf.ctypes.data,
                                         len(tid2pdf) - 1, 0, C.byref(h))
    if rc == 0:
        capi.lib().vbgpu_decoder_destroy(h)
    return rc, capi.lib().vbgpu_last_error().decode()


def small(arcs, S=3, start=0, finals=(np.inf, np.inf, 0.0)):
    a = np.array(arcs, np.float64).reshape(-1, 5)
    return dict(num_states=S, start=start, final_cost=np.array(finals, np.float32), arc_src=a[:, 0].astype(np.int32),
                arc_dst=a[:, 1].astype(np.int32), arc_ilabel=a[:, 2].astype(np.int32),
                arc_olabel=a[:, 3].astype(np.int32), arc_weight=a[:, 4].astype(np.float32))


@pytest.mark.parametrize("case", ["dst", "src", "start", "ilabel", "olabel", "tid2pdf", "weight_nan", "weight_neginf",
                                  "final_nan", "eps_cycle"])
def test_create_rejects_bad_graphs(case):
    """Invalid graphs are rejected on the host before any device work (so with or without a GPU)."""
    tid2pdf = np.array([0, 0, 1], np.int32)
    ok = [(0, 1, 1, 4, -0.5), (1, 2, 0, 3, -1.0), (2, 2, 2, 0, 0.0)]  # negative weights are fine
    assert create(small(ok), tid2pdf)[0] in (0, capi.ERR_CUDA)
    g, want = small(ok), {"dst": "outside", "src": "outside", "start": "start state", "ilabel": "ilabel 3 outside",
                          "olabel": "olabel -1", "tid2pdf": "negative", "weight_nan": "NaN or -inf",
                          "weight_neginf": "NaN or -inf", "final_nan": "NaN or -inf", "eps_cycle": "cycle"}[case]
    if case == "dst":
        g = small(ok + [(2, 3, 1, 0, 0.0)])
    elif case == "src":
        g = small(ok + [(-1, 0, 1, 0, 0.0)])
    elif case == "start":
        g["start"] = 3
    elif case == "ilabel":
        g = small(ok + [(2, 0, 3, 0, 0.0)])
    elif case == "olabel":
        g = small(ok + [(2, 0, 1, -1, 0.0)])
    elif case == "tid2pdf":
        tid2pdf = np.array([0, 0, -1], np.int32)
    elif case == "weight_nan":
        g["arc_weight"][1] = np.nan
    elif case == "weight_neginf":
        g["arc_weight"][0] = -np.inf
    elif case == "final_nan":
        g["final_cost"][0] = np.nan
    else:
        g = small(ok + [(2, 1, 0, 0, 0.0)])
    rc, msg = create(g, tid2pdf)
    assert rc == capi.ERR_INVALID, (rc, msg)
    assert want in msg, msg
