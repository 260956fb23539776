"""The float64 restatement of lattice generation (tests/latgen_ref.py) without a GPU: against brute-force path
enumeration on tiny graphs with dyadic costs, against a Kaldi-style prune that iterates each frame until nothing
changes, nesting over lattice beams, and the shortest path through the lattice against beam_decode_ref."""
import numpy as np
import pytest

from tests.decode_ref import beam_decode_ref
from tests.latgen_ref import latgen_ref, prune_lattice, raw_lattice
from tests.test_decode_ref import tiny_graph
from voicebridge_b200 import synth

INF_ACTIVE = 2**31 - 1
SCALE = 0.5  # with log-likelihoods in halves, every acoustic cost and every FP64 sum below is exact


def dyadic_case(seed, n_tids=4, T=3, neg=True):
    rng = np.random.default_rng(seed)
    g = tiny_graph(rng, n_tids, neg)
    tid2pdf = np.r_[0, rng.integers(0, 3, n_tids)].astype(np.int32)
    ll = (rng.integers(-8, 1, (T, 3)) * 0.5).astype(np.float32)
    return g, tid2pdf, ll


def brute_links(g, ll, tid2pdf, status):
    """Every complete path: {(f_src, src, arc): best path cost through it}, {(f, s): likewise}, best cost."""
    ac = (-(np.float32(SCALE) * ll)).astype(np.float32).astype(np.float64)
    T = ll.shape[0]
    links, toks, best = {}, {}, [np.inf]

    def walk(s, r, cost, path, states):
        f = float(g["final_cost"][s]) if status == 0 else 0.0
        if r == T and f < np.inf:
            c = cost + f
            best[0] = min(best[0], c)
            for k in path:
                links[k] = min(links.get(k, np.inf), c)
            for k in states + [(r, s)]:
                toks[k] = min(toks.get(k, np.inf), c)
        for a in range(len(g["arc_src"])):
            if g["arc_src"][a] != s:
                continue
            d, lab, w = int(g["arc_dst"][a]), int(g["arc_ilabel"][a]), float(g["arc_weight"][a])
            if lab == 0:
                walk(d, r, cost + w, path + [(r, s, a)], states + [(r, s)])
            elif r < T:
                walk(d, r + 1, (cost + w) + ac[r, tid2pdf[lab]], path + [(r, s, a)], states + [(r, s)])

    walk(int(g["start"]), 0, 0.0, [], [])
    return links, toks, best[0]


def arc_ids(g, lat):
    """(frame of source, source graph state, arc index) of every lattice arc."""
    fr, st = lat["state_frame"], lat["state_graph"]
    out = set()
    for i in range(len(lat["arc_src"])):
        s = int(lat["arc_src"][i])
        # the arc index: the graph arc of that source state with this label pair and destination state
        cands = [a for a in range(len(g["arc_src"])) if g["arc_src"][a] == st[s] and g["arc_dst"][a] ==
                 st[lat["arc_dst"][i]] and g["arc_ilabel"][a] == lat["arc_ilabel"][i] and
                 g["arc_olabel"][a] == lat["arc_olabel"][i] and g["arc_weight"][a] == lat["arc_graph_cost"][i]]
        out |= {(int(fr[s]), int(st[s]), a) for a in cands}
    return out


@pytest.mark.parametrize("lattice_beam", [0.0, 0.5, 1.5, np.inf])
@pytest.mark.parametrize("finals", ["some", "none"])
def test_exact_lattice_equals_brute_force(lattice_beam, finals):
    checked = {0: 0, 1: 0}
    for seed in range(60):
        g, tid2pdf, ll = dyadic_case(seed)
        if finals == "none":
            g["final_cost"] = np.full(g["num_states"], np.inf, np.float32)
        one, lat = latgen_ref(g, ll, tid2pdf, SCALE, np.inf, INF_ACTIVE, 1 << 20, lattice_beam)
        if one[0] >= 2:
            assert len(lat["state_frame"]) == 0
            continue
        links, toks, best = brute_links(g, ll, tid2pdf, one[0])
        assert best == one[1]
        want_t = {k for k, c in toks.items() if c - best <= lattice_beam}
        want_a = {k for k, c in links.items() if c - best <= lattice_beam}
        assert set(zip(lat["state_frame"].tolist(), lat["state_graph"].tolist())) == want_t, seed
        assert arc_ids(g, lat) == want_a, seed
        # numbering: (frame, level, state) order, start first, arcs by (source, arc), topological
        assert (lat["state_frame"][0], lat["state_graph"][0]) == (0, g["start"])
        assert np.all(np.diff(lat["arc_src"]) >= 0)
        assert np.all(lat["arc_dst"] > lat["arc_src"]) or len(lat["arc_src"]) == 0
        checked[one[0]] += 1
    assert checked[0 if finals == "some" else 1] >= 15


def kaldi_prune(g, one, frames, links, lattice_beam):
    """PruneForwardLinks(Final) as LatticeFasterDecoder writes it: per frame from the last, sweep the frame's tokens
    until no extra cost changes.  Returns the kept link indices."""
    status, tot = one[0], one[1]
    T = len(frames) - 1
    final = np.asarray(g["final_cost"], np.float32)
    extra = {}
    out = {}
    for i, lk in enumerate(links):
        out.setdefault((lk[0], lk[1]), []).append(i)
    kept = set()
    for f in range(T, -1, -1):
        for s in frames[f]:
            extra[(f, s)] = np.inf
        changed = True
        while changed:
            changed = False
            for s, a in frames[f].items():
                e = np.inf
                if f == T:
                    e = (a + float(final[s])) - tot if status == 0 else a - tot
                for i in out.get((f, s), []):
                    le = extra[(links[i][2], links[i][3])] + links[i][7]
                    if le < np.inf and le <= lattice_beam:
                        kept.add(i)
                        e = min(e, le)
                    else:
                        kept.discard(i)
                if e > lattice_beam:
                    e = np.inf
                if e != extra[(f, s)]:
                    extra[(f, s)], changed = e, True
    return kept


@pytest.mark.parametrize("beam,max_active", [(np.inf, INF_ACTIVE), (6.0, 40), (3.0, 8)])
def test_level_ordered_prune_equals_kaldi_iteration(beam, max_active):
    topo = synth.phone_topology(6)
    for seed in range(3):
        g = synth.make_decoding_graph(topo, 12, 30, seed)
        ll = np.random.default_rng(seed).normal(-20, 6, (12, 30)).astype(np.float32)
        one, frames, links = raw_lattice(g, ll, g["tid2pdf"], 0.1, beam, max_active)
        assert one[0] <= 1
        for lb in (0.0, 2.0, 8.0, np.inf):
            _, kept = prune_lattice(g, one, frames, links, lb)
            assert kept == kaldi_prune(g, one, frames, links, lb), (seed, lb)


def test_larger_lattice_beams_nest():
    topo = synth.phone_topology(6)
    g = synth.make_decoding_graph(topo, 12, 30, 5)
    ll = np.random.default_rng(5).normal(-20, 6, (15, 30)).astype(np.float32)
    one, frames, links = raw_lattice(g, ll, g["tid2pdf"], 0.1, 8.0, 30)
    prev, sizes = set(), []
    for lb in (0.0, 0.5, 2.0, 5.0, 10.0, np.inf):
        _, kept = prune_lattice(g, one, frames, links, lb)
        assert prev <= kept
        prev = kept
        sizes.append(len(kept))
    assert sizes[0] < sizes[-1]


def shortest_path(lat, final_status):
    """Best path through a numbered lattice (states topological), costs summed as the search sums them."""
    ns = len(lat["state_frame"])
    dist, back = np.full(ns, np.inf), np.full(ns, -1)
    dist[0] = 0.0
    for i in range(len(lat["arc_src"])):
        s, d = lat["arc_src"][i], lat["arc_dst"][i]
        c = dist[s] + float(lat["arc_graph_cost"][i])
        if lat["arc_ilabel"][i]:
            c += float(lat["arc_ac_cost"][i])
        if c < dist[d]:
            dist[d], back[d] = c, i
    end = dist + lat["state_final"].astype(np.float64)
    s = int(np.argmin(end))
    arcs = []
    while back[s] >= 0:
        arcs.append(int(back[s]))
        s = int(lat["arc_src"][back[s]])
    arcs = arcs[::-1]
    ali = [int(lat["arc_ilabel"][i]) for i in arcs if lat["arc_ilabel"][i]]
    words = [int(lat["arc_olabel"][i]) for i in arcs if lat["arc_olabel"][i]]
    return float(end.min()), ali, words


@pytest.mark.parametrize("beam,max_active,lattice_beam", [(8.0, 30, 4.0), (5.0, 10, 0.0), (np.inf, INF_ACTIVE, 6.0)])
def test_shortest_path_is_the_one_best(beam, max_active, lattice_beam):
    topo = synth.phone_topology(8)
    for seed in range(4):
        g = synth.make_decoding_graph(topo, 20, 40, 10 + seed)
        ll = np.random.default_rng(seed).normal(-20, 6, (25, 40)).astype(np.float32)
        one, lat = latgen_ref(g, ll, g["tid2pdf"], 0.1, beam, max_active, 65536, lattice_beam)
        want = beam_decode_ref(g, ll, g["tid2pdf"], 0.1, beam, max_active, 65536)
        assert one[0] == want[0] and one[1] == want[1] and np.array_equal(one[2], want[2])
        assert one[0] <= 1
        cost, ali, words = shortest_path(lat, one[0])
        assert cost == one[1]
        assert ali == one[2].tolist() and words == list(one[4])
        assert np.all(lat["state_frame"][lat["arc_dst"]] == lat["state_frame"][lat["arc_src"]] +
                      (lat["arc_ilabel"] > 0))
