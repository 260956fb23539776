"""Float64 restatement of forced alignment (vbgpu_align_*, include/vbgpu.h) for the tests and tools/bench_align.py:
the pdf subset the device scores for each utterance, and the Viterbi search with the device's operation order, epsilon
levels and tie rule."""
import numpy as np


def align_subsets(graphs, tid2pdf):
    """Per utterance, the pdfs the device scores for it: the distinct tid2pdf of its emitting arcs, increasing."""
    ao, lab = graphs["arc_offsets"], np.asarray(graphs["arc_ilabel"])
    out = []
    for u in range(len(ao) - 1):
        l = lab[ao[u]:ao[u + 1]]
        out.append(np.unique(np.asarray(tid2pdf)[l[l > 0]]).astype(np.int32))
    return out


def _levels(S, esrc, edst):
    """Longest epsilon path into each state (Kahn); None when the epsilon arcs form a cycle."""
    level, indeg = np.zeros(S, np.int64), np.bincount(edst, minlength=S)
    out = [[] for _ in range(S)]
    for a, b in zip(esrc, edst):
        out[a].append(b)
    queue = [s for s in range(S) if indeg[s] == 0]
    for s in queue:
        for d in out[s]:
            level[d] = max(level[d], level[s] + 1)
            indeg[d] -= 1
            if indeg[d] == 0:
                queue.append(d)
    return level if len(queue) == S else None


def _padded(arcs, dests, rows):
    """[len(rows), K] indices of the arcs into each state of rows (arc order within a row), -1 padding."""
    pos = {int(s): i for i, s in enumerate(rows)}
    lists = [[] for _ in rows]
    for a, d in zip(arcs, dests):
        if int(d) in pos:
            lists[pos[int(d)]].append(int(a))
    m = np.full((len(rows), max([len(v) for v in lists] + [1])), -1, np.int64)
    for i, v in enumerate(lists):
        m[i, :len(v)] = v
    return m


def viterbi_align_ref(graphs, u, ll, pdfs, tid2pdf, tid_cost=None, acoustic_scale=0.1, path=None):
    """float64 restatement of vbgpu_align for utterance u (include/vbgpu.h): ll [T_u, len(pdfs)] holds the log-likelihoods
    of the pdfs `pdfs` (align_subsets order).  Same operation order as the device: arc weights plus tid_cost in float32,
    ac = -(acoustic_scale * ll) in float32, emitting cost (prev + w) + ac and epsilon cost prev + w in float64; the
    epsilon closure level by level (longest epsilon path into a state), first-in-arc-order wins ties, an epsilon
    relaxation only when strictly lower, the lowest state among equal final costs.
    Returns (tot_cost, ali[T_u] transition-ids, pdf_ids[T_u]); (+inf, zeros, -1s) when no final state is reachable.
    path (a list) receives the arcs of the best path, epsilon arcs included, in order, as arc indices of utterance u."""
    so, ao = graphs["state_offsets"], graphs["arc_offsets"]
    S, a0, a1 = int(so[u + 1] - so[u]), int(ao[u]), int(ao[u + 1])
    src, dst = np.asarray(graphs["arc_src"][a0:a1], np.int64), np.asarray(graphs["arc_dst"][a0:a1], np.int64)
    lab = np.asarray(graphs["arc_ilabel"][a0:a1], np.int64)
    w = np.asarray(graphs["arc_weight"][a0:a1], np.float32)
    if tid_cost is not None:
        tc = np.asarray(tid_cost, np.float32)
        w = np.where(lab > 0, w + tc[lab], w).astype(np.float32)
    w64 = w.astype(np.float64)
    final = np.asarray(graphs["final_cost"][so[u]:so[u + 1]], np.float32).astype(np.float64)
    tid2pdf = np.asarray(tid2pdf)
    ll = np.asarray(ll, np.float32)
    T = ll.shape[0]
    ac = (-(np.float32(acoustic_scale) * ll)).astype(np.float32).astype(np.float64)
    ac = np.concatenate([ac, np.zeros((T, 1))], axis=1)  # (a column for the padding of E to index)
    col = np.full(max(int(tid2pdf.max()) + 1, 1), -1, np.int64)
    col[np.asarray(pdfs, np.int64)] = np.arange(len(pdfs))
    emit = lab > 0
    acol = np.where(emit, col[tid2pdf[lab]], -1)
    ei, xi = np.flatnonzero(emit), np.flatnonzero(~emit)
    E = _padded(ei, dst[ei], np.arange(S))
    level = _levels(S, src[~emit], dst[~emit])
    assert level is not None, "epsilon cycle"
    lvl_states = [np.flatnonzero(level == l) for l in range(1, int(level.max(initial=0)) + 1)]
    X = [_padded(xi, dst[xi], st) for st in lvl_states]
    tb = np.full((T + 1, S), -1, np.int64)
    inf = np.inf
    psrc, pw, pcol = np.r_[src, 0], np.r_[w64, 0.0], np.r_[acol, -1]  # index -1 (padding) reads the extra entry

    def closure(c, tbr):
        for st, m in zip(lvl_states, X):
            v = np.where(m >= 0, c[psrc[m]] + pw[m], inf)
            cand = np.concatenate([c[st][:, None], v], axis=1)
            k = np.argmin(np.where(np.isnan(cand), inf, cand), axis=1)
            ch = k > 0
            c[st[ch]] = cand[ch, k[ch]]
            tbr[st[ch]] = m[ch, k[ch] - 1]

    c = np.full(S, inf)
    c[int(graphs["start"][u])] = 0.0
    closure(c, tb[0])
    for t in range(T):
        v = np.where(E >= 0, (c[psrc[E]] + pw[E]) + ac[t, pcol[E]], inf)
        v = np.where(np.isnan(v), inf, v)
        k = np.argmin(v, axis=1)
        best = v[np.arange(S), k]
        c = best.copy()
        tb[t + 1] = np.where(best < inf, E[np.arange(S), k], -1)
        closure(c, tb[t + 1])
    tot = c + final
    s = int(np.argmin(tot))
    if not tot[s] < inf:
        return inf, np.zeros(T, np.int32), np.full(T, -1, np.int32)
    ali, r, arcs = np.zeros(T, np.int32), T, []
    while tb[r, s] >= 0:
        a = int(tb[r, s])
        arcs.append(a)
        if lab[a]:
            r -= 1
            ali[r] = lab[a]
        s = int(src[a])
    assert r == 0
    if path is not None:
        path.extend(arcs[::-1])
    return float(tot[int(np.argmin(tot))]), ali, tid2pdf[ali].astype(np.int32)
