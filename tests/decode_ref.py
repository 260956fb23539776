"""Float64 restatement of one-best decoding (vbgpu_decoder_*, include/vbgpu.h) for the tests and tools/bench_decode.py:
the same cost arithmetic, epsilon levels, prune rule, tie rules, status rules and output rules as the device."""
import numpy as np

from tests.align_ref import _levels


def beam_decode_ref(g, ll, tid2pdf, acoustic_scale=0.1, beam=16.0, max_active=2**31 - 1, max_tokens=65536,
                    max_words=None, stats=None, ties=None):
    """Decodes one utterance: ll [T, P] float32 log-likelihoods in pdf order.  Returns (status, tot_cost, ali[T],
    pdf_ids[T], words (all of them; the caller truncates), num_words).  stats (a list) receives the size of every
    frame's token set.  ties (a collections.Counter) counts the ties the tie rules decided: "arcs" equal candidates into
    one state within a relaxation, "emit_kept" epsilon candidates equal to an emitting token's cost, "eps_equal"
    epsilon candidates equal to an earlier epsilon back-pointer's cost, "best" frames whose best cost is held by
    several tokens, "boundary" frames where c_(max_active) = c_(max_active+1), "final" ends with several best states."""
    ties = ties if ties is not None else {}
    S = int(g["num_states"])
    src, dst = np.asarray(g["arc_src"], np.int64), np.asarray(g["arc_dst"], np.int64)
    lab, ol = np.asarray(g["arc_ilabel"], np.int64), np.asarray(g["arc_olabel"], np.int64)
    w64 = np.asarray(g["arc_weight"], np.float32).astype(np.float64)
    final = np.asarray(g["final_cost"], np.float32).astype(np.float64)
    tid2pdf = np.asarray(tid2pdf)
    ll = np.asarray(ll, np.float32)
    T = ll.shape[0]
    emit = lab > 0
    level = _levels(S, src[~emit], dst[~emit])
    assert level is not None, "epsilon cycle"
    L = int(level.max(initial=0))
    e_out, x_out = [[] for _ in range(S)], [[] for _ in range(S)]
    for a in range(len(src)):  # arc order within each list
        (e_out if emit[a] else x_out)[src[a]].append(a)
    beam64 = float(np.float32(beam))
    scale = np.float32(acoustic_scale)

    # a token: state -> [cost, arc of its back-pointer (-1 none), previous node]; a node is (arc, node) or None
    def relax(tok, cands, eps):
        """cands: (v, arc, parent node) per arc; the minimum per destination, lowest arc among equal costs."""
        best = {}
        for v, a, node in cands:
            if not v < np.inf:
                continue
            d = int(dst[a])
            if d in best and v == best[d][0]:
                ties["arcs"] = ties.get("arcs", 0) + 1
            if d not in best or v < best[d][0] or (v == best[d][0] and a < best[d][1]):
                best[d] = (v, a, node)
        for d, (v, a, node) in best.items():
            if d not in tok:
                tok[d] = [v, a, (a, node), eps]
            elif v == tok[d][0]:
                k = "eps_equal" if tok[d][3] else "emit_kept"
                ties[k] = ties.get(k, 0) + 1
            if d in tok and (v < tok[d][0] or (v == tok[d][0] and eps and tok[d][3] and a < tok[d][1])):
                tok[d] = [v, a, (a, node), eps]
        return len(tok) <= max_tokens

    def closure(tok, cut):
        for lv in range(L):
            srcs = [s for s in tok if level[s] == lv and tok[s][0] < cut]
            cands = [(tok[s][0] + w64[a], a, tok[s][2]) for s in srcs for a in x_out[s]]
            if not relax(tok, cands, True):
                return False
        return True

    tok = {int(g["start"]): [0.0, -1, None, False]}
    status = 0 if closure(tok, np.inf) else 3
    for t in range(T if status == 0 else 0):
        if stats is not None:
            stats.append(len(tok))
        costs = sorted(v[0] for v in tok.values())
        c1 = costs[0]
        cut = c1 + beam64
        if len(tok) > max_active:
            ck = costs[max_active]
            if ck == costs[max_active - 1]:
                ties["boundary"] = ties.get("boundary", 0) + 1
            cut = ck if ck < cut else cut
        surv = [s for s in tok if tok[s][0] < cut or tok[s][0] == c1]
        if costs[1:2] == [c1]:
            ties["best"] = ties.get("best", 0) + 1
        if len(surv) > max_active:
            status = 3
            break
        ac = (-(scale * ll[t])).astype(np.float32).astype(np.float64)
        cands = [((tok[s][0] + w64[a]) + ac[tid2pdf[lab[a]]], a, tok[s][2]) for s in surv for a in e_out[s]]
        tok = {}
        if not relax(tok, cands, False):
            status = 3
            break
        if not tok:
            status = 2
            break
        if not closure(tok, min(v[0] for v in tok.values()) + beam64):
            status = 3
            break
    if status >= 2:
        return status, np.inf, np.zeros(T, np.int32), np.full(T, -1, np.int32), [], 0
    fin = [(tok[s][0] + final[s], s) for s in tok if final[s] < np.inf]
    if not fin:
        status = 1
        fin = [(v[0], s) for s, v in tok.items()]
    cost, s = min(fin)
    if sum(c == cost for c, _ in fin) > 1:
        ties["final"] = ties.get("final", 0) + 1
    arcs, node = [], tok[s][2]
    while node is not None:
        arcs.append(node[0])
        node = node[1]
    arcs = np.asarray(arcs[::-1], np.int64)
    ali = lab[arcs][emit[arcs]].astype(np.int32)
    assert len(ali) == T
    words = [int(o) for o in ol[arcs] if o]
    return status, float(cost), ali, tid2pdf[ali].astype(np.int32), words, len(words)


def loglikes_in_pdf_order(ll_cols, col_of_pdf):
    """[T, P] pdf-order view of a device column-order matrix."""
    return np.ascontiguousarray(np.asarray(ll_cols)[:, np.asarray(col_of_pdf)])
