"""Float64 restatement of lattice generation (vbgpu_decode_lattice*, include/vbgpu.h) for the tests and
tools/bench_latgen.py: beam_decode_ref's search, run unchanged while its relaxations and finished token sets are
observed, then the same exact final prune and output numbering as the device."""
import sys

import numpy as np

from tests.align_ref import _levels
from tests.decode_ref import beam_decode_ref

LATTICE_KEYS = ("state_frame", "state_graph", "state_final", "arc_src", "arc_dst", "arc_ilabel", "arc_olabel",
                "arc_graph_cost", "arc_ac_cost")


def _observe(run, start, dst):
    """Calls run() (a beam_decode_ref call) and watches its nested functions through sys.setprofile: every call of
    relax(tok, cands, eps) gives the candidates (cost, arc, node of the source token) of one relaxation, every return
    of closure(tok, cut) the finished token set of one frame.  Returns (run's result, frames {state: cost},
    relaxations (frame of the source, source state, arc, candidate cost, epsilon))."""
    code = beam_decode_ref.__code__.co_filename
    frames, rel, cur = [], [], [0]
    prev = sys.getprofile()

    def hook(frame, event, arg):
        c = frame.f_code
        if c.co_filename != code:
            return
        if event == "call" and c.co_name == "relax":
            loc = frame.f_locals
            eps = bool(loc["eps"])
            if not eps:
                cur[0] = len(frames)  # the emitting step out of the last finished frame
            f = cur[0] if eps else cur[0] - 1
            for v, a, node in loc["cands"]:
                rel.append((f, start if node is None else int(dst[node[0]]), int(a), float(v), eps))
        elif event == "return" and c.co_name == "closure":
            frames.append({s: t[0] for s, t in frame.f_locals["tok"].items()})

    sys.setprofile(hook)
    try:
        out = run()
    finally:
        sys.setprofile(prev)
    return out, frames, rel


def raw_lattice(g, ll, tid2pdf, acoustic_scale=0.1, beam=16.0, max_active=2**31 - 1, max_tokens=65536):
    """Runs the search and returns (one-best tuple of beam_decode_ref, frames, links).  frames[f] = {state: cost}
    (empty when the status is 2 or 3); links: (f_src, src, f_dst, dst, arc, graph cost float32, acoustic cost float32,
    term) with term the FP64 candidate cost minus the destination's cost, in the search's operation order."""
    dst, lab = np.asarray(g["arc_dst"], np.int64), np.asarray(g["arc_ilabel"], np.int64)
    one, frames, rel = _observe(lambda: beam_decode_ref(g, ll, tid2pdf, acoustic_scale, beam, max_active, max_tokens),
                                int(g["start"]), dst)
    if one[0] >= 2:
        return one, [], []
    w32 = np.asarray(g["arc_weight"], np.float32)
    scale, ll = np.float32(acoustic_scale), np.asarray(ll, np.float32)
    tid2pdf = np.asarray(tid2pdf)
    links = []
    for f, s, a, v, eps in rel:
        if not v < np.inf:
            continue
        fd, d = (f if eps else f + 1), int(dst[a])
        ac = np.float32(0.0) if eps else np.float32(-(scale * ll[f][tid2pdf[lab[a]]]))
        links.append((f, s, fd, d, a, w32[a], ac, v - frames[fd][d]))
    return one, frames, links


def prune_lattice(g, one, frames, links, lattice_beam):
    """The exact final prune in one pass (frames from the last, epsilon levels from the highest): returns
    (extra {(f, s): extra}, kept link indices)."""
    status, tot = one[0], one[1]
    S = int(g["num_states"])
    src, dst, lab = (np.asarray(g[k], np.int64) for k in ("arc_src", "arc_dst", "arc_ilabel"))
    level = _levels(S, src[lab == 0], dst[lab == 0])
    final = np.asarray(g["final_cost"], np.float32)
    lb = float(np.float32(lattice_beam))
    T = len(frames) - 1
    extra = {}
    for s, a in frames[T].items():
        e = (a + float(final[s])) - tot if status == 0 else a - tot
        extra[(T, s)] = e if e <= lb else np.inf
    by_src = {}
    for i, lk in enumerate(links):
        f, s, fd = lk[0], lk[1], lk[2]
        key = (f, -1 if fd > f else int(level[s]))
        by_src.setdefault(key, []).append(i)
    kept = set()
    L = int(level.max(initial=0))
    for f in range(T, -1, -1):
        for lv in [-1] + list(range(L - 1, -1, -1)):
            for i in by_src.get((f, lv), []):
                fs, s, fd, d, _, _, _, term = links[i]
                e = extra.get((fd, d), np.inf) + term
                if e < np.inf and e <= lb:
                    kept.add(i)
                    if e < extra.get((fs, s), np.inf):
                        extra[(fs, s)] = e
                else:
                    extra.setdefault((fs, s), np.inf)
    return extra, kept


def number_lattice(g, one, frames, links, extra, kept):
    """The numbered output: a dict of the LATTICE_KEYS arrays (states by (frame, level, state), arcs by (source
    state, original arc index))."""
    S = int(g["num_states"])
    src, dst, lab = (np.asarray(g[k], np.int64) for k in ("arc_src", "arc_dst", "arc_ilabel"))
    level = _levels(S, src[lab == 0], dst[lab == 0])
    final = np.asarray(g["final_cost"], np.float32)
    ol = np.asarray(g["arc_olabel"], np.int64)
    T = len(frames) - 1
    toks = sorted(((f, int(level[s]), s) for f in range(T + 1) for s in frames[f]
                   if extra.get((f, s), np.inf) < np.inf))
    num = {(f, s): n for n, (f, _, s) in enumerate(toks)}
    arcs = sorted((num[(lk[0], lk[1])], lk[4], i) for i, lk in enumerate(links) if i in kept)
    out = {"state_frame": np.array([t[0] for t in toks], np.int32),
           "state_graph": np.array([t[2] for t in toks], np.int32),
           "state_final": np.array([np.float32(np.inf) if f < T else final[s] if one[0] == 0 else np.float32(0.0)
                                    for f, _, s in toks], np.float32),
           "arc_src": np.array([a[0] for a in arcs], np.int32),
           "arc_dst": np.array([num[(links[i][2], links[i][3])] for _, _, i in arcs], np.int32),
           "arc_ilabel": np.array([lab[a] for _, a, _ in arcs], np.int32),
           "arc_olabel": np.array([ol[a] for _, a, _ in arcs], np.int32),
           "arc_graph_cost": np.array([links[i][5] for _, _, i in arcs], np.float32),
           "arc_ac_cost": np.array([links[i][6] for _, _, i in arcs], np.float32)}
    return out


def empty_lattice():
    return {k: np.zeros(0, np.float32 if k in ("state_final", "arc_graph_cost", "arc_ac_cost") else np.int32)
            for k in LATTICE_KEYS}


def latgen_ref(g, ll, tid2pdf, acoustic_scale=0.1, beam=16.0, max_active=2**31 - 1, max_tokens=65536,
               lattice_beam=10.0):
    """One utterance: ll [T, P] float32 log-likelihoods in pdf order.  Returns (one-best tuple as beam_decode_ref,
    lattice dict of LATTICE_KEYS arrays; empty under status 2 / 3)."""
    one, frames, links = raw_lattice(g, ll, tid2pdf, acoustic_scale, beam, max_active, max_tokens)
    if one[0] >= 2:
        return one, empty_lattice()
    extra, kept = prune_lattice(g, one, frames, links, lattice_beam)
    return one, number_lattice(g, one, frames, links, extra, kept)
