"""Tree statistics on the device (vbgpu_tree_*, host.TreeStatsGpu) and the per transition-id tables of a model file
(vbgpu_io_mdl_transitions, kaldi_io.read_transitions).

The truth is a Python restatement of AccumulateTreeStats (hmm/tree-accu.cc), SplitToPhones / IsReordered
(hmm/hmm-utils.cc) and GaussClusterable::AddStats (tree/clusterable-classes.cc), written from the rules as the project
documents them (include/vbgpu.h).  It has not been checked against the compiled reference: the reference's sources are
needed for that.  Sums are float64 over the same float32 rows, so only the order of the FP64 additions may differ: counts
must be exact and every sum within 1e-11 of the sum of the absolute values of its terms."""
import ctypes as C
import struct

import numpy as np
import pytest

from tests.common import recipe_opts
from voicebridge_b200 import capi, host, kaldi_io, synth

TOL = 1e-11


# ---- the restatement -----------------------------------------------------------------------------------------------------
def is_reordered(ali, t):
    sl = lambda k: bool(t["flags"][ali[k]] & capi.TID_SELF_LOOP)  # noqa: E731
    ts = t["trans_state"]
    for i in range(len(ali) - 1):
        if ts[ali[i]] != ts[ali[i + 1]]:
            if sl(i):
                return True
            if sl(i + 1):
                return False
    if len(ali) and sl(0):
        return False
    return bool(len(ali) and sl(len(ali) - 1))


def split_to_phones(ali, t):
    """Phone segments [(begin, end)] of a good alignment, None for a bad one."""
    n = len(ali)
    if any(a < 1 or a >= len(t["phone"]) for a in ali):
        return None
    fl, ts, ph = t["flags"], t["trans_state"], t["phone"]
    reordered = is_reordered(ali, t)
    ends, ok, i = [], True, 0
    while i < n:
        if fl[ali[i]] & capi.TID_FINAL:
            if reordered:
                while i + 1 < n and fl[ali[i + 1]] & capi.TID_SELF_LOOP:
                    i += 1
            ends.append(i + 1)
        elif i + 1 == n:
            ok = False
            ends.append(i + 1)
        elif ts[ali[i]] != ts[ali[i + 1]] and ph[ali[i]] != ph[ali[i + 1]]:
            ok = False
            ends.append(i + 1)
        i += 1
    segs, b = [], 0
    for e in ends:
        if fl[ali[b]] & capi.TID_STATE0_EMITTING and t["hmm_state"][ali[b]] != 0:
            ok = False
        segs.append((b, e))
        b = e
    return segs if ok else None


def event_types(ali, t, N, P, ci):
    """EventType of every frame of a good alignment (None for a bad one)."""
    segs = split_to_phones(ali, t)
    if segs is None:
        return None
    phones = [int(t["phone"][ali[b]]) for b, _ in segs]
    out = []
    for s, (b, e) in enumerate(segs):
        c = phones[s]
        ctx = [phones[s - P + j] if 0 <= s - P + j < len(segs) else 0 for j in range(N)]
        pairs = [(P, c)] if c in ci else [(j, ctx[j]) for j in range(N)]
        for k in range(b, e):
            out.append(tuple(sorted(pairs + [(-1, int(t["pdf_class"][ali[k]]))])))
    return out


def restate(feats, tids, fo, t, N, P, ci, D):
    """{EventType: [count, sum_x, sum_x2, sum |x|, sum x^2]} and the number of bad utterances."""
    stats, bad = {}, 0
    for u in range(len(fo) - 1):
        ali = tids[fo[u]:fo[u + 1]]
        evs = event_types(ali, t, N, P, ci)
        if evs is None:
            bad += 1
            continue
        for k, ev in enumerate(evs):
            x = feats[fo[u] + k, :D].astype(np.float64)
            st = stats.setdefault(ev, [0, np.zeros(D), np.zeros(D), np.zeros(D), np.zeros(D)])
            st[0] += 1
            st[1] += x
            st[2] += x * x
            st[3] += np.abs(x)
            st[4] += x * x
    return stats, bad


def assert_stats(got, want, keys=None):
    """got: TreeStatsGpu.stats(); want: restate()[0].  keys: compare only these (table overflow)."""
    if keys is None:
        assert set(got) == set(want), (sorted(set(got) ^ set(want))[:5], len(got), len(want))
    assert list(got) == sorted(got), "download order is not the EventType order"
    for ev in (got if keys is None else keys):
        c, sx, sx2 = got[ev]
        w = want[ev]
        assert c == w[0], ev
        assert np.isfinite(sx).all() and np.isfinite(sx2).all(), ev
        assert (np.abs(sx - w[1]) <= TOL * w[3]).all(), (ev, np.abs(sx - w[1]).max())
        assert (np.abs(sx2 - w[2]) <= TOL * w[4]).all(), (ev, np.abs(sx2 - w[2]).max())


# ---- hand-worked examples (no device needed) -----------------------------------------------------------------------------
TOPO = synth.phone_topology(5)  # phone 1: 1 state; phones 2 ... 5: 3 states


def ten_frames(reordered):
    """phone 2 (state frames 1, 2, 1), phone 3 (2, 1, 1), phone 1 (2 frames)."""
    return synth.phone_alignment(TOPO, [2, 3, 1], [[1, 2, 1], [2, 1, 1], [2]], reordered)


@pytest.mark.parametrize("reordered", [False, True])
def test_restatement_hand_worked_triphones(reordered):
    ali = ten_frames(reordered)
    assert len(ali) == 10 and is_reordered(ali, TOPO) == reordered
    assert split_to_phones(ali, TOPO) == [(0, 4), (4, 8), (8, 10)]
    evs = event_types(ali, TOPO, 3, 1, [])
    left, mid, right = ((0, 0), (1, 2), (2, 3)), ((0, 2), (1, 3), (2, 1)), ((0, 3), (1, 1), (2, 0))  # edges: phone 0
    assert evs == [((-1, 0),) + left, ((-1, 1),) + left, ((-1, 1),) + left, ((-1, 2),) + left,
                   ((-1, 0),) + mid, ((-1, 0),) + mid, ((-1, 1),) + mid, ((-1, 2),) + mid,
                   ((-1, 0),) + right, ((-1, 0),) + right]
    # a context-independent central phone keeps only (P, c)
    evs = event_types(ali, TOPO, 3, 1, [1])
    assert evs[8:] == [((-1, 0), (1, 1))] * 2 and evs[:8] == event_types(ali, TOPO, 3, 1, [])[:8]
    # monophone windows, and a right-biased one
    assert event_types(ali, TOPO, 1, 0, [])[4] == ((-1, 0), (0, 3))
    assert event_types(ali, TOPO, 2, 1, [])[9] == ((-1, 0), (0, 3), (1, 1))


def test_restatement_drops_bad_alignments():
    tid = TOPO["tid"]
    good = ten_frames(False)
    # phone 2 leaves from state 1 to phone 3 without a final transition
    no_final = np.array([tid[(2, 0, False)], tid[(2, 1, False)], tid[(3, 0, False)], tid[(3, 1, False)],
                         tid[(3, 2, False)]], np.int32)
    mid_phone = good[:6]  # ends inside phone 3
    state1_start = np.concatenate([[tid[(2, 1, True)], tid[(2, 1, False)], tid[(2, 2, False)]], good[4:]]).astype(np.int32)
    for ali in (no_final, mid_phone, state1_start):
        assert split_to_phones(ali, TOPO) is None
    assert split_to_phones(good, TOPO) is not None
    assert split_to_phones(np.zeros(0, np.int32), TOPO) == []
    assert split_to_phones(np.array([tid[(1, 0, False)]], np.int32), TOPO) == [(0, 1)]
    assert split_to_phones(np.array([tid[(1, 0, True)]], np.int32), TOPO) is None


# ---- model-file tables -----------------------------------------------------------------------------------------------
def _tok(t):
    return t.encode() + b" "


def _i(v):
    return b"\x04" + struct.pack("<i", v)


def _ivec(v):
    return b"\x04" + struct.pack("<i", len(v)) + struct.pack("<%di" % len(v), *v)


def model_bytes(topo, tuples_form, D=2):
    """A binary model file (TransitionModel + AmDiagGmm) for topo: <Triples> with an HMM topology, or <Tuples> with
    the non-HMM topology form that stores self-loop pdf classes."""
    entries, tuples = topo["entries"], topo["tuples"]
    phones = sorted(topo["phone2entry"])
    phone2idx = [-1] * (max(phones) + 1)
    for p in phones:
        phone2idx[p] = topo["phone2entry"][p]
    b = b"\0B" + _tok("<TransitionModel>") + _tok("<Topology>") + _ivec(phones) + _ivec(phone2idx)
    if tuples_form:
        b += _i(-1)
    b += _i(len(entries))
    for e in entries:
        b += _i(len(e))
        for fwd, slf, dsts in e:
            b += _i(fwd) + (_i(slf) if tuples_form else b"") + _i(len(dsts))
            for d in dsts:
                b += _i(d) + b"\x04" + struct.pack("<f", 1.0 / len(dsts))
    b += _tok("</Topology>") + _tok("<Tuples>" if tuples_form else "<Triples>") + _i(len(tuples))
    for p, s, f, sl in tuples:
        b += _i(p) + _i(s) + _i(f) + (_i(sl) if tuples_form else b"")
    nt = len(topo["phone"])
    b += _tok("</Tuples>" if tuples_form else "</Triples>") + _tok("<LogProbs>") + _tok("FV") + _i(nt)
    b += struct.pack("<%df" % nt, *([-0.5] * nt)) + _tok("</LogProbs>") + _tok("</TransitionModel>")
    b += _tok("<DIMENSION>") + _i(D) + _tok("<NUMPDFS>") + _i(len(tuples))
    for _ in tuples:
        b += _tok("<DiagGMM>") + _tok("<WEIGHTS>") + _tok("FV") + _i(1) + struct.pack("<f", 1.0)
        b += _tok("<MEANS_INVVARS>") + _tok("FM") + _i(1) + _i(D) + struct.pack("<%df" % D, *([0.0] * D))
        b += _tok("<INV_VARS>") + _tok("FM") + _i(1) + _i(D) + struct.pack("<%df" % D, *([1.0] * D))
        b += _tok("</DiagGMM>")
    return b


def pdf_of_phone_class_is_a_function(tables, tid2pdf):
    seen = {}
    for t in range(1, len(tid2pdf)):
        k = (int(tables["phone"][t]), int(tables["pdf_class"][t]))
        if seen.setdefault(k, int(tid2pdf[t])) != int(tid2pdf[t]):
            return False
    return True


@pytest.mark.parametrize("tuples_form", [False, True])
def test_model_file_tables(tuples_form):
    topo = synth.phone_topology(4)
    want = {k: topo[k].copy() for k in ("phone", "hmm_state", "pdf_class", "trans_state", "flags")}
    if tuples_form:  # a self-loop pdf class of its own in state 1 of the 3-state phones
        topo = dict(topo, entries=[topo["entries"][0], [(0, 0, [0, 1]), (1, 3, [1, 2]), (2, 2, [2, 3]), (-1, -1, [])]])
        sl1 = (want["hmm_state"] == 1) & ((want["flags"] & capi.TID_SELF_LOOP) != 0) & (want["phone"] > 1)
        want["pdf_class"][sl1] = 3
    b = model_bytes(topo, tuples_form)
    got = kaldi_io.read_transitions(b)
    for k, v in want.items():
        assert np.array_equal(got[k], v), k
    m = kaldi_io.read_mdl(b)
    assert len(m["tid2pdf"]) == len(want["phone"])
    if not tuples_form:
        assert pdf_of_phone_class_is_a_function(got, m["tid2pdf"])
    with pytest.raises(capi.VbgpuError):
        kaldi_io.read_transitions(b[:100])  # inside the topology


def test_model_file_tables_of_the_reference_writer(ref):
    m = synth.make_model(12, 30, 4, 5)
    b = ref.io_write_mdl(m, 4)
    got = kaldi_io.read_transitions(b)
    assert pdf_of_phone_class_is_a_function(got, kaldi_io.read_mdl(b)["tid2pdf"])


# ---- argument checks and no fallback (no device needed) ------------------------------------------------------------------
def tree_args(N=3, P=1, ci=(), topo=TOPO):
    tabs = {k: np.ascontiguousarray(topo[k], np.int32) for k in ("phone", "hmm_state", "pdf_class", "trans_state", "flags")}
    ci = np.asarray(ci, np.int32)
    t = capi.TidTables(len(tabs["phone"]) - 1, *(tabs[k].ctypes.data for k in
                                                  ("phone", "hmm_state", "pdf_class", "trans_state", "flags")))
    o = capi.TreeOpts(N, P, ci.ctypes.data if len(ci) else None, len(ci))
    return o, t, (tabs, ci)


def test_argument_errors_need_no_gpu():
    lib = capi.lib()
    h = C.c_void_p()

    def create(o, t, dim=13, max_keys=100):
        return lib.vbgpu_tree_create(C.byref(o) if o is not None else None, C.byref(t) if t is not None else None, dim,
                                     max_keys, 0, C.byref(h))
    for N, P in ((5, 1), (0, 0), (3, 3), (2, -1)):
        o, t, keep = tree_args(N, P)
        assert create(o, t) == capi.ERR_INVALID, (N, P)
    o, t, keep = tree_args()
    assert create(None, t) == capi.ERR_INVALID
    assert create(o, None) == capi.ERR_INVALID
    for dim in (0, 257):
        assert create(o, t, dim=dim) == capi.ERR_INVALID
        assert b"dim" in lib.vbgpu_last_error()
    assert create(o, t, max_keys=0) == capi.ERR_INVALID
    big = dict(TOPO, phone=TOPO["phone"].copy())
    big["phone"][3] = 4096
    o2, t2, keep2 = tree_args(topo=big)
    assert create(o2, t2) == capi.ERR_INVALID and b"4095" in lib.vbgpu_last_error()
    cls = dict(TOPO, pdf_class=TOPO["pdf_class"].copy())
    cls["pdf_class"][2] = 256
    o3, t3, keep3 = tree_args(topo=cls)
    assert create(o3, t3) == capi.ERR_INVALID
    o4, t4, keep4 = tree_args(ci=(3, 1))
    assert create(o4, t4) == capi.ERR_INVALID  # ci_phones not sorted
    t.phone = None
    assert create(o, t) == capi.ERR_INVALID
    assert lib.vbgpu_tree_create(C.byref(o), C.byref(t), 13, 100, 0, None) == capi.ERR_INVALID
    fo = np.array([0, 4], np.int64)
    assert lib.vbgpu_tree_accumulate(None, None, 13, None, fo.ctypes.data, 1) == capi.ERR_INVALID
    assert lib.vbgpu_tree_accumulate_dev(None, None, 13, None, fo.ctypes.data, 1, None) == capi.ERR_INVALID
    assert lib.vbgpu_tree_zero(None) == capi.ERR_INVALID
    assert lib.vbgpu_tree_download(None, None, None, None, None, None) == capi.ERR_INVALID
    assert lib.vbgpu_tree_add(None, 0, None, None, None, None, None) == capi.ERR_INVALID
    assert lib.vbgpu_tree_bad_count(None, None, None) == capi.ERR_INVALID
    assert lib.vbgpu_io_mdl_transitions(None, 0, None, None, None, None, None) == capi.ERR_INVALID


def test_no_cpu_fallback():
    lib = capi.lib()
    n = C.c_int(0)
    if lib.vbgpu_device_count(C.byref(n)) == 0 and n.value > 0:
        pytest.skip("a GPU is present")
    o, t, keep = tree_args()
    h = C.c_void_p()
    assert lib.vbgpu_tree_create(C.byref(o), C.byref(t), 13, 100, 0, C.byref(h)) == capi.ERR_CUDA
    with pytest.raises(capi.VbgpuError):
        host.TreeStatsGpu(TOPO, 13, 100)


# ---- on the device ------------------------------------------------------------------------------------------------------
def gpu_or_skip():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def make_batch(D, stride, reordered, seed, n_phones=12):
    """Utterances of 0 ... 80 frames (a 0-frame and a 1-frame one among them) and three bad ones with NaN rows."""
    rng = np.random.default_rng(seed)
    lens = [37, 0, 1, 80, 12, 55, 3, 64, 20, 41]
    fo = np.zeros(len(lens) + 1, np.int64)
    fo[1:] = np.cumsum(lens)
    topo, tids, _ = synth.make_phone_alignment(n_phones, fo, seed, reordered=reordered, zipf=0.8, mean_state_frames=2.5)
    tid = topo["tid"]

    def ali(phones, durs):
        return synth.phone_alignment(topo, phones, durs, reordered)
    # a phone change without a final transition, a phone starting at hmm-state 1, an utterance ending mid-phone
    tids[fo[3]:fo[4]] = np.concatenate([[tid[(2, 0, False)], tid[(2, 1, False)]], ali([3, 1], [[1, 1, 1], [75]])])
    tids[fo[5]:fo[6]] = np.concatenate([[tid[(3, 1, False)], tid[(3, 2, False)]], ali([1], [[53]])])
    tids[fo[7]:fo[8]] = ali([2], [[30, 34, 1]])[:-1]
    X = np.full((int(fo[-1]), stride), np.nan, np.float32)
    X[:, :D] = (rng.standard_normal((int(fo[-1]), D)) * 2.0 + rng.uniform(-3, 3, D)).astype(np.float32)
    for u in (3, 5, 7):
        X[fo[u]:fo[u + 1]] = np.nan  # rows of bad utterances are never read
    return topo, tids, fo, X


@pytest.mark.gpu
@pytest.mark.parametrize("reordered", [False, True])
@pytest.mark.parametrize("NP", [(3, 1), (1, 0), (2, 1), (4, 2)])
@pytest.mark.parametrize("D", [1, 13, 39, 40, 117, 256])
def test_matches_restatement(D, NP, reordered):
    torch = gpu_or_skip()
    N, P = NP
    ci = (1, 5)
    topo, tids, fo, X = make_batch(D, D + 3, reordered, 100 * D + 10 * N + reordered)
    want, bad = restate(X, tids, fo, topo, N, P, ci, D)
    assert bad == 3
    ts = host.TreeStatsGpu(topo, D, 4096, N, P, ci)
    ts.AccumulateTreeStats(X, tids, fo)
    assert ts.NumKeys() == len(want)
    assert_stats(ts.stats(), want)
    assert ts.bad_count() == (bad, 0)
    assert ts.bad_count() == (0, 0)
    ts.ZeroAccumulators()
    assert ts.NumKeys() == 0 and ts.stats() == {}
    ts.accumulate_dev(torch.from_numpy(X).cuda(), D + 3, torch.from_numpy(tids).cuda(), fo)
    torch.cuda.synchronize()
    assert_stats(ts.stats(), want)
    assert ts.bad_count() == (bad, 0)


@pytest.mark.gpu
def test_split_calls_equal_one_call_and_merging():
    torch = gpu_or_skip()
    D, N, P = 39, 3, 1
    topo = synth.phone_topology(30)
    rng = np.random.default_rng(3)
    lens = rng.integers(20, 300, 40)
    fo = np.zeros(len(lens) + 1, np.int64)
    fo[1:] = np.cumsum(lens)
    _, tids, _ = synth.make_phone_alignment(30, fo, 4, reordered=True)
    X = rng.standard_normal((int(fo[-1]), D)).astype(np.float32)
    want, bad = restate(X, tids, fo, topo, N, P, (1,), D)
    one = host.TreeStatsGpu(topo, D, 1 << 15, N, P, (1,))
    one.accumulate_dev(torch.from_numpy(X).cuda(), D, torch.from_numpy(tids).cuda(), fo)
    all_stats = one.stats()
    assert_stats(all_stats, want)

    # the same batch in three calls: keys first seen in later calls get later dense ids
    split = host.TreeStatsGpu(topo, D, 1 << 15, N, P, (1,))
    for a, b in ((0, 5), (5, 6), (6, 40)):
        sub = fo[a:b + 1] - fo[a]
        split.accumulate_dev(torch.from_numpy(X[fo[a]:fo[b]]).cuda(), D, torch.from_numpy(tids[fo[a]:fo[b]]).cuda(), sub)
    assert_stats(split.stats(), want)

    # two handles, half the utterances each (devices 0 and 1 when there are two), merged key by key
    devs = (0, 1) if torch.cuda.device_count() >= 2 else (0, 0)
    halves = []
    for dev, (a, b) in zip(devs, ((0, 20), (20, 40))):
        h = host.TreeStatsGpu(topo, D, 1 << 15, N, P, (1,), device=dev)
        h.AccumulateTreeStats(X[fo[a]:fo[b]], tids[fo[a]:fo[b]], fo[a:b + 1] - fo[a])
        halves.append(h.stats())
    merged = host.TreeStatsGpu(topo, D, 1 << 15, N, P, (1,))
    merged.Add(halves[0])
    merged.Add(halves[1])
    assert_stats(merged.stats(), want)
    assert merged.bad_count() == (0, 0)


@pytest.mark.gpu
def test_table_overflow_is_counted():
    torch = gpu_or_skip()
    D = 13
    topo, tids, fo, X = make_batch(D, D, False, 9)
    want, bad = restate(X, tids, fo, topo, 3, 1, (), D)
    small = 8
    assert len(want) > small
    ts = host.TreeStatsGpu(topo, D, small, 3, 1, ())
    with pytest.raises(capi.VbgpuError) as e:
        ts.AccumulateTreeStats(X, tids, fo)
    assert e.value.code == capi.ERR_NUMERIC
    got = ts.stats()
    assert ts.NumKeys() == small == len(got)
    assert_stats(got, want, keys=list(got))  # the keys that found room hold all their frames
    n_bad, dropped = ts.bad_count()
    assert n_bad == bad and dropped == sum(w[0] for k, w in want.items() if k not in got)
    ts.accumulate_dev(torch.from_numpy(X).cuda(), D, torch.from_numpy(tids).cuda(), fo)
    assert ts.bad_count()[1] == dropped
    with pytest.raises(capi.VbgpuError):
        ts.Add({k: (w[0], w[1], w[2]) for k, w in want.items()})


@pytest.mark.gpu
def test_end_to_end_mfcc_deltas_tree_stats():
    """PCM -> MFCC -> CMVN + deltas (vbgpu_feat_run_dev, the train_deltas chain) -> tree statistics, against the
    restatement over the host form's rows (vbgpu_feat_run)."""
    torch = gpu_or_skip()
    n_spk = 3
    pcm, so, u2s = synth.make_corpus(n_spk, 3, 1.0, 2.5, 31)
    mfcc = host.Mfcc(recipe_opts(capi))
    fo = mfcc.frame_offsets(so)
    T = int(fo[-1])
    s = torch.cuda.current_stream()
    d_mf = torch.zeros((T, 16), dtype=torch.float32, device="cuda")
    mfcc.compute_dev(torch.from_numpy(np.asarray(pcm, np.int16)).cuda(), so, d_mf, 16, stream=s)
    torch.cuda.synchronize()
    mf = d_mf[:, :13].cpu().numpy()
    fp = host.FeaturePipeline(capi.default_feat_opts(), 13)
    st = fp.cmvn_stats(mf, fo, u2s, n_spk)
    d_x = torch.zeros((T, 40), dtype=torch.float32, device="cuda")
    fp.run_dev(d_mf, 16, fo, d_x, 40, u2s, n_spk, cmvn_stats=st, stream=s)
    feats = fp.run(mf, fo, u2s, n_spk, cmvn_stats=st)
    topo, tids, _ = synth.make_phone_alignment(40, fo, 32)
    ts = host.TreeStatsGpu(topo, 39, 1 << 14, 3, 1, (1,))
    ts.accumulate_dev(d_x, 40, torch.from_numpy(tids).cuda(), fo, stream=s)
    want, bad = restate(feats, tids, fo, topo, 3, 1, (1,), 39)
    assert bad == 0
    assert_stats(ts.stats(), want)
    assert ts.bad_count() == (0, 0)
