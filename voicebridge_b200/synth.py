"""Seeded synthetic inputs for the parity tests and bench.py (SURVEY.md §8d).

Distributions follow the reference's own test helpers (gmm/model-test-common.cc:91-108
`InitRandDiagGmm`: weights = softmax(N(0,1)), means = N(0,1)/(1+d), vars = exp(N(0,1))/(1+d) + 0.01 ...)
scaled to the LibriSpeech-shape configs; #Gaussians per pdf follows the power-law mix-up rule of
`AmDiagGmm::SplitByCount` (am-diag-gmm.cc, power 0.25).
"""
from dataclasses import dataclass

import numpy as np

LOG_2PI = 1.8378770664093454835606594728112


@dataclass
class GmmModel:
    """Flattened AmDiagGmm: pdf p owns Gaussians [pdf_offsets[p], pdf_offsets[p+1])."""
    pdf_offsets: np.ndarray  # int32 [P+1]
    weights: np.ndarray      # f32 [N]
    means: np.ndarray        # f32 [N, D]
    iv: np.ndarray           # f32 [N, D]  inverse variances (DiagGmm::inv_vars_)
    miv: np.ndarray          # f32 [N, D]  means * inverse variances (DiagGmm::means_invvars_)
    gconsts: np.ndarray      # f32 [N]

    @property
    def num_pdfs(self):
        return len(self.pdf_offsets) - 1

    @property
    def num_gauss(self):
        return len(self.gconsts)

    @property
    def dim(self):
        return self.means.shape[1]


def compute_gconsts(weights, miv, iv):
    """DiagGmm::ComputeGconsts (gmm/diag-gmm.cc:114-152), float accumulation over d."""
    D = miv.shape[1]
    gc = (np.log(weights.astype(np.float32)) + np.float32(-0.5 * LOG_2PI * D)).astype(np.float32)
    term = (0.5 * np.log(iv.astype(np.float32)).astype(np.float64)
            - 0.5 * miv.astype(np.float64) * miv.astype(np.float64) / iv.astype(np.float64))
    for d in range(D):
        gc = (gc.astype(np.float64) + term[:, d]).astype(np.float32)
    gc = np.where(np.isposinf(gc), -np.inf, gc).astype(np.float32)
    return gc


def pdf_sizes(P, N, rng, power=0.25):
    """#Gaussians per pdf ∝ occupancy^power with occupancies ~ lognormal, min 1, exactly N in total."""
    occ = rng.lognormal(mean=0.0, sigma=2.0, size=P)
    t = occ ** power
    sizes = np.maximum(1, np.floor(t / t.sum() * N)).astype(np.int64)
    # distribute the remainder to the largest targets, deterministically
    rem = N - int(sizes.sum())
    order = np.argsort(-t, kind="stable")
    i = 0
    while rem != 0:
        p = order[i % P]
        if rem > 0:
            sizes[p] += 1
            rem -= 1
        elif sizes[p] > 1:
            sizes[p] -= 1
            rem += 1
        i += 1
    return sizes.astype(np.int32)


def make_model(P, N, D, seed, spread=1.0):
    """Random AmDiagGmm in the style of InitRandDiagGmm, but with speech-like scaling: per-dimension
    scale 1/(1+0.1 d), means ~ spread * N(0,1) * scale_d, variances exp(0.5 N(0,1)) * scale_d^2."""
    rng = np.random.default_rng(seed)
    sizes = pdf_sizes(P, N, rng) if N > P else np.ones(P, np.int32)
    offs = np.zeros(P + 1, np.int32)
    offs[1:] = np.cumsum(sizes)
    Ntot = int(offs[-1])
    scale = (1.0 / (1.0 + 0.1 * np.arange(D))).astype(np.float32)
    centers = rng.standard_normal((P, D)).astype(np.float32) * spread
    means = np.repeat(centers, sizes, axis=0) + 0.5 * rng.standard_normal((Ntot, D)).astype(np.float32)
    means = (means * scale).astype(np.float32)
    var = (np.exp(0.5 * rng.standard_normal((Ntot, D))) * 0.6 + 0.01).astype(np.float32) * scale * scale
    iv = (1.0 / var).astype(np.float32)
    w = np.exp(rng.standard_normal(Ntot)).astype(np.float32)
    for p in range(P):  # softmax per pdf
        s = slice(offs[p], offs[p + 1])
        w[s] = w[s] / w[s].sum()
    miv = (means * iv).astype(np.float32)
    return GmmModel(offs, w, means, iv, miv, compute_gconsts(w, miv, iv))


def make_feats(model, T, seed):
    """Frames drawn near the model: pick a Gaussian, sample from it (like RandDiagGaussFeatures)."""
    rng = np.random.default_rng(seed)
    g = rng.integers(0, model.num_gauss, size=T)
    std = np.sqrt(1.0 / model.iv[g])
    return (model.means[g] + std * rng.standard_normal((T, model.dim))).astype(np.float32)


def make_alignment(P, T, seed, seg=7):
    """Random pdf id per ~seg-frame segment (SURVEY §8d cfg 5)."""
    rng = np.random.default_rng(seed)
    nseg = (T + seg - 1) // seg
    return np.repeat(rng.integers(0, P, size=nseg), seg)[:T].astype(np.int32)


def make_wave(n_samples, seed, samp_freq=16000.0):
    """Speech-like synthetic PCM: a few amplitude-modulated harmonic tones + Gaussian noise, int16."""
    rng = np.random.default_rng(seed)
    t = np.arange(n_samples, dtype=np.float64) / samp_freq
    x = np.zeros(n_samples)
    f0 = rng.uniform(90, 250)
    for h in range(1, 9):
        amp = rng.uniform(200, 3000) / h
        x += amp * np.sin(2 * np.pi * f0 * h * t * (1.0 + 0.02 * np.sin(2 * np.pi * rng.uniform(1, 4) * t)) + rng.uniform(0, 6.28))
    env = 0.55 + 0.45 * np.sin(2 * np.pi * rng.uniform(1.5, 4.0) * t + rng.uniform(0, 6.28))
    x = x * env + rng.standard_normal(n_samples) * 500.0 + rng.uniform(-200, 200)
    return np.clip(np.round(x), -32768, 32767).astype(np.int16)


def make_corpus(n_spk, utts_per_spk, min_s, max_s, seed, samp_freq=16000.0, fast=False):
    """Concatenated int16 PCM + sample offsets + utt2spk.  fast=True tiles a few base waves (for the
    large bench batches, where generation cost matters and content does not)."""
    rng = np.random.default_rng(seed)
    n_utts = n_spk * utts_per_spk
    lens = (rng.uniform(min_s, max_s, size=n_utts) * samp_freq).astype(np.int64)
    offs = np.zeros(n_utts + 1, np.int64)
    offs[1:] = np.cumsum(lens)
    pcm = np.empty(int(offs[-1]), np.int16)
    if fast:
        base = [make_wave(int(max_s * samp_freq), seed + 1000 + k, samp_freq) for k in range(8)]
    for u in range(n_utts):
        n = int(lens[u])
        if fast:
            b = base[u % len(base)]
            shift = int(rng.integers(0, 1000))
            pcm[offs[u]:offs[u + 1]] = np.roll(b, shift)[:n]
        else:
            pcm[offs[u]:offs[u + 1]] = make_wave(n, seed + 17 * u + 1, samp_freq)
    utt2spk = np.repeat(np.arange(n_spk, dtype=np.int32), utts_per_spk)
    return pcm, offs, utt2spk


def make_fmllr(n_spk, D, seed):
    """Per-speaker affine transforms A = I + 0.05 N(0,1), b = 0.1 N(0,1), laid out D x (D+1) (SURVEY §8d)."""
    rng = np.random.default_rng(seed)
    A = np.zeros((n_spk, D, D + 1), np.float32)
    A[:, :, :D] = np.eye(D, dtype=np.float32) + 0.05 * rng.standard_normal((n_spk, D, D)).astype(np.float32)
    A[:, :, D] = 0.1 * rng.standard_normal((n_spk, D)).astype(np.float32)
    return A


def make_lda(rows, cols, seed):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((rows, cols)) / np.sqrt(cols)).astype(np.float32)


def make_model_from_feats(feats, P, N, seed):
    """A model matched to given feature frames (as a trained model would be): pdf centres are random
    frames, Gaussians scatter around their pdf centre, variances are the global variance times a
    log-normal factor.  Keeps |loglike| in the realistic O(10^2) range on those features."""
    rng = np.random.default_rng(seed)
    feats = np.asarray(feats, np.float32)
    D = feats.shape[1]
    sizes = pdf_sizes(P, N, rng) if N > P else np.ones(P, np.int32)
    offs = np.zeros(P + 1, np.int32)
    offs[1:] = np.cumsum(sizes)
    Ntot = int(offs[-1])
    gstd = feats.std(axis=0).astype(np.float32) + 1e-3
    centers = feats[rng.integers(0, feats.shape[0], size=P)]
    means = np.repeat(centers, sizes, axis=0) + 0.5 * gstd * rng.standard_normal((Ntot, D)).astype(np.float32)
    means = means.astype(np.float32)
    var = (gstd * gstd * (0.6 * np.exp(0.5 * rng.standard_normal((Ntot, D))) + 0.01)).astype(np.float32)
    iv = (1.0 / var).astype(np.float32)
    w = np.exp(rng.standard_normal(Ntot)).astype(np.float32)
    for p in range(P):
        s = slice(offs[p], offs[p + 1])
        w[s] = w[s] / w[s].sum()
    miv = (means * iv).astype(np.float32)
    return GmmModel(offs, w, means, iv, miv, compute_gconsts(w, miv, iv))


def make_pitch_wave(n_samples, seed, samp_freq=16000.0):
    """Voiced stretches with a gliding fundamental (70..320 Hz), separated by noise-only pauses: exercises the
    voiced / unvoiced decisions of a pitch tracker.  int16."""
    rng = np.random.default_rng(seed)
    t = np.arange(n_samples, dtype=np.float64) / samp_freq
    f0 = rng.uniform(80, 260) * (1.0 + 0.25 * np.sin(2 * np.pi * rng.uniform(0.3, 1.2) * t + rng.uniform(0, 6.28)))
    ph = 2 * np.pi * np.cumsum(f0) / samp_freq
    x = np.zeros(n_samples)
    for h in range(1, 7):
        x += rng.uniform(0.3, 1.0) / h * np.sin(h * ph + rng.uniform(0, 6.28))
    gate = (np.sin(2 * np.pi * rng.uniform(0.6, 1.6) * t + rng.uniform(0, 6.28)) > -0.25).astype(np.float64)
    k = int(0.01 * samp_freq)
    if n_samples > k:
        gate = np.convolve(gate, np.ones(k) / k, mode="same")
    x = 4000.0 * x * gate + rng.standard_normal(n_samples) * 250.0 + rng.uniform(-100, 100)
    return np.clip(np.round(x), -32768, 32767).astype(np.int16)


def phone_topology(n_phones):
    """A Kaldi-style HMM topology and its per transition-id tables: phone 1 is a 1-state phone, phones 2 ... n_phones are
    3-state left-to-right phones (pdf classes 0, 1, 2; each emitting state has a self-loop, then a forward transition;
    the last state is final, non-emitting).  Every (phone, state) has its own pdf, so <Triples> and <Tuples> agree.
    Returns a dict: the tables of vbgpu_tid_tables (phone, hmm_state, pdf_class, trans_state, flags, [num_tids + 1]),
    entries (per topology entry: [(forward_pdf_class, self_loop_pdf_class, [destination, ...]), ...]), phone2entry,
    tuples [(phone, hmm_state, forward_pdf, self_loop_pdf)] and tid {(phone, state, is_self_loop): transition-id}."""
    one = [(0, 0, [0, 1]), (-1, -1, [])]
    three = [(0, 0, [0, 1]), (1, 1, [1, 2]), (2, 2, [2, 3]), (-1, -1, [])]
    entries = [one, three]
    phone2entry = {p: (0 if p == 1 else 1) for p in range(1, n_phones + 1)}
    tuples, cols, tid = [], {k: [0] for k in ("phone", "hmm_state", "pdf_class", "trans_state", "flags")}, {}
    for p in range(1, n_phones + 1):
        e = entries[phone2entry[p]]
        for s, (fwd, slf, dsts) in enumerate(e):
            if fwd < 0:
                continue
            tuples.append((p, s, len(tuples), len(tuples)))
            for d in dsts:
                is_self = d == s
                tid[(p, s, is_self)] = len(cols["phone"])
                cols["phone"].append(p)
                cols["hmm_state"].append(s)
                cols["pdf_class"].append(slf if is_self else fwd)
                cols["trans_state"].append(len(tuples))
                cols["flags"].append((1 if is_self else 0) | (2 if d + 1 == len(e) else 0) | (4 if e[0][0] >= 0 else 0))
    out = {k: np.asarray(v, np.int32) for k, v in cols.items()}
    out.update(entries=entries, phone2entry=phone2entry, tuples=tuples, tid=tid)
    return out


def phone_alignment(topo, phones, durations, reordered=False):
    """Transition-ids of a phone sequence: durations[i] holds the frames of each emitting state of phones[i] (>= 1 each).
    Plain: a state's self-loops, then its forward transition; reordered: the forward transition first."""
    out = []
    for p, durs in zip(phones, durations):
        for s, d in enumerate(durs):
            run = [topo["tid"][(p, s, True)]] * (d - 1)
            fwd = topo["tid"][(p, s, False)]
            out += ([fwd] + run) if reordered else (run + [fwd])
    return np.asarray(out, np.int32)


def make_phone_alignment(n_phones, frame_offsets, seed, reordered=False, zipf=1.0, mean_state_frames=3.0):
    """Alignments that fill every utterance of a packed batch exactly: phones drawn with Zipf-like frequencies
    (p(rank r) ~ 1 / r^zipf, so that triphone keys repeat as in speech), state durations 1 + Poisson(mean - 1); the
    last phone of an utterance is shortened to fit, or is the 1-state phone.  Returns (topology, tids[T], phone
    sequence per utterance)."""
    rng = np.random.default_rng(seed)
    topo = phone_topology(n_phones)
    freq = 1.0 / np.arange(1, n_phones + 1) ** zipf
    freq /= freq.sum()
    rank2phone = rng.permutation(np.arange(1, n_phones + 1))
    fo = np.asarray(frame_offsets, np.int64)
    tids, seqs = [], []
    for u in range(len(fo) - 1):
        rem = int(fo[u + 1] - fo[u])
        phones, durs = [], []
        while rem > 0:
            p = int(rank2phone[rng.choice(n_phones, p=freq)])
            ns = len(topo["entries"][topo["phone2entry"][p]]) - 1
            d = list(1 + rng.poisson(mean_state_frames - 1.0, ns))
            if sum(d) > rem:
                if rem >= ns:
                    d = [1] * ns
                    d[-1] += rem - ns
                else:
                    p, d = 1, [rem]
            phones.append(p)
            durs.append(d)
            rem -= sum(d)
        seqs.append(phones)
        tids.append(phone_alignment(topo, phones, durs, reordered))
    return topo, (np.concatenate(tids) if tids else np.zeros(0, np.int32)).astype(np.int32), seqs


def make_training_graphs(topo, phone_seqs, num_pdfs, seed, alt_prob=0.1, self_loop_scale=0.1, max_word_phones=3):
    """Training graphs (what compile-train-graphs makes of a transcript) for the phone sequences of make_phone_alignment,
    over `topo` (phone_topology), packed as vbgpu_align_create takes them.  Per utterance, the phones are cut into words of
    1 ... max_word_phones phones; the graph is
        start -eps-> J  word  J  word ... word  J -> pre -eps-> end
    where every J is a junction with an optional 1-state silence (phone 1): J -eps-> next, J -eps-> sil, sil -> next.  Each
    emitting HMM state gets a self-loop and a forward arc (transition-ids of topo["tid"], costs -s log 0.75 / -s log 0.25
    with s = self_loop_scale); with probability alt_prob a phone gets an alternative pronunciation (another 3-state phone in
    parallel, both joining the next state), so that such states have several incoming arcs.  `end` is final with cost 0,
    `pre` with cost 0.5.  The generating alignment (phone_alignment of the same sequence) is a path through the graph.
    tid2pdf maps every (phone, state) tuple to a distinct pdf of a num_pdfs-pdf model (at random).
    Returns a dict: state_offsets, start, final_cost, arc_offsets, arc_src, arc_dst, arc_ilabel, arc_weight, tid2pdf,
    num_tids."""
    rng = np.random.default_rng(seed)
    tid = topo["tid"]
    n_tuples = len(topo["tuples"])
    pdf_of_tuple = rng.permutation(num_pdfs)[:n_tuples] if n_tuples <= num_pdfs else rng.integers(0, num_pdfs, n_tuples)
    ts = topo["trans_state"]
    tid2pdf = np.zeros(len(ts), np.int32)
    tid2pdf[1:] = pdf_of_tuple[ts[1:] - 1]
    phones = sorted(topo["phone2entry"])
    w_self = float(np.float32(-self_loop_scale * np.log(0.75)))
    w_fwd = float(np.float32(-self_loop_scale * np.log(0.25)))
    w_sil = float(np.float32(-np.log(0.5)))
    w_alt, w_main = float(np.float32(-np.log(alt_prob or 1.0))), float(np.float32(-np.log(1.0 - alt_prob)))
    so, ao, start, finals, src, dst, lab, wt = [0], [0], [], [], [], [], [], []
    for seq in phone_seqs:
        fin = []

        def new(final=np.inf):
            fin.append(final)
            return len(fin) - 1

        def arc(a, b, label, w):
            src.append(a), dst.append(b), lab.append(label), wt.append(w)

        def connect(pending, s):
            for a, label, w in pending:
                arc(a, s, label, w)

        def phone(pending, p, extra=0.0):
            pending = [(a, label, w + extra) for a, label, w in pending]
            for i in range(len(topo["entries"][topo["phone2entry"][p]]) - 1):
                s = new()
                connect(pending, s)
                arc(s, s, tid[(p, i, True)], w_self)
                pending = [(s, tid[(p, i, False)], w_fwd)]
            return pending

        def junction(pending):
            j, sil = new(), new()
            connect(pending, j)
            arc(j, sil, 0, w_sil)
            arc(sil, sil, tid[(1, 0, True)], w_self)
            return [(j, 0, w_sil), (sil, tid[(1, 0, False)], w_fwd)]

        s0 = new()
        start.append(s0)
        pending = junction([(s0, 0, 0.0)])
        k = 0
        while k < len(seq):
            n = int(rng.integers(1, max_word_phones + 1))
            for p in seq[k:k + n]:
                if p != 1 and alt_prob > 0 and rng.random() < alt_prob:
                    q = int(rng.choice([x for x in phones if x not in (1, p)]))
                    pending = phone(pending, p, w_main) + phone(pending, q, w_alt)
                else:
                    pending = phone(pending, p)
            pending = junction(pending)
            k += n
        pre = new(0.5)
        connect(pending, pre)
        end = new(0.0)
        arc(pre, end, 0, 0.0)
        finals += fin
        so.append(len(finals))
        ao.append(len(src))
    return dict(state_offsets=np.asarray(so, np.int32), start=np.asarray(start, np.int32),
                final_cost=np.asarray(finals, np.float32), arc_offsets=np.asarray(ao, np.int64),
                arc_src=np.asarray(src, np.int32), arc_dst=np.asarray(dst, np.int32), arc_ilabel=np.asarray(lab, np.int32),
                arc_weight=np.asarray(wt, np.float32), tid2pdf=tid2pdf, num_tids=len(tid2pdf) - 1)


def make_decoding_graph(topo, n_words, num_pdfs, seed, phones_per_word=(1, 3), n_bigram=3, eps_olabel_frac=0.2,
                        self_loop_scale=0.1):
    """A decoding graph (HCLG-like, what mkgraph makes of a lexicon and a bigram grammar) over `topo` (phone_topology),
    as vbgpu_decoder_create takes it.  Word ids 1 ... n_words each get a distinct pronunciation of phones_per_word 3-state
    phones and one HMM chain E_w -> c_1 ... c_m (the arc into c_i emits the forward transition-id of its HMM state, a
    self-loop at c_i its self-loop transition-id).  Grammar: the backoff state G (the start state) has an epsilon arc
    to every E_w (unigram cost) and to an optional silence (phone 1) that returns to G; the end of word w goes by
    epsilon to its history state H_w, which has epsilon arcs to n_bigram successors' E_v and an epsilon backoff arc to
    G whose weight may be negative.  A fraction eps_olabel_frac of the words carries its olabel on the epsilon arcs into
    E_w, the others on their first emitting arc.  G and every H_w are final (several final states); the epsilon levels
    are c_m 0, H_w 1, G 2, E_w 3.  tid2pdf maps every (phone, state) tuple to a distinct pdf (at random) where the
    model has enough.  Returns a dict: num_states, start, final_cost, arc_src, arc_dst, arc_ilabel, arc_olabel,
    arc_weight, tid2pdf, num_tids, n_words, prons."""
    rng = np.random.default_rng(seed)
    tid = topo["tid"]
    n_tuples = len(topo["tuples"])
    pdf_of_tuple = rng.permutation(num_pdfs)[:n_tuples] if n_tuples <= num_pdfs else rng.integers(0, num_pdfs, n_tuples)
    ts = topo["trans_state"]
    tid2pdf = np.zeros(len(ts), np.int32)
    tid2pdf[1:] = pdf_of_tuple[ts[1:] - 1]
    phones = [p for p in sorted(topo["phone2entry"]) if p != 1]
    w_self = float(np.float32(-self_loop_scale * np.log(0.75)))
    w_fwd = float(np.float32(-self_loop_scale * np.log(0.25)))
    src, dst, ilab, olab, wt, fin = [], [], [], [], [], []

    def new(final=np.inf):
        fin.append(final)
        return len(fin) - 1

    def arc(a, b, i, o, w):
        src.append(a), dst.append(b), ilab.append(i), olab.append(o), wt.append(float(np.float32(w)))

    G = new(float(np.float32(rng.uniform(1.0, 3.0))))
    prons, seen = [], set()
    while len(prons) < n_words:
        pr = tuple(int(p) for p in rng.choice(phones, int(rng.integers(phones_per_word[0], phones_per_word[1] + 1))))
        if pr not in seen:
            seen.add(pr)
            prons.append(pr)
    uni = 1.0 / np.arange(1, n_words + 1)
    uni = -np.log(uni[rng.permutation(n_words)] / uni.sum())
    eps_ol = rng.random(n_words) < eps_olabel_frac
    entry, hist = [], []
    for k, pr in enumerate(prons):
        w = k + 1
        E = new()
        entry.append(E)
        prev, first = E, True
        for p in pr:
            for j in range(len(topo["entries"][topo["phone2entry"][p]]) - 1):
                c = new()
                arc(prev, c, tid[(p, j, False)], w if first and not eps_ol[k] else 0, w_fwd)
                arc(c, c, tid[(p, j, True)], 0, w_self)
                prev, first = c, False
        H = new(float(np.float32(rng.uniform(0.5, 4.0))))
        hist.append(H)
        arc(prev, H, 0, 0, 0.0)
    for k in range(n_words):
        arc(G, entry[k], 0, k + 1 if eps_ol[k] else 0, uni[k])
    for k in range(n_words):
        for v in rng.choice(n_words, min(n_bigram, n_words), replace=False):
            arc(hist[k], entry[v], 0, int(v) + 1 if eps_ol[v] else 0, rng.uniform(0.2, 2.0))
        arc(hist[k], G, 0, 0, rng.uniform(-0.5, 1.0))
    SE = new()
    arc(G, SE, 0, 0, -np.log(0.3))
    s1 = new()
    arc(SE, s1, tid[(1, 0, False)], 0, w_fwd)
    arc(s1, s1, tid[(1, 0, True)], 0, w_self)
    arc(s1, G, 0, 0, 0.0)
    return dict(num_states=len(fin), start=G, final_cost=np.asarray(fin, np.float32), arc_src=np.asarray(src, np.int32),
                arc_dst=np.asarray(dst, np.int32), arc_ilabel=np.asarray(ilab, np.int32),
                arc_olabel=np.asarray(olab, np.int32), arc_weight=np.asarray(wt, np.float32), tid2pdf=tid2pdf,
                num_tids=len(tid2pdf) - 1, n_words=n_words, prons=prons)


def sample_decoding_path(graph, seed, min_frames, self_loop_prob=0.5):
    """A random path of a decoding graph from the start state to a final state with at least min_frames emitting arcs:
    at each state a self-loop is taken with probability self_loop_prob (when there is one), else one of the other
    outgoing arcs uniformly; the walk stops at the first final state once min_frames frames are emitted.  Returns
    (words: the nonzero olabels along the path, tids[T]: its transition-ids, arcs: the arc indices of the path)."""
    rng = np.random.default_rng(seed)
    S = int(graph["num_states"])
    src, dst = np.asarray(graph["arc_src"]), np.asarray(graph["arc_dst"])
    lab, ol = np.asarray(graph["arc_ilabel"]), np.asarray(graph["arc_olabel"])
    order = np.argsort(src, kind="stable")
    off = np.searchsorted(src[order], np.arange(S + 1))
    s, arcs, T = int(graph["start"]), [], 0
    while not (T >= min_frames and graph["final_cost"][s] < np.inf):
        out = order[off[s]:off[s + 1]]
        loops = [a for a in out if dst[a] == s]
        other = [a for a in out if dst[a] != s]
        a = int(loops[0]) if loops and (not other or rng.random() < self_loop_prob) else int(rng.choice(other))
        arcs.append(a)
        T += lab[a] > 0
        s = int(dst[a])
    arcs = np.asarray(arcs, np.int64)
    return ([int(o) for o in ol[arcs] if o], lab[arcs][lab[arcs] > 0].astype(np.int32), arcs)
