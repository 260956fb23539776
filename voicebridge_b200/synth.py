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
