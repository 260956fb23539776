"""gmm-latgen-faster on the device (raw lattices), measured on the bench batch of one rank (bench.rank_corpus(1, 0)).

  python tools/bench_latgen.py [--iters 2] [--words 20000] [--workspace-gib 120] [--out FILE]

The batch, features, model and 20 000-word graph are tools/bench_decode.py's; beam 13, max_active 7000, lattice beam 6.
Times are CUDA events over --iters calls after a warm-up: vbgpu_decode_lattice_dev (features -> one-best + lattices)
and, in the same run, the one-best vbgpu_decode_dev.  The split into scoring, search, traceback and the lattice pass
(final prune and output) comes from a separate torch.profiler run, which also counts the workspace groups (search
launches per call).  Lattice states and arcs per frame, and the lattice store's peak per utterance, come from the
call's outputs.  One seeded utterance among the shortest is checked against tests/latgen_ref.py on the device's own
log-likelihoods (the restatement is slow).  Prints one JSON line (and writes it to --out)."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
from bench_align import card, event_ms  # noqa: E402
from tests.decode_ref import loglikes_in_pdf_order  # noqa: E402
from tests.latgen_ref import LATTICE_KEYS, latgen_ref  # noqa: E402
from voicebridge_b200 import capi, host, synth  # noqa: E402

N_PHONES, D, SCALE, MAX_WORDS = 200, 39, 0.1, 256
BEAM, MAX_ACTIVE, LATTICE_BEAM = 13.0, 7000, 6.0


def kernel_split(fn):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out, groups = {"scoring": 0.0, "search": 0.0, "traceback": 0.0, "lattice": 0.0, "other": 0.0}, 0
    for e in prof.events():
        if not str(getattr(e, "device_type", "")).endswith("CUDA") or "Memcpy" in e.name or "Memset" in e.name:
            continue
        k = ("search" if "decode_search_kernel" in e.name else "traceback" if "decode_traceback_kernel" in e.name
             else "lattice" if "decode_lattice_kernel" in e.name else "other" if "decode_" in e.name else "scoring")
        groups += k == "search"
        out[k] += e.time_range.elapsed_us() / 1000.0
    return out, groups


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=2)
    ap.add_argument("--words", type=int, default=20000)
    ap.add_argument("--workspace-gib", type=float, default=120.0)
    ap.add_argument("--arena-tokens", type=int, default=8192)
    ap.add_argument("--arena-links", type=int, default=24576)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_latgen needs a CUDA device"
    dev = torch.device("cuda", 0)
    s = torch.cuda.current_stream()
    info = card()

    pcm, so, u2s, n_spk, audio_s = bench.rank_corpus(1, 0)
    mfcc = host.Mfcc(capi.default_mfcc_opts(dither=0.0, use_energy=0))
    fo = mfcc.frame_offsets(so)
    T, n_utts = int(fo[-1]), len(so) - 1
    d_pcm = torch.from_numpy(pcm).to(dev)
    d_mf = torch.zeros((T, 16), dtype=torch.float32, device=dev)
    mfcc.compute_dev(d_pcm, so, d_mf, 16, stream=s)
    fp = host.FeaturePipeline(capi.default_feat_opts(), 13)
    cmvn = fp.cmvn_stats(d_mf[:, :13].cpu().numpy(), fo, u2s, n_spk)
    d_x = torch.zeros((T, D), dtype=torch.float32, device=dev)
    fp.run_dev(d_mf, 16, fo, d_x, D, u2s, n_spk, cmvn_stats=cmvn, stream=s)
    X = d_x.cpu().numpy()
    am = host.AmDiagGmmGpu.from_model(bench.make_bench_model(X[:200000]))
    g = synth.make_decoding_graph(synth.phone_topology(N_PHONES), args.words, bench.P_PDFS, bench.SEED + 41)
    C = am.NumCols()

    lo = capi.default_lattice_opts(lattice_beam=LATTICE_BEAM, arena_tokens=args.arena_tokens,
                                   arena_links=args.arena_links)
    lens = np.diff(fo)
    max_states, max_arcs = int(lens.max() + 1) * 64, int(lens.max() + 1) * 256  # lattice_status 2 beyond
    lo.max_states, lo.max_arcs = max_states, max_arcs
    z = lambda k, t=torch.int32: torch.zeros(k, dtype=t, device=dev)  # noqa: E731
    o = dict(d_ali=z(T), d_pdf_ids=z(T), d_words=z(n_utts * MAX_WORDS), d_num_words=z(n_utts),
             d_tot_cost=z(n_utts, torch.float64), d_status=z(n_utts))
    o1 = {k: torch.zeros_like(v) for k, v in o.items()}
    lat = {}
    for k, t, per_state in host.GmmDecodeFasterGpu.LATTICE_ARRAYS:
        lat[k] = torch.zeros(n_utts * (max_states if per_state else max_arcs),
                             dtype=torch.float32 if t == np.float32 else torch.int32, device=dev)
    for k in ("num_states", "num_arcs", "lattice_status"):
        lat[k] = z(n_utts)
    lat["arena_peak"] = z(2 * n_utts)

    dec = host.GmmDecodeFasterGpu(g, g["tid2pdf"], beam=BEAM, max_active=MAX_ACTIVE, max_tokens=65536)
    dec.set_workspace(int(args.workspace_gib * 2**30))

    def feats_to_lattices():
        dec.decode_lattice_dev(am, d_x, D, fo, max_words=MAX_WORDS, lattice=lat, lattice_opts=lo,
                               acoustic_scale=SCALE, stream=s, **o)

    def feats_to_words():
        dec.decode_dev(am, d_x, D, fo, max_words=MAX_WORDS, acoustic_scale=SCALE, stream=s, **o1)

    lat_ms = event_ms(feats_to_lattices, args.iters, s)
    one_ms = event_ms(feats_to_words, args.iters, s)
    split, groups = kernel_split(feats_to_lattices)
    torch.cuda.synchronize()
    same_one_best = all(torch.equal(o[k], o1[k]) for k in o)
    arr = {k: v.cpu().numpy() for k, v in lat.items()}
    st, ls = o["d_status"].cpu().numpy(), arr["lattice_status"]
    ok = (st <= 1) & (ls == 0)
    frames = lens + 1
    sp = arr["num_states"][ok] / frames[ok]
    ap_ = arr["num_arcs"][ok] / frames[ok]
    peak_t, peak_l = arr["arena_peak"][0::2], arr["arena_peak"][1::2]

    # one seeded utterance among the shortest tenth, against the restatement on the device's own log-likelihoods
    short = np.flatnonzero(lens <= np.quantile(lens, 0.1))
    u = int(np.random.default_rng(bench.SEED + 43).choice(short))
    n = int(lens[u])
    d_l2 = torch.zeros((n, C), dtype=torch.float32, device=dev)
    am.score_cols_dev(d_x[int(fo[u]):int(fo[u + 1])], n, D, d_l2, C, stream=s)
    torch.cuda.synchronize()
    ll = loglikes_in_pdf_order(d_l2.cpu().numpy(), am.col_of_pdf())
    t0 = time.perf_counter()
    r_one, r_lat = latgen_ref(g, ll, g["tid2pdf"], SCALE, BEAM, MAX_ACTIVE, 65536, LATTICE_BEAM)
    got = host.GmmDecodeFasterGpu.split_lattices(arr, n_utts, max_states, max_arcs)[u]
    identical = bool(r_one[0] == st[u] and np.array_equal(r_one[2], o["d_ali"].cpu().numpy()[fo[u]:fo[u + 1]]) and
                     all(np.array_equal(got[k].view(np.int32), r_lat[k].view(np.int32)) for k in LATTICE_KEYS))

    def rate(ms):
        return {"ms": round(ms, 3), "audio_s_per_s": round(T / 100.0 / (ms * 1e-3), 1) if ms > 0 else None}

    res = {"tool": "tools/bench_latgen.py", "gpu": info, "frames": T, "utterances": n_utts,
           "audio_s": round(audio_s, 1), "dim": D, "model": {"pdfs": bench.P_PDFS, "gaussians": bench.N_GAUSS},
           "graph": {"words": args.words, "states": int(g["num_states"]), "arcs": len(g["arc_src"])},
           "beam": BEAM, "max_active": MAX_ACTIVE, "lattice_beam": LATTICE_BEAM, "acoustic_scale": SCALE,
           "arena_tokens_per_frame": args.arena_tokens, "arena_links_per_frame": args.arena_links,
           "workspace_cap_gib": args.workspace_gib, "groups": groups, "iters": args.iters,
           "features_to_lattices": rate(lat_ms), "features_to_words_one_best": rate(one_ms),
           "kernels_profiler": {k: rate(v) for k, v in split.items()},
           "one_best_identical_to_decode": same_one_best,
           "status_counts": {str(k): int((st == k).sum()) for k in range(4)},
           "lattice_status_counts": {str(k): int((ls == k).sum()) for k in range(3)},
           "lattice_states_per_frame": {"mean": round(float(sp.mean()), 2), "max": round(float(sp.max()), 2)},
           "lattice_arcs_per_frame": {"mean": round(float(ap_.mean()), 2), "max": round(float(ap_.max()), 2)},
           "arena_peak_per_utterance": {"tokens_mean": round(float(peak_t.mean())), "tokens_max": int(peak_t.max()),
                                        "links_mean": round(float(peak_l.mean())), "links_max": int(peak_l.max()),
                                        "tokens_per_frame_max": round(float((peak_t / frames).max()), 1),
                                        "links_per_frame_max": round(float((peak_l / frames).max()), 1)},
           "sample_vs_restatement": {"utterance": u, "frames": n, "identical": identical,
                                     "states": int(got["num_states"]), "arcs": int(got["num_arcs"]),
                                     "restatement_s": round(time.perf_counter() - t0, 1)}}
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    assert same_one_best and identical, "correctness check failed"


if __name__ == "__main__":
    main()
