"""gmm-decode-faster on the device, measured on the bench batch of one rank (bench.rank_corpus(1, 0): 1 024 utterances).

  python tools/bench_decode.py [--iters 3] [--sample 2] [--words 20000] [--out FILE]

Features: MFCC -> per-speaker CMVN + delta + delta-delta (vbgpu_feat_run_dev, D = 39), the cfg 3 model
(bench.make_bench_model: P = 4000, N = 40000).  Graph: synth.make_decoding_graph over 200 phones with --words words
(1-3 phones each, bigram grammar with 3 successors per word and epsilon backoff).  Two operating points: beam 13 /
max_active 7000 (the decode scripts' settings) and beam 16 / unlimited max_active (gmm-decode-faster's defaults); the
token capacity is 65536 per frame, and utterances that outgrow it (status 3) are counted.  Times are CUDA events over
--iters calls after a warm-up: vbgpu_decode_dev (features -> words) and PCM -> vbgpu_pipeline_score_cols_dev ->
vbgpu_decode_loglikes_dev (PCM -> words).  The split into scoring, search and traceback comes from a separate
torch.profiler run.  At the first point a seeded sample of utterances is checked against tests/decode_ref.py beam_decode_ref on the
device's own log-likelihoods, which also gives tokens per frame.  The CPU gmm-decode-faster of the reference is not
measured.  Prints one JSON line (and writes it to --out)."""
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
from tests.align_ref import _levels  # noqa: E402
from tests.decode_ref import beam_decode_ref, loglikes_in_pdf_order  # noqa: E402
from voicebridge_b200 import capi, host, synth  # noqa: E402

N_PHONES, D, SCALE, MAX_WORDS = 200, 39, 0.1, 256


def kernel_split(fn, iters):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
    out = {"scoring": 0.0, "search": 0.0, "traceback": 0.0, "other": 0.0}
    for e in prof.events():
        if not str(getattr(e, "device_type", "")).endswith("CUDA") or "Memcpy" in e.name or "Memset" in e.name:
            continue
        k = ("search" if "decode_search_kernel" in e.name else "traceback" if "decode_traceback_kernel" in e.name
             else "other" if "decode_" in e.name else "scoring")
        out[k] += e.time_range.elapsed_us() / 1000.0 / iters
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--sample", type=int, default=2)
    ap.add_argument("--words", type=int, default=20000)
    ap.add_argument("--workspace-gib", type=float, default=64.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_decode needs a CUDA device"
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
    pipe = host.ScoringPipeline(mfcc, fp, am)

    t0 = time.perf_counter()
    g = synth.make_decoding_graph(synth.phone_topology(N_PHONES), args.words, bench.P_PDFS, bench.SEED + 41)
    graph_s = time.perf_counter() - t0
    emit = g["arc_ilabel"] > 0
    levels = int(_levels(g["num_states"], g["arc_src"][~emit], g["arc_dst"][~emit]).max())
    C = am.NumCols()
    d_ll = torch.zeros((T, C), dtype=torch.float32, device=dev)
    z = lambda k, t=torch.int32: torch.zeros(k, dtype=t, device=dev)  # noqa: E731
    o = dict(d_ali=z(T), d_pdf_ids=z(T), d_words=z(n_utts * MAX_WORDS), d_num_words=z(n_utts),
             d_tot_cost=z(n_utts, torch.float64), d_status=z(n_utts))
    ll_sample = None
    sample = sorted(np.random.default_rng(bench.SEED + 42).choice(n_utts, args.sample, replace=False).tolist())

    def rate(ms):
        return {"ms": round(ms, 3), "audio_s_per_s": round(T / 100.0 / (ms * 1e-3), 1) if ms > 0 else None}

    points = []
    for beam, max_active in ((13.0, 7000), (16.0, 2**31 - 1)):
        dec = host.GmmDecodeFasterGpu(g, g["tid2pdf"], beam=beam, max_active=max_active, max_tokens=65536)
        dec.set_workspace(int(args.workspace_gib * 2**30))

        def feats_to_words():
            dec.decode_dev(am, d_x, D, fo, max_words=MAX_WORDS, acoustic_scale=SCALE, stream=s, **o)

        def pcm_to_words():
            pipe.score_cols_dev(d_pcm, so, u2s, n_spk, None, 0, d_ll, C, stream=s)
            dec.decode_loglikes_dev(am, d_ll, C, fo, max_words=MAX_WORDS, acoustic_scale=SCALE, stream=s, **o)

        f_ms = event_ms(feats_to_words, args.iters, s)
        split = kernel_split(feats_to_words, 1)
        torch.cuda.synchronize()
        st = o["d_status"].cpu().numpy()
        ali, nw, cost = o["d_ali"].cpu().numpy(), o["d_num_words"].cpu().numpy(), o["d_tot_cost"].cpu().numpy()
        p_ms = event_ms(pcm_to_words, args.iters, s)
        if ll_sample is None:  # the device's own log-likelihoods of the features the feature form scored
            ll_sample, cop = {}, am.col_of_pdf()
            for u in sample:
                n = int(fo[u + 1] - fo[u])
                d_l2 = torch.zeros((n, C), dtype=torch.float32, device=dev)
                am.score_cols_dev(d_x[int(fo[u]):int(fo[u + 1])], n, D, d_l2, C, stream=s)
                torch.cuda.synchronize()
                ll_sample[u] = loglikes_in_pdf_order(d_l2.cpu().numpy(), cop)
        check = None
        if not points:  # the restatement is slow: the first point only
            same, max_rel, tok = True, 0.0, []
            for u in sample:
                rows = slice(int(fo[u]), int(fo[u + 1]))
                r = beam_decode_ref(g, ll_sample[u], g["tid2pdf"], SCALE, beam, max_active, 65536, stats=tok)
                same &= bool(r[0] == st[u] and np.array_equal(r[2], ali[rows]) and r[5] == nw[u])
                if np.isfinite(r[1]):
                    max_rel = max(max_rel, abs(cost[u] - r[1]) / max(abs(r[1]), 1.0))
            check = {"utterances": sample, "identical": same, "max_rel_cost_diff": max_rel,
                     "tokens_per_frame_mean": round(float(np.mean(tok)), 1) if tok else None,
                     "tokens_per_frame_max": int(np.max(tok)) if tok else None}
        points.append({"beam": beam, "max_active": max_active, "max_tokens": 65536,
                       "features_to_words": rate(f_ms), "pcm_to_words": rate(p_ms),
                       "kernels_profiler": {k: rate(v) for k, v in split.items()},
                       "status_counts": {str(k): int((st == k).sum()) for k in range(4)},
                       "words_mean": round(float(nw.mean()), 1),
                       "sample_vs_restatement": check if check else "not checked"})
        dec.close()
        print(json.dumps(points[-1]), flush=True)

    res = {"tool": "tools/bench_decode.py", "gpu": info, "frames": T, "utterances": n_utts, "audio_s": round(audio_s, 1),
           "dim": D, "model": {"pdfs": bench.P_PDFS, "gaussians": bench.N_GAUSS, "plan_note": am.plan_note()},
           "acoustic_scale": SCALE,
           "graph": {"words": args.words, "phones": N_PHONES, "states": int(g["num_states"]), "arcs": len(g["arc_src"]),
                     "epsilon_levels": levels, "synth_s": round(graph_s, 2)},
           "workspace_cap_gib": args.workspace_gib, "iters": args.iters, "points": points,
           "cpu_reference_gmm_decode_faster": "not measured"}
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    checks = [p["sample_vs_restatement"] for p in points if isinstance(p["sample_vs_restatement"], dict)]
    assert checks and all(c["identical"] and c["max_rel_cost_diff"] <= 1e-12 for c in checks), "correctness sample failed"


if __name__ == "__main__":
    main()
