"""gmm-align-compiled on the device, measured on the bench batch of one rank (bench.rank_corpus(1, 0): 1 024 utterances).

  python tools/bench_align.py [--iters 5] [--sample 8] [--out FILE]

The realign chain of the training recipes: MFCC -> per-speaker CMVN + Δ + ΔΔ (vbgpu_feat_run_dev, D = 39) -> forced
alignment (vbgpu_align_dev) with the cfg 3 model (bench.make_bench_model: P = 4000, N = 40000) and transition costs.  The
training graphs come from synth.make_training_graphs over the phone sequences of synth.make_phone_alignment (200 phones):
optional silence between words, 10 % alternative pronunciations.
Times come from CUDA events over --iters calls after a warm-up; the split into subset scoring (every kernel that is not an
align_* kernel), Viterbi, traceback and the per-call arc weights comes from a separate torch.profiler run.  The host form
(vbgpu_align from host rows) is timed with a host clock; the device-resident realign + accumulate iteration is
vbgpu_align_dev -> vbgpu_acc_accumulate_dev + vbgpu_acc_accumulate_transitions_dev, timed with events.  A seeded sample of
--sample utterances is checked against tests/align_ref.py viterbi_align_ref on the device's own subset log-likelihoods
(identical alignments, costs to 1e-12 relative).  The CPU gmm-align-compiled of the reference is not measured (its sources
are needed to build it).  Prints one JSON line (and writes it to --out)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from tests.align_ref import align_subsets, viterbi_align_ref  # noqa: E402
from voicebridge_b200 import capi, host, synth  # noqa: E402

N_PHONES, D, SCALE = 200, 39, 0.1


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True).stdout.strip()
    name, power, clock = [v.strip() for v in q.split(",")]
    return {"name": name, "power_limit": power, "clocks_max_sm": clock}


def event_ms(fn, iters, stream):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(iters):
        fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def kernel_split(fn, iters):
    """Device time per group of kernels (ms per call) from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
    out = {"subset_scoring": 0.0, "viterbi": 0.0, "traceback": 0.0, "arc_weights": 0.0}
    for e in prof.events():
        if not str(getattr(e, "device_type", "")).endswith("CUDA") or "Memcpy" in e.name or "Memset" in e.name:
            continue
        k = ("viterbi" if "align_viterbi_kernel" in e.name else "traceback" if "align_traceback_kernel" in e.name
             else "arc_weights" if "align_weights_kernel" in e.name else "subset_scoring")
        out[k] += e.time_range.elapsed_us() / 1000.0 / iters
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--sample", type=int, default=8)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_align needs a CUDA device"
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

    t0 = time.perf_counter()
    topo, _, seqs = synth.make_phone_alignment(N_PHONES, fo, bench.SEED + 31)
    g = synth.make_training_graphs(topo, seqs, bench.P_PDFS, bench.SEED + 32)
    graph_s = time.perf_counter() - t0
    tid2pdf = g["tid2pdf"]
    tc = np.random.default_rng(bench.SEED + 33).uniform(0.0, 3.0, g["num_tids"] + 1).astype(np.float32)
    t0 = time.perf_counter()
    al = host.GmmAlignCompiledGpu(g, tid2pdf)
    create_s = time.perf_counter() - t0

    d_ali = torch.zeros(T, dtype=torch.int32, device=dev)
    d_pdf = torch.zeros(T, dtype=torch.int32, device=dev)
    d_cost = torch.zeros(n_utts, dtype=torch.float64, device=dev)

    def align():
        al.align_dev(am, d_x, D, fo, d_ali, d_pdf, d_cost, tid_cost=tc, acoustic_scale=SCALE, stream=s)
    align_ms = event_ms(align, args.iters, s)
    split = kernel_split(align, 2)
    bad = am.bad_count()

    acc = host.AccumAmDiagGmmGpu(am, num_tids=g["num_tids"])

    def iteration():
        align()
        acc.accumulate_dev(d_x, T, D, d_pdf, stream=s)
        acc.accumulate_transitions_dev(d_ali, T, stream=s)
    iter_ms = event_ms(iteration, args.iters, s)

    ali_dev, cost_dev = d_ali.cpu().numpy(), d_cost.cpu().numpy()
    al.Align(am, X, fo, tid_cost=tc, acoustic_scale=SCALE)  # warm-up (staging buffers)
    t0 = time.perf_counter()
    ali_h, pdf_h, cost_h = al.Align(am, X, fo, tid_cost=tc, acoustic_scale=SCALE)
    host_ms = (time.perf_counter() - t0) * 1e3
    host_same = bool(np.array_equal(ali_h, ali_dev) and np.array_equal(cost_h, cost_dev))

    # correctness sample: the restatement on the device's own subset log-likelihoods of the same features
    subs = align_subsets(g, tid2pdf)
    sample = sorted(np.random.default_rng(bench.SEED + 34).choice(n_utts, args.sample, replace=False).tolist())
    same_ali, max_rel = True, 0.0
    for u in sample:
        rows = slice(int(fo[u]), int(fo[u + 1]))
        blk = am.score_subset(X[rows], [0, fo[u + 1] - fo[u]], [subs[u]])[0]
        c, a, _ = viterbi_align_ref(g, u, blk, subs[u], tid2pdf, tc, SCALE)
        same_ali &= bool(np.array_equal(a, ali_dev[rows]))
        max_rel = max(max_rel, abs(cost_dev[u] - c) / abs(c))

    S = np.diff(g["state_offsets"]).astype(np.int64)
    A = np.diff(g["arc_offsets"])
    Tu = np.diff(fo)
    nsub = np.array([len(x) for x in subs], np.int64)
    tb_bytes = 2 if A.max() < 32768 else 4

    def rate(ms):
        return {"ms": round(ms, 4), "audio_s_per_s": round(T / 100.0 / (ms * 1e-3), 1)}

    res = {"tool": "tools/bench_align.py", "gpu": info, "frames": T, "utterances": n_utts, "audio_s": round(audio_s, 1),
           "dim": D, "model": {"pdfs": bench.P_PDFS, "gaussians": bench.N_GAUSS, "plan_note": am.plan_note()},
           "phones": N_PHONES, "acoustic_scale": SCALE, "tid_cost": "uniform [0, 3)",
           "graphs": {"states_mean": round(float(S.mean()), 1), "states_max": int(S.max()), "arcs_mean": round(float(A.mean()), 1),
                      "subset_mean": round(float(nsub.mean()), 1), "subset_max": int(nsub.max()),
                      "traceback_bytes": int(((Tu + 1) * S).sum() * tb_bytes), "subset_ll_bytes": int((Tu * nsub).sum() * 4),
                      "synth_s": round(graph_s, 2), "handle_create_s": round(create_s, 3)},
           "iters": args.iters,
           "align_dev": rate(align_ms),
           "align_kernels_profiler": {k: rate(v) for k, v in split.items()},
           "align_host_form": dict(rate(host_ms), note="host clock around the synchronous call: PCIe copy of the rows, "
                                                       "then the same work, alignments and costs back"),
           "host_form_same_as_dev": host_same,
           "realign_accumulate_iteration_dev": rate(iter_ms),
           "nonfinite_loglikes": bad,
           "unreachable_utterances": int(np.isinf(cost_dev).sum()),
           "sample_vs_restatement": {"utterances": sample, "alignments_identical": same_ali, "max_rel_cost_diff": max_rel},
           "cpu_reference_gmm_align_compiled": "not measured"}
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    assert same_ali and max_rel <= 1e-12 and host_same, "correctness sample failed"


if __name__ == "__main__":
    main()
