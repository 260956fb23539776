"""acc-lda on the device, measured on the bench batch of one rank (bench.rank_corpus(1, 0): 1 024 utterances).

  python tools/bench_lda.py [--iters 10] [--out FILE]

The LDA+MLLT recipe's statistics pass: MFCC -> per-speaker CMVN + splice +-3 (vbgpu_feat_run_dev, identity 91 x 91
transform) -> LDA class statistics (vbgpu_lda_accumulate_dev), C = 2 500 classes (cfg 4's pdf count), labels from
bench.synth_alignment and weight 0 for a fixed tenth of the classes ("silence").  Times come from CUDA events over
--iters launches after a warm-up; the split of the statistics into sort / class sums / triangle comes from a separate
torch.profiler run.  The host form (vbgpu_lda_accumulate from host spliced features) is timed with a host clock: it
copies 364 B per frame over PCIe and synchronises.  Prints one JSON line (and writes it to --out)."""
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
from voicebridge_b200 import capi, host  # noqa: E402

C_CLASSES, SPLICE = 2500, 3


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
    groups = {"sort": ("acc_hist_kernel", "acc_scan_kernel", "acc_scatter_kernel", "Memset"),
              "class_sums": ("lda_class_kernel",), "triangle": ("lda_tri_kernel",)}
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
    out = {k: 0.0 for k in groups}
    for e in prof.events():
        if str(getattr(e, "device_type", "")).endswith("CUDA"):
            us = e.time_range.elapsed_us()
            for k, names in groups.items():
                if any(n in e.name for n in names):
                    out[k] += us / 1000.0 / iters
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_lda needs a CUDA device"
    dev = torch.device("cuda", 0)
    s = torch.cuda.current_stream()
    info = card()

    pcm, so, u2s, n_spk, audio_s = bench.rank_corpus(1, 0)
    mfcc = host.Mfcc(capi.default_mfcc_opts(dither=0.0, use_energy=0))
    fo = mfcc.frame_offsets(so)
    T = int(fo[-1])
    K = 13 * (2 * SPLICE + 1)
    d_pcm = torch.from_numpy(pcm).to(dev)
    d_mf = torch.zeros((T, 16), dtype=torch.float32, device=dev)
    mfcc_ms = event_ms(lambda: mfcc.compute_dev(d_pcm, so, d_mf, 16, stream=s), args.iters, s)

    fp = host.FeaturePipeline(capi.default_feat_opts(mode=1, splice_left=SPLICE, splice_right=SPLICE), 13,
                              transform=np.eye(K, dtype=np.float32))
    cmvn = fp.cmvn_stats(d_mf[:, :13].cpu().numpy(), fo, u2s, n_spk)
    d_sp = torch.zeros((T, K), dtype=torch.float32, device=dev)
    feat_ms = event_ms(lambda: fp.run_dev(d_mf, 16, fo, d_sp, K, u2s, n_spk, cmvn_stats=cmvn, stream=s), args.iters, s)

    pdf, _ = bench.synth_alignment(C_CLASSES, fo, bench.SEED + 11)
    w = np.where(pdf % 10 == 0, 0.0, 1.0).astype(np.float32)
    d_ids, d_w = torch.from_numpy(pdf).to(dev), torch.from_numpy(w).to(dev)
    est = host.LdaEstimateGpu(C_CLASSES, K)
    lda_ms = event_ms(lambda: est.accumulate_dev(d_sp, T, K, d_ids, d_w, stream=s), args.iters, s)
    split = kernel_split(lambda: est.accumulate_dev(d_sp, T, K, d_ids, d_w, stream=s), 3)

    # the host form on host spliced features, checked against the device form
    feats = d_sp.cpu().numpy()
    est.ZeroAccumulators()
    est.accumulate_dev(d_sp, T, K, d_ids, d_w, stream=s)
    want = est.stats()
    est.ZeroAccumulators()
    est.Accumulate(feats, pdf, w)  # warm-up (staging buffers)
    est.ZeroAccumulators()
    t0 = time.perf_counter()
    est.Accumulate(feats, pdf, w)
    host_ms = (time.perf_counter() - t0) * 1e3
    got = est.stats()
    host_vs_dev = max(float(np.abs(g - h).max() / max(np.abs(h).max(), 1e-300)) for g, h in zip(got, want))

    fma = T * K * (K + 1) / 2
    stats_ms = sum(split.values())

    def rate(ms):
        return {"ms": round(ms, 4), "audio_s_per_s": round(T / 100.0 / (ms * 1e-3), 1)}

    res = {"tool": "tools/bench_lda.py", "gpu": info, "frames": T, "utterances": len(so) - 1, "speakers": int(n_spk),
           "audio_s": round(audio_s, 1), "classes": C_CLASSES, "dim": K, "zero_weight_frames": int((w == 0).sum()),
           "iters": args.iters,
           "mfcc": rate(mfcc_ms),
           "feat_run_dev_cmvn_splice": rate(feat_ms),
           "lda_accumulate_dev": rate(lda_ms),
           "lda_kernels_profiler": {k: rate(v) for k, v in split.items()},
           "lda_kernels_sum_ms": round(stats_ms, 4),
           "triangle_fp64_fma_per_s": fma / (split["triangle"] * 1e-3) if split["triangle"] else None,
           "triangle_fp64_tflops": 2 * fma / (split["triangle"] * 1e-3) / 1e12 if split["triangle"] else None,
           "triangle_algorithmic_fma": fma,
           "lda_accumulate_host_form": dict(rate(host_ms), bytes_per_frame=K * 4 + 8,
                                            note="host clock around the synchronous call: PCIe copy of features, ids "
                                                 "and weights, then the same kernels"),
           "host_form_vs_dev_form_max_rel_diff": host_vs_dev,
           "stats_kernels_faster_than_mfcc": bool(stats_ms < mfcc_ms)}
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
