"""acc-tree-stats on the device, measured on the bench batch of one rank (bench.rank_corpus(1, 0): 1 024 utterances).

  python tools/bench_tree_stats.py [--iters 10] [--out FILE]

The train_deltas chain: MFCC -> per-speaker CMVN + Δ + ΔΔ (vbgpu_feat_run_dev, D = 39) -> tree statistics
(vbgpu_tree_accumulate_dev), N = 3, P = 1, phone 1 context-independent.  Alignments are reordered (the recipes' default)
and drawn by synth.make_phone_alignment over 200 phones with Zipf-like frequencies (exponent 1.6: about 60 000 keys,
a quarter of the 2^18 key table), so that keys repeat as in speech.
Times come from CUDA events over --iters calls after a warm-up; the split into the per-utterance kernel (phones, keys,
hash table), the counting sort and the moments kernel comes from a separate torch.profiler run.  The sort runs over the
handle's whole id range (max_keys), so the profiler run is repeated with a handle sized 1.1 times the key count: what a
sort over the key count alone (read back per call) would cost, less the read-back.  The host form (vbgpu_tree_accumulate
from host rows) is timed with a host clock.  The CPU acc-tree-stats of the reference is not measured (its sources are
needed to build it).  Prints one JSON line (and writes it to --out)."""
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
from voicebridge_b200 import capi, host, synth  # noqa: E402

N_PHONES, ZIPF, MAX_KEYS, D = 200, 1.6, 1 << 18, 39


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
    groups = {"utterances_keys_hash": ("tree_utt_kernel",),
              "sort": ("acc_hist_kernel", "acc_scan_kernel", "acc_scatter_kernel", "Memset"),
              "moments": ("tree_moments_kernel",)}
    fn()
    torch.cuda.synchronize()
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
    assert torch.cuda.is_available(), "bench_tree_stats needs a CUDA device"
    dev = torch.device("cuda", 0)
    s = torch.cuda.current_stream()
    info = card()

    pcm, so, u2s, n_spk, audio_s = bench.rank_corpus(1, 0)
    mfcc = host.Mfcc(capi.default_mfcc_opts(dither=0.0, use_energy=0))
    fo = mfcc.frame_offsets(so)
    T = int(fo[-1])
    d_pcm = torch.from_numpy(pcm).to(dev)
    d_mf = torch.zeros((T, 16), dtype=torch.float32, device=dev)
    mfcc_ms = event_ms(lambda: mfcc.compute_dev(d_pcm, so, d_mf, 16, stream=s), args.iters, s)

    fp = host.FeaturePipeline(capi.default_feat_opts(), 13)
    cmvn = fp.cmvn_stats(d_mf[:, :13].cpu().numpy(), fo, u2s, n_spk)
    d_x = torch.zeros((T, D), dtype=torch.float32, device=dev)
    feat_ms = event_ms(lambda: fp.run_dev(d_mf, 16, fo, d_x, D, u2s, n_spk, cmvn_stats=cmvn, stream=s), args.iters, s)

    topo, tids, _ = synth.make_phone_alignment(N_PHONES, fo, bench.SEED + 21, reordered=True, zipf=ZIPF)
    d_tids = torch.from_numpy(tids).to(dev)
    ts = host.TreeStatsGpu(topo, D, MAX_KEYS, 3, 1, (1,))

    def run(h):
        return lambda: h.accumulate_dev(d_x, D, d_tids, fo, stream=s)
    tree_ms = event_ms(run(ts), args.iters, s)
    keys = ts.NumKeys()
    bad = ts.bad_count()
    split = kernel_split(run(ts), 3)
    tight_keys = (int(keys * 1.1) + 1023) // 1024 * 1024
    tight = host.TreeStatsGpu(topo, D, tight_keys, 3, 1, (1,))
    split_tight = kernel_split(run(tight), 3)

    # the host form on host rows, checked against the device form
    feats = d_x.cpu().numpy()
    ts.ZeroAccumulators()
    ts.accumulate_dev(d_x, D, d_tids, fo, stream=s)
    want = ts.download()
    ts.ZeroAccumulators()
    ts.AccumulateTreeStats(feats, tids, fo)  # warm-up (staging buffers)
    ts.ZeroAccumulators()
    t0 = time.perf_counter()
    ts.AccumulateTreeStats(feats, tids, fo)
    host_ms = (time.perf_counter() - t0) * 1e3
    got = ts.download()
    same_keys = bool(np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]) and np.array_equal(got[2], want[2]))
    host_vs_dev = max(float(np.abs(g - w).max() / max(np.abs(w).max(), 1e-300)) for g, w in zip(got[3:], want[3:]))

    def rate(ms):
        return {"ms": round(ms, 4), "audio_s_per_s": round(T / 100.0 / (ms * 1e-3), 1)}

    moments_bytes = T * D * 4 + T * 4  # rows (read once, gathered by key) and the sorted frame order
    res = {"tool": "tools/bench_tree_stats.py", "gpu": info, "frames": T, "utterances": len(so) - 1,
           "speakers": int(n_spk), "audio_s": round(audio_s, 1), "dim": D, "phones": N_PHONES,
           "context_width": 3, "central_position": 1, "alignment": "reordered, phone p(rank r) ~ 1 / r^%g" % ZIPF,
           "distinct_keys": keys, "max_keys": MAX_KEYS,
           "bad_utterances_and_dropped_frames_per_call": [b // (args.iters + 1) for b in bad],
           "iters": args.iters,
           "mfcc": rate(mfcc_ms),
           "feat_run_dev_cmvn_deltas": rate(feat_ms),
           "tree_accumulate_dev": rate(tree_ms),
           "tree_kernels_profiler": {k: rate(v) for k, v in split.items()},
           "tree_kernels_profiler_tight_table": dict({k: rate(v) for k, v in split_tight.items()}, max_keys=tight_keys),
           "moments_bytes_per_call": moments_bytes,
           "moments_gb_per_s": moments_bytes / (split["moments"] * 1e-3) / 1e9 if split["moments"] else None,
           "tree_accumulate_host_form": dict(rate(host_ms), bytes_per_frame=D * 4 + 4,
                                             note="host clock around the synchronous call: PCIe copy of rows and "
                                                  "transition-ids, then the same kernels"),
           "host_form_same_keys_and_counts": same_keys,
           "host_form_vs_dev_form_max_rel_diff": host_vs_dev,
           "cpu_reference_acc_tree_stats": "not measured"}
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
