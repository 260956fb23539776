#!/usr/bin/env python
"""bench.py — audio-seconds/second of the acoustic-scoring hot path (PCM -> per-frame per-pdf diag-GMM loglikes).

  python bench.py --gpus N --steps K --warmup W            our arm (CUDA path through the C ABI)
  python bench.py --impl reference --gpus N --steps K ...  the reference's own CPU implementation on the host cores
  python bench.py ... --dump-outputs DIR                    also save a seeded sample of the last timed step's outputs

Workload (BASELINE.json configs[2], SURVEY.md §8d cfg 3 — the headline config): LibriSpeech-shape DELTA+SAT,
16 kHz synthetic int16 audio, 13 MFCC -> per-speaker CMVN -> delta+delta-delta (39) -> per-speaker fMLLR ->
P=4000 pdfs / N=40000 Gaussians.  One step = one pass over a batch of 32 speakers x 32 utterances of 5..20 s per GPU
(~1.28e6 frames, ~12 800 audio-seconds).  Weak scaling: every rank owns 32 whole speakers (speaker-level sharding,
voicebridge_b200/shard.py); scoring needs no collective.

`value`   : whole-job audio-s/s with PCM resident in HBM, loglikes written to HBM (device-timed, max over ranks).
`e2e`     : the same through vbgpu_pipeline_score_i16 with HOST buffers (pinned), H2D of the PCM and D2H of the
            [frames x 4000] float32 loglike matrix inside the timed region.
`roofline`: the scoring kernel alone, algorithmic FLOPs = 2*(2D+1)*N per frame, timed with CUDA events on the
            launching stream, against the measured dense bf16 tensor peak in MEASURED_PEAKS.json (and the TF32 line,
            half of it, which SURVEY.md §8d names).
`parity`  : 256 frames of the timed batch itself, all pdfs, against the reference's own CPU code (outside the timed region).
`e2e_align`: the same host-buffer path for a consumer that reads a pdf subset per utterance (forced alignment):
            vbgpu_pipeline_score_subset_i16, D2H = the subset only.
`em`      : BASELINE configs[4]: PCM + alignment -> GMM + transition statistics -> ONE NCCL all-reduce per pass.
Diagnostics: `ms_per_step_by_rank` / `roofline.kernel_ms_by_rank` (which rank set the max), `clocks.by_gpu` (every GPU of the job),
`rescored_frames_last_step` (frames the tensor-core path handed to the FP32 kernel: a slow step usually means broken input).
The loglike matrix of `value` is in DEVICE COLUMN ORDER (include/vbgpu.h: column col_of_pdf[p] holds pdf p; every consumer
goes through tid2pdf already); `value_pdf_order` is the same with the gather kernel that restores the model's pdf order.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SAMP = 16000.0
P_PDFS, N_GAUSS, DIM = 4000, 40000, 39
SPK_PER_GPU, UTT_PER_SPK, MIN_S, MAX_S = 32, 32, 5.0, 20.0
SEED = 1234 + 3
METRIC = "audio_sec_per_sec_pcm_to_gmm_loglikes"
UNIT = "audio-s/s"


def workload_config(n_gpus):
    return {
        "workload": "librispeech_delta_sat_scoring (BASELINE configs[2] / SURVEY cfg 3)",
        "sample_rate_hz": 16000, "mfcc": "13 ceps, 23 mel, povey 25ms/10ms, dither=0, use_energy=false",
        "features": "per-speaker CMVN + delta+delta-delta (39) + per-speaker fMLLR 39x40",
        "loglike_layout": "device column order [frames x n_cols] + col_of_pdf map (include/vbgpu.h); value_pdf_order adds the gather",
        "pdfs": P_PDFS, "gaussians": N_GAUSS, "dim": DIM,
        "batch_per_gpu": "%d speakers x %d utterances of %g..%g s" % (SPK_PER_GPU, UTT_PER_SPK, MIN_S, MAX_S),
        "parallelism": "speaker-sharded x%d, no collective" % n_gpus,
        "l2": "no flush needed: per step 0.4 GB of PCM in and 20 GB of loglikes out, both >> 126 MB L2",
    }


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return None


# ----------------------------------------------------------------------------------------------------------------------
# corpus: lengths for the whole job, speaker-sharded; each rank synthesises only its own audio
# ----------------------------------------------------------------------------------------------------------------------
def job_layout(n_gpus):
    rng = np.random.default_rng(SEED)
    n_spk = SPK_PER_GPU * n_gpus
    utt2spk = np.repeat(np.arange(n_spk, dtype=np.int32), UTT_PER_SPK)
    lens = (rng.uniform(MIN_S, MAX_S, size=len(utt2spk)) * SAMP).astype(np.int64)
    return utt2spk, lens


def rank_corpus(n_gpus, rank):
    from voicebridge_b200 import shard, synth
    utt2spk, lens = job_layout(n_gpus)
    frames = 1 + (lens - 400) // 160
    mine = shard.shard_speakers(utt2spk, frames, n_gpus)[rank]
    so = np.zeros(len(mine) + 1, np.int64)
    so[1:] = np.cumsum(lens[mine])
    base = [synth.make_wave(int(MAX_S * SAMP), SEED + 1000 + k, SAMP) for k in range(8)]
    pcm = np.empty(int(so[-1]), np.int16)
    rng = np.random.default_rng(SEED + 77 + rank)
    for i, u in enumerate(mine):
        n = int(lens[u])
        pcm[so[i]:so[i + 1]] = np.roll(base[int(u) % 8], int(rng.integers(0, 4000)))[:n]
    spk_ids, local = np.unique(utt2spk[mine], return_inverse=True)
    return pcm, so, local.astype(np.int32), len(spk_ids), float(so[-1]) / SAMP


def sample_corpus(n_spk, utts, secs, seed):
    """Bounded CPU sample of the same workload: n_spk speakers x utts utterances x secs seconds."""
    from voicebridge_b200 import synth
    base = [synth.make_wave(int(secs * SAMP), SEED + 1000 + k, SAMP) for k in range(8)]
    n = int(secs * SAMP)
    pcm = np.empty(n_spk * utts * n, np.int16)
    rng = np.random.default_rng(seed)
    for u in range(n_spk * utts):
        pcm[u * n:(u + 1) * n] = np.roll(base[u % 8], int(rng.integers(0, 4000)))
    so = np.arange(n_spk * utts + 1, dtype=np.int64) * n
    return pcm, so, np.repeat(np.arange(n_spk, dtype=np.int32), utts)


def ncu_traffic(frames):
    """dram__bytes_read.sum + dram__bytes_write.sum of the scoring kernel per launch, from the committed ncu --set full
    capture of this launch (a number taken under the profiler is evidence, never a bench value).  The capture was taken
    at 1 262 745 frames (the N=1 batch); the kernel's DRAM traffic is linear in the frame count (features in, loglikes
    out; the 12.8 MB model image stays in L2), so other batch sizes are scaled by frames and flagged as such."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_score_tc_final.json")))
        total = d["dram_bytes_read"] + d["dram_bytes_write"]
        if d["frames"] == frames:
            return total, "measured at this launch size"
        return total * frames / d["frames"], "scaled by frames from the capture at %d frames" % d["frames"]
    except Exception:
        return None, "no capture"


def make_bench_model(feats_sample):
    from voicebridge_b200 import synth
    return synth.make_model_from_feats(feats_sample, P_PDFS, N_GAUSS, SEED)


# ----------------------------------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi sampling (every 25 ms) of the job's GPUs from rank 0.  The clocks line is GPU `device`'s; with several
    GPUs `by_gpu` carries the same figures for each of them, so a rank that sets the max-over-ranks time can be matched with
    a throttled device."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, device, n_gpus=1):
        self.proc, self.lines, self.device = None, [], int(device)
        ids = ",".join(str(i) for i in range(n_gpus)) if n_gpus > 1 else str(device)
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", ids, "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    @classmethod
    def _summary(cls, rows):
        sm, mx, pw = [r[0] for r in rows], [r[1] for r in rows], [r[2] for r in rows]
        reasons = sorted({nm for r in rows for nm in r[3]})
        busy = [c for c, p in zip(sm, pw) if p >= 0.5 * max(pw)] or sm
        return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": float(max(mx)), "reasons": reasons,
                "power_w_max": float(max(pw)), "samples": len(sm)}

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        by_gpu = {}
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                row = (float(f[1]), float(f[2]), float(f[3]), [nm for nm, v in zip(self.NAMES, f[4:8]) if v == "Active"])
                by_gpu.setdefault(int(f[0]), []).append(row)
            except ValueError:
                continue
        if self.device not in by_gpu:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        out = self._summary(by_gpu[self.device])
        if len(by_gpu) > 1:
            out["by_gpu"] = [dict(gpu=g, **self._summary(by_gpu[g])) for g in sorted(by_gpu)]
            out["reasons"] = sorted({r for g in out["by_gpu"] for r in g["reasons"]})
        return out


# ----------------------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's own code (oracle/_ref) or, failing that, the oracle port
# ----------------------------------------------------------------------------------------------------------------------
def cpu_reference_run(steps, warmup, target_s=12.0):
    """Times PCM -> loglikes on the host cores.  Returns dict(value, cores, kind, sample, ms_per_step, audio_s)."""
    import ctypes as C
    from oracle import pyoracle as po
    from voicebridge_b200 import synth
    cores = os.cpu_count() or 1
    o = po.default_opts(dither=0.0, use_energy=0)
    try:
        ref = po.load("ref") if po.have_ref() else None
    except OSError:
        ref = None
    orc = po.load("orc")
    # a model matched to the data, built with the CPU chain itself
    w = synth.make_wave(int(8 * SAMP), SEED + 1000, SAMP).astype(np.float32)
    mf = orc.mfcc(o, w)
    fs = orc.deltas(orc.cmvn_apply(orc.cmvn_acc(mf), mf))
    model = make_bench_model(fs)
    if ref is not None:
        kind, nj = "reference", cores
        # ~10 audio-s/s/core at N=40k (BASELINE.md §2): size the sample for ~target_s seconds per step
        secs_per_spk = max(10.0, 8.0 * target_s)
        utts = max(1, int(round(secs_per_spk / 10.0)))
        pcm, so, u2s = sample_corpus(nj, utts, 10.0, SEED + 5)
        fm = synth.make_fmllr(nj, DIM, SEED + 6)
        h = ref.ref_model(model.pdf_offsets, model.weights, model.means, model.iv)
        fo = np.zeros(len(so), np.int64)
        fo[1:] = np.cumsum([ref.num_frames(int(so[i + 1] - so[i]), o) for i in range(len(so) - 1)])

        def step():
            n = ref.lib.ref_pcm_to_loglikes(C.byref(o), C.c_void_p(h), pcm.ctypes.data_as(C.c_void_p),
                                            so.ctypes.data_as(C.c_void_p), C.c_int32(len(so) - 1),
                                            u2s.ctypes.data_as(C.c_void_p), C.c_int32(nj), C.c_int32(0), C.c_int32(0),
                                            C.c_int32(2), C.c_int32(2), None, C.c_int32(0), C.c_int32(0),
                                            fm.ctypes.data_as(C.c_void_p), C.c_int32(nj), None,
                                            fo.ctypes.data_as(C.c_void_p), C.c_int32(P_PDFS))
            assert n == fo[-1], n
        audio_s = float(so[-1]) / SAMP
        sample = "%d speakers x %d utts x 10 s (%.0f audio-s), nj=%d threads, OpenBLAS 1 thread/worker" % (
            nj, utts, audio_s, nj)
    else:
        kind, nj = "port", 1
        pcm, so, u2s = sample_corpus(1, 1, 2.0 * target_s / 12.0 + 1.0, SEED + 5)
        fm = synth.make_fmllr(1, DIM, SEED + 6)

        def step():
            mfc = orc.mfcc(o, pcm.astype(np.float32))
            f = orc.transform(orc.deltas(orc.cmvn_apply(orc.cmvn_acc(mfc), mfc)), fm[0])
            orc.gmm_loglikes(model, f)
        audio_s = float(so[-1]) / SAMP
        sample = "1 utterance of %.1f s, scalar C port, 1 thread" % audio_s
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    return {"value": audio_s / dt, "unit": UNIT, "cores": nj, "kind": kind, "sample": sample,
            "ms_per_step": dt * 1e3, "audio_s": audio_s}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = args.steps
    warm = 1 if args.warmup > 0 else 0
    r = cpu_reference_run(steps, warm, target_s=8.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args.gpus),
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
                         "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "steps_requested": args.steps, "warmup_requested": args.warmup,
        "note": "the reference's CPU path uses the host cores only: the same number is reported for every --gpus; warmup "
                "is CAPPED at 1 (each step is ~8 s of CPU work on a bounded sample of the workload)",
    }
    print(json.dumps(line), flush=True)


def nccl_comm(rank, world, device):
    """A raw ncclComm_t for vbgpu_acc_allreduce (the C-ABI path a C++ host uses): the unique id is made on rank 0 and
    shared through torch.distributed."""
    import ctypes as C
    import glob
    import torch
    import torch.distributed as dist
    cands = glob.glob(os.path.join(os.path.dirname(torch.__file__), "..", "nvidia", "nccl", "lib", "libnccl.so.2"))
    lib = C.CDLL(cands[0] if cands else "libnccl.so.2", mode=C.RTLD_GLOBAL)

    class UniqueId(C.Structure):
        _fields_ = [("internal", C.c_byte * 128)]
    uid = UniqueId()
    if rank == 0:
        assert lib.ncclGetUniqueId(C.byref(uid)) == 0
    t = torch.frombuffer(bytearray(bytes(uid.internal)), dtype=torch.uint8).clone().cuda(device)
    dist.broadcast(t, 0)
    C.memmove(C.byref(uid), bytes(t.cpu().numpy().tobytes()), 128)
    comm = C.c_void_p()
    lib.ncclCommInitRank.argtypes = [C.POINTER(C.c_void_p), C.c_int, UniqueId, C.c_int]
    assert lib.ncclCommInitRank(C.byref(comm), world, uid, rank) == 0
    return lib, comm


def synth_alignment(P, fo, seed):
    """Per-frame pdf ids and transition ids of a synthetic alignment: a new pdf every ~7 frames inside each utterance;
    transition-id = 2 * pdf + 1 (self-loop) or 2 * pdf + 2 (the segment's last frame), NumTransitionIds() = 2 P."""
    from voicebridge_b200 import synth
    T = int(fo[-1])
    pdf = synth.make_alignment(P, T, seed)
    last = np.ones(T, bool)
    last[:-1] = pdf[1:] != pdf[:-1]
    last[np.asarray(fo[1:], np.int64) - 1] = True
    return pdf, (2 * pdf + 1 + last).astype(np.int32)


def bind_to_gpu_numa(local):
    """Multi-rank runs only: pin this rank's host threads (hence its first-touch pinned buffers) to the NUMA node its GPU
    hangs off, the way a production job launcher binds one job per GPU.  With 8 ranks each returning 20 GB of loglikes per
    step, host-memory placement decides the end-to-end rate.  Returns the node, or None when nothing was changed."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


# ----------------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from voicebridge_b200 import capi, host, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    numa_node = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL_DEBUG=VERSION / WARN make NCCL print its version banner on stdout, where the bench prints ONE line: drop those
        # levels (INFO and above are left alone: whoever sets them wants the log)
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
            del os.environ["NCCL_DEBUG"]
        numa_node = bind_to_gpu_numa(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    n_gpus = world

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def all_ranks(x):
        """x of every rank, in rank order (diagnostics: which rank set the max)."""
        if world == 1:
            return [float(x)]
        t = torch.zeros(world, dtype=torch.float64, device=dev)
        t[rank] = x
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [round(float(v), 3) for v in t.tolist()]

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- build the job ----
    opts = capi.default_mfcc_opts(dither=0.0, use_energy=0)
    mfcc = host.Mfcc(opts, device=local)
    fp = host.FeaturePipeline(capi.default_feat_opts(), 13, device=local)
    pcm, so, u2s, n_spk, audio_s = rank_corpus(n_gpus, rank)
    fo = mfcc.frame_offsets(so)
    T = int(fo[-1])
    # model matched to the data (same on every rank): features of 8 s of the shared base audio
    w = synth.make_wave(int(8 * SAMP), SEED + 1000, SAMP)
    mf, mfo = mfcc.compute_batch(w, [0, len(w)])
    fs = fp.run(mf, mfo, cmvn_stats=fp.cmvn_stats(mf, mfo))
    model = make_bench_model(fs)
    am = host.AmDiagGmmGpu.from_model(model, device=local)
    if args.kernel:
        am.set_kernel(args.kernel)
    pipe = host.ScoringPipeline(mfcc, fp, am)
    fm = synth.make_fmllr(n_spk, DIM, SEED + 6 + rank)

    d_pcm = torch.from_numpy(pcm).to(dev)
    d_fm = torch.from_numpy(fm).to(dev)
    n_cols = am.NumCols()            # device column order: n_cols >= P, column col_of_pdf[p] holds pdf p
    col_of_pdf = am.col_of_pdf()
    d_ll = torch.empty((T, n_cols), dtype=torch.float32, device=dev)
    d_feats = torch.empty((T, 40), dtype=torch.float32, device=dev)
    stream = torch.cuda.current_stream()

    def step():
        pipe.score_cols_dev(d_pcm, so, u2s, n_spk, d_fm, DIM + 1, d_ll, n_cols, d_feats, 40, stream)

    # ---- device-resident throughput (`value`) ----
    # nvidia-smi needs ~0.2 s to start: launch it before the warm-up so that it is sampling (every 25 ms) by the time
    # the timed region runs; samples taken under load (power >= half the maximum seen) make the clocks line.
    sampler = ClockSampler(local, world) if rank == 0 else None
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    barrier()
    ms_local = e0.elapsed_time(e1) / args.steps
    ms = max_over_ranks(ms_local)
    ms_by_rank = all_ranks(ms_local)
    bad = am.bad_count()
    rescored = int(sum_over_ranks(am.rescored_frames()))   # frames of the last step the FP32 kernel had to re-score
    total_audio = sum_over_ranks(audio_s)
    value = total_audio / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d_ll, d_feats, col_of_pdf, T)

    # ---- parity on the timed batch itself (outside the timed region): 256 frames, all pdfs, vs the reference's CPU code ----
    parity = None
    if rank == 0:
        try:
            from oracle import pyoracle as po
            chk, kind = (po.load("ref"), "reference (oracle/_ref/libvbref.so)") if po.have_ref() else (po.load("orc"), "oracle port")
            rows = np.sort(np.random.default_rng(SEED).choice(T, 256, replace=False))
            x = d_feats[torch.from_numpy(rows).to(dev)][:, :DIM].cpu().numpy()
            got = d_ll[torch.from_numpy(rows).to(dev)].cpu().numpy()[:, col_of_pdf]
            rc, want = chk.gmm_loglikes(model, x)
            err, mag = np.abs(got - want), np.abs(want)
            bins = {}
            for lo, hi in ((0, 500), (500, 1000), (1000, 2000), (2000, 1e9)):
                sel = (mag >= lo) & (mag < hi)
                if sel.any():  # the reference computes in FP32: its own ulp is 6e-5 at |ll| = 500 and 4.9e-4 at 5000
                    bins["|ll| in [%d, %s)" % (lo, "inf" if hi > 1e8 else "%d" % hi)] = {
                        "share": float(sel.mean()), "max_abs_err": float(err[sel].max())}
            parity = {"frames": 256, "pdfs": P_PDFS, "checker": kind, "max_abs_err": float(err.max()),
                      "max_abs_ll": float(mag.max()), "median_abs_ll": float(np.median(mag)),
                      "by_magnitude": bins, "tolerance": 1e-3, "rc": int(rc),
                      "note": "the timed batch scores fMLLR-transformed features against a model built on untransformed ones: "
                              "a share of its log-likelihoods lies thousands of nats out, where 1e-3 absolute is ~2 ulp of the "
                              "reference's own FP32 result"}
        except Exception as ex:  # the checker must never take the bench line down
            parity = {"error": repr(ex)}

    # ---- dominant kernel alone: scoring on the resident features (roofline) ----
    k_iters = max(3, min(args.steps, 10))
    am.score_cols_dev(d_feats, T, 40, d_ll, n_cols, stream)
    torch.cuda.synchronize()
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k0.record(stream)
    for _ in range(k_iters):
        am.score_cols_dev(d_feats, T, 40, d_ll, n_cols, stream)
    k1.record(stream)
    torch.cuda.synchronize()
    k_ms = k0.elapsed_time(k1) / k_iters
    k_ms_by_rank = all_ranks(k_ms)
    # the same step with the model's pdf order restored on the device (one extra gather kernel over the matrix)
    d_ll_pdf = torch.empty((T, P_PDFS), dtype=torch.float32, device=dev)
    pipe.score_dev(d_pcm, so, u2s, n_spk, d_fm, DIM + 1, d_ll_pdf, P_PDFS, d_feats, 40, stream)
    torch.cuda.synchronize()
    k0.record(stream)
    for _ in range(2):
        pipe.score_dev(d_pcm, so, u2s, n_spk, d_fm, DIM + 1, d_ll_pdf, P_PDFS, d_feats, 40, stream)
    k1.record(stream)
    torch.cuda.synchronize()
    ms_pdf = max_over_ranks(k0.elapsed_time(k1) / 2)
    del d_ll_pdf
    clocks = sampler.stop() if sampler else None  # covers the timed steps and the kernel-alone loop (same load)
    flops = 2.0 * (2 * DIM + 1) * N_GAUSS * T
    pk = peaks()
    peak_tf = (pk or {}).get("bf16_tflops_sustained", 1400.0)
    achieved = flops / (k_ms * 1e-3) / 1e12
    roofline = {"bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                "frac_of_tf32_line": achieved / (0.5 * peak_tf),
                "note": "kind::f16 MMAs, 3 products per result: the pipe executes 3x the algorithmic FLOPs, so this scheme "
                        "tops out at 1/3 of the bf16 line (2/3 of the TF32 line SURVEY.md 8d names); measured MMA-only floor "
                        "of this kernel: profiles/r2_score_tc_final_timing.txt",
                "traffic": ncu_traffic(T)[0],
                "traffic_unit": "dram bytes per launch (ncu --set full, %s)" % ncu_traffic(T)[1],
                "executed_tensor_tflops": 3.0 * achieved, "kernel": "gmm scoring (%s)" % ("tcgen05" if args.kernel != 1 and am_is_tc(am) else "fp32 simt"),
                "kernel_ms": k_ms, "kernel_ms_by_rank": k_ms_by_rank, "share_of_step": k_ms / ms,
                "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if pk else "fallback 1400 (of fallback)",
                "algorithmic_flops_per_frame": 2 * (2 * DIM + 1) * N_GAUSS}
    # front end alone (HBM-bound by the rulebook; instruction-bound in practice)
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    d_mf = torch.empty((T, 16), dtype=torch.float32, device=dev)
    mfcc.compute_dev(d_pcm, so, d_mf, 16, stream=stream)
    torch.cuda.synchronize()
    f0.record(stream)
    for _ in range(k_iters):
        mfcc.compute_dev(d_pcm, so, d_mf, 16, stream=stream)
    f1.record(stream)
    torch.cuda.synchronize()
    f_ms = f0.elapsed_time(f1) / k_iters
    hbm = (pk or {}).get("hbm_gbs", 6650.0)
    fe_bytes = T * (2 * 160 + 64)
    frontend = {"bound": "hbm", "achieved": fe_bytes / (f_ms * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
                "frac": fe_bytes / (f_ms * 1e-3) / 1e9 / hbm, "kernel": "mfcc (pcm -> 13 ceps)", "kernel_ms": f_ms,
                "algorithmic_bytes_per_frame": 2 * 160 + 64}

    # ---- end to end through the host-buffer C-ABI call (`e2e`) ----
    grp = 4  # speakers per call: the reference runs one decode job per speaker split
    groups = []
    for s0 in range(0, n_spk, grp):
        utts = np.flatnonzero((u2s >= s0) & (u2s < s0 + grp))
        a, b = int(utts[0]), int(utts[-1]) + 1  # utterances of a speaker are contiguous
        groups.append((a, b, so[a:b + 1] - so[a], (u2s[a:b] - s0).astype(np.int32), s0, int(fo[b] - fo[a])))
    pin_pcm = torch.from_numpy(pcm).pin_memory()
    max_frames = max(g[5] for g in groups)
    pin_out = torch.empty((max_frames, P_PDFS), dtype=torch.float32).pin_memory()

    def e2e_step():
        for a, b, gso, gu2s, s0, nfr in groups:
            pipe.score(pin_pcm[int(so[a]):int(so[b])], gso, gu2s, min(grp, n_spk - s0), fmllr=fm[s0:s0 + grp],
                       out=pin_out)

    e2e_steps = max(1, min(args.steps, 3))
    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / e2e_steps
    e2e = {"value": total_audio / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(pcm.nbytes + fm.nbytes),
           "d2h_bytes_per_step": int(T) * P_PDFS * 4, "ms_per_step": e2e_ms, "steps": e2e_steps,
           "api": "vbgpu_pipeline_score_i16, %d calls/step (4 speakers each), pinned host buffers" % len(groups),
           "host_numa_node_of_rank0": numa_node}

    # ---- end to end for a consumer that reads a pdf subset per utterance (forced alignment, SURVEY.md 8f n3) ----
    # gmm-align-compiled reads only the pdfs of the utterance's training graph: 200 of the 4000 here (an utterance of
    # 5..20 s has a few hundred distinct HMM states).  Host PCM in, host [frames x 200] blocks out.
    SUB = 200
    rng_s = np.random.default_rng(SEED + 11 + rank)
    n_utts = len(so) - 1
    sub_o = np.arange(n_utts + 1, dtype=np.int64) * SUB
    sub_p = np.concatenate([rng_s.choice(P_PDFS, SUB, replace=False) for _ in range(n_utts)]).astype(np.int32)
    pin_sub = torch.empty(T * SUB, dtype=torch.float32).pin_memory()

    def align_step():
        return pipe.score_subset(pin_pcm, so, sub_o, sub_p, u2s, n_spk, fmllr=fm, out=pin_sub)

    _, oo = align_step()
    # spot check against the dense matrix scored above (same rows, the utterance's own columns): bit-identical
    u_chk = n_utts // 2
    a, b = int(fo[u_chk]), int(fo[u_chk + 1])
    blk = pin_sub[int(oo[u_chk]):int(oo[u_chk + 1])].view(b - a, SUB).numpy()
    cols = torch.from_numpy(col_of_pdf[sub_p[u_chk * SUB:(u_chk + 1) * SUB]].astype(np.int64)).to(dev)
    align_ok = bool(np.array_equal(blk, d_ll[a:b][:, cols].cpu().numpy()))
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        align_step()
    torch.cuda.synchronize()
    al_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / e2e_steps
    e2e_align = {"value": total_audio / (al_ms * 1e-3), "unit": UNIT, "ms_per_step": al_ms, "steps": e2e_steps,
                 "h2d_bytes_per_step": int(pcm.nbytes + fm.nbytes + sub_p.nbytes),
                 "d2h_bytes_per_step": int(T) * SUB * 4, "d2h_fraction_of_dense": SUB / float(P_PDFS),
                 "pdfs_per_utterance": SUB, "identical_to_dense": align_ok,
                 "api": "vbgpu_pipeline_score_subset_i16, one call per step, pinned host buffers"}

    # ---- EM pass (BASELINE configs[4]): PCM + alignment -> GMM and transition statistics -> one all-reduce ----
    pdf_ali, tid_ali = synth_alignment(P_PDFS, fo, SEED + 21 + rank)
    d_pdf, d_tid = torch.from_numpy(pdf_ali).to(dev), torch.from_numpy(tid_ali).to(dev)
    acc = host.AccumAmDiagGmmGpu(am, num_tids=2 * P_PDFS)
    comm = nccl_comm(rank, world, local)[1] if world > 1 else None
    acc_ptr, acc_n = acc.buffer()

    def em_pass(reduce=True):
        acc.as_tensor().zero_()
        pipe.accumulate_dev(acc, d_pcm, so, u2s, n_spk, d_fm, DIM + 1, d_pdf, stream=stream)
        acc.accumulate_transitions_dev(d_tid, T, stream=stream)
        if reduce and comm is not None:
            capi.check(capi.lib().vbgpu_acc_allreduce(acc.h, comm, stream.cuda_stream))

    for _ in range(2):
        em_pass()
    barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    em_iters = max(2, min(args.steps, 5))
    t_acc = t_red = 0.0
    for _ in range(em_iters):
        ev[0].record(stream)
        em_pass(reduce=False)
        ev[1].record(stream)
        if comm is not None:
            capi.check(capi.lib().vbgpu_acc_allreduce(acc.h, comm, stream.cuda_stream))
        ev[2].record(stream)
        barrier()
        t_acc += max_over_ranks(ev[0].elapsed_time(ev[1]))
        t_red += max_over_ranks(ev[1].elapsed_time(ev[2]))
    t_acc, t_red = t_acc / em_iters, t_red / em_iters
    merged = acc.as_tensor().clone()
    # host-buffer form: PCM and the alignment go up, the merged statistics come back
    pin_pdf, pin_tid = torch.from_numpy(pdf_ali).pin_memory(), torch.from_numpy(tid_ali).pin_memory()
    pin_acc = torch.empty(acc_n, dtype=torch.float64).pin_memory()

    def em_e2e():
        d_pcm.copy_(pin_pcm, non_blocking=True)
        d_pdf.copy_(pin_pdf, non_blocking=True)
        d_tid.copy_(pin_tid, non_blocking=True)
        em_pass()
        pin_acc.copy_(acc.as_tensor(), non_blocking=True)
        torch.cuda.synchronize()

    em_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        em_e2e()
    em_e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / e2e_steps
    # merged statistics vs ONE GPU accumulating every rank's shard (rank 0; FP64 sums: 1e-10)
    em_err, em_frames_ok = None, None
    if rank == 0:
        single = host.AccumAmDiagGmmGpu(am, num_tids=2 * P_PDFS)
        for r in range(world):
            if r == 0:
                p_r, so_r, u_r, n_r, fo_r = d_pcm, so, u2s, n_spk, fo
                fm_r = d_fm
            else:
                pc, so_r, u_r, n_r, _ = rank_corpus(n_gpus, r)
                p_r, fo_r = torch.from_numpy(pc).to(dev), mfcc.frame_offsets(so_r)
                fm_r = torch.from_numpy(synth.make_fmllr(n_r, DIM, SEED + 6 + r)).to(dev)
            pa, ta = synth_alignment(P_PDFS, fo_r, SEED + 21 + r)
            pipe.accumulate_dev(single, p_r, so_r, u_r, n_r, fm_r, DIM + 1, torch.from_numpy(pa).to(dev), stream=stream)
            single.accumulate_transitions_dev(torch.from_numpy(ta).to(dev), int(fo_r[-1]), stream=stream)
            torch.cuda.synchronize()
        want = single.as_tensor()
        em_err = float((merged - want).abs().max().item() / want.abs().max().item())
        n_stats = am.NumGauss() * (2 * DIM + 1)
        em_frames_ok = bool(merged[n_stats + 1].item() == want[n_stats + 1].item() and
                            merged[n_stats + 2:].sum().item() == want[n_stats + 2:].sum().item())
        del single
    em = {"value": total_audio / ((t_acc + t_red) * 1e-3), "unit": UNIT, "accumulate_ms": t_acc, "allreduce_ms": t_red,
          "allreduce_bytes": int(acc_n) * 8, "passes_timed": em_iters,
          "buffer": "[occ | mean | var | tot_like | tot_frames | transition accs]: %d doubles, one ncclAllReduce" % acc_n,
          "merged_vs_single_gpu_rel_err": em_err, "frame_and_transition_counts_equal": em_frames_ok,
          "e2e": {"value": total_audio / (em_e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": em_e2e_ms,
                  "h2d_bytes_per_step": int(pcm.nbytes + pdf_ali.nbytes + tid_ali.nbytes), "d2h_bytes_per_step": int(acc_n) * 8},
          "api": "vbgpu_pipeline_accumulate_dev + vbgpu_acc_accumulate_transitions_dev + vbgpu_acc_allreduce (raw ncclComm_t)"}
    del acc

    # ---- the other BASELINE configs on this GPU (device-resident, a few steps each; rank 0 at N=1 only) ----
    others = None
    if rank == 0 and world == 1 and not args.no_others:
        others = []
        del d_ll
        torch.cuda.empty_cache()
        for name, P2, N2, lda in (("cfg2 tri-delta", 2000, 10000, False), ("cfg4 LDA+MLLT", 2500, 15000, True)):
            fo2 = capi.default_feat_opts()
            mat = None
            if lda:
                fo2.mode = 1
                mat = synth.make_lda(40, 91, 7)
            fp2 = host.FeaturePipeline(fo2, 13, transform=mat, device=local)
            D2 = 40 if lda else 39
            fs2 = fp2.run(mf, mfo, cmvn_stats=fp2.cmvn_stats(mf, mfo))
            model2 = synth.make_model_from_feats(fs2, P2, N2, SEED)
            am2 = host.AmDiagGmmGpu.from_model(model2, device=local)
            pipe2 = host.ScoringPipeline(mfcc, fp2, am2)
            nc2 = am2.NumCols()
            d_ll2 = torch.empty((T, nc2), dtype=torch.float32, device=dev)

            def step2():
                pipe2.score_cols_dev(d_pcm, so, u2s, n_spk, None, 0, d_ll2, nc2, d_feats, 40, stream)
            for _ in range(3):
                step2()
            torch.cuda.synchronize()
            k0.record(stream)
            for _ in range(3):
                step2()
            k1.record(stream)
            torch.cuda.synchronize()
            ms2 = k0.elapsed_time(k1) / 3
            rows = np.sort(np.random.default_rng(SEED + 1).choice(T, 64, replace=False))
            par2 = None
            try:
                from oracle import pyoracle as po
                chk = po.load("ref") if po.have_ref() else po.load("orc")
                x2 = d_feats[torch.from_numpy(rows).to(dev)][:, :D2].cpu().numpy()
                got2 = d_ll2[torch.from_numpy(rows).to(dev)].cpu().numpy()[:, am2.col_of_pdf()]
                par2 = float(np.abs(got2 - chk.gmm_loglikes(model2, x2)[1]).max())
            except Exception as ex:
                par2 = repr(ex)
            others.append({"config": name, "pdfs": P2, "gaussians": N2, "dim": D2, "ms_per_step": ms2,
                           "value": audio_s / (ms2 * 1e-3), "unit": UNIT, "kernel_note": am2.plan_note() or "tcgen05",
                           "parity_max_abs_err_64_frames": par2, "nonfinite": am2.bad_count()})
            del d_ll2, pipe2, am2
            torch.cuda.empty_cache()

    # ---- cpu baseline (rank 0, N=1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            r = cpu_reference_run(1, 0, target_s=12.0)
            cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]}
        except Exception as ex:  # the baseline must never take the bench line down
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "failed: %r" % (ex,)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32" if not am_is_tc(am) or args.kernel == 1 else "f16x3 split (f32 accumulate)",
            "data": "synthetic",
            "config": dict(workload_config(n_gpus), frames_per_step_per_gpu=T, audio_s_per_step_per_gpu=audio_s),
            "value_pdf_order": total_audio / (ms_pdf * 1e-3), "ms_per_step_pdf_order": ms_pdf,
            "ms_per_step_by_rank": ms_by_rank, "roofline": roofline, "roofline_frontend": frontend, "cpu_baseline": cpu, "e2e": e2e, "e2e_align": e2e_align,
            "em": em, "parity": parity, "other_configs": others,
            "gpu_launches": 8 * args.steps, "clocks": clocks, "rescored_frames_last_step": rescored, "nonfinite_loglikes": bad,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


DUMP_ROWS = 2048  # 2048 frames x 4000 pdfs x 4 bytes = 33 MB: the dump stays under 64 MB


def dump_outputs(out_dir, d_ll, d_feats, col_of_pdf, T):
    """What the timed step hands its caller, on a fixed seeded sample of DUMP_ROWS frames of rank 0's batch, so that two
    builds run with the same arguments can be compared output for output:
      loglikes.npy    [rows x P_PDFS] float32, in the model's pdf order (the device column order mapped back)
      feats.npy       [rows x DIM]    float32, the fMLLR-transformed features the loglikes were scored on
      frame_rows.npy  [rows]          float64, the frame index of each sampled row"""
    import torch
    rows = np.sort(np.random.default_rng(SEED + 31).choice(T, min(DUMP_ROWS, T), replace=False))
    idx = torch.from_numpy(rows).to(d_ll.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loglikes.npy"), np.ascontiguousarray(d_ll[idx].cpu().numpy()[:, col_of_pdf]))
    np.save(os.path.join(out_dir, "feats.npy"), np.ascontiguousarray(d_feats[idx][:, :DIM].cpu().numpy()))
    np.save(os.path.join(out_dir, "frame_rows.npy"), rows.astype(np.float64))


def am_is_tc(am):
    """True when the tensor-core scorer serves this model (set_kernel(2) is accepted only then)."""
    from voicebridge_b200 import capi
    try:
        am.set_kernel(2)
        am.set_kernel(0)
        return True
    except capi.VbgpuError:
        return False


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--kernel", type=int, default=0, help="0 auto, 1 fp32 simt, 2 tcgen05")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-others", action="store_true", help="skip the other_configs leg (cfg 2 / cfg 4)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a seeded sample of rank 0's loglikes and features of the last step "
                         "as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs saves the CUDA path's outputs: it does not apply to --impl reference")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
