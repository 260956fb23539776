"""Kaldi pitch on the device (SURVEY.md §8f n4: ComputeKaldiPitch, ProcessPitch, ComputeAndProcessKaldiPitch) against the
plain-C oracle, the reference's own code (oracle/_ref, where it is built) and the committed dumps of the compiled
reference (tests/golden/pitch_golden.npz).  Tolerances: see tests.common.assert_pitch_close."""
import os

import numpy as np
import pytest

from oracle import pyoracle as po
from tests.common import assert_pitch_close, assert_process_pitch_close, copy_opts
from tests.golden.make_pitch_golden import PROCESS_VARIANT
from voicebridge_b200 import capi, host, synth

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def orc_opts(o):
    return copy_opts(o, po.PitchOpts)


def orc_popts(o):
    return copy_opts(o, po.ProcessPitchOpts)


PITCH_VARIANTS = [
    dict(), dict(snip_edges=0), dict(preemph_coeff=0.5), dict(samp_freq=8000.0), dict(samp_freq=22050.0),
    dict(min_f0=60.0, max_f0=300.0, delta_pitch=0.01), dict(frame_shift_ms=5.0, frame_length_ms=20.0),
    dict(resample_freq=3000.0, lowpass_cutoff=800.0, upsample_filter_width=3, lowpass_filter_width=2),
    dict(nccf_ballast=100.0, soft_min_f0=30.0, penalty_factor=0.3), dict(recompute_frame=100),
]


@pytest.mark.parametrize("kw", PITCH_VARIANTS, ids=lambda d: ",".join("%s=%s" % kv for kv in d.items()) or "default")
def test_pitch_single_utterance(orc, kw):
    o = capi.default_pitch_opts(**kw)
    p = host.Pitch(o)
    for secs, seed in ((2.3, 1), (6.1, 2)):
        w = synth.make_pitch_wave(int(secs * o.samp_freq), seed, o.samp_freq)
        got = p.Compute(w)
        want = orc.pitch(orc_opts(o), w.astype(np.float32))
        assert got.shape == want.shape == (p.NumFrames(len(w)), 2)
        assert_pitch_close(got, want, what="pitch %s %gs" % (kw, secs))
        assert np.array_equal(got, p.Compute(w.astype(np.float32)))  # int16 and float input: same samples, same result
        assert np.array_equal(got, p.Compute(w))                     # and deterministic


def test_pitch_golden_dumps_of_the_reference():
    g = dict(np.load(os.path.join(GOLDEN, "pitch_golden.npz")))
    pcm = np.load(os.path.join(GOLDEN, "htk_golden.npz"))["pcm"]
    p = host.Pitch()
    raw = p.Compute(pcm)
    assert_pitch_close(raw, g["raw16"], "test.wav")
    assert_pitch_close(host.Pitch(capi.default_pitch_opts(snip_edges=0)).Compute(pcm), g["raw16_nosnip"], "no snip")
    assert_pitch_close(p.Compute(pcm[:9000]), g["raw16_short"], "short")
    p8 = host.Pitch(capi.default_pitch_opts(samp_freq=8000.0, min_f0=60.0, max_f0=350.0))
    assert_pitch_close(p8.Compute(g["wave8"]), g["raw8"], "8 kHz")
    pp = capi.default_process_pitch_opts(delta_pitch_noise_stddev=0.0)
    assert_process_pitch_close(p.Process(pp, g["raw16"]), g["proc16"])
    pv = capi.default_process_pitch_opts(delta_pitch_noise_stddev=0.0, **PROCESS_VARIANT)
    assert_process_pitch_close(p.Process(pv, g["raw16"]), g["proc16_variant"])


@pytest.mark.parametrize("kw", [PITCH_VARIANTS[0], PITCH_VARIANTS[1], PITCH_VARIANTS[6]],
                         ids=lambda d: ",".join("%s=%s" % kv for kv in d.items()) or "default")
def test_pitch_ragged_batch(orc, kw):
    """Empty, shorter-than-a-window, one-frame and long utterances in one packed batch: every utterance equals the oracle
    run on it alone (no leakage across utterance boundaries), and the reference's own code where it is built."""
    o = capi.default_pitch_opts(**kw)
    lens = [0, 300, 399, 400, 560, 1700, 16000, 48000, 0, 131072, 7777]
    so = np.zeros(len(lens) + 1, np.int64)
    so[1:] = np.cumsum(lens)
    pcm = np.concatenate([synth.make_pitch_wave(n, 40 + i) for i, n in enumerate(lens)])
    p = host.Pitch(o)
    got, ro = p.compute_batch(pcm, so)
    oo = orc_opts(o)
    checkers = [("oracle", orc)] + ([("reference", po.load("ref"))] if po.have_ref() else [])
    for name, chk in checkers:
        n_diff = 0
        for u, n in enumerate(lens):
            want = chk.pitch(oo, pcm[so[u]:so[u + 1]].astype(np.float32))
            assert ro[u + 1] - ro[u] == len(want) == p.NumFrames(n)
            n_diff += assert_pitch_close(got[ro[u]:ro[u + 1]], want, what="utt %d (%d samples) vs %s" % (u, n, name)) or 0
        assert n_diff <= 0.03 * len(got), "%s: %d of %d frames on a different lag state" % (name, n_diff, len(got))


def test_pitch_energy_correction(orc):
    """RecomputeBacktraces: a burst in the flushed tail changes the energy estimate by more than 1%."""
    o = capi.default_pitch_opts()
    w = synth.make_pitch_wave(16000, 5).astype(np.float32) * 0.3
    w[-12:] = 32000.0
    assert_pitch_close(host.Pitch(o).Compute(w), orc.pitch(orc_opts(o), w), what="energy correction")


@pytest.mark.parametrize("kw", [dict(), PROCESS_VARIANT, dict(add_pov_feature=0, add_delta_pitch=0),
                                dict(pov_offset=1.0, pitch_scale=1.0, delay=1)],
                         ids=lambda d: ",".join("%s=%s" % kv for kv in d.items()) or "default")
def test_process_pitch(orc, kw):
    pp = capi.default_process_pitch_opts(delta_pitch_noise_stddev=0.0, **kw)
    o = capi.default_pitch_opts()
    p = host.Pitch(o)
    lens = [16000 * 3, 600, 0, 16000]
    so = np.zeros(len(lens) + 1, np.int64)
    so[1:] = np.cumsum(lens)
    pcm = np.concatenate([synth.make_pitch_wave(n, 60 + i) for i, n in enumerate(lens)])
    raw, ro = p.compute_batch(pcm, so)
    # ProcessPitch on rows the caller supplies, several matrices at once
    got = p.Process(pp, raw, ro)
    want = [orc.process_pitch(orc_popts(pp), raw[ro[u]:ro[u + 1]]) for u in range(len(lens)) if ro[u + 1] > ro[u]]
    assert_process_pitch_close(got, np.concatenate(want))
    # ComputeAndProcessKaldiPitch in one call gives the same rows
    both, ro2 = p.compute_batch(pcm, so, pp)
    assert np.array_equal(both, got) and ro2[-1] == len(got)


def test_delta_pitch_noise_is_gaussian_with_the_requested_spread():
    """The reference adds RandGauss() * stddev from rand(); ours comes from a counter-based generator: same distribution,
    different stream (documented in include/vbgpu.h)."""
    p = host.Pitch()
    raw = p.Compute(synth.make_pitch_wave(16000 * 20, 9))
    quiet = p.Process(capi.default_process_pitch_opts(delta_pitch_noise_stddev=0.0), raw)
    noisy = p.Process(capi.default_process_pitch_opts(delta_pitch_noise_stddev=0.005), raw)
    assert np.array_equal(quiet[:, :2], noisy[:, :2])
    d = (noisy[:, 2] - quiet[:, 2]) / 10.0  # delta_pitch_scale
    assert abs(d.mean()) < 5e-4 and 0.0045 < d.std() < 0.0055 and np.abs(d).max() < 0.03


def test_pitch_argument_errors():
    p = host.Pitch()
    with pytest.raises(capi.VbgpuError):
        p.compute_batch(np.zeros(100, np.int16), np.array([5, 100], np.int64))   # offsets must start at 0
    with pytest.raises(capi.VbgpuError):
        p.Process(capi.default_process_pitch_opts(add_pov_feature=0, add_normalized_log_pitch=0, add_delta_pitch=0),
                  np.ones((4, 2), np.float32))                                    # no output column selected
    with pytest.raises(capi.VbgpuError):
        p.Process(capi.default_process_pitch_opts(), np.zeros((4, 2), np.float32))  # pitch must be > 0
    with pytest.raises(capi.VbgpuError):
        host.Pitch(capi.default_pitch_opts(delta_pitch=0.0005))                  # > 1024 lag states
    assert p.Compute(np.zeros(0, np.int16)).shape == (0, 2)
    z = p.Compute(np.zeros(16000, np.int16))  # digital silence: NCCF 0/0 -> 0, a flat path
    assert z.shape == (p.NumFrames(16000), 2) and np.isfinite(z).all() and not z[:, 0].any()


def test_pitch_device_buffers():
    """PCM already in HBM and rows left in HBM (cudaMemcpyDefault on both sides): same numbers as the host-buffer call."""
    import ctypes as C
    import torch
    p = host.Pitch()
    w = synth.make_pitch_wave(16000 * 2, 3)
    want = p.Compute(w)
    d_w = torch.from_numpy(w).cuda()
    d_out = torch.zeros((len(want), 2), dtype=torch.float32, device="cuda")
    so = np.array([0, len(w)], np.int64)
    torch.cuda.synchronize()
    capi.check(capi.lib().vbgpu_pitch_compute_i16(p.h, d_w.data_ptr(), so.ctypes.data, 1, None, d_out.data_ptr(), 2))
    assert np.array_equal(d_out.cpu().numpy(), want)


def test_make_mfcc_pitch(orc):
    """steps/make_mfcc_pitch: MFCC and processed pitch pasted with --length-tolerance=2 (the pitch extractor yields one
    or two frames more than the MFCC front end with snip-edges)."""
    from tests.gpu_common import to_orc_opts
    from tests.common import assert_feats_close
    mo = capi.default_mfcc_opts(dither=0.0)
    pp = capi.default_process_pitch_opts(delta_pitch_noise_stddev=0.0)
    lens = [16000 * 2, 300, 5000, 0, 16000]
    so = np.zeros(len(lens) + 1, np.int64)
    so[1:] = np.cumsum(lens)
    pcm = np.concatenate([synth.make_pitch_wave(n, 80 + i) for i, n in enumerate(lens)])
    m, p = host.Mfcc(mo), host.Pitch()
    out = host.make_mfcc_pitch(m, p, pcm, so, pp)
    assert len(out) == len(lens) and out[1] is None and out[3] is None  # too short for a frame / empty: dropped
    for u in (0, 2, 4):
        w = pcm[so[u]:so[u + 1]].astype(np.float32)
        a = orc.mfcc(to_orc_opts(mo), w)
        raw = orc.pitch(orc_opts(capi.default_pitch_opts()), w)
        b = orc.process_pitch(orc_popts(pp), raw)
        assert 0 <= len(b) - len(a) <= 2 and out[u].shape == (len(a), 16)
        assert_feats_close(out[u][:, :13], a, what="mfcc part")
        same = np.abs(p.Compute(w)[:len(a), 1] - raw[:len(a), 1]) <= 1e-6 * raw[:len(a), 1]
        assert same.mean() >= 0.9


@pytest.mark.parametrize("seed", range(16))
def test_pitch_random_options(orc, seed):
    """Random valid option sets (sample rates 8..44.1 kHz, resampling / search / framing options) and lengths."""
    from tests.common import random_pitch_opts
    rng = np.random.default_rng(2000 + seed)
    kw = random_pitch_opts(rng)
    o = capi.default_pitch_opts(**kw)
    w = synth.make_pitch_wave(int(rng.uniform(0.2, 3.0) * o.samp_freq), seed, o.samp_freq)
    assert_pitch_close(host.Pitch(o).Compute(w), orc.pitch(orc_opts(o), w.astype(np.float32)), what=str(kw))


@pytest.mark.parametrize("groups,states", [(3, 1), (4, 2), (2, 4)])
def test_pitch_upload_groups_and_states_per_thread(orc, monkeypatch, groups, states):
    """Large batches upload the PCM in groups of utterances overlapped with the first kernels, and the Viterbi kernel keeps
    1, 2 or 4 lag states per thread depending on the batch size: forced here on a small ragged batch, every variant gives
    the rows of the default path."""
    lens = [7000, 0, 16000, 400, 23000, 9000, 300, 12000]
    so = np.zeros(len(lens) + 1, np.int64)
    so[1:] = np.cumsum(lens)
    pcm = np.concatenate([synth.make_pitch_wave(n, 90 + i) for i, n in enumerate(lens)])
    p = host.Pitch()
    pp = capi.default_process_pitch_opts(delta_pitch_noise_stddev=0.0)
    want, ro = p.compute_batch(pcm, so, pp)
    monkeypatch.setenv("VBGPU_PITCH_UPLOAD_GROUPS", str(groups))
    monkeypatch.setenv("VBGPU_PITCH_STATES_PER_THREAD", str(states))
    got, ro2 = p.compute_batch(pcm, so, pp)
    assert np.array_equal(ro, ro2) and np.array_equal(got, want)
    u = 4
    raw = orc.pitch(orc_opts(capi.default_pitch_opts()), pcm[so[u]:so[u + 1]].astype(np.float32))
    assert_process_pitch_close(got[ro[u]:ro[u + 1]], orc.process_pitch(orc_popts(pp), raw), atol=2e-3)
