"""Host-side mirror of the reference's interface for the hot path, on top of the C ABI (capi.py).

Class / method names and argument meaning follow the Kaldi types VoiceBridge links
(paths relative to /root/reference/kaldi-master/src):

  Mfcc                     OfflineFeatureTpl<MfccComputer>          feat/feature-common.h:110-178
  FeaturePipeline          apply-cmvn | add-deltas | splice-feats | transform-feats   (VB/scr/steps/decode_gmm.cpp:395-571)
  AmDiagGmmGpu             AmDiagGmm                                 gmm/am-diag-gmm.h:36-105
  DecodableAmDiagGmmGpu    DecodableAmDiagGmmScaled                  gmm/decodable-am-diag-gmm.h:121-160
  AccumAmDiagGmmGpu        AccumAmDiagGmm                            gmm/mle-am-diag-gmm.h:34-108
  LdaEstimateGpu           LdaEstimate (accumulation)                transform/lda-estimate.h
  TreeStatsGpu             AccumulateTreeStats (acc-tree-stats)      hmm/tree-accu.cc
  GmmAlignCompiledGpu      AlignUtteranceWrapper + FasterDecoder (gmm-align-compiled)   decoder/decoder-wrappers.cc
  GmmDecodeFasterGpu       FasterDecoder Decode / ReachedFinal / GetBestPath (gmm-decode-faster)  decoder/faster-decoder.cc
  ScoringPipeline          the fused PCM -> loglikes job (compute-mfcc-feats ... gmm-latgen-faster's decodable)

Errors surface as capi.VbgpuError (the reference throws std::runtime_error from KALDI_ERR).
numpy arrays are host buffers; torch CUDA tensors are passed by device pointer.  This module never computes
on the CPU: every method is a call into libvbgpu.so.
"""
import ctypes as C

import numpy as np

from . import capi
from .capi import check


def kaldi_stride(cols):
    """Stride of kaldi::Matrix<float>: cols rounded up to 16 bytes (matrix/kaldi-matrix.cc:797-808)."""
    return (cols + 3) // 4 * 4


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return a.data_ptr()  # torch tensor


def _np(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


def _stream_ptr(stream):
    if stream is None:
        import torch
        return torch.cuda.current_stream().cuda_stream
    return stream if isinstance(stream, int) else stream.cuda_stream


class _Handle:
    _destroy = None

    def __init__(self):
        self.h = C.c_void_p()

    def close(self):
        if getattr(self, "h", None) is not None and self.h.value:
            getattr(capi.lib(), self._destroy)(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class WaveData:
    """WaveData (feat/wave-reader.h:115-190) over an in-memory RIFF/RIFX image: SampFreq(), Data() as int16
    [channels, samples] (the reference holds the same values as float), Duration()."""

    def __init__(self, image):
        buf = np.frombuffer(bytes(image), np.uint8)
        info = capi.WaveInfo()
        check(capi.lib().vbgpu_wave_parse(buf.ctypes.data, buf.size, C.byref(info)))
        self.info = info
        self._data = np.zeros((info.num_channels, info.num_samples), np.int16)
        for ch in range(info.num_channels):
            check(capi.lib().vbgpu_wave_channel_i16(buf.ctypes.data, buf.size, C.byref(info), ch,
                                                    self._data[ch].ctypes.data))

    @classmethod
    def Read(cls, path):
        with open(path, "rb") as f:
            return cls(f.read())

    def SampFreq(self):
        return float(self.info.samp_freq)

    def Data(self):
        return self._data

    def Duration(self):
        return self._data.shape[1] / self.SampFreq()


class Downsampler(_Handle):
    """DownsampleWaveForm (feat/resample.cc:368-376) for one (orig_freq, new_freq) pair."""
    _destroy = "vbgpu_downsample_destroy"

    def __init__(self, orig_freq, new_freq, device=0):
        super().__init__()
        check(capi.lib().vbgpu_downsample_create(float(orig_freq), float(new_freq), device, C.byref(self.h)))

    def NumOut(self, n_in):
        return check(capi.lib().vbgpu_downsample_num_out(self.h, int(n_in)))

    def __call__(self, wave):
        w = _np(wave, np.float32)
        out = np.zeros(max(self.NumOut(len(w)), 1), np.float32)
        check(capi.lib().vbgpu_downsample_f32(self.h, w.ctypes.data, len(w), out.ctypes.data))
        return out[:self.NumOut(len(w))]


class Mfcc(_Handle):
    """MFCC computer.  `opts` is a capi.MfccOpts (MfccOptions); allow_downsample is FrameExtractionOptions::allow_downsample
    (feat/feature-window.h:46), a switch of ComputeFeatures, not of the computation."""
    _destroy = "vbgpu_mfcc_destroy"

    def __init__(self, opts=None, device=0, allow_downsample=False):
        super().__init__()
        self.opts = opts if opts is not None else capi.default_mfcc_opts()
        check(capi.lib().vbgpu_mfcc_create(C.byref(self.opts), device, C.byref(self.h)))
        self.device = device
        self.allow_downsample = bool(allow_downsample)
        self._down = {}

    def Dim(self):
        return check(capi.lib().vbgpu_mfcc_dim(self.h))

    def NumFrames(self, num_samples):
        return check(capi.lib().vbgpu_mfcc_num_frames(self.h, num_samples))

    def frame_offsets(self, sample_offsets):
        so = _np(sample_offsets, np.int64)
        fo = np.zeros_like(so)
        check(capi.lib().vbgpu_mfcc_frame_offsets(self.h, so.ctypes.data, len(so) - 1, fo.ctypes.data))
        return fo

    def ComputeFeatures(self, wave, sample_freq=None, vtln_warp=1.0):
        """One utterance, like OfflineFeatureTpl::ComputeFeatures(wave, sample_freq, vtln_warp, &out).
        wave: int16 or float32 samples in int16 range.  Returns float32 [NumFrames, Dim]."""
        if sample_freq is not None and float(sample_freq) != float(self.opts.samp_freq):
            new = float(self.opts.samp_freq)
            if new < float(sample_freq):  # feature-common-inl.h:37-48
                if not self.allow_downsample:
                    raise capi.VbgpuError(capi.ERR_INVALID, "Waveform and config sample Frequency mismatch: %s .vs %s "
                                          "( use --allow_downsample=true option to allow downsampling the waveform)." %
                                          (sample_freq, new))
                key = float(sample_freq)
                if key not in self._down:
                    self._down[key] = Downsampler(key, new, self.device)
                wave = self._down[key](np.asarray(wave, np.float32))
            else:                         # feature-common-inl.h:49-53: up-sampling is never done
                raise capi.VbgpuError(capi.ERR_INVALID, "New sample Frequency %s is larger than waveform original sampling "
                                      "frequency %s" % (new, sample_freq))
        wave = np.asarray(wave)
        offs = np.array([0, len(wave)], np.int64)
        return self.compute_batch(wave, offs, None if vtln_warp == 1.0 else [vtln_warp])[0]

    def compute_batch(self, wave, sample_offsets, vtln_warp=None, out_stride=None):
        """Batched ComputeFeatures over packed utterances.  Returns (feats [T, Dim], frame_offsets)."""
        so = _np(sample_offsets, np.int64)
        n_utts = len(so) - 1
        fo = self.frame_offsets(so)
        T, D = int(fo[-1]), self.Dim()
        st = out_stride or kaldi_stride(D)
        out = np.zeros((max(T, 1), st), np.float32)
        vt = _np(vtln_warp, np.float32) if vtln_warp is not None else None
        wave = np.asarray(wave)
        if wave.dtype == np.int16:
            w = np.ascontiguousarray(wave)
            fn = capi.lib().vbgpu_mfcc_compute_i16
        else:
            w = _np(wave, np.float32)
            fn = capi.lib().vbgpu_mfcc_compute_f32
        check(fn(self.h, w.ctypes.data, so.ctypes.data, n_utts, _ptr(vt), out.ctypes.data, st))
        return out[:T, :D], fo

    def compute_dev(self, d_pcm, sample_offsets, d_out, out_stride, is_f32=False, stream=None):
        so = _np(sample_offsets, np.int64)
        check(capi.lib().vbgpu_mfcc_compute_dev(self.h, _ptr(d_pcm), int(is_f32), so.ctypes.data, len(so) - 1, None,
                                                _ptr(d_out), out_stride, _stream_ptr(stream)))


class Fbank(Mfcc):
    """OfflineFeatureTpl<FbankComputer> (feat/feature-fbank.cc): mel filterbank energies, num_bins (+1 with use_energy)
    columns.  Frame / mel / energy / htk_compat options come from the same options struct as MFCC."""

    def __init__(self, opts=None, use_log_fbank=True, use_power=True, device=0):
        _Handle.__init__(self)
        self.opts = opts if opts is not None else capi.default_mfcc_opts(use_energy=0)
        check(capi.lib().vbgpu_fbank_create(C.byref(self.opts), int(use_log_fbank), int(use_power), device,
                                            C.byref(self.h)))
        self.device = device


class Plp(Mfcc):
    """OfflineFeatureTpl<PlpComputer> (feat/feature-plp.cc): num_ceps PLP cepstra per frame."""

    def __init__(self, opts=None, lpc_order=12, compress_factor=0.33333, cepstral_scale=1.0, device=0):
        _Handle.__init__(self)
        self.opts = opts if opts is not None else capi.default_mfcc_opts()
        check(capi.lib().vbgpu_plp_create(C.byref(self.opts), int(lpc_order), float(compress_factor),
                                          float(cepstral_scale), device, C.byref(self.h)))
        self.device = device


class Pitch(_Handle):
    """Kaldi pitch for batches of utterances: ComputeKaldiPitch, ProcessPitch and ComputeAndProcessKaldiPitch
    (feat/pitch-functions.cc:1291, 1581, 1597), offline mode."""
    _destroy = "vbgpu_pitch_destroy"

    def __init__(self, opts=None, device=0):
        super().__init__()
        self.opts = opts if opts is not None else capi.default_pitch_opts()
        check(capi.lib().vbgpu_pitch_create(C.byref(self.opts), device, C.byref(self.h)))
        self.device = device

    def NumFrames(self, num_samples):
        return check(capi.lib().vbgpu_pitch_num_frames(self.h, int(num_samples)))

    def NumStates(self):
        return check(capi.lib().vbgpu_pitch_num_states(self.h))

    @staticmethod
    def process_dim(process_opts):
        return sum(1 for k in ("add_pov_feature", "add_normalized_log_pitch", "add_delta_pitch", "add_raw_log_pitch")
                   if getattr(process_opts, k))

    def compute_batch(self, wave, sample_offsets, process_opts=None):
        """Packed utterances -> (rows, row_offsets).  process_opts None: rows are (NCCF, pitch Hz) like
        ComputeKaldiPitch; otherwise the ProcessPitch features (ComputeAndProcessKaldiPitch)."""
        so = _np(sample_offsets, np.int64)
        n_utts = len(so) - 1
        delay = process_opts.delay if process_opts is not None else 0
        ro = np.zeros(n_utts + 1, np.int64)
        for u in range(n_utts):
            T = self.NumFrames(int(so[u + 1] - so[u]))
            ro[u + 1] = ro[u] + (T + delay if T > 0 else 0)
        dim = 2 if process_opts is None else self.process_dim(process_opts)
        out = np.zeros((max(int(ro[-1]), 1), max(dim, 1)), np.float32)
        wave = np.asarray(wave)
        if wave.dtype == np.int16:
            w = np.ascontiguousarray(wave)
            fn = capi.lib().vbgpu_pitch_compute_i16
        else:
            w = _np(wave, np.float32)
            fn = capi.lib().vbgpu_pitch_compute_f32
        check(fn(self.h, w.ctypes.data, so.ctypes.data, n_utts,
                 C.byref(process_opts) if process_opts is not None else None, out.ctypes.data, out.shape[1]))
        return out[:int(ro[-1])], ro

    def Compute(self, wave, process_opts=None):
        """One utterance: ComputeKaldiPitch(opts, wave, &out) / ComputeAndProcessKaldiPitch."""
        wave = np.asarray(wave)
        return self.compute_batch(wave, np.array([0, len(wave)], np.int64), process_opts)[0]

    def Process(self, process_opts, raw, frame_offsets=None):
        """ProcessPitch(opts, raw, &out) for one [T, 2] matrix or several packed ones."""
        raw = _np(raw, np.float32)
        fo = _np(frame_offsets, np.int64) if frame_offsets is not None else np.array([0, raw.shape[0]], np.int64)
        rows = sum((int(fo[u + 1] - fo[u]) + process_opts.delay) if fo[u + 1] > fo[u] else 0 for u in range(len(fo) - 1))
        dim = self.process_dim(process_opts)
        out = np.zeros((max(rows, 1), max(dim, 1)), np.float32)
        check(capi.lib().vbgpu_pitch_process(self.h, C.byref(process_opts), raw.ctypes.data, raw.shape[1] if raw.ndim == 2 else 2,
                                             fo.ctypes.data, len(fo) - 1, out.ctypes.data, out.shape[1]))
        return out[:rows]


def paste_feats(mats, length_tolerance=0):
    """AppendFeats of paste-feats (VB/src/featbin/paste-feats.cpp:25-65): column-wise concatenation of one utterance's
    feature matrices, trimmed to the shortest when the lengths differ by at most `length_tolerance` frames; None when they
    differ by more or one of them is empty (the reference warns and drops the utterance)."""
    lens = [int(m.shape[0]) for m in mats]
    if max(lens) - min(lens) > length_tolerance or min(lens) == 0:
        return None
    n = min(lens)
    return np.concatenate([np.asarray(m, np.float32)[:n] for m in mats], axis=1)


def make_mfcc_pitch(mfcc, pitch, wave, sample_offsets, process_opts=None, length_tolerance=2):
    """steps/make_mfcc_pitch (VB/scr/steps/make_mfcc_pitch.cpp:150-210): compute-mfcc-feats, compute-kaldi-pitch-feats |
    process-kaldi-pitch-feats and paste-feats --length-tolerance=2 for a packed batch of utterances.  `mfcc` is a Mfcc /
    Fbank / Plp, `pitch` a Pitch.  Returns one [frames, mfcc_dim + pitch_dim] matrix per utterance (None where paste-feats
    would drop it)."""
    if process_opts is None:
        process_opts = capi.default_process_pitch_opts()
    a, fo = mfcc.compute_batch(wave, sample_offsets)
    b, ro = pitch.compute_batch(wave, sample_offsets, process_opts)
    return [paste_feats([a[fo[u]:fo[u + 1]], b[ro[u]:ro[u + 1]]], length_tolerance) for u in range(len(fo) - 1)]


class FeaturePipeline(_Handle):
    """apply-cmvn -> add-deltas | splice-feats + transform-feats [-> per-speaker fMLLR]."""
    _destroy = "vbgpu_feat_destroy"

    def __init__(self, opts=None, in_dim=13, transform=None, device=0):
        super().__init__()
        self.opts = opts if opts is not None else capi.default_feat_opts()
        self.in_dim = in_dim
        t = _np(transform, np.float32) if transform is not None else None
        rows, cols = (t.shape if t is not None else (0, 0))
        check(capi.lib().vbgpu_feat_create(C.byref(self.opts), in_dim, _ptr(t), rows, cols, device, C.byref(self.h)))

    def out_dim(self):
        return check(capi.lib().vbgpu_feat_out_dim(self.h))

    def cmvn_stats(self, feats, frame_offsets, utt2spk=None, n_spk=None, stats=None):
        """AccCmvnStats per speaker -> float64 [n_spk, 2, dim+1] (added to `stats` if given)."""
        feats = _np(feats, np.float32)
        fo = _np(frame_offsets, np.int64)
        n_utts = len(fo) - 1
        u2s = _np(utt2spk, np.int32) if utt2spk is not None else None
        if n_spk is None:
            n_spk = n_utts if u2s is None else int(u2s.max()) + 1 if len(u2s) else 0
        if stats is None:
            stats = np.zeros((n_spk, 2, self.in_dim + 1), np.float64)
        check(capi.lib().vbgpu_cmvn_stats(self.h, feats.ctypes.data, feats.shape[1], fo.ctypes.data, n_utts, _ptr(u2s),
                                          n_spk, stats.ctypes.data))
        return stats

    def run(self, feats, frame_offsets, utt2spk=None, n_spk=None, cmvn_stats=None, fmllr=None):
        feats = _np(feats, np.float32)
        fo = _np(frame_offsets, np.int64)
        n_utts = len(fo) - 1
        u2s = _np(utt2spk, np.int32) if utt2spk is not None else None
        if n_spk is None:
            n_spk = n_utts if u2s is None else int(u2s.max()) + 1 if len(u2s) else 0
        st = _np(cmvn_stats, np.float64) if cmvn_stats is not None else None
        fm = _np(fmllr, np.float32) if fmllr is not None else None
        fcols = fm.shape[-1] if fm is not None else 0
        T, OD = int(fo[-1]), self.out_dim()
        ost = kaldi_stride(OD)
        out = np.zeros((max(T, 1), ost), np.float32)
        check(capi.lib().vbgpu_feat_run(self.h, feats.ctypes.data, feats.shape[1], fo.ctypes.data, n_utts, _ptr(u2s),
                                        n_spk, _ptr(st), _ptr(fm), fcols, out.ctypes.data, ost))
        return out[:T, :OD]

    def run_dev(self, d_feats, in_stride, frame_offsets, d_out, out_stride, utt2spk=None, n_spk=None, cmvn_stats=None,
                d_fmllr=None, fmllr_cols=0, stream=None):
        """vbgpu_feat_run_dev: device features in and out (d_out [T x out_stride]); frame_offsets, utt2spk and cmvn_stats
        are host arrays.  Enqueued on `stream` (default: torch's current stream)."""
        fo = _np(frame_offsets, np.int64)
        n_utts = len(fo) - 1
        u2s = _np(utt2spk, np.int32) if utt2spk is not None else None
        if n_spk is None:
            n_spk = n_utts if u2s is None else int(u2s.max()) + 1 if len(u2s) else 0
        st = _np(cmvn_stats, np.float64) if cmvn_stats is not None else None
        check(capi.lib().vbgpu_feat_run_dev(self.h, _ptr(d_feats), in_stride, fo.ctypes.data, n_utts, _ptr(u2s), n_spk,
                                            _ptr(st), _ptr(d_fmllr), fmllr_cols, _ptr(d_out), out_stride,
                                            _stream_ptr(stream)))


class AmDiagGmmGpu(_Handle):
    """Device-resident AmDiagGmm, flattened: pdf p owns Gaussians [pdf_offsets[p], pdf_offsets[p+1])."""
    _destroy = "vbgpu_gmm_destroy"

    def __init__(self, pdf_offsets, gconsts, means_invvars, inv_vars, device=0):
        super().__init__()
        po = _np(pdf_offsets, np.int32)
        gc, miv, iv = _np(gconsts, np.float32), _np(means_invvars, np.float32), _np(inv_vars, np.float32)
        check(capi.lib().vbgpu_gmm_create(len(po) - 1, miv.shape[1], po.ctypes.data, gc.ctypes.data, miv.ctypes.data,
                                          iv.ctypes.data, miv.shape[1], device, C.byref(self.h)))
        self.device = device

    @classmethod
    def from_mdl(cls, mdl_bytes, device=0):
        """A model file as the recipes write it (final.mdl: TransitionModel + AmDiagGmm, binary) -> (scorer, tid2pdf).
        tid2pdf is 1-based like transition-ids (entry 0 unused); empty for a bare AmDiagGmm."""
        from . import kaldi_io
        m = kaldi_io.read_mdl(mdl_bytes)
        am = cls(m["pdf_offsets"], m["gconsts"], m["means_invvars"], m["inv_vars"], device=device)
        return am, m["tid2pdf"]

    @classmethod
    def from_model(cls, m, device=0):
        return cls(m.pdf_offsets, m.gconsts, m.miv, m.iv, device)

    def NumPdfs(self):
        return check(capi.lib().vbgpu_gmm_num_pdfs(self.h))

    def NumGauss(self):
        return check(capi.lib().vbgpu_gmm_num_gauss(self.h))

    def Dim(self):
        return check(capi.lib().vbgpu_gmm_dim(self.h))

    def set_kernel(self, kind):
        """0 auto, 1 FP32 SIMT, 2 tcgen05."""
        check(capi.lib().vbgpu_gmm_set_kernel(self.h, kind))

    def set_gconsts(self, gconsts):
        gc = _np(gconsts, np.float32)
        check(capi.lib().vbgpu_gmm_set_gconsts(self.h, gc.ctypes.data))

    def score(self, feats):
        """Dense all-pdf log-likelihoods [T, P] (what the decodable would compute lazily)."""
        feats = _np(feats, np.float32)
        T, P = feats.shape[0], self.NumPdfs()
        out = np.zeros((max(T, 1), P), np.float32)
        check(capi.lib().vbgpu_gmm_score(self.h, feats.ctypes.data, T, feats.shape[1], out.ctypes.data, P))
        return out[:T]

    def score_dev(self, d_feats, T, stride, d_ll, ll_stride, stream=None):
        check(capi.lib().vbgpu_gmm_score_dev(self.h, _ptr(d_feats), T, stride, _ptr(d_ll), ll_stride,
                                             _stream_ptr(stream)))

    def NumCols(self):
        """Columns of the score matrix in DEVICE COLUMN ORDER (>= NumPdfs(); see include/vbgpu.h)."""
        return check(capi.lib().vbgpu_gmm_num_cols(self.h))

    def col_of_pdf(self):
        """int32 [NumPdfs()]: the column of the device-order score matrix that holds each pdf."""
        out = np.zeros(self.NumPdfs(), np.int32)
        check(capi.lib().vbgpu_gmm_col_of_pdf(self.h, out.ctypes.data))
        return out

    def plan_note(self):
        """'' when the model is scored by the tcgen05 kernel, else the reason it is not."""
        return capi.lib().vbgpu_gmm_plan_note(self.h).decode()

    def score_cols_dev(self, d_feats, T, stride, d_ll, ll_stride, stream=None):
        """Device column order: d_ll[t, col_of_pdf()[p]] (ll_stride >= NumCols()); no gather kernel."""
        check(capi.lib().vbgpu_gmm_score_cols_dev(self.h, _ptr(d_feats), T, stride, _ptr(d_ll), ll_stride,
                                                  _stream_ptr(stream)))

    def score_subset(self, feats, frame_offsets, subsets):
        """Forced-alignment form: utterance u (rows frame_offsets[u]:frame_offsets[u+1]) is scored against the pdfs
        subsets[u] only.  Returns a list of [T_u, len(subsets[u])] arrays (columns in the order given)."""
        feats = _np(feats, np.float32)
        fo = _np(frame_offsets, np.int64)
        so = np.zeros(len(subsets) + 1, np.int64)
        so[1:] = np.cumsum([len(x) for x in subsets])
        pdfs = _np(np.concatenate([np.asarray(x, np.int32) for x in subsets]) if so[-1] else np.zeros(1, np.int32), np.int32)
        oo = np.zeros(len(subsets) + 1, np.int64)
        total = int(sum((fo[u + 1] - fo[u]) * len(subsets[u]) for u in range(len(subsets))))
        out = np.zeros(max(total, 1), np.float32)
        check(capi.lib().vbgpu_gmm_score_subset(self.h, feats.ctypes.data, feats.shape[0], feats.shape[1], fo.ctypes.data,
                                                len(subsets), so.ctypes.data, pdfs.ctypes.data, out.ctypes.data,
                                                oo.ctypes.data))
        return [out[oo[u]:oo[u + 1]].reshape(int(fo[u + 1] - fo[u]), len(subsets[u])) for u in range(len(subsets))]

    def score_gather(self, feats, frames, pdfs):
        """Lattice-rescoring form: one log-likelihood per (frame, pdf) pair."""
        feats = _np(feats, np.float32)
        fr, pd = _np(frames, np.int32), _np(pdfs, np.int32)
        out = np.zeros(max(len(fr), 1), np.float32)
        check(capi.lib().vbgpu_gmm_score_gather(self.h, feats.ctypes.data, feats.shape[0], feats.shape[1], fr.ctypes.data,
                                                pd.ctypes.data, len(fr), out.ctypes.data))
        return out[:len(fr)]

    def ComponentPosteriors(self, feats, pdf_ids, pdf_offsets, weights=None):
        """DiagGmm::ComponentPosteriors of every frame's aligned pdf (gmm-post-to-gpost): returns (post, offsets,
        loglikes) with frame t's posteriors at post[offsets[t]:offsets[t+1]]."""
        feats = _np(feats, np.float32)
        ids = _np(pdf_ids, np.int32)
        sizes = np.diff(np.asarray(pdf_offsets))[ids]
        offs = np.zeros(len(ids) + 1, np.int64)
        offs[1:] = np.cumsum(sizes)
        post = np.zeros(int(offs[-1]), np.float32)
        ll = np.zeros(len(ids), np.float32)
        w = _np(weights, np.float32) if weights is not None else None
        check(capi.lib().vbgpu_gmm_component_posteriors(self.h, feats.ctypes.data, feats.shape[0], feats.shape[1],
                                                        ids.ctypes.data, _ptr(w), post.ctypes.data, ll.ctypes.data))
        return post, offs, ll

    def rescored_frames(self):
        """Frames of the last launch re-scored by the FP32 kernel (outside the fp16 plan / scores at the padding level)."""
        n = C.c_int64(0)
        check(capi.lib().vbgpu_gmm_rescored_frames(self.h, C.byref(n)))
        return int(n.value)

    def bad_count(self):
        n = C.c_int64(0)
        check(capi.lib().vbgpu_gmm_bad_count(self.h, C.byref(n)))
        return n.value


class DecodableAmDiagGmmGpu:
    """DecodableInterface (itf/decodable-itf.h:83-119) over a dense device-computed score matrix.

    Like DecodableAmDiagGmmScaled (gmm/decodable-am-diag-gmm.h:121-160): LogLikelihood(frame, tid) returns
    scale * loglike(frame, pdf(tid)); tids are 1-based, `tid2pdf[tid]` is TransitionModel::TransitionIdToPdf."""

    def __init__(self, am, tid2pdf, feats, scale=1.0):
        self.scale = np.float32(scale)
        self.tid2pdf = _np(tid2pdf, np.int32)  # index 0 unused
        self.loglikes = am.score(feats)        # one launch scores every (frame, pdf)

    def LogLikelihood(self, frame, tid):
        return float(self.scale * self.loglikes[frame, self.tid2pdf[tid]])

    def NumFramesReady(self):
        return self.loglikes.shape[0]

    def IsLastFrame(self, frame):
        assert frame < self.NumFramesReady()
        return frame == self.NumFramesReady() - 1

    def NumIndices(self):
        return len(self.tid2pdf) - 1


class AccumAmDiagGmmGpu(_Handle):
    """AccumAmDiagGmm with flags kGmmAll; statistics live in one FP64 device buffer."""
    _destroy = "vbgpu_acc_destroy"

    def __init__(self, am, num_tids=0):
        """num_tids > 0 adds the transition accumulators of gmm-acc-stats-ali (TransitionModel::NumTransitionIds()) to the
        same buffer, so that one all-reduce merges everything an EM pass produces."""
        super().__init__()
        self.am, self.num_tids = am, int(num_tids)
        check(capi.lib().vbgpu_acc_create_with_transitions(am.h, self.num_tids, C.byref(self.h)))

    def AccumulateTransitions(self, tids):
        """transition_accs[tid] += 1 for every frame's transition-id (gmm-acc-stats-ali.cpp:92)."""
        t = _np(tids, np.int32)
        check(capi.lib().vbgpu_acc_accumulate_transitions(self.h, t.ctypes.data, len(t)))

    def accumulate_transitions_dev(self, d_tids, T, stream=None):
        check(capi.lib().vbgpu_acc_accumulate_transitions_dev(self.h, _ptr(d_tids), T, _stream_ptr(stream)))

    def transition_accs(self):
        out = np.zeros(self.num_tids + 1)
        check(capi.lib().vbgpu_acc_download_transitions(self.h, out.ctypes.data))
        return out

    def SetZero(self):
        check(capi.lib().vbgpu_acc_zero(self.h))

    def AccumulateForUtterance(self, feats, pdf_ids, weights=None, feats2=None):
        """AccumulateForGmm (or ...Twofeats when feats2 is given) for every frame; returns sum of weight*loglike."""
        feats = _np(feats, np.float32)
        ids = _np(pdf_ids, np.int32)
        w = _np(weights, np.float32) if weights is not None else None
        f2 = _np(feats2, np.float32) if feats2 is not None else None
        tl = C.c_double(0.0)
        check(capi.lib().vbgpu_acc_accumulate(self.h, feats.ctypes.data, _ptr(f2), feats.shape[0], feats.shape[1],
                                              ids.ctypes.data, _ptr(w), C.byref(tl)))
        return tl.value

    def accumulate_dev(self, d_feats, T, stride, d_pdf_ids, d_weights=None, d_feats2=None, stream=None):
        check(capi.lib().vbgpu_acc_accumulate_dev(self.h, _ptr(d_feats), _ptr(d_feats2), T, stride, _ptr(d_pdf_ids),
                                                  _ptr(d_weights), _stream_ptr(stream)))

    def Add(self, scale, other):
        check(capi.lib().vbgpu_acc_add(self.h, float(scale), other.h))

    def buffer(self):
        """(device pointer, n_doubles) of [occ | mean | var | tot_like | tot_frames]."""
        p, n = C.c_void_p(), C.c_int64(0)
        check(capi.lib().vbgpu_acc_buffer(self.h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def as_tensor(self):
        """Zero-copy torch.float64 view of the accumulator buffer (for torch.distributed.all_reduce over NCCL)."""
        import torch
        ptr, n = self.buffer()

        class _Arr:
            __cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False), "version": 3}
        return torch.as_tensor(_Arr(), device="cuda:%d" % self.am.device)

    def AllReduce(self, group=None):
        """One in-place sum all-reduce per EM iteration (replaces gmm-sum-accs over x.JOBID.acc files)."""
        import torch.distributed as dist
        dist.all_reduce(self.as_tensor(), op=dist.ReduceOp.SUM, group=group)

    def download(self):
        N, D = self.am.NumGauss(), self.am.Dim()
        occ, mean, var = np.zeros(N), np.zeros((N, D)), np.zeros((N, D))
        tl, tf = C.c_double(0.0), C.c_double(0.0)
        check(capi.lib().vbgpu_acc_download(self.h, occ.ctypes.data, mean.ctypes.data, var.ctypes.data, C.byref(tl),
                                            C.byref(tf)))
        return occ, mean, var, tl.value, tf.value

    def TotLogLike(self):
        return self.download()[3]

    def TotCount(self):
        return self.download()[4]


class FmllrDiagGmmAccsGpu(_Handle):
    """n_spk independent FmllrDiagGmmAccs (transform/fmllr-diag-gmm.h:61-150, update_type "full"): beta, K, G per
    speaker on the device, accumulated for a whole batch of utterances per call (gmm-est-fmllr.cpp:40-55).  The solver
    (FmllrDiagGmmAccs::Update) stays on the host: hand it stats(spk)."""
    _destroy = "vbgpu_fmllr_destroy"

    def __init__(self, am, n_spk=1):
        super().__init__()
        self.am, self.n_spk = am, int(n_spk)
        check(capi.lib().vbgpu_fmllr_create(am.h, self.n_spk, C.byref(self.h)))

    def SetZero(self):
        check(capi.lib().vbgpu_fmllr_zero(self.h))

    def AccumulateForUtterances(self, feats, pdf_ids, frame_offsets=None, utt2spk=None, weights=None):
        """AccumulateForGmm for every frame of a packed batch; returns the sum of the frames' log-likelihoods."""
        feats = _np(feats, np.float32)
        ids = _np(pdf_ids, np.int32)
        T = feats.shape[0]
        fo = _np(frame_offsets if frame_offsets is not None else [0, T], np.int64)
        u2s = _np(utt2spk, np.int32) if utt2spk is not None else None
        w = _np(weights, np.float32) if weights is not None else None
        tl = C.c_double(0.0)
        check(capi.lib().vbgpu_fmllr_accumulate(self.h, feats.ctypes.data, T, feats.shape[1], ids.ctypes.data, _ptr(w),
                                                fo.ctypes.data, len(fo) - 1, _ptr(u2s), C.byref(tl)))
        return tl.value

    def accumulate_dev(self, d_feats, T, stride, d_pdf_ids, frame_offsets, utt2spk=None, d_weights=None, stream=None):
        fo = _np(frame_offsets, np.int64)
        u2s = _np(utt2spk, np.int32) if utt2spk is not None else None
        check(capi.lib().vbgpu_fmllr_accumulate_dev(self.h, _ptr(d_feats), T, stride, _ptr(d_pdf_ids), _ptr(d_weights),
                                                    fo.ctypes.data, len(fo) - 1, _ptr(u2s), _stream_ptr(stream)))

    def stats(self, spk=0):
        """(beta, K[D, D+1], G[D, (D+1)(D+2)/2]) of one speaker; G[i] in SpMatrix packing."""
        D = self.am.Dim()
        beta = C.c_double(0.0)
        K, G = np.zeros((D, D + 1)), np.zeros((D, (D + 1) * (D + 2) // 2))
        check(capi.lib().vbgpu_fmllr_download(self.h, int(spk), C.byref(beta), K.ctypes.data, G.ctypes.data))
        return beta.value, K, G


class MlltAccsGpu:
    """MlltAccs (transform/mllt.h:42-100, rand_prune = 0): beta and G[D, D(D+1)/2] accumulated on the device per call
    (gmm-acc-mllt.cpp:100-112); MlltAccs::Update (the solver) stays on the host."""

    def __init__(self, am):
        self.am = am
        D = am.Dim()
        self.beta, self.G = 0.0, np.zeros((D, D * (D + 1) // 2))

    def AccumulateForUtterance(self, feats, pdf_ids, weights=None):
        feats = _np(feats, np.float32)
        ids = _np(pdf_ids, np.int32)
        w = _np(weights, np.float32) if weights is not None else None
        beta, tl = C.c_double(self.beta), C.c_double(0.0)
        check(capi.lib().vbgpu_mllt_accumulate(self.am.h, feats.ctypes.data, feats.shape[0], feats.shape[1], ids.ctypes.data,
                                               _ptr(w), C.byref(beta), self.G.ctypes.data, C.byref(tl)))
        self.beta = beta.value
        return tl.value


class LdaEstimateGpu(_Handle):
    """The accumulation half of LdaEstimate (transform/lda-estimate.h): zero-, first- and second-order class statistics in
    one FP64 device buffer [zero C | first C*D | second D(D+1)/2].  Every frame is accumulated (no rand_prune); the solver
    (LdaEstimate::Estimate) stays on the host: hand it stats()."""
    _destroy = "vbgpu_lda_destroy"

    def __init__(self, num_classes, dim, device=0):
        super().__init__()
        self.C, self.D, self.device = int(num_classes), int(dim), int(device)
        check(capi.lib().vbgpu_lda_create(self.C, self.D, self.device, C.byref(self.h)))

    def NumClasses(self):
        return self.C

    def Dim(self):
        return self.D

    def ZeroAccumulators(self):
        check(capi.lib().vbgpu_lda_zero(self.h))

    def Accumulate(self, feats, class_ids, weights=None):
        """Accumulate(row t, class_ids[t], weights[t] or 1.0) for every row; a weight of 0 skips the frame.  Raises
        VbgpuError (ERR_NUMERIC) after adding every valid frame when a class id is outside [0, NumClasses())."""
        feats = _np(feats, np.float32)
        ids = _np(class_ids, np.int32)
        w = _np(weights, np.float32) if weights is not None else None
        check(capi.lib().vbgpu_lda_accumulate(self.h, feats.ctypes.data, feats.shape[0], feats.shape[1], ids.ctypes.data,
                                              _ptr(w)))

    def accumulate_dev(self, d_feats, T, stride, d_class_ids, d_weights=None, stream=None):
        check(capi.lib().vbgpu_lda_accumulate_dev(self.h, _ptr(d_feats), T, stride, _ptr(d_class_ids), _ptr(d_weights),
                                                  _stream_ptr(stream)))

    def bad_count(self):
        """Invalid class ids seen by accumulate_dev since the last query (the count is reset)."""
        n = C.c_int64(0)
        check(capi.lib().vbgpu_lda_bad_count(self.h, C.byref(n)))
        return n.value

    def stats(self):
        """(zero[C], first[C, D], second packed [D(D+1)/2], SpMatrix order)."""
        zero, first, second = np.zeros(self.C), np.zeros((self.C, self.D)), np.zeros(self.D * (self.D + 1) // 2)
        check(capi.lib().vbgpu_lda_download(self.h, zero.ctypes.data, first.ctypes.data, second.ctypes.data))
        return zero, first, second

    def TotCount(self):
        zero = np.zeros(self.C)
        check(capi.lib().vbgpu_lda_download(self.h, zero.ctypes.data, None, None))
        return float(zero.sum())

    def buffer(self):
        """(device pointer, n_doubles) of [zero | first | second]."""
        p, n = C.c_void_p(), C.c_int64(0)
        check(capi.lib().vbgpu_lda_buffer(self.h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def allreduce(self, comm, stream=None):
        """In-place sum all-reduce of the statistics over a raw ncclComm_t (replaces est-lda summing the job files)."""
        c = comm.value if isinstance(comm, C.c_void_p) else comm
        check(capi.lib().vbgpu_lda_allreduce(self.h, c, _stream_ptr(stream)))


class TreeStatsGpu(_Handle):
    """The statistics of acc-tree-stats (AccumulateTreeStats, hmm/tree-accu.cc) on the device: one GaussClusterable
    (count, sum x, sum x^2 in FP64) per EventType, in a device hash table of at most max_keys keys.  `tables` is the dict
    of kaldi_io.read_transitions (or synth.make_phone_alignment); EventTypes are tuples of sorted (key, value) pairs,
    (-1, pdf-class) first, as the reference's std::map holds them."""
    _destroy = "vbgpu_tree_destroy"

    def __init__(self, tables, dim, max_keys, context_width=3, central_position=1, ci_phones=(), device=0):
        super().__init__()
        self.N, self.P, self.D, self.device = int(context_width), int(central_position), int(dim), int(device)
        self._tables = {k: _np(tables[k], np.int32) for k in ("phone", "hmm_state", "pdf_class", "trans_state", "flags")}
        self._ci = _np(sorted(ci_phones), np.int32)
        t = capi.TidTables(len(self._tables["phone"]) - 1, *(self._tables[k].ctypes.data for k in
                                                              ("phone", "hmm_state", "pdf_class", "trans_state", "flags")))
        o = capi.TreeOpts(self.N, self.P, self._ci.ctypes.data if len(self._ci) else None, len(self._ci))
        check(capi.lib().vbgpu_tree_create(C.byref(o), C.byref(t), self.D, int(max_keys), self.device, C.byref(self.h)))

    def ZeroAccumulators(self):
        check(capi.lib().vbgpu_tree_zero(self.h))

    def AccumulateTreeStats(self, feats, tids, frame_offsets):
        """Host form over a packed batch: feats [T, >= dim] rows, tids[T], utterance u = rows frame_offsets[u] ... [u+1].
        Raises VbgpuError (ERR_NUMERIC) after adding everything else when a frame found no room in the key table."""
        feats = _np(feats, np.float32)
        tids, fo = _np(tids, np.int32), _np(frame_offsets, np.int64)
        check(capi.lib().vbgpu_tree_accumulate(self.h, feats.ctypes.data, feats.shape[1], tids.ctypes.data,
                                               fo.ctypes.data, len(fo) - 1))

    def accumulate_dev(self, d_feats, stride, d_tids, frame_offsets, stream=None):
        fo = _np(frame_offsets, np.int64)
        check(capi.lib().vbgpu_tree_accumulate_dev(self.h, _ptr(d_feats), stride, _ptr(d_tids), fo.ctypes.data,
                                                   len(fo) - 1, _stream_ptr(stream)))

    def bad_count(self):
        """(bad utterances, frames without room in the key table) since the last query; resets both."""
        b, d = C.c_int64(0), C.c_int64(0)
        check(capi.lib().vbgpu_tree_bad_count(self.h, C.byref(b), C.byref(d)))
        return b.value, d.value

    def NumKeys(self):
        n = C.c_int32(0)
        check(capi.lib().vbgpu_tree_num_keys(self.h, C.byref(n)))
        return n.value

    def download(self):
        """(pdf_class[K], phones[K, N] with -1 for absent positions, count[K], sum_x[K, D], sum_x2[K, D]) in EventType order."""
        K = self.NumKeys()
        pc, ph = np.zeros(K, np.int32), np.zeros((K, self.N), np.int32)
        cnt, sx, sx2 = np.zeros(K), np.zeros((K, self.D)), np.zeros((K, self.D))
        check(capi.lib().vbgpu_tree_download(self.h, pc.ctypes.data, ph.ctypes.data, cnt.ctypes.data, sx.ctypes.data,
                                             sx2.ctypes.data))
        return pc, ph, cnt, sx, sx2

    def stats(self):
        """dict EventType -> (count, sum_x[D], sum_x2[D]), inserted in the reference's std::map order."""
        pc, ph, cnt, sx, sx2 = self.download()
        out = {}
        for k in range(len(pc)):
            ev = ((-1, int(pc[k])),) + tuple((j, int(p)) for j, p in enumerate(ph[k]) if p >= 0)
            out[ev] = (float(cnt[k]), sx[k], sx2[k])
        return out

    def Add(self, other_stats):
        """Adds a dict of the form stats() returns, key by key (sum-tree-stats; merging handles of several GPUs)."""
        evs = list(other_stats)
        n = len(evs)
        pc, ph = np.zeros(n, np.int32), np.full((n, self.N), -1, np.int32)
        cnt, sx, sx2 = np.zeros(n), np.zeros((n, self.D)), np.zeros((n, self.D))
        for k, ev in enumerate(evs):
            for key, val in ev:
                if key == -1:
                    pc[k] = val
                else:
                    ph[k, key] = val
            cnt[k], sx[k], sx2[k] = other_stats[ev]
        check(capi.lib().vbgpu_tree_add(self.h, n, pc.ctypes.data, ph.ctypes.data, cnt.ctypes.data, sx.ctypes.data,
                                        sx2.ctypes.data))


class GmmAlignCompiledGpu(_Handle):
    """gmm-align-compiled on the device: exact Viterbi over each utterance's training graph (include/vbgpu.h,
    vbgpu_align_*).  `graphs` is a dict of packed arrays (synth.make_training_graphs builds one): state_offsets, start,
    final_cost, arc_offsets, arc_src, arc_dst, arc_ilabel, arc_weight.  The handle holds the graphs, not the model: create
    it once per training stage and align with each iteration's model (and its transition costs, tid_cost)."""
    _destroy = "vbgpu_align_destroy"
    _KEYS = (("state_offsets", np.int32), ("start", np.int32), ("final_cost", np.float32), ("arc_offsets", np.int64),
             ("arc_src", np.int32), ("arc_dst", np.int32), ("arc_ilabel", np.int32), ("arc_weight", np.float32))

    def __init__(self, graphs, tid2pdf, device=0):
        super().__init__()
        self._g = {k: _np(graphs[k], t) for k, t in self._KEYS}
        self.tid2pdf = _np(tid2pdf, np.int32)
        self.n_utts = len(self._g["start"])
        self.device = device
        check(capi.lib().vbgpu_align_create(self.n_utts, *(_ptr(self._g[k]) for k, _ in self._KEYS), self.tid2pdf.ctypes.data,
                                            len(self.tid2pdf) - 1, device, C.byref(self.h)))

    def set_workspace(self, nbytes):
        """Cap of the per-group workspace in bytes (<= 0: the default)."""
        check(capi.lib().vbgpu_align_set_workspace(self.h, int(nbytes)))

    def _tc(self, tid_cost):
        if tid_cost is None:
            return None
        tc = _np(tid_cost, np.float32)
        if len(tc) != len(self.tid2pdf):
            raise ValueError("tid_cost has %d entries, expected num_tids + 1 = %d" % (len(tc), len(self.tid2pdf)))
        return tc

    def Align(self, am, feats, frame_offsets, tid_cost=None, acoustic_scale=0.1):
        """Host form: returns (ali[T] transition-ids, pdf_ids[T], tot_cost[n_utts]); tot_cost = +inf (ali 0, pdf -1)
        where no final state is reachable.  Raises VbgpuError (ERR_NUMERIC) on non-finite log-likelihoods."""
        feats = _np(feats, np.float32)
        fo = _np(frame_offsets, np.int64)
        tc = self._tc(tid_cost)
        T = int(fo[-1])
        ali, pdf, tot = np.zeros(max(T, 1), np.int32), np.zeros(max(T, 1), np.int32), np.zeros(len(fo) - 1)
        check(capi.lib().vbgpu_align(self.h, am.h, _ptr(tc), float(acoustic_scale), feats.ctypes.data,
                                     feats.shape[1] if feats.ndim == 2 else 0, fo.ctypes.data, len(fo) - 1,
                                     ali.ctypes.data, pdf.ctypes.data, tot.ctypes.data))
        return ali[:T], pdf[:T], tot

    def align_dev(self, am, d_feats, stride, frame_offsets, d_ali, d_pdf_ids, d_tot_cost, tid_cost=None,
                  acoustic_scale=0.1, stream=None):
        """Device form: d_ali / d_pdf_ids (nullable) [T] int32, d_tot_cost [n_utts] float64 device buffers."""
        fo = _np(frame_offsets, np.int64)
        tc = self._tc(tid_cost)
        check(capi.lib().vbgpu_align_dev(self.h, am.h, _ptr(tc), float(acoustic_scale), _ptr(d_feats), stride,
                                         fo.ctypes.data, len(fo) - 1, _ptr(d_ali), _ptr(d_pdf_ids), _ptr(d_tot_cost),
                                         _stream_ptr(stream)))


class GmmDecodeFasterGpu(_Handle):
    """gmm-decode-faster on the device: one-best beam search over one decoding graph (HCLG) shared by every utterance
    (include/vbgpu.h, vbgpu_decoder_*).  `graph` is a dict (synth.make_decoding_graph builds one): num_states, start,
    final_cost, arc_src, arc_dst, arc_ilabel, arc_olabel, arc_weight.  The handle holds the graph, not the model.
    Options are FasterDecoderOptions' beam and max_active, plus max_tokens (a frame's token capacity).  On a large graph
    the defaults (beam 16, unlimited max_active) outgrow max_tokens: pass a finite max_active (the decode scripts use
    7000) or max_tokens >= the graph's state count."""
    _destroy = "vbgpu_decoder_destroy"
    _KEYS = (("arc_src", np.int32), ("arc_dst", np.int32), ("arc_ilabel", np.int32), ("arc_olabel", np.int32),
             ("arc_weight", np.float32))

    def __init__(self, graph, tid2pdf, beam=16.0, max_active=2**31 - 1, max_tokens=65536, device=0):
        super().__init__()
        self._g = {k: _np(graph[k], t) for k, t in self._KEYS}
        self.final_cost = _np(graph["final_cost"], np.float32)
        self.tid2pdf = _np(tid2pdf, np.int32)
        self.device = device
        self.opts = capi.default_decoder_opts(beam=beam, max_active=max_active, max_tokens=max_tokens)
        check(capi.lib().vbgpu_decoder_create(int(graph["num_states"]), int(graph["start"]), self.final_cost.ctypes.data,
                                              len(self._g["arc_src"]), *(self._g[k].ctypes.data for k, _ in self._KEYS),
                                              self.tid2pdf.ctypes.data, len(self.tid2pdf) - 1, device, C.byref(self.h)))

    def set_workspace(self, nbytes):
        """Cap of the per-group workspace in bytes (<= 0: the default)."""
        check(capi.lib().vbgpu_decoder_set_workspace(self.h, int(nbytes)))

    def Decode(self, am, feats, frame_offsets, acoustic_scale=0.1, max_words=64):
        """Host form (Decode + ReachedFinal + GetBestPath per utterance): returns (ali[T] transition-ids, pdf_ids[T],
        words per utterance (lists, at most max_words each), num_words[n_utts], tot_cost[n_utts], status[n_utts]).
        status: 0 reached a final state, 1 did not (partial best path), 2 no token left, 3 over max_tokens.  Raises
        VbgpuError (ERR_NUMERIC) on non-finite log-likelihoods."""
        feats = _np(feats, np.float32)
        fo = _np(frame_offsets, np.int64)
        n, T = len(fo) - 1, int(fo[-1])
        ali, pdf = np.zeros(max(T, 1), np.int32), np.zeros(max(T, 1), np.int32)
        words, nw = np.zeros(max(n * max_words, 1), np.int32), np.zeros(max(n, 1), np.int32)
        tot, st = np.zeros(max(n, 1)), np.zeros(max(n, 1), np.int32)
        check(capi.lib().vbgpu_decode(self.h, am.h, C.byref(self.opts), float(acoustic_scale), feats.ctypes.data,
                                      feats.shape[1] if feats.ndim == 2 else 0, fo.ctypes.data, n, ali.ctypes.data,
                                      pdf.ctypes.data, words.ctypes.data, max_words, nw.ctypes.data, tot.ctypes.data,
                                      st.ctypes.data))
        wl = [words[u * max_words:u * max_words + min(int(nw[u]), max_words)].tolist() for u in range(n)]
        return ali[:T], pdf[:T], wl, nw[:n], tot[:n], st[:n]

    def decode_dev(self, am, d_feats, stride, frame_offsets, d_ali, d_pdf_ids, d_words, max_words, d_num_words,
                   d_tot_cost, d_status, acoustic_scale=0.1, stream=None):
        """Feature form on device buffers: d_ali / d_pdf_ids (nullable) [T], d_words [n_utts * max_words],
        d_num_words / d_status [n_utts] int32, d_tot_cost [n_utts] float64."""
        fo = _np(frame_offsets, np.int64)
        check(capi.lib().vbgpu_decode_dev(self.h, am.h, C.byref(self.opts), float(acoustic_scale), _ptr(d_feats), stride,
                                          fo.ctypes.data, len(fo) - 1, _ptr(d_ali), _ptr(d_pdf_ids), _ptr(d_words),
                                          max_words, _ptr(d_num_words), _ptr(d_tot_cost), _ptr(d_status),
                                          _stream_ptr(stream)))

    def decode_loglikes_dev(self, am, d_loglikes, ll_stride, frame_offsets, d_ali, d_pdf_ids, d_words, max_words,
                            d_num_words, d_tot_cost, d_status, acoustic_scale=0.1, stream=None):
        """Log-likelihood form: d_loglikes [T x ll_stride] in the model's device column order."""
        fo = _np(frame_offsets, np.int64)
        check(capi.lib().vbgpu_decode_loglikes_dev(self.h, am.h, C.byref(self.opts), float(acoustic_scale),
                                                   _ptr(d_loglikes), ll_stride, fo.ctypes.data, len(fo) - 1, _ptr(d_ali),
                                                   _ptr(d_pdf_ids), _ptr(d_words), max_words, _ptr(d_num_words),
                                                   _ptr(d_tot_cost), _ptr(d_status), _stream_ptr(stream)))


    # lattice arrays of vbgpu_lattice_out: (name, dtype, per state (True) or per arc)
    LATTICE_ARRAYS = (("state_frame", np.int32, True), ("state_graph", np.int32, True), ("state_final", np.float32, True),
                      ("arc_src", np.int32, False), ("arc_dst", np.int32, False), ("arc_ilabel", np.int32, False),
                      ("arc_olabel", np.int32, False), ("arc_graph_cost", np.float32, False),
                      ("arc_ac_cost", np.float32, False))

    @staticmethod
    def lattice_out(arrays):
        """vbgpu_lattice_out over a dict of arrays (numpy or torch): the LATTICE_ARRAYS names plus num_states,
        num_arcs, lattice_status and optionally arena_peak."""
        return capi.LatticeOut(**{k: _ptr(arrays.get(k)) for k, _ in capi.LatticeOut._fields_})

    def DecodeLattice(self, am, feats, frame_offsets, acoustic_scale=0.1, max_words=64, lattice_beam=10.0,
                      max_states=131072, max_arcs=524288, arena_tokens=8192, arena_links=24576):
        """Host form of lattice generation (LatticeFasterDecoder up to GetRawLattice): returns Decode's tuple plus a
        list with one dict per utterance: state_frame, state_graph, state_final (per state), arc_src, arc_dst,
        arc_ilabel, arc_olabel, arc_graph_cost, arc_ac_cost (per arc), num_states, num_arcs, lattice_status (0 written,
        1 lattice store overflow, 2 over max_states / max_arcs: counts only) and arena_peak (tokens, links)."""
        feats = _np(feats, np.float32)
        fo = _np(frame_offsets, np.int64)
        n, T = len(fo) - 1, int(fo[-1])
        lo = capi.default_lattice_opts(lattice_beam=lattice_beam, max_states=max_states, max_arcs=max_arcs,
                                       arena_tokens=arena_tokens, arena_links=arena_links)
        ali, pdf = np.zeros(max(T, 1), np.int32), np.zeros(max(T, 1), np.int32)
        words, nw = np.zeros(max(n * max_words, 1), np.int32), np.zeros(max(n, 1), np.int32)
        tot, st = np.zeros(max(n, 1)), np.zeros(max(n, 1), np.int32)
        arr = {k: np.zeros(max(n * (max_states if per_state else max_arcs), 1), t)
               for k, t, per_state in self.LATTICE_ARRAYS}
        for k in ("num_states", "num_arcs", "lattice_status"):
            arr[k] = np.zeros(max(n, 1), np.int32)
        arr["arena_peak"] = np.zeros(max(2 * n, 2), np.int32)
        out = self.lattice_out(arr)
        check(capi.lib().vbgpu_decode_lattice(self.h, am.h, C.byref(self.opts), C.byref(lo), float(acoustic_scale),
                                              feats.ctypes.data, feats.shape[1] if feats.ndim == 2 else 0,
                                              fo.ctypes.data, n, ali.ctypes.data, pdf.ctypes.data, words.ctypes.data,
                                              max_words, nw.ctypes.data, tot.ctypes.data, st.ctypes.data, C.byref(out)))
        wl = [words[u * max_words:u * max_words + min(int(nw[u]), max_words)].tolist() for u in range(n)]
        return ali[:T], pdf[:T], wl, nw[:n], tot[:n], st[:n], self.split_lattices(arr, n, max_states, max_arcs)

    @classmethod
    def split_lattices(cls, arr, n, max_states, max_arcs):
        """Per-utterance dicts from the flat arrays of a call (numpy)."""
        lats = []
        for u in range(n):
            ns, na, ls = int(arr["num_states"][u]), int(arr["num_arcs"][u]), int(arr["lattice_status"][u])
            d = {"num_states": ns, "num_arcs": na, "lattice_status": ls}
            if "arena_peak" in arr and arr["arena_peak"] is not None:
                d["arena_peak"] = (int(arr["arena_peak"][2 * u]), int(arr["arena_peak"][2 * u + 1]))
            for k, _, per_state in cls.LATTICE_ARRAYS:
                cap, cnt = (max_states, ns) if per_state else (max_arcs, na)
                d[k] = np.asarray(arr[k][u * cap:u * cap + (cnt if ls == 0 else 0)]).copy()
            lats.append(d)
        return lats

    def _lattice_opts(self, lattice_opts):
        return lattice_opts if lattice_opts is not None else capi.default_lattice_opts()

    def decode_lattice_dev(self, am, d_feats, stride, frame_offsets, d_ali, d_pdf_ids, d_words, max_words,
                           d_num_words, d_tot_cost, d_status, lattice, lattice_opts=None, acoustic_scale=0.1,
                           stream=None):
        """Feature form of lattice generation on device buffers: the decode_dev arguments plus `lattice`, a dict of
        device arrays (lattice_out) sized by lattice_opts (capi.default_lattice_opts)."""
        fo = _np(frame_offsets, np.int64)
        out = self.lattice_out(lattice)
        check(capi.lib().vbgpu_decode_lattice_dev(self.h, am.h, C.byref(self.opts),
                                                  C.byref(self._lattice_opts(lattice_opts)), float(acoustic_scale),
                                                  _ptr(d_feats), stride, fo.ctypes.data, len(fo) - 1, _ptr(d_ali),
                                                  _ptr(d_pdf_ids), _ptr(d_words), max_words, _ptr(d_num_words),
                                                  _ptr(d_tot_cost), _ptr(d_status), C.byref(out), _stream_ptr(stream)))

    def decode_lattice_loglikes_dev(self, am, d_loglikes, ll_stride, frame_offsets, d_ali, d_pdf_ids, d_words,
                                    max_words, d_num_words, d_tot_cost, d_status, lattice, lattice_opts=None,
                                    acoustic_scale=0.1, stream=None):
        """Log-likelihood form of lattice generation: d_loglikes [T x ll_stride] in the model's device column order."""
        fo = _np(frame_offsets, np.int64)
        out = self.lattice_out(lattice)
        check(capi.lib().vbgpu_decode_lattice_loglikes_dev(self.h, am.h, C.byref(self.opts),
                                                           C.byref(self._lattice_opts(lattice_opts)),
                                                           float(acoustic_scale), _ptr(d_loglikes), ll_stride,
                                                           fo.ctypes.data, len(fo) - 1, _ptr(d_ali), _ptr(d_pdf_ids),
                                                           _ptr(d_words), max_words, _ptr(d_num_words),
                                                           _ptr(d_tot_cost), _ptr(d_status), C.byref(out),
                                                           _stream_ptr(stream)))


class ScoringPipeline(_Handle):
    """PCM -> per-frame per-pdf log-likelihoods in one call (MFCC -> CMVN -> deltas|LDA -> fMLLR -> GMM scoring)."""
    _destroy = "vbgpu_pipeline_destroy"

    def __init__(self, mfcc, feat, am):
        super().__init__()
        self.mfcc, self.feat, self.am = mfcc, feat, am
        check(capi.lib().vbgpu_pipeline_create(mfcc.h, feat.h, am.h, C.byref(self.h)))

    def score(self, pcm, sample_offsets, utt2spk=None, n_spk=None, cmvn_stats=None, fmllr=None, out=None,
              return_feats=False):
        """Host buffers in, host loglikes [T, P] out (H2D and D2H inside).  `pcm`/`out` may be pinned torch tensors."""
        so = _np(sample_offsets, np.int64)
        n_utts = len(so) - 1
        u2s = _np(utt2spk, np.int32) if utt2spk is not None else None
        if n_spk is None:
            n_spk = n_utts if u2s is None else int(u2s.max()) + 1 if len(u2s) else 0
        T = int(self.mfcc.frame_offsets(so)[-1])
        P, D = self.am.NumPdfs(), self.am.Dim()
        if out is None:
            out = np.zeros((max(T, 1), P), np.float32)
        st = _np(cmvn_stats, np.float64) if cmvn_stats is not None else None
        fm = _np(fmllr, np.float32) if fmllr is not None else None
        fcols = fm.shape[-1] if fm is not None else 0
        fo, fst = None, 0
        if return_feats:
            fst = kaldi_stride(D)
            fo = np.zeros((max(T, 1), fst), np.float32)
        pcm_arr = pcm if not isinstance(pcm, np.ndarray) else np.ascontiguousarray(pcm, np.int16)
        ll_stride = out.shape[1] if hasattr(out, "shape") else P
        check(capi.lib().vbgpu_pipeline_score_i16(self.h, _ptr(pcm_arr), so.ctypes.data, n_utts, _ptr(u2s), n_spk,
                                                  _ptr(st), _ptr(fm), fcols, _ptr(out), ll_stride, _ptr(fo), fst))
        res = out[:T]
        return (res, fo[:T, :D]) if return_feats else res

    def _host_args(self, pcm, sample_offsets, utt2spk, n_spk, cmvn_stats, fmllr):
        so = _np(sample_offsets, np.int64)
        n_utts = len(so) - 1
        u2s = _np(utt2spk, np.int32) if utt2spk is not None else None
        if n_spk is None:
            n_spk = n_utts if u2s is None else int(u2s.max()) + 1 if len(u2s) else 0
        st = _np(cmvn_stats, np.float64) if cmvn_stats is not None else None
        fm = _np(fmllr, np.float32) if fmllr is not None else None
        pcm_arr = pcm if not isinstance(pcm, np.ndarray) else np.ascontiguousarray(pcm, np.int16)
        return so, n_utts, u2s, n_spk, st, fm, (fm.shape[-1] if fm is not None else 0), pcm_arr

    def score_subset(self, pcm, sample_offsets, subset_offsets, subset_pdfs, utt2spk=None, n_spk=None, cmvn_stats=None,
                     fmllr=None, out=None):
        """Host PCM in, the per-utterance pdf subsets' log-likelihoods out (packed; returns (out, out_offsets)).
        `out` may be a pinned torch tensor / numpy array of sum(T_u * |S_u|) floats."""
        so, n_utts, u2s, n_spk, st, fm, fcols, pcm_arr = self._host_args(pcm, sample_offsets, utt2spk, n_spk, cmvn_stats, fmllr)
        sub_o = _np(subset_offsets, np.int64)
        sub_p = subset_pdfs if not isinstance(subset_pdfs, np.ndarray) else _np(subset_pdfs, np.int32)
        fo = self.mfcc.frame_offsets(so)
        oo = np.zeros(n_utts + 1, np.int64)
        if out is None:
            out = np.zeros(max(int(np.sum(np.diff(fo) * np.diff(sub_o))), 1), np.float32)
        check(capi.lib().vbgpu_pipeline_score_subset_i16(self.h, _ptr(pcm_arr), so.ctypes.data, n_utts, _ptr(u2s), n_spk,
                                                         _ptr(st), _ptr(fm), fcols, sub_o.ctypes.data, _ptr(sub_p),
                                                         _ptr(out), oo.ctypes.data))
        return out, oo

    def score_gather(self, pcm, sample_offsets, frames, pdfs, utt2spk=None, n_spk=None, cmvn_stats=None, fmllr=None):
        """Host PCM in, one log-likelihood per (frame, pdf) arc out."""
        so, n_utts, u2s, n_spk, st, fm, fcols, pcm_arr = self._host_args(pcm, sample_offsets, utt2spk, n_spk, cmvn_stats, fmllr)
        fr, pd = _np(frames, np.int32), _np(pdfs, np.int32)
        out = np.zeros(max(len(fr), 1), np.float32)
        check(capi.lib().vbgpu_pipeline_score_gather_i16(self.h, _ptr(pcm_arr), so.ctypes.data, n_utts, _ptr(u2s), n_spk,
                                                         _ptr(st), _ptr(fm), fcols, fr.ctypes.data, pd.ctypes.data, len(fr),
                                                         out.ctypes.data))
        return out[:len(fr)]

    def score_dev(self, d_pcm, sample_offsets, utt2spk, n_spk, d_fmllr, fmllr_cols, d_ll, ll_stride, d_feats=None,
                  feats_stride=0, stream=None):
        so = _np(sample_offsets, np.int64)
        u2s = _np(utt2spk, np.int32) if utt2spk is not None else None
        check(capi.lib().vbgpu_pipeline_score_dev(self.h, _ptr(d_pcm), so.ctypes.data, len(so) - 1, _ptr(u2s), n_spk,
                                                  _ptr(d_fmllr), fmllr_cols, _ptr(d_ll), ll_stride, _ptr(d_feats),
                                                  feats_stride, _stream_ptr(stream)))

    def score_cols_dev(self, d_pcm, sample_offsets, utt2spk, n_spk, d_fmllr, fmllr_cols, d_ll, ll_stride, d_feats=None,
                       feats_stride=0, stream=None):
        """score_dev with the log-likelihoods in device column order (AmDiagGmmGpu.col_of_pdf)."""
        so = _np(sample_offsets, np.int64)
        u2s = _np(utt2spk, np.int32) if utt2spk is not None else None
        check(capi.lib().vbgpu_pipeline_score_cols_dev(self.h, _ptr(d_pcm), so.ctypes.data, len(so) - 1, _ptr(u2s), n_spk,
                                                       _ptr(d_fmllr), fmllr_cols, _ptr(d_ll), ll_stride, _ptr(d_feats),
                                                       feats_stride, _stream_ptr(stream)))

    def accumulate_dev(self, acc, d_pcm, sample_offsets, utt2spk, n_spk, d_fmllr, fmllr_cols, d_pdf_ids, stream=None):
        so = _np(sample_offsets, np.int64)
        u2s = _np(utt2spk, np.int32) if utt2spk is not None else None
        check(capi.lib().vbgpu_pipeline_accumulate_dev(self.h, acc.h, _ptr(d_pcm), so.ctypes.data, len(so) - 1,
                                                       _ptr(u2s), n_spk, _ptr(d_fmllr), fmllr_cols, _ptr(d_pdf_ids),
                                                       _stream_ptr(stream)))
