"""ctypes binding of libvbgpu.so (include/vbgpu.h) — the only way Python code reaches the CUDA path.

There is no CPU fallback: importing this module fails loudly when the in-tree library has not been built
(`python -c "import __graft_entry__ as g; g.build()"` or `make -C voicebridge_b200/csrc`).
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libvbgpu.so")

OK, ERR_INVALID, ERR_CUDA, ERR_NUMERIC, ERR_NOMEM = 0, -1, -2, -3, -4


class VbgpuError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("vbgpu error %d: %s" % (code, msg))
        self.code = code


class MfccOpts(C.Structure):
    """vbgpu_mfcc_opts (mirror of Kaldi's MfccOptions, feat/feature-mfcc.h:38-78)."""
    _fields_ = [
        ("samp_freq", C.c_float), ("frame_shift_ms", C.c_float), ("frame_length_ms", C.c_float),
        ("dither", C.c_float), ("preemph_coeff", C.c_float), ("remove_dc_offset", C.c_int32),
        ("window_type", C.c_int32), ("round_to_power_of_two", C.c_int32), ("blackman_coeff", C.c_float),
        ("snip_edges", C.c_int32), ("num_bins", C.c_int32), ("low_freq", C.c_float), ("high_freq", C.c_float),
        ("vtln_low", C.c_float), ("vtln_high", C.c_float), ("htk_mode", C.c_int32), ("num_ceps", C.c_int32),
        ("use_energy", C.c_int32), ("energy_floor", C.c_float), ("raw_energy", C.c_int32),
        ("cepstral_lifter", C.c_float), ("htk_compat", C.c_int32),
    ]


class PitchOpts(C.Structure):
    """vbgpu_pitch_opts (mirror of PitchExtractionOptions, feat/pitch-functions.h:43-123)."""
    _fields_ = [
        ("samp_freq", C.c_float), ("frame_shift_ms", C.c_float), ("frame_length_ms", C.c_float),
        ("preemph_coeff", C.c_float), ("min_f0", C.c_float), ("max_f0", C.c_float), ("soft_min_f0", C.c_float),
        ("penalty_factor", C.c_float), ("lowpass_cutoff", C.c_float), ("resample_freq", C.c_float),
        ("delta_pitch", C.c_float), ("nccf_ballast", C.c_float), ("lowpass_filter_width", C.c_int32),
        ("upsample_filter_width", C.c_int32), ("recompute_frame", C.c_int32), ("snip_edges", C.c_int32),
    ]


class ProcessPitchOpts(C.Structure):
    """vbgpu_process_pitch_opts (mirror of ProcessPitchOptions, feat/pitch-functions.h:216-255)."""
    _fields_ = [
        ("pitch_scale", C.c_float), ("pov_scale", C.c_float), ("pov_offset", C.c_float),
        ("delta_pitch_scale", C.c_float), ("delta_pitch_noise_stddev", C.c_float),
        ("normalization_left_context", C.c_int32), ("normalization_right_context", C.c_int32),
        ("delta_window", C.c_int32), ("delay", C.c_int32), ("add_pov_feature", C.c_int32),
        ("add_normalized_log_pitch", C.c_int32), ("add_delta_pitch", C.c_int32), ("add_raw_log_pitch", C.c_int32),
    ]


class FeatOpts(C.Structure):
    """vbgpu_feat_opts."""
    _fields_ = [("norm_means", C.c_int32), ("norm_vars", C.c_int32), ("mode", C.c_int32), ("delta_order", C.c_int32),
                ("delta_window", C.c_int32), ("splice_left", C.c_int32), ("splice_right", C.c_int32)]


class WaveInfo(C.Structure):
    """vbgpu_wave_info."""
    _fields_ = [("samp_freq", C.c_float), ("num_channels", C.c_int32), ("num_samples", C.c_int64),
                ("data_offset", C.c_int64), ("reverse_bytes", C.c_int32)]


_vp, _i32, _i64, _f, _d = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_double
_pi = C.POINTER(C.c_int)

class IoInfo(C.Structure):
    """vbgpu_io_info (include/vbgpu.h)."""
    _fields_ = [("kind", C.c_int32), ("rows", C.c_int32), ("cols", C.c_int32), ("min_value", C.c_float),
                ("range", C.c_float), ("header_bytes", C.c_int64), ("total_bytes", C.c_int64)]


class TidTables(C.Structure):
    """vbgpu_tid_tables: per transition-id arrays of num_tids + 1 (entry 0 unused)."""
    _fields_ = [("num_tids", C.c_int32), ("phone", _vp), ("hmm_state", _vp), ("pdf_class", _vp), ("trans_state", _vp),
                ("flags", _vp)]


class TreeOpts(C.Structure):
    """vbgpu_tree_opts (acc-tree-stats --context-width / --central-position / --ci-phones)."""
    _fields_ = [("context_width", C.c_int32), ("central_position", C.c_int32), ("ci_phones", _vp),
                ("num_ci_phones", C.c_int32)]


TID_SELF_LOOP, TID_FINAL, TID_STATE0_EMITTING = 1, 2, 4

# name -> (restype, argtypes).  Pointers to data are passed as void* (integers / numpy .ctypes.data / torch .data_ptr()).
_SIGS = {
    "vbgpu_version": (C.c_int, []),
    "vbgpu_last_error": (C.c_char_p, []),
    "vbgpu_device_count": (C.c_int, [_pi]),
    "vbgpu_wave_parse": (C.c_int, [_vp, C.c_size_t, C.POINTER(WaveInfo)]),
    "vbgpu_wave_channel_i16": (C.c_int, [_vp, C.c_size_t, C.POINTER(WaveInfo), _i32, _vp]),
    "vbgpu_downsample_create": (C.c_int, [C.c_float, C.c_float, _i32, C.POINTER(_vp)]),
    "vbgpu_downsample_destroy": (None, [_vp]),
    "vbgpu_downsample_num_out": (_i64, [_vp, _i64]),
    "vbgpu_downsample_f32": (C.c_int, [_vp, _vp, _i64, _vp]),
    "vbgpu_downsample_dev": (C.c_int, [_vp, _vp, _i64, _vp, _vp]),
    "vbgpu_mfcc_opts_default": (None, [C.POINTER(MfccOpts)]),
    "vbgpu_mfcc_create": (C.c_int, [C.POINTER(MfccOpts), C.c_int, C.POINTER(_vp)]),
    "vbgpu_fbank_create": (C.c_int, [C.POINTER(MfccOpts), _i32, _i32, C.c_int, C.POINTER(_vp)]),
    "vbgpu_plp_create": (C.c_int, [C.POINTER(MfccOpts), _i32, _f, _f, C.c_int, C.POINTER(_vp)]),
    "vbgpu_mfcc_destroy": (C.c_int, [_vp]),
    "vbgpu_pitch_opts_default": (None, [C.POINTER(PitchOpts)]),
    "vbgpu_process_pitch_opts_default": (None, [C.POINTER(ProcessPitchOpts)]),
    "vbgpu_pitch_create": (C.c_int, [C.POINTER(PitchOpts), C.c_int, C.POINTER(_vp)]),
    "vbgpu_pitch_destroy": (None, [_vp]),
    "vbgpu_pitch_num_states": (_i32, [_vp]),
    "vbgpu_pitch_num_frames": (_i64, [_vp, _i64]),
    "vbgpu_pitch_compute_f32": (C.c_int, [_vp, _vp, _vp, _i32, C.POINTER(ProcessPitchOpts), _vp, _i32]),
    "vbgpu_pitch_compute_i16": (C.c_int, [_vp, _vp, _vp, _i32, C.POINTER(ProcessPitchOpts), _vp, _i32]),
    "vbgpu_pitch_process": (C.c_int, [_vp, C.POINTER(ProcessPitchOpts), _vp, _i32, _vp, _i32, _vp, _i32]),
    "vbgpu_mfcc_dim": (C.c_int, [_vp]),
    "vbgpu_mfcc_num_frames": (_i64, [_vp, _i64]),
    "vbgpu_mfcc_frame_offsets": (_i64, [_vp, _vp, _i32, _vp]),
    "vbgpu_mfcc_compute_i16": (C.c_int, [_vp, _vp, _vp, _i32, _vp, _vp, _i32]),
    "vbgpu_mfcc_compute_f32": (C.c_int, [_vp, _vp, _vp, _i32, _vp, _vp, _i32]),
    "vbgpu_mfcc_compute_dev": (C.c_int, [_vp, _vp, _i32, _vp, _i32, _vp, _vp, _i32, _vp]),
    "vbgpu_feat_opts_default": (None, [C.POINTER(FeatOpts)]),
    "vbgpu_feat_create": (C.c_int, [C.POINTER(FeatOpts), _i32, _vp, _i32, _i32, C.c_int, C.POINTER(_vp)]),
    "vbgpu_feat_destroy": (C.c_int, [_vp]),
    "vbgpu_feat_out_dim": (C.c_int, [_vp]),
    "vbgpu_cmvn_stats": (C.c_int, [_vp, _vp, _i32, _vp, _i32, _vp, _i32, _vp]),
    "vbgpu_feat_run": (C.c_int, [_vp, _vp, _i32, _vp, _i32, _vp, _i32, _vp, _vp, _i32, _vp, _i32]),
    "vbgpu_feat_run_dev": (C.c_int, [_vp, _vp, _i32, _vp, _i32, _vp, _i32, _vp, _vp, _i32, _vp, _i32, _vp]),
    "vbgpu_gmm_create": (C.c_int, [_i32, _i32, _vp, _vp, _vp, _vp, _i32, C.c_int, C.POINTER(_vp)]),
    "vbgpu_gmm_destroy": (C.c_int, [_vp]),
    "vbgpu_gmm_num_pdfs": (C.c_int, [_vp]),
    "vbgpu_gmm_num_gauss": (C.c_int, [_vp]),
    "vbgpu_gmm_dim": (C.c_int, [_vp]),
    "vbgpu_gmm_set_gconsts": (C.c_int, [_vp, _vp]),
    "vbgpu_gmm_set_kernel": (C.c_int, [_vp, _i32]),
    "vbgpu_gmm_score": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _i32]),
    "vbgpu_gmm_score_dev": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _i32, _vp]),
    "vbgpu_gmm_num_cols": (C.c_int, [_vp]),
    "vbgpu_gmm_col_of_pdf": (C.c_int, [_vp, _vp]),
    "vbgpu_gmm_plan_note": (C.c_char_p, [_vp]),
    "vbgpu_gmm_score_cols_dev": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _i32, _vp]),
    "vbgpu_debug_tc_layout": (C.c_int, [_i32, _i32, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _i64, _vp, _i32, _vp, _i32,
                                        _vp, _vp, _i32, _vp, _vp, _vp, _vp]),
    "vbgpu_debug_live_bytes": (C.c_int, [C.POINTER(_i64), C.POINTER(_i64)]),
    "vbgpu_gmm_score_subset": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _i32, _vp, _vp, _vp, _vp]),
    "vbgpu_gmm_score_subset_dev": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _i32, _vp, _vp, _vp, _vp, _vp]),
    "vbgpu_gmm_score_gather": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _vp, _i64, _vp]),
    "vbgpu_gmm_score_gather_dev": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _vp, _i64, _vp, _vp]),
    "vbgpu_gmm_bad_count": (C.c_int, [_vp, C.POINTER(_i64)]),
    "vbgpu_gmm_rescored_frames": (C.c_int, [_vp, C.POINTER(_i64)]),
    "vbgpu_gmm_component_posteriors": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp]),
    "vbgpu_acc_create": (C.c_int, [_vp, C.POINTER(_vp)]),
    "vbgpu_acc_create_with_transitions": (C.c_int, [_vp, _i32, C.POINTER(_vp)]),
    "vbgpu_acc_accumulate_transitions": (C.c_int, [_vp, _vp, _i64]),
    "vbgpu_acc_accumulate_transitions_dev": (C.c_int, [_vp, _vp, _i64, _vp]),
    "vbgpu_acc_download_transitions": (C.c_int, [_vp, _vp]),
    "vbgpu_acc_destroy": (C.c_int, [_vp]),
    "vbgpu_acc_zero": (C.c_int, [_vp]),
    "vbgpu_acc_accumulate": (C.c_int, [_vp, _vp, _vp, _i64, _i32, _vp, _vp, C.POINTER(_d)]),
    "vbgpu_acc_accumulate_dev": (C.c_int, [_vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp]),
    "vbgpu_acc_buffer": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_i64)]),
    "vbgpu_acc_allreduce": (C.c_int, [_vp, _vp, _vp]),
    "vbgpu_acc_add": (C.c_int, [_vp, _d, _vp]),
    "vbgpu_acc_download": (C.c_int, [_vp, _vp, _vp, _vp, C.POINTER(_d), C.POINTER(_d)]),
    "vbgpu_fmllr_create": (C.c_int, [_vp, _i32, C.POINTER(_vp)]),
    "vbgpu_fmllr_destroy": (C.c_int, [_vp]),
    "vbgpu_fmllr_zero": (C.c_int, [_vp]),
    "vbgpu_fmllr_accumulate": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _vp, _vp, _i32, _vp, C.POINTER(_d)]),
    "vbgpu_fmllr_accumulate_dev": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _vp, _vp, _i32, _vp, _vp]),
    "vbgpu_fmllr_download": (C.c_int, [_vp, _i32, C.POINTER(_d), _vp, _vp]),
    "vbgpu_mllt_accumulate": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _vp, C.POINTER(_d), _vp, C.POINTER(_d)]),
    "vbgpu_lda_create": (C.c_int, [_i32, _i32, C.c_int, C.POINTER(_vp)]),
    "vbgpu_lda_destroy": (C.c_int, [_vp]),
    "vbgpu_lda_zero": (C.c_int, [_vp]),
    "vbgpu_lda_accumulate": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _vp]),
    "vbgpu_lda_accumulate_dev": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _vp, _vp]),
    "vbgpu_lda_bad_count": (C.c_int, [_vp, C.POINTER(_i64)]),
    "vbgpu_lda_download": (C.c_int, [_vp, _vp, _vp, _vp]),
    "vbgpu_lda_buffer": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_i64)]),
    "vbgpu_lda_allreduce": (C.c_int, [_vp, _vp, _vp]),
    "vbgpu_tree_create": (C.c_int, [C.POINTER(TreeOpts), C.POINTER(TidTables), _i32, _i32, C.c_int, C.POINTER(_vp)]),
    "vbgpu_tree_destroy": (C.c_int, [_vp]),
    "vbgpu_tree_zero": (C.c_int, [_vp]),
    "vbgpu_tree_accumulate": (C.c_int, [_vp, _vp, _i32, _vp, _vp, _i32]),
    "vbgpu_tree_accumulate_dev": (C.c_int, [_vp, _vp, _i32, _vp, _vp, _i32, _vp]),
    "vbgpu_tree_bad_count": (C.c_int, [_vp, C.POINTER(_i64), C.POINTER(_i64)]),
    "vbgpu_tree_num_keys": (C.c_int, [_vp, C.POINTER(_i32)]),
    "vbgpu_tree_download": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "vbgpu_tree_add": (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp]),
    "vbgpu_io_object_info": (C.c_int, [_vp, _i64, C.POINTER(IoInfo)]),
    "vbgpu_io_read_matrix": (C.c_int, [_vp, _i64, _vp, _i32]),
    "vbgpu_io_read_vector": (C.c_int, [_vp, _i64, _vp]),
    "vbgpu_io_read_int32_vector": (C.c_int, [_vp, _i64, _vp, _i32]),
    "vbgpu_io_write_matrix": (_i64, [_vp, _i32, _i32, _i32, _vp, _i64]),
    "vbgpu_io_write_int32_vector": (_i64, [_vp, _i32, _vp, _i64]),
    "vbgpu_io_ark_next": (C.c_int, [_vp, _i64, _i64, _vp, _i32, C.POINTER(_i64), C.POINTER(_i64), C.POINTER(IoInfo)]),
    "vbgpu_io_mdl_info": (C.c_int, [_vp, _i64, C.POINTER(_i32), C.POINTER(_i32), C.POINTER(_i32), C.POINTER(_i32)]),
    "vbgpu_io_mdl_read": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "vbgpu_io_mdl_transitions": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    "vbgpu_io_write_acc": (_i64, [_i32, _i32, _vp, _vp, _i32, _vp, _vp, _vp, _d, _d, _vp, _i64]),
    "vbgpu_io_matrix_to_device": (C.c_int, [_vp, _i64, _vp, _i32, _vp, _i64, _vp]),
    "vbgpu_pipeline_create": (C.c_int, [_vp, _vp, _vp, C.POINTER(_vp)]),
    "vbgpu_pipeline_destroy": (C.c_int, [_vp]),
    "vbgpu_pipeline_score_i16": (C.c_int, [_vp, _vp, _vp, _i32, _vp, _i32, _vp, _vp, _i32, _vp, _i32, _vp, _i32]),
    "vbgpu_pipeline_score_dev": (C.c_int, [_vp, _vp, _vp, _i32, _vp, _i32, _vp, _i32, _vp, _i32, _vp, _i32, _vp]),
    "vbgpu_pipeline_score_cols_dev": (C.c_int, [_vp, _vp, _vp, _i32, _vp, _i32, _vp, _i32, _vp, _i32, _vp, _i32, _vp]),
    "vbgpu_pipeline_score_subset_i16": (C.c_int, [_vp, _vp, _vp, _i32, _vp, _i32, _vp, _vp, _i32, _vp, _vp, _vp, _vp]),
    "vbgpu_pipeline_score_gather_i16": (C.c_int, [_vp, _vp, _vp, _i32, _vp, _i32, _vp, _vp, _i32, _vp, _vp, _i64, _vp]),
    "vbgpu_pipeline_accumulate_dev": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _vp, _i32, _vp, _i32, _vp, _vp]),
}

EXPORTS = tuple(sorted(_SIGS))

_lib = None


def lib():
    """The loaded library (loads on first use; raises if the CUDA extension has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "%s is missing: the CUDA extension has not been built and there is no CPU fallback. "
                "Run `python -c 'import __graft_entry__ as g; g.build()'` at the repo root." % LIB_PATH)
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(l, name)  # AttributeError here = header and library disagree
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc):
    if rc < 0:
        raise VbgpuError(rc, lib().vbgpu_last_error().decode("utf-8", "replace"))
    return rc


def default_mfcc_opts(**kw):
    o = MfccOpts()
    lib().vbgpu_mfcc_opts_default(C.byref(o))
    for k, v in kw.items():
        if not hasattr(o, k):
            raise KeyError(k)
        setattr(o, k, v)
    return o


def _with(o, kw):
    for k, v in kw.items():
        if not hasattr(o, k):
            raise KeyError(k)
        setattr(o, k, v)
    return o


def default_pitch_opts(**kw):
    o = PitchOpts()
    lib().vbgpu_pitch_opts_default(C.byref(o))
    return _with(o, kw)


def default_process_pitch_opts(**kw):
    o = ProcessPitchOpts()
    lib().vbgpu_process_pitch_opts_default(C.byref(o))
    return _with(o, kw)


def default_feat_opts(**kw):
    o = FeatOpts()
    lib().vbgpu_feat_opts_default(C.byref(o))
    for k, v in kw.items():
        if not hasattr(o, k):
            raise KeyError(k)
        setattr(o, k, v)
    return o
