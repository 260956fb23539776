"""The C-ABI library: loads, exports exactly what include/vbgpu.h declares, and fails loudly without a GPU."""
import ctypes as C
import os
import re

import pytest

from voicebridge_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    txt = open(os.path.join(ROOT, "include", "vbgpu.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(vbgpu_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    lib = capi.lib()
    names = declared_symbols()
    assert len(names) >= 40
    for n in names:
        assert hasattr(lib, n), "libvbgpu.so does not export %s" % n
    # the Python binding covers the same set
    assert sorted(capi.EXPORTS) == names


def test_option_struct_layout_matches_oracle():
    from oracle import pyoracle as po
    assert C.sizeof(capi.MfccOpts) == C.sizeof(po.MfccOpts) == 22 * 4
    assert [f[0] for f in capi.MfccOpts._fields_] == [f[0] for f in po.MfccOpts._fields_]
    a, b = capi.default_mfcc_opts(), po.default_opts()
    for name, _ in capi.MfccOpts._fields_:
        assert getattr(a, name) == getattr(b, name), name
    for mine, theirs, a, b in ((capi.PitchOpts, po.PitchOpts, capi.default_pitch_opts(), po.default_pitch_opts()),
                               (capi.ProcessPitchOpts, po.ProcessPitchOpts, capi.default_process_pitch_opts(),
                                po.default_process_pitch_opts(delta_pitch_noise_stddev=0.005))):
        assert C.sizeof(mine) == C.sizeof(theirs)
        assert [f[0] for f in mine._fields_] == [f[0] for f in theirs._fields_]
        for name, _ in mine._fields_:
            assert getattr(a, name) == getattr(b, name), name
    f = capi.default_feat_opts()
    assert (f.norm_means, f.norm_vars, f.mode, f.delta_order, f.delta_window, f.splice_left, f.splice_right) == \
        (1, 0, 0, 2, 2, 3, 3)


def test_version_and_argument_errors_need_no_gpu():
    lib = capi.lib()
    assert lib.vbgpu_version() >= 100
    h = C.c_void_p()
    o = capi.default_mfcc_opts(round_to_power_of_two=0)
    assert lib.vbgpu_mfcc_create(C.byref(o), 0, C.byref(h)) == capi.ERR_INVALID
    assert b"round_to_power_of_two" in lib.vbgpu_last_error()
    o = capi.default_mfcc_opts(num_bins=40)
    assert lib.vbgpu_mfcc_create(C.byref(o), 0, C.byref(h)) == capi.ERR_INVALID
    fo = capi.default_feat_opts(mode=7)
    assert lib.vbgpu_feat_create(C.byref(fo), 13, None, 0, 0, 0, C.byref(h)) == capi.ERR_INVALID
    assert lib.vbgpu_gmm_create(0, 39, None, None, None, None, 39, 0, C.byref(h)) == capi.ERR_INVALID
    assert lib.vbgpu_mfcc_dim(None) == capi.ERR_INVALID
    po_ = capi.default_pitch_opts(lowpass_cutoff=3000.0)  # LinearResample asserts cutoff * 2 <= resample_freq (resample.cc:45)
    assert lib.vbgpu_pitch_create(C.byref(po_), 0, C.byref(h)) == capi.ERR_INVALID
    po_ = capi.default_pitch_opts(min_f0=400.0, max_f0=50.0)
    assert lib.vbgpu_pitch_create(C.byref(po_), 0, C.byref(h)) == capi.ERR_INVALID
    # destroying a NULL handle is a no-op that succeeds
    destroys = [n for n in capi.EXPORTS if n.endswith("_destroy") and capi._SIGS[n][0] is C.c_int]
    assert len(destroys) >= 8
    for n in destroys:
        assert getattr(lib, n)(None) == 0, n


def test_no_cpu_fallback():
    """Without a CUDA device every create call must fail with VBGPU_ERR_CUDA — never compute on the host."""
    lib = capi.lib()
    n = C.c_int(0)
    rc = lib.vbgpu_device_count(C.byref(n))
    if rc == 0 and n.value > 0:
        pytest.skip("a GPU is present")
    h = C.c_void_p()
    o = capi.default_mfcc_opts()
    assert lib.vbgpu_mfcc_create(C.byref(o), 0, C.byref(h)) == capi.ERR_CUDA
    assert b"no CPU fallback" in lib.vbgpu_last_error()
    po_ = capi.default_pitch_opts()
    assert lib.vbgpu_pitch_create(C.byref(po_), 0, C.byref(h)) == capi.ERR_CUDA
    assert b"no CPU fallback" in lib.vbgpu_last_error()
    assert lib.vbgpu_downsample_create(16000.0, 8000.0, 0, C.byref(h)) == capi.ERR_CUDA
    assert b"no CPU fallback" in lib.vbgpu_last_error()
    from voicebridge_b200 import host
    with pytest.raises(capi.VbgpuError):
        host.Mfcc()
    with pytest.raises(capi.VbgpuError):
        host.Pitch()
