"""Kaldi wire / disk formats over the C ABI (vbgpu_io_*, csrc/kaldi_io.cu): what the recipe scripts exchange through
archives and temp files on either side of the hot path (SURVEY.md §8f n2).  Binary forms only."""
import ctypes as C

import numpy as np

from . import capi
from .capi import check

KINDS = {1: "FM", 2: "DM", 3: "CM", 4: "CM2", 5: "CM3", 6: "FV", 7: "DV", 8: "IV"}


def _buf(b):
    a = np.frombuffer(b, np.uint8) if not isinstance(b, np.ndarray) else np.ascontiguousarray(b, np.uint8)
    return a, a.ctypes.data, a.size


def object_info(b, offset=0):
    a, p, n = _buf(b)
    info = capi.IoInfo()
    check(capi.lib().vbgpu_io_object_info(p + offset, n - offset, C.byref(info)))
    return info


def read_matrix(b, offset=0):
    """Matrix<BaseFloat>::Read of an FM / DM / CM / CM2 / CM3 object -> float32 [rows, cols]."""
    a, p, n = _buf(b)
    info = object_info(a, offset)
    out = np.zeros((info.rows, info.cols), np.float32)
    check(capi.lib().vbgpu_io_read_matrix(p + offset, n - offset, out.ctypes.data, max(info.cols, 0)))
    return out


def read_vector(b, offset=0):
    a, p, n = _buf(b)
    info = object_info(a, offset)
    out = np.zeros(info.cols, np.float64)
    check(capi.lib().vbgpu_io_read_vector(p + offset, n - offset, out.ctypes.data))
    return out


def read_int32_vector(b, offset=0):
    a, p, n = _buf(b)
    info = object_info(a, offset)
    out = np.zeros(info.cols, np.int32)
    check(capi.lib().vbgpu_io_read_int32_vector(p + offset, n - offset, out.ctypes.data, info.cols))
    return out


def write_matrix(m):
    m = np.ascontiguousarray(m, np.float32)
    rows, cols = m.shape
    n = check(capi.lib().vbgpu_io_write_matrix(m.ctypes.data, rows, cols, cols, None, 0))
    out = np.zeros(n, np.uint8)
    check(capi.lib().vbgpu_io_write_matrix(m.ctypes.data, rows, cols, cols, out.ctypes.data, n))
    return out.tobytes()


def write_int32_vector(v):
    v = np.ascontiguousarray(v, np.int32)
    n = check(capi.lib().vbgpu_io_write_int32_vector(v.ctypes.data, len(v), None, 0))
    out = np.zeros(n, np.uint8)
    check(capi.lib().vbgpu_io_write_int32_vector(v.ctypes.data, len(v), out.ctypes.data, n))
    return out.tobytes()


def write_ark_entry(key, obj_bytes):
    """One archive entry as the table writers emit it: key, a space, the (\\0B-marked) object."""
    return key.encode() + b" " + obj_bytes


def read_ark(b):
    """Iterates a binary archive: yields (key, info, object offset); read the object with read_matrix(b, offset) etc."""
    a, p, n = _buf(b)
    pos = 0
    key = C.create_string_buffer(256)
    while True:
        info = capi.IoInfo()
        op, nx = C.c_int64(0), C.c_int64(0)
        rc = check(capi.lib().vbgpu_io_ark_next(p, n, pos, key, 256, C.byref(op), C.byref(nx), C.byref(info)))
        if rc == 1:
            return
        yield key.value.decode("utf-8", "replace"), info, op.value
        pos = nx.value


def read_mdl(b):
    """A final.mdl / x.mdl (TransitionModel + AmDiagGmm) or a bare AmDiagGmm -> dict with the flattened model that
    vbgpu_gmm_create takes, tid2pdf (1-based; empty without a transition model) and the transition log-probs."""
    a, p, n = _buf(b)
    D, P, N, nt = C.c_int32(0), C.c_int32(0), C.c_int32(0), C.c_int32(0)
    check(capi.lib().vbgpu_io_mdl_info(p, n, C.byref(D), C.byref(P), C.byref(N), C.byref(nt)))
    D, P, N, nt = D.value, P.value, N.value, nt.value
    out = dict(dim=D, pdf_offsets=np.zeros(P + 1, np.int32), gconsts=np.zeros(N, np.float32),
               weights=np.zeros(N, np.float32), means_invvars=np.zeros((N, D), np.float32),
               inv_vars=np.zeros((N, D), np.float32), tid2pdf=np.zeros(nt + 1 if nt else 0, np.int32),
               trans_log_probs=np.zeros(nt + 1 if nt else 0, np.float32))
    out["num_inf_gconsts"] = check(capi.lib().vbgpu_io_mdl_read(
        p, n, out["pdf_offsets"].ctypes.data, out["gconsts"].ctypes.data, out["weights"].ctypes.data,
        out["means_invvars"].ctypes.data, out["inv_vars"].ctypes.data,
        out["tid2pdf"].ctypes.data if nt else None, out["trans_log_probs"].ctypes.data if nt else None))
    return out


def read_transitions(b):
    """The per transition-id tables of a model file's TransitionModel: dict of int32 arrays phone, hmm_state, pdf_class,
    trans_state and flags (capi.TID_*), num_tids + 1 each with entry 0 unused, as vbgpu_tree_create takes them."""
    a, p, n = _buf(b)
    nt = check(capi.lib().vbgpu_io_mdl_transitions(p, n, None, None, None, None, None))
    out = {k: np.zeros(nt + 1, np.int32) for k in ("phone", "hmm_state", "pdf_class", "trans_state", "flags")}
    check(capi.lib().vbgpu_io_mdl_transitions(p, n, *(out[k].ctypes.data for k in
                                                      ("phone", "hmm_state", "pdf_class", "trans_state", "flags"))))
    return out


def write_acc(pdf_offsets, occ, mean_acc, var_acc, tot_like, tot_frames, trans_accs=None):
    """The bytes of a gmm-acc-stats-ali output file (x.JOBID.acc) from downloaded statistics."""
    po = np.ascontiguousarray(pdf_offsets, np.int32)
    occ, mean_acc, var_acc = (np.ascontiguousarray(v, np.float64) for v in (occ, mean_acc, var_acc))
    ta = np.ascontiguousarray(trans_accs, np.float64) if trans_accs is not None else None
    args = (len(po) - 1, mean_acc.shape[1], po.ctypes.data, ta.ctypes.data if ta is not None else None,
            len(ta) if ta is not None else 0, occ.ctypes.data, mean_acc.ctypes.data, var_acc.ctypes.data,
            float(tot_like), float(tot_frames))
    n = check(capi.lib().vbgpu_io_write_acc(*args, None, 0))
    out = np.zeros(n, np.uint8)
    check(capi.lib().vbgpu_io_write_acc(*args, out.ctypes.data, n))
    return out.tobytes()


def matrix_to_device(b, d_out, out_stride, d_scratch=None, stream=None, offset=0):
    """Expands a matrix object (host bytes) into a device float tensor; packed kinds cross PCIe as stored."""
    a, p, n = _buf(b)
    sp = d_scratch.data_ptr() if d_scratch is not None else None
    sb = d_scratch.numel() * d_scratch.element_size() if d_scratch is not None else 0
    st = stream.cuda_stream if stream is not None else None
    check(capi.lib().vbgpu_io_matrix_to_device(p + offset, n - offset, d_out.data_ptr(), out_stride, sp, sb, st))
