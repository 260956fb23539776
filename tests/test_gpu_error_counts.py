"""Error counts of the host forms (synchronous calls on host buffers) and of the _dev calls on one model.

The _dev calls cannot return their errors, so they add them to the model's running count (vbgpu_gmm_bad_count).  A host
form reports the errors of its own call through its return code and leaves that count alone: a count left pending by a
_dev call survives a clean host call, and a failing host call names only the frames it saw itself.  Each host form is
checked once with clean input and once with bad input: an invalid pdf-id, a NaN feature row, -inf gconsts over a whole
pdf (the pipeline forms, whose input is PCM) or out-of-range transition-ids."""
import re

import numpy as np
import pytest

from tests.common import recipe_opts
from voicebridge_b200 import capi, host, synth

pytestmark = pytest.mark.gpu

P, N, D, T = 20, 80, 39, 300
K = 3          # counts left pending on the model before the host call
N_TIDS = 20


def leave_pending(am, k=K):
    """k out-of-range transition-ids through accumulate_transitions_dev: k counts on the model, finished before the return
    (the host forms run on streams of their own)."""
    import torch
    acc = host.AccumAmDiagGmmGpu(am, num_tids=N_TIDS)
    d_tids = torch.full((k,), N_TIDS + 1, dtype=torch.int32, device="cuda")
    acc.accumulate_transitions_dev(d_tids, k)
    torch.cuda.synchronize()
    acc.close()


def failure(call):
    """(code, count) of a failing call: the count is the number its message starts with."""
    with pytest.raises(capi.VbgpuError) as e:
        call()
    m = re.match(r"vbgpu error -?\d+: (\d+) ", str(e.value))
    assert m, str(e.value)
    return e.value.code, int(m.group(1))


def model(bad_pdf=False):
    m = synth.make_model(P, N, D, 3)
    gc = m.gconsts.copy()
    if bad_pdf:
        gc[m.pdf_offsets[1]:m.pdf_offsets[2]] = -np.inf
    return m, host.AmDiagGmmGpu(m.pdf_offsets, gc, m.miv, m.iv)


def feats(m, bad):
    X = synth.make_feats(m, T, 4)
    if bad:
        X[7] = np.nan
    return X


def ali(bad):
    a = synth.make_alignment(P, T, 5)
    if bad:
        a[[3, 50, 51, 200]] = [-1, P, 10 ** 6, -7]
    return a


# ---- every host form: (model handle, a call of the form on clean or bad input) --------------------------------------------
def gmm_score(bad):
    m, am = model()
    X = feats(m, bad)
    return am, lambda: am.score(X)


def gmm_score_subset(bad):
    m, am = model()
    X = feats(m, bad)
    return am, lambda: am.score_subset(X, np.array([0, 100, T], np.int64), [[0, 5, 7], [1, 2, 19]])


def gmm_score_gather(bad):
    m, am = model()
    X = feats(m, bad)
    fr = np.arange(0, T, 3, dtype=np.int32)
    return am, lambda: am.score_gather(X, fr, fr % P)


def pipeline(bad):
    pcm, so, u2s = synth.make_corpus(2, 2, 0.5, 1.0, 7)
    _, am = model(bad_pdf=bad)
    pipe = host.ScoringPipeline(host.Mfcc(recipe_opts(capi)), host.FeaturePipeline(in_dim=13), am)
    return am, pipe, np.asarray(pcm, np.int16), so, u2s


def pipeline_score(bad):
    am, pipe, pcm, so, u2s = pipeline(bad)
    return am, lambda: pipe.score(pcm, so, u2s)


def pipeline_score_subset(bad):
    am, pipe, pcm, so, u2s = pipeline(bad)
    sub_o = np.arange(len(so), dtype=np.int64) * 2
    sub_p = np.arange(2 * (len(so) - 1), dtype=np.int32) % P
    return am, lambda: pipe.score_subset(pcm, so, sub_o, sub_p, u2s)


def pipeline_score_gather(bad):
    am, pipe, pcm, so, u2s = pipeline(bad)
    fr = np.arange(0, 40, dtype=np.int32)
    return am, lambda: pipe.score_gather(pcm, so, fr, fr % P, u2s)


def acc_accumulate(bad):
    m, am = model()
    acc, X, a = host.AccumAmDiagGmmGpu(am), feats(m, False), ali(bad)
    return am, lambda: acc.AccumulateForUtterance(X, a)


def acc_accumulate_transitions(bad):
    _, am = model()
    acc = host.AccumAmDiagGmmGpu(am, num_tids=N_TIDS)
    tids = np.arange(T, dtype=np.int32) % N_TIDS + 1
    if bad:
        tids[[0, 9, 10, 150, 299]] = [0, N_TIDS + 1, N_TIDS + 1, -4, 1000]
    return am, lambda: acc.AccumulateTransitions(tids)


def fmllr_accumulate(bad):
    m, am = model()
    f, X, a = host.FmllrDiagGmmAccsGpu(am), feats(m, False), ali(bad)
    return am, lambda: f.AccumulateForUtterances(X, a)


def mllt_accumulate(bad):
    m, am = model()
    X, a = feats(m, False), ali(bad)
    return am, lambda: host.MlltAccsGpu(am).AccumulateForUtterance(X, a)


def component_posteriors(bad):
    # (ComponentPosteriors indexes pdf_offsets with the ids on the host, so its bad input is a NaN row)
    m, am = model()
    X, a = feats(m, bad), ali(False)
    return am, lambda: am.ComponentPosteriors(X, a, m.pdf_offsets)


FORMS = {f.__name__: f for f in (gmm_score, gmm_score_subset, gmm_score_gather, pipeline_score, pipeline_score_subset,
                                 pipeline_score_gather, acc_accumulate, acc_accumulate_transitions, fmllr_accumulate,
                                 mllt_accumulate, component_posteriors)}


@pytest.mark.parametrize("form", sorted(FORMS))
def test_pending_count_survives_a_clean_host_call(form):
    am, call = FORMS[form](bad=False)
    leave_pending(am)
    call()  # returns 0: the pending counts are not this call's
    assert am.bad_count() == K


@pytest.mark.parametrize("form", sorted(FORMS))
def test_host_call_reports_only_its_own_errors(form):
    am, call = FORMS[form](bad=True)
    code, m = failure(call)
    assert code == (capi.ERR_INVALID if form == "acc_accumulate_transitions" else capi.ERR_NUMERIC)
    assert m >= 1 and m != K
    assert am.bad_count() == 0  # the host call reported its errors through the return code only
    leave_pending(am)
    assert failure(call) == (code, m)
    assert am.bad_count() == K
