"""One handle walked through traces of different forms: the rows trace, a sharded trace, the hashed tally, host output and the
one-device gather of rthx_trace_exchange_multi.  Whatever came before, the handle must behave as a fresh handle that ran only the last
trace: every read-out that state allows returns the same arrays bit for bit, every read-out it does not allow fails with the same
message, and trace_continue is accepted or rejected alike."""

import numpy as np
import pytest

R1, R2 = 700, 500


def _listed(tr):
    """Every surface row (so that the crop n = Ns is traced in full) and two volume rows."""
    ns, N = tr.flat.n_surfaces, tr.n_elements
    return list(range(ns)) + [ns + 3, N - 1]


def _traces():
    from rthx._lib import trace_multi
    return {
        "rows": lambda tr: tr.trace_rows(_listed(tr), R1, dense=False, seed=11),
        "rows_host": lambda tr: tr.trace_rows(_listed(tr), R1, seed=12),
        "sharded": lambda tr: tr.trace(R1, dense=False, seed=13, emitter_rank=1, emitter_world=2),
        "hashed": lambda tr: tr.trace_sparse(R1, seed=14),
        "gather": lambda tr: trace_multi([tr], R1, dense=False, seed=15),
    }


def _state(rthx_mod, tr, rtm):
    """Every read-out of bin 0 of the resident counts (the smoothings whole and cropped to the surfaces): its arrays, or the message it
    was rejected with."""
    ns = tr.flat.n_surfaces
    w = rthx_mod.get_w(rtm)
    wn, wc = w / w.min(), w[:ns] / w[:ns].min()

    def run(f):
        try:
            return [np.array(x, copy=True) for x in f()]
        except rthx_mod.RthxError as e:
            return str(e)

    def dense(ww, n):
        F, st = tr.smooth(ww, n=n)
        return F, st["iterations"], st["delta"]

    def sparse(ww, n):
        F, st = tr.smooth_sparse(ww, n=n)
        return F.indptr, F.indices, F.data, st["iterations"], st["delta"]

    return dict(stats=run(lambda: tr.counts_stats(0)), csr=run(lambda: tr.counts_csr(0)),
                csc=run(lambda: tr.counts_csc(0, values=True, pinned=False)),
                smooth=run(lambda: dense(wn, None)), smooth_crop=run(lambda: dense(wc, ns)),
                smooth_sparse=run(lambda: sparse(wn, None)), smooth_sparse_crop=run(lambda: sparse(wc, ns)))


def _assert_same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        x, y = a[k], b[k]
        if isinstance(x, str) or isinstance(y, str):
            assert x == y, k
        else:
            assert len(x) == len(y) and all(np.array_equal(u, v) for u, v in zip(x, y)), k


def _continued(rthx_mod, tr, rtm):
    """The state after trace_continue(R2), or the message it was rejected with (under "continue_")."""
    try:
        tr.trace_continue(R2)
    except rthx_mod.RthxError as e:
        return dict(continue_=str(e))
    return _state(rthx_mod, tr, rtm)


def _two_handles(rthx_mod):
    from rthx._lib import create_multi
    rtm = rthx_mod.meshes.square_domain(11, kappa=1.0)
    flat = rthx_mod.flatten_domain(rtm)
    (mixed,), (fresh,) = create_multi(flat, [0]), create_multi(flat, [0])
    return rtm, mixed, fresh


@pytest.mark.gpu
@pytest.mark.parametrize("before, last, rejected", [
    ("rows", "sharded", None),
    ("rows", "hashed", None),
    ("hashed", "rows", None),
    ("hashed", "rows_host", "host-output"),
    ("rows", "gather", "several devices"),                  # rthx_trace_exchange_multi on one device
])
def test_a_handle_behaves_as_after_its_last_trace_alone(rthx_mod, cuda_lib, before, last, rejected):
    rtm, mixed, fresh = _two_handles(rthx_mod)
    traces = _traces()
    traces[before](mixed)
    traces[last](mixed)
    traces[last](fresh)
    _assert_same(_state(rthx_mod, mixed, rtm), _state(rthx_mod, fresh, rtm))
    got, want = _continued(rthx_mod, mixed, rtm), _continued(rthx_mod, fresh, rtm)
    if rejected:
        assert "(1)" in want["continue_"] and rejected in want["continue_"]
    else:
        assert "continue_" not in want, want
    _assert_same(got, want)


@pytest.mark.gpu
def test_a_rejected_rows_trace_leaves_the_hashed_counts(rthx_mod, cuda_lib):
    rtm, mixed, fresh = _two_handles(rthx_mod)
    traces = _traces()
    traces["hashed"](mixed)
    with pytest.raises(rthx_mod.RthxError, match=r"\(1\).*strictly ascending"):
        mixed.trace_rows([3, 2], R1, dense=False, seed=11)
    traces["hashed"](fresh)
    _assert_same(_state(rthx_mod, mixed, rtm), _state(rthx_mod, fresh, rtm))
    _assert_same(_continued(rthx_mod, mixed, rtm), _continued(rthx_mod, fresh, rtm))
