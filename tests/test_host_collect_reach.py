"""Host collects (`mdim_collect_host`) upload what each host operand reaches, and nothing a collect needs is left out.

A host collect copies each host operand into device staging: whole (resident), or in slabs along axis 0 when the collect is
cut into chunks.  Which elements an operand reaches comes from the planner's hull (plan.cpp: `operand_reach` over the ranges
of `node_axis_ranges`), and those ranges follow the planner's own children of every node.  The init view of a fold
(`rows().map(Fold(B, init_view))`, a FOLD node with two children) is the case here: it reaches one element per output, so a
hull that missed it would upload a single element and the other outputs would read whatever follows in the staging arena.

Each fold runs resident (the default 128 MB chunks) and chunked (MDIM_HOST_CHUNK_MB=1, read when the context is created),
against a numpy sequential fold in f32 (Sub: the order matters).  A TUPLE root has several output runs, which a host collect
does not take: it is refused with MDIM_ERR_INVALID.
"""
import os

import numpy as np
import pytest

from helpers import assert_same_bits
import multidimension_b200 as P
from multidimension_b200 import _ffi as F
from multidimension_b200 import lowering as L
from test_eval_routes import Subject, axes, fold, leaf, src

_ctx = {}


def context(chunk_mb):
    """One context per chunk size: MDIM_HOST_CHUNK_MB is read by mdim_init."""
    if chunk_mb not in _ctx:
        old = os.environ.get("MDIM_HOST_CHUNK_MB")
        os.environ["MDIM_HOST_CHUNK_MB"] = str(chunk_mb)
        try:
            _ctx[chunk_mb] = P.Context(0)
        finally:
            if old is None:
                del os.environ["MDIM_HOST_CHUNK_MB"]
            else:
                os.environ["MDIM_HOST_CHUNK_MB"] = old
    return _ctx[chunk_mb]


def init_fold(out_lens, red_len, init_offset):
    """FOLD(Sub, init view, body) over the last axis: init[o] at init_offset + o (row-major over the outputs), body x[o, k] dense.
    -> (Subject, numpy reference)."""
    *out, r = axes(*out_lens, red_len)
    n_out = int(np.prod(out_lens))
    st, acc = {}, 1
    for a in reversed(out):
        st[a] = acc
        acc *= a.length
    init_buf = src(f"reach-init-{out_lens}", "f32", init_offset + n_out + 8)
    body_buf = src(f"reach-body-{out_lens}-{red_len}", "f32", n_out * red_len + 8)
    init = leaf("f32", init_buf, init_offset, st)
    body = leaf("f32", body_buf, 0, {**{a: s * red_len for a, s in st.items()}, r: 1})
    subject = Subject(fold("f32", F.SUB, body, [r], init_view=init), out)
    x = body_buf.host[:n_out * red_len].reshape(n_out, red_len)
    want = init_buf.host[init_offset:init_offset + n_out].copy()
    for k in range(red_len):  # sequential, in index order, rounded to f32 at every step
        want = np.subtract(want, x[:, k], dtype=np.float32)
    return subject, want


# (output lengths, reduction length, offset of the init view): ~4 MB of body, so 1 MB chunks cut axis 0 into several
FOLDS = {"rank1-init": ((20000,), 48, 3), "rank2-init": ((2000, 12), 40, 5)}


@pytest.mark.parametrize("name", FOLDS)
def test_reference_matches_oracle(name):
    subject, want = init_fold(*FOLDS[name])
    (got,), err = subject.oracle()
    assert err is None, err
    assert_same_bits(got, want, name)


@pytest.mark.gpu
@pytest.mark.parametrize("chunk_mb", [128, 1], ids=["resident", "chunked"])
@pytest.mark.parametrize("name", FOLDS)
def test_fold_init_view(name, chunk_mb):
    subject, want = init_fold(*FOLDS[name])
    em = L.emit(subject.root(), subject.axes, "host")
    got = np.full(em.out_len, np.nan, np.float32)
    context(chunk_mb).collect_host(em.expr, got.ctypes.data)
    assert_same_bits(got, want, f"{name} ({chunk_mb} MB chunks)")


@pytest.mark.gpu
def test_tuple_root_refused():
    o, = axes(1000)
    a = leaf("f32", src("reach-tuple-a", "f32", 1008), 0, {o: 1})
    b = leaf("u32", src("reach-tuple-b", "u32", 1008), 0, {o: 1})
    em = L.emit([a, b], [o], "host")
    out = np.zeros(em.out_len * 2, np.uint32)
    with pytest.raises(F.MdimError) as e:
        context(128).collect_host(em.expr, out.ctypes.data)
    assert e.value.status == F.ERR_INVALID
