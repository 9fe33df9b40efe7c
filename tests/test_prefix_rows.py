"""Canonical rows (bark_api.cu run_coarse, "Prefix reuse"): row p of a causal evaluation does not depend on the call's n_kv as
long as p < n_kv & ~31, so a coarse window may start from the cached rows of the previous window.  Checked here on the CPU
on the C restatement, whose from-scratch logits must equal the UNMODIFIED reference's (tests/golden/ref_checks.npz, where the
reference passed the same tail checks): evaluating the tail of a sequence on top of the cached canonical rows gives
bit-identical logits to evaluating the whole sequence from n_past = 0 — and a non-canonical row (p >= n_kv & ~31 of the call
that produced it) does not."""
import hashlib
import os

import numpy as np
import pytest

from conftest import GOLDEN_DIR, bits


@pytest.mark.parametrize("ftype", ["f32", "f16"])
def test_tail_on_canonical_rows_equals_from_scratch(orc, weights_file, ftype):
    path = weights_file("mini", ftype)
    rng = np.random.default_rng(21)
    full = np.concatenate([rng.integers(0, 10000, 256), [12050], rng.integers(10000, 12048, 75)]).astype(np.int32)
    e = orc.Oracle(path)
    scratch, p = e.gpt_eval(1, full, 0, False)
    assert p == full.size
    for cut in (256, 288, 320):
        _, p = e.gpt_eval(1, full[:cut + 5], 0, False)          # rows [0, cut) canonical ((cut + 5) & ~31 == cut)
        tail, p = e.gpt_eval(1, full[cut:], cut, False)
        assert p == full.size
        assert np.array_equal(bits(tail), bits(scratch)), f"oracle: tail after {cut} cached rows: {int((tail != scratch).sum())} logits differ"
    # the decode path of the same thing: one id on top of a cache whose last rows came from single-token steps is how the
    # reference's own windows end; starting the NEXT window from those rows would not be exact
    want = str(np.load(os.path.join(GOLDEN_DIR, "ref_checks.npz"))[f"prefix_rows_{ftype}_sha1"])
    assert hashlib.sha1(bits(scratch).tobytes()).hexdigest() == want, "from-scratch logits differ from the reference's"


def test_rows_written_by_decode_steps_are_not_canonical(orc, weights_file):
    """Negative control, f32 so nothing is hidden by operand rounding: rows written one token at a time (n_kv = p + 1, the row's
    own last columns sit in the scalar leftovers of the P.V dot) differ in the last bits from the same rows of a batch."""
    path = weights_file("mini", "f32")
    rng = np.random.default_rng(22)
    full = np.concatenate([rng.integers(0, 10000, 256), [12050], rng.integers(10000, 12048, 60)]).astype(np.int32)
    o = orc.Oracle(path)
    scratch, _ = o.gpt_eval(1, full, 0, False)
    _, p = o.gpt_eval(1, full[:257], 0, False)
    for t in full[257:]:
        stepwise, p = o.gpt_eval(1, np.array([t], np.int32), p, False)
    assert p == full.size
    assert not np.array_equal(bits(stepwise), bits(scratch)), "decode-written rows happened to be canonical here: pick another seed"
    assert np.allclose(stepwise, scratch, rtol=0, atol=1e-3)
