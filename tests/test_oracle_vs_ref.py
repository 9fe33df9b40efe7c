"""CPU: the C oracle against the unmodified reference, bit for bit.  The reference's answers for these inputs are stored in
tests/golden/ref_checks.npz (tests/golden/make_golden_ref_checks.py runs the reference on the same inputs)."""
import hashlib
import os

import numpy as np
import pytest

from conftest import GOLDEN_DIR, bits


def sha(a):
    return hashlib.sha1(bits(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(GOLDEN_DIR, "ref_checks.npz"))


@pytest.fixture(scope="module")
def oracle(orc, weights_file):
    return orc.Oracle(weights_file("tiny", "f16"), seed=0, n_steps=16)


def test_gelu_table(orc, golden):
    o, _ = orc.gelu_tables()
    assert hashlib.sha1(o.tobytes()).hexdigest() == str(golden["vs_ref_gelu_sha1"])


def test_tokenizer(oracle, golden):
    texts = ["hello world", "", "Hello, world! 123 café zz", "ÀÉÎõü ñ ç", "a" * 600, "x,y;z...", "日本語 text", "tab\there"]
    for text, want in zip(texts, golden["vs_ref_tokenize"], strict=True):
        assert np.array_equal(oracle.tokenize(text), want), text


def test_causal_eval_bit_exact(oracle, golden):
    o = oracle
    rng = np.random.default_rng(1)
    for which, first, merge in ((0, None, True), (1, np.concatenate([rng.integers(0, 10000, 256), [12050], rng.integers(10000, 12048, 37)]).astype(np.int32), False)):
        toks = o.tokenize("hello world") if first is None else first
        po = 0
        for step in range(40):
            lo, po = o.gpt_eval(which, toks, po, merge)
            assert po == golden[f"vs_ref_causal{which}_n_past"][step], (which, step)
            assert sha(lo) == str(golden[f"vs_ref_causal{which}_sha1"][step]), \
                (which, step, f"first {int((bits(lo[:32]) != bits(golden[f'vs_ref_causal{which}_head'][step])).sum())} of 32 logits differ")
            toks = np.array([int(np.argmax(lo[:10000])) if which == 0 else 10000 + int(np.argmax(lo[10000:12048]))], np.int32)


def test_fine_eval_bit_exact(oracle, golden):
    rng = np.random.default_rng(2)
    buf = rng.integers(0, 1024, (8, 1024)).astype(np.int32)
    for nn in (2, 7):
        x = buf.copy(); x[nn:, :] = 1024
        assert sha(oracle.fine_eval(x, nn)) == str(golden[f"vs_ref_fine{nn}_sha1"]), nn


def test_sampler(oracle, golden):
    rng = np.random.default_rng(3)
    oracle.reseed(9)
    for i in range(150):
        lg = (rng.standard_normal((10048, 1024)[i % 2]) * 4).astype(np.float32)
        temp = (0.7, 0.5, 0.0)[i % 3]
        t, e = oracle.sample(lg, temp)
        assert t == golden["vs_ref_sample_token"][i] and bits(np.float32(e)) == bits(golden["vs_ref_sample_eos"][i]), i


def test_encodec_bit_exact(oracle, golden):
    rng = np.random.default_rng(4)
    for T in (7, 40):
        codes = rng.integers(0, 1024, (8, T)).astype(np.int32)
        a = oracle.encodec_decode(codes)
        assert a.size == golden[f"vs_ref_encodec{T}_size"] and sha(a) == str(golden[f"vs_ref_encodec{T}_sha1"]), T


def test_full_generate(oracle, golden):
    oracle.reseed(0)
    a = oracle.generate("hello world")
    for k in ("semantic", "coarse", "fine"):
        assert np.array_equal(a[k], golden[f"vs_ref_generate_{k}"]), k
    assert np.array_equal(bits(a["audio"]), bits(golden["vs_ref_generate_audio"]))
