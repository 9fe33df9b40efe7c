"""q4_0 files (BASELINE configs[3]): the native bark_model_quantize (csrc/quantize.cu, host only) must write the very bytes the
reference tool writes (bark.cpp:2300-2377), and the C oracle's q4_0 arithmetic (quantize_row_q8_0 + ggml_vec_dot_q4_0_q8_0 of
the pinned AVX2 build, get_rows dequantisation) must reproduce the unmodified reference on such a file bit for bit.  The
reference's files and results are stored in tests/golden/ref_checks.npz (tests/golden/make_golden_ref_checks.py)."""
import hashlib
import os

import numpy as np
import pytest

from conftest import FIXTURE_DIR, GOLDEN_DIR, bits

GGML_FTYPE_MOSTLY_Q4_0 = 2


def q4_file(pkg, weights_file, config, src_ftype):
    src = weights_file(config, src_ftype)
    dst = os.path.join(FIXTURE_DIR, f"{config}_{src_ftype}_1234_q4_0.bin")
    if not os.path.exists(dst):
        assert pkg.lib().bark_model_quantize(src.encode(), (dst + ".tmp").encode(), GGML_FTYPE_MOSTLY_Q4_0)
        os.replace(dst + ".tmp", dst)
    return src, dst


def reference(config, src_ftype, qname):
    """What the unmodified reference produced for this file (tests/golden/make_golden_ref_checks.py)."""
    g = np.load(os.path.join(GOLDEN_DIR, "ref_checks.npz"))
    prefix = f"quant_{config}_{src_ftype}_{qname}_"
    return {k[len(prefix):]: g[k] for k in g.files if k.startswith(prefix)}


def sha(a):
    return hashlib.sha1(bits(a).tobytes()).hexdigest()


FTYPES = {"q4_0": 2, "q4_1": 3, "q8_0": 7, "q5_0": 8, "q5_1": 9}      # enum ggml_ftype (ggml.h:388-417), the five types the reference tool's README lists


@pytest.mark.parametrize("qname", sorted(FTYPES))
@pytest.mark.parametrize("config,src_ftype", [("tiny", "f16"), ("mini", "f32")])
def test_quantized_file_is_byte_identical_to_the_reference_tool(pkg, weights_file, tmp_path, config, src_ftype, qname):
    src = weights_file(config, src_ftype)
    ours = str(tmp_path / "ours.bin")
    assert pkg.lib().bark_model_quantize(src.encode(), ours.encode(), FTYPES[qname])
    ref = reference(config, src_ftype, qname)
    a = open(ours, "rb").read()
    assert len(a) == int(ref["file_size"]) and hashlib.sha1(a).hexdigest() == str(ref["file_sha1"])
    assert len(a) < os.path.getsize(src)


def test_quantize_rejects_what_it_cannot_do(pkg, weights_file, tmp_path):
    src = weights_file("tiny", "f16")
    L = pkg.lib()
    assert not L.bark_model_quantize(src.encode(), str(tmp_path / "x.bin").encode(), 12)          # q4_K: k-quants are not implemented here
    assert not L.bark_model_quantize(b"/nonexistent/in.bin", str(tmp_path / "y.bin").encode(), GGML_FTYPE_MOSTLY_Q4_0)
    bad = tmp_path / "bad.bin"; bad.write_bytes(b"\x00" * 64)
    assert not L.bark_model_quantize(str(bad).encode(), str(tmp_path / "z.bin").encode(), GGML_FTYPE_MOSTLY_Q4_0)


@pytest.mark.parametrize("qname", sorted(FTYPES))
@pytest.mark.parametrize("config,src_ftype", [("tiny", "f16"), ("mini", "f32")])
def test_quantised_oracle_matches_the_reference(pkg, orc, weights_file, tmp_path, config, src_ftype, qname):
    """Pins the oracle's quantised paths (q8_0 / q8_1 activation blocks, the 8-lane integer dots, hsum_float_8, get_rows
    dequantisation): teacher-forced logits (merged prompt, decode, ragged coarse prefill), a fine pass and a whole generation,
    oracle vs the unmodified reference on the same quantised file."""
    src = weights_file(config, src_ftype)
    path = str(tmp_path / f"{qname}.bin")
    assert pkg.lib().bark_model_quantize(src.encode(), path.encode(), FTYPES[qname])
    o, ref = orc.Oracle(path, seed=0, n_steps=10), reference(config, src_ftype, qname)
    assert int(o.hparams(0)[9]) % 1000 == FTYPES[qname]
    rng = np.random.default_rng(17)
    toks, po = o.tokenize("Hello, world"), 0
    for step in range(4):
        lo, po = o.gpt_eval(0, toks, po, True)
        assert sha(lo) == str(ref["semantic_sha1"][step]), f"semantic step {step}: logits differ from the reference's"
        toks = np.array([int(np.argmax(lo[:10000]))], np.int32)
    toks = np.concatenate([rng.integers(0, 10000, 256), [12050], rng.integers(10000, 12048, 21)]).astype(np.int32)
    po = 0
    for step in range(3):
        lo, po = o.gpt_eval(1, toks, po, False)
        assert sha(lo) == str(ref["coarse_sha1"][step]), f"coarse step {step}: logits differ from the reference's"
        toks = np.array([10000 + int(np.argmax(lo[10000:12048]))], np.int32)
    buf = rng.integers(0, 1024, (8, 1024)).astype(np.int32); buf[:, 300:] = 1024; buf[4:, :] = 1024
    assert sha(o.fine_eval(buf, 4)) == str(ref["fine_sha1"])
    go = o.generate("hello world")
    for k in ("semantic", "coarse", "fine"):
        assert np.array_equal(go[k], ref[f"generate_{k}"]), k
    assert sha(go["audio"]) == str(ref["generate_audio_sha1"])
