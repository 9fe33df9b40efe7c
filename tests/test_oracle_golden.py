"""CPU: the C oracle (oracle/bark_oracle.c) against the committed golden vectors, which were produced by the
unmodified reference (tests/golden/make_golden.py).  This is what pins the oracle on machines where
/root/reference does not exist (the GPU box)."""
import glob
import hashlib
import os

import numpy as np
import pytest

from conftest import GOLDEN_DIR, bits


def sha(a):
    return hashlib.sha1(np.ascontiguousarray(a).tobytes()).hexdigest()


# small_* / large_*: true-size fixtures (tests/test_baseline_config0.py, tests/test_true_size_gpu.py); minutes of CPU time each on the oracle.
# ref_checks.npz: the reference's answers for the inputs of other tests (tests/golden/make_golden_ref_checks.py)
GOLDENS = sorted(p for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")) if "gelu" not in p and not os.path.basename(p).startswith(("small_", "large_", "ref_checks")))


def test_goldens_present():
    assert len(GOLDENS) >= 5


@pytest.mark.parametrize("path", GOLDENS, ids=[os.path.basename(p) for p in GOLDENS])
def test_oracle_reproduces_reference_golden(pkg, orc, weights_file, tmp_path, path):
    g = np.load(path)
    wpath = weights_file(str(g["config"]), str(g["ftype"]), int(g["weight_seed"]))
    if "quant" in g.files and str(g["quant"]) == "q4_0":     # the fixture's file came from the reference's quantizer: ours must write the same bytes
        qpath = str(tmp_path / "q4_0.bin")
        assert pkg.lib().bark_model_quantize(wpath.encode(), qpath.encode(), 2)
        wpath = qpath
    assert hashlib.sha1(open(wpath, "rb").read()).hexdigest() == str(g["weights_sha1"]), "weight generator / quantizer is not reproducible"
    o = orc.Oracle(wpath, seed=int(g["seed"]), n_steps=int(g["n_steps"]))
    prompt = o.tokenize(str(g["prompt"]))
    assert np.array_equal(prompt, g["prompt_ids"])
    toks, n_past = prompt, 0
    for i in range(4):
        lg, n_past = o.gpt_eval(0, toks, n_past, True)
        assert sha(lg) == str(g["sem_logits_sha1"][i]), f"teacher-forced semantic logits differ at step {i}"
        assert np.array_equal(bits(lg[:256]), bits(g["sem_logits_head"][i]))
        toks = np.array([int(np.argmax(lg[:10000]))], np.int32)
    rng = np.random.default_rng(3)
    buf = rng.integers(0, 1024, (8, 1024)).astype(np.int32); buf[:, 700:] = 1024; buf[3:, :] = 1024
    fl = o.fine_eval(buf, 2)
    assert sha(fl) == str(g["fine_logits_sha1"])
    o.reseed(int(g["seed"]))
    r = o.generate(str(g["prompt"]))
    assert np.array_equal(r["semantic"], g["semantic"])
    assert np.array_equal(r["coarse"], g["coarse"])
    assert np.array_equal(r["fine"], g["fine"])
    assert np.array_equal(bits(r["audio"]), bits(g["audio"])), "oracle waveform is not bit-identical to the reference's"


def test_gelu_table_matches_reference(orc):
    ours, _ = orc.gelu_tables()
    ref = np.load(os.path.join(GOLDEN_DIR, "gelu_table_f16.npz"))["table"]
    assert np.array_equal(ours, ref)


def test_vec_dot_lane_order(orc):
    """Unit pins of the dot-product restatement: known answers that only the 4x8-lane order produces."""
    o = orc.Oracle  # noqa: F841  (ensures the library is built)
    import ctypes as C
    L = C.CDLL(orc.ORACLE_SO)
    L.orc_vec_dot_f32.restype = C.c_float
    L.orc_vec_dot_f32.argtypes = [C.c_int, C.c_void_p, C.c_void_p]
    # lane 0 gets 1e8 then -1e8, every other element is 1: a sequential float sum would lose the ones, the lane sum keeps them
    x = np.ones(64, np.float32); y = np.ones(64, np.float32); x[0] = 1e8; x[32] = -1e8
    assert L.orc_vec_dot_f32(64, x.ctypes.data, y.ctypes.data) == 62.0
    # empty and ragged lengths
    assert L.orc_vec_dot_f32(0, x.ctypes.data, y.ctypes.data) == 0.0
    z = np.arange(1, 8, dtype=np.float32)
    assert L.orc_vec_dot_f32(7, z.ctypes.data, z.ctypes.data) == float((z * z).sum())
    # f16 conversion: ties to even, subnormals, overflow to inf
    L.orc_f32_to_f16.restype = C.c_uint16; L.orc_f32_to_f16.argtypes = [C.c_float]
    L.orc_f16_to_f32.restype = C.c_float; L.orc_f16_to_f32.argtypes = [C.c_uint16]
    vals = np.array([0.0, -0.0, 1.0, 1.0009765625, 1.00048828125, 65504.0, 65520.0, 1e-8, 6e-8, 5.96e-8, 3.0e-5, -2.5, 1e6], np.float32)
    for v in vals:
        assert L.orc_f32_to_f16(float(v)) == int(np.float16(v).view(np.uint16)), v
    allh = np.arange(65536, dtype=np.uint16)
    finite = np.isfinite(allh.view(np.float16))
    for h in allh[finite][::97]:
        assert L.orc_f16_to_f32(int(h)) == float(np.array([h], np.uint16).view(np.float16)[0])


def test_mt19937_and_v_expf(orc):
    import ctypes as C
    import random
    L = C.CDLL(orc.ORACLE_SO)
    st = (C.c_uint32 * 625)()
    L.orc_mt_seed(st, 5489)
    L.orc_mt_next.restype = C.c_uint32
    for _ in range(9999):
        L.orc_mt_next(st)
    assert L.orc_mt_next(st) == 4123659995          # the C++ standard's check value for mt19937 (10000th draw)
    L.orc_v_expf.restype = C.c_float; L.orc_v_expf.argtypes = [C.c_float]
    for x in (0.0, -1.0, -10.5, -87.0, -100.0, -200.0, float("-inf")):
        got = L.orc_v_expf(x)
        want = np.exp(np.float64(x))
        assert abs(got - want) <= 3e-7 * max(want, 1e-38) + 1e-45
