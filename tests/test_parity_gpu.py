"""GPU parity: the CUDA path, called through the C-ABI (libbark_b200.so), against the CPU oracle.

Token ids and teacher-forced logits must be BIT-exact (north_star: "bit-exactly for token ids"); the
waveform must be within 1e-3 relative (north_star).  For the full-size (bark-small) case the checker is the unmodified
reference itself, through its outputs stored in tests/golden/ref_checks.npz.
"""
import numpy as np
import pytest

from conftest import bits

pytestmark = pytest.mark.gpu

WAV_RTOL = 1e-3          # BASELINE.json north_star: "within 1e-3 relative for the final fp32 waveform"


def wav_rel(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


CASES = [("tiny", "f16"), ("mini", "f32"), ("mini", "f16")]


@pytest.mark.parametrize("config,ftype", CASES)
def test_teacher_forced_logits_bit_exact(pkg, orc, weights_file, config, ftype):
    path = weights_file(config, ftype)
    o = orc.Oracle(path)
    rng = np.random.default_rng(7)
    with pkg.Bark(path) as b:
        # semantic: merged 513-id prompt (257 positions), then single-token decode steps
        prompt = o.tokenize("Hello, world! 123 café")
        assert np.array_equal(prompt, b.tokenize("Hello, world! 123 café"))
        toks, pg, po = prompt, 0, 0
        for step in range(20):
            lg, pg = b.gpt_eval(0, toks, pg, True)
            lo, po = o.gpt_eval(0, toks, po, True)
            assert pg == po
            assert np.array_equal(bits(lg), bits(lo)), f"semantic step {step}: {int((lg != lo).sum())} logits differ, max {np.abs(lg - lo).max():.3e}"
            toks = np.array([int(np.argmax(lo[:10000]))], np.int32)
        # coarse: ragged prefill (n_kv % 8 != 0 and % 32 != 0 -> libm expf tail, scalar dot leftovers), decode across the boundaries
        toks = np.concatenate([rng.integers(0, 10000, 256), [12050], rng.integers(10000, 12048, 37)]).astype(np.int32)
        pg = po = 0
        for step in range(45):
            lg, pg = b.gpt_eval(1, toks, pg, False)
            lo, po = o.gpt_eval(1, toks, po, False)
            assert np.array_equal(bits(lg), bits(lo)), f"coarse step {step} (n_past {po}): {int((lg != lo).sum())} logits differ, max {np.abs(lg - lo).max():.3e}"
            toks = np.array([10000 + int(np.argmax(lo[10000:12048]))], np.int32)
        # a multi-row evaluation on top of a filled cache (a coarse window start with prefix reuse): rows below n_kv & ~31 of
        # an evaluation do not depend on its n_kv (bark_api.cu run_coarse), so evaluating the tail on top of them must equal
        # the oracle's from-scratch evaluation of the whole sequence
        full = np.concatenate([rng.integers(0, 10000, 256), [12050], rng.integers(10000, 12048, 75)]).astype(np.int32)
        for cut in (256, 288, 320):
            _, pg = b.gpt_eval(1, full[:cut + 5], 0, False)          # leaves rows [0, cut) canonical, rows cut .. cut+4 are overwritten below
            lg, pg = b.gpt_eval(1, full[cut:], cut, False)
            lo, po = o.gpt_eval(1, full, 0, False)
            assert pg == po == full.size
            assert np.array_equal(bits(lg), bits(lo)), f"suffix evaluation after {cut} cached rows: {int((lg != lo).sum())} logits differ"


@pytest.mark.parametrize("config,ftype", [("tiny", "f16"), ("mini", "f32")])
def test_fine_pass_logits_bit_exact(pkg, orc, weights_file, config, ftype):
    path = weights_file(config, ftype)
    o = orc.Oracle(path)
    rng = np.random.default_rng(3)
    buf = rng.integers(0, 1024, (8, 1024)).astype(np.int32)
    buf[:, 700:] = 1024                      # time padding like a 700-frame clip
    with pkg.Bark(path) as b:
        for nn in (2, 5, 7):
            x = buf.copy(); x[nn:, :] = 1024
            lg, lo = b.fine_eval(x, nn), o.fine_eval(x, nn)
            assert np.array_equal(bits(lg), bits(lo)), f"fine nn={nn}: {int((lg != lo).sum())} logits differ, max {np.abs(lg - lo).max():.3e}"


def test_host_sampler_matches_oracle(pkg, orc, weights_file):
    path = weights_file("tiny", "f16")
    o = orc.Oracle(path)
    rng = np.random.default_rng(11)
    with pkg.Bark(path) as b:
        b.reseed(42); o.reseed(42)
        for i in range(200):
            n = (10048, 1024)[i % 2]
            lg = (rng.standard_normal(n) * 5).astype(np.float32)
            temp = (0.7, 0.5, 0.0)[i % 3]
            assert b.sample(0, lg, temp) == o.sample(lg, temp)


def test_device_sampler_matches_oracle(pkg, orc, weights_file):
    """sample_rows_kernel (the sampler the stages use) against gpt_sample of the oracle: same tokens, same RNG stream."""
    path = weights_file("tiny", "f16")
    o = orc.Oracle(path)
    rng = np.random.default_rng(13)
    with pkg.Bark(path) as b:
        b.reseed(9); o.reseed(9)
        replays = 0
        for case, (rows, n, scale, temp) in enumerate([(1024, 1024, 5.0, 0.5), (1, 10048, 5.0, 0.7), (1, 1024, 0.01, 0.7), (64, 1024, 40.0, 0.7),
                                                        (7, 1056, 1.0, 0.0), (1, 10048, 3.0, 0.0), (33, 777, 8.0, 1.3)]):
            lg = (rng.standard_normal((rows, n)) * scale).astype(np.float32)
            if case == 3:
                lg[:, -1] += 200.0               # one dominant logit: everything else underflows to 0
            tok, eos, r = b.sample_rows(lg, temp)
            replays += r
            for i in range(rows):
                t, e = o.sample(lg[i], temp)
                assert tok[i] == t, f"case {case} row {i}: device {tok[i]} oracle {t}"
                assert bits(np.float32(eos[i])) == bits(np.float32(e))
        assert replays < 8                        # flagged rows are the rare exception, not the path


def test_sampler_paths_agree(pkg, weights_file, monkeypatch):
    """Device sampler (chained decode), forced host replays inside the chain, and the plain host sampler: same tokens and
    same RNG state afterwards (second clip on the same context)."""
    path = weights_file("mini", "f16")
    runs = []
    for env in ({}, {"BARK_B200_SAMPLE_FLAG_EVERY": "5"}, {"BARK_B200_SAMPLE": "host"}, {"BARK_B200_DECODE": "multi"}, {"BARK_B200_KV_REUSE": "0"},
                {"BARK_B200_KV_REUSE": "0", "BARK_B200_SAMPLE": "host"}):
        for k in ("BARK_B200_SAMPLE_FLAG_EVERY", "BARK_B200_SAMPLE", "BARK_B200_DECODE", "BARK_B200_KV_REUSE"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        with pkg.Bark(path, seed=3, n_steps_text_encoder=70) as b:
            a1 = b.generate("one two three"); t1 = [b.tokens(i).copy() for i in range(3)]
            a2 = b.generate("four"); t2 = [b.tokens(i).copy() for i in range(3)]
        runs.append((a1, t1, a2, t2))
    for a1, t1, a2, t2 in runs[1:]:
        for i in range(3):
            assert np.array_equal(t1[i], runs[0][1][i]) and np.array_equal(t2[i], runs[0][3][i])
        assert np.array_equal(bits(a1), bits(runs[0][0])) and np.array_equal(bits(a2), bits(runs[0][2]))


def test_coarse_prefix_reuse_on_a_long_clip(pkg, weights_file, monkeypatch):
    """230 semantic tokens -> 690 coarse steps in 12 windows: the semantic window start moves (semantic_idx > 209) and the
    coarse history saturates at 630, so window prompts stop being extensions of the cache.  Prefix reuse (default) must give
    the tokens of the reference's full re-prefill (BARK_B200_KV_REUSE=0; that path is the one pinned against the oracle)."""
    path = weights_file("tiny", "f16")
    runs = []
    for reuse in ("1", "0"):
        monkeypatch.setenv("BARK_B200_KV_REUSE", reuse)
        with pkg.Bark(path, seed=5, n_steps_text_encoder=230) as b:
            a = b.generate("a long clip")
            runs.append((a, [b.tokens(i).copy() for i in range(3)]))
    assert runs[0][1][1].shape[0] == 345
    for i in range(3):
        assert np.array_equal(runs[0][1][i], runs[1][1][i])
    assert np.array_equal(bits(runs[0][0]), bits(runs[1][0]))


def test_semantic_early_stop_inside_a_batch(pkg, orc, weights_file):
    """min_eos_p low enough that the stop test fires mid-batch: the device path runs ahead, then must drop the surplus
    steps and rewind the RNG so the coarse and fine stages draw what the reference draws."""
    path = weights_file("tiny", "f16")
    hit = 0
    for seed, eos in ((0, 7.0e-6), (1, 1.2e-5), (2, 3.6e-6)):      # stops after 39, 85 and 37 tokens (batches are 64 steps)
        ref = orc.Oracle(path, seed=seed, n_steps=150, min_eos_p=eos).generate("hello world")
        with pkg.Bark(path, seed=seed, n_steps_text_encoder=150, min_eos_p=eos) as b:
            b.generate("hello world")
            assert np.array_equal(b.tokens(0), ref["semantic"])
            assert np.array_equal(b.tokens(1), ref["coarse"])
            assert np.array_equal(b.tokens(2), ref["fine"])
        hit += 0 < len(ref["semantic"]) < 150
    assert hit == 3, "no early stop happened: adjust min_eos_p in this test"


@pytest.mark.parametrize("config,ftype,n_steps", [("tiny", "f16", 20), ("mini", "f32", 45), ("mini", "f16", 30)])
def test_generate_tokens_bit_exact_and_waveform(pkg, orc, weights_file, config, ftype, n_steps):
    path = weights_file(config, ftype)
    ref = orc.Oracle(path, seed=0, n_steps=n_steps).generate("hello world")
    with pkg.Bark(path, seed=0, n_steps_text_encoder=n_steps) as b:
        audio = b.generate("hello world")
        assert np.array_equal(b.tokens(0), ref["semantic"])
        assert np.array_equal(b.tokens(1), ref["coarse"])
        assert np.array_equal(b.tokens(2), ref["fine"])
        assert audio.shape == ref["audio"].shape
        assert wav_rel(audio, ref["audio"]) < WAV_RTOL             # the contract
        assert np.array_equal(bits(audio), bits(ref["audio"]))      # what the lane-ordered codec actually delivers
        # second call on the same context: RNG is NOT reseeded (bark.cpp:1179), sample counters accumulate
        audio2 = b.generate("hello world")
        assert audio2.shape[0] % 320 == 0


def test_encodec_decode_within_tolerance(pkg, orc, weights_file):
    path = weights_file("tiny", "f16")
    o = orc.Oracle(path)
    rng = np.random.default_rng(5)
    with pkg.Bark(path) as b:
        for T in (7, 33, 96):
            codes = rng.integers(0, 1024, (8, T)).astype(np.int32)
            a, r = b.encodec_decode(codes), o.encodec_decode(codes)
            assert a.shape == r.shape == (320 * T,)
            assert wav_rel(a, r) < WAV_RTOL                      # the contract
            assert np.array_equal(bits(a), bits(r)), f"T={T}: codec is expected to be bit-exact, rel err {wav_rel(a, r):.3e}"


def test_full_size_against_the_reference_itself(pkg, weights_file):
    """bark-small dimensions (E=768, L=12, H=12, f16): CUDA vs the unmodified reference, teacher-forced and free-running.  The
    reference's logits (sha1 of their bits), ids and waveform are stored in tests/golden/ref_checks.npz."""
    import hashlib
    import os
    from conftest import GOLDEN_DIR
    g = np.load(os.path.join(GOLDEN_DIR, "ref_checks.npz"))
    path = weights_file("small", "f16")
    with pkg.Bark(path, seed=0, n_steps_text_encoder=12) as b:
        prompt = b.tokenize("hello world")
        assert np.array_equal(prompt, g["small_prompt_ids"])
        toks, pg = prompt, 0
        for step in range(6):
            lg, pg = b.gpt_eval(0, toks, pg, True)
            head = g["small_semantic_head"][step]
            assert hashlib.sha1(bits(lg).tobytes()).hexdigest() == str(g["small_semantic_sha1"][step]), \
                f"semantic step {step}: logits differ from the reference's ({int((bits(lg[:head.size]) != bits(head)).sum())} of the first {head.size})"
            toks = np.array([int(np.argmax(lg[:10000]))], np.int32)
        audio = b.generate("hello world")
        assert np.array_equal(b.tokens(0), g["small_generate_semantic"])
        assert np.array_equal(b.tokens(1), g["small_generate_coarse"])
        assert np.array_equal(b.tokens(2), g["small_generate_fine"])
        assert audio.shape == g["small_generate_audio"].shape
        assert wav_rel(audio, g["small_generate_audio"]) < WAV_RTOL


# ---- q4_0 GPT weights (BASELINE configs[3]: q4_0 GPT + f16 codec) --------------------------------------------------------
def _q4_path(pkg, weights_file, config, src_ftype):
    import os
    from conftest import FIXTURE_DIR
    src = weights_file(config, src_ftype)
    dst = os.path.join(FIXTURE_DIR, f"{config}_{src_ftype}_1234_q4_0.bin")
    if not os.path.exists(dst):
        assert pkg.lib().bark_model_quantize(src.encode(), (dst + ".tmp").encode(), 2)      # the library's own quantizer (tests/test_quantize.py pins it)
        os.replace(dst + ".tmp", dst)
    return dst


@pytest.mark.parametrize("config,src_ftype,n_steps", [("tiny", "f16", 16), ("mini", "f32", 30)])
def test_q4_0_logits_tokens_and_waveform(pkg, orc, weights_file, config, src_ftype, n_steps):
    """q4_0 mul_mat (q8_0 activation blocks, 8 int lanes per block, hsum_float_8) and q4_0 get_rows against the oracle, whose
    q4_0 path is pinned bit-exactly against the unmodified reference (tests/test_quantize.py)."""
    path = _q4_path(pkg, weights_file, config, src_ftype)
    o = orc.Oracle(path, seed=0, n_steps=n_steps)
    rng = np.random.default_rng(19)
    with pkg.Bark(path, seed=0, n_steps_text_encoder=n_steps) as b:
        assert int(b.hparams(0)[9]) % 1000 == 2
        toks, pg, po = o.tokenize("Hello, world"), 0, 0
        for step in range(6):
            lg, pg = b.gpt_eval(0, toks, pg, True)
            lo, po = o.gpt_eval(0, toks, po, True)
            assert np.array_equal(bits(lg), bits(lo)), f"semantic step {step}: {int((lg != lo).sum())} logits differ, max {np.abs(lg - lo).max():.3e}"
            toks = np.array([int(np.argmax(lo[:10000]))], np.int32)
        toks = np.concatenate([rng.integers(0, 10000, 256), [12050], rng.integers(10000, 12048, 37)]).astype(np.int32)
        pg = po = 0
        for step in range(8):
            lg, pg = b.gpt_eval(1, toks, pg, False)
            lo, po = o.gpt_eval(1, toks, po, False)
            assert np.array_equal(bits(lg), bits(lo)), f"coarse step {step}: {int((lg != lo).sum())} logits differ"
            toks = np.array([10000 + int(np.argmax(lo[10000:12048]))], np.int32)
        buf = rng.integers(0, 1024, (8, 1024)).astype(np.int32); buf[:, 500:] = 1024
        for nn in (2, 6):
            x = buf.copy(); x[nn:, :] = 1024
            assert np.array_equal(bits(b.fine_eval(x, nn)), bits(o.fine_eval(x, nn))), f"fine nn={nn}"
        ref = o.generate("hello world")
        audio = b.generate("hello world")
        assert np.array_equal(b.tokens(0), ref["semantic"])
        assert np.array_equal(b.tokens(1), ref["coarse"])
        assert np.array_equal(b.tokens(2), ref["fine"])
        assert wav_rel(audio, ref["audio"]) < WAV_RTOL


def test_bark_large_widths(pkg, orc, weights_file):
    """E=1024 / 16 heads / K=4096 (bark-large widths, BASELINE configs[2]) at 2 layers: decode rows too long for the staging
    area are streamed from global memory, 64 soft_max CTAs, two LayerNorm elements per thread — all against the oracle."""
    path = weights_file("wide", "f16")
    o = orc.Oracle(path, seed=0, n_steps=8)
    rng = np.random.default_rng(23)
    with pkg.Bark(path, seed=0, n_steps_text_encoder=8) as b:
        toks, pg, po = o.tokenize("hello world"), 0, 0
        for step in range(12):
            lg, pg = b.gpt_eval(0, toks, pg, True)
            lo, po = o.gpt_eval(0, toks, po, True)
            assert np.array_equal(bits(lg), bits(lo)), f"semantic step {step}: {int((lg != lo).sum())} logits differ, max {np.abs(lg - lo).max():.3e}"
            toks = np.array([int(np.argmax(lo[:10000]))], np.int32)
        toks = np.concatenate([rng.integers(0, 10000, 256), [12050], rng.integers(10000, 12048, 45)]).astype(np.int32)
        pg = po = 0
        for step in range(12):
            lg, pg = b.gpt_eval(1, toks, pg, False)
            lo, po = o.gpt_eval(1, toks, po, False)
            assert np.array_equal(bits(lg), bits(lo)), f"coarse step {step}: {int((lg != lo).sum())} logits differ"
            toks = np.array([10000 + int(np.argmax(lo[10000:12048]))], np.int32)
        buf = rng.integers(0, 1024, (8, 1024)).astype(np.int32); buf[:, 600:] = 1024; buf[3:, :] = 1024
        assert np.array_equal(bits(b.fine_eval(buf, 3)), bits(o.fine_eval(buf, 3)))      # one 1024-row pass (a whole generation costs the CPU oracle a minute)


@pytest.mark.parametrize("config,ftype", [("tiny", "f16"), ("mini", "f32"), ("mini", "f16")])
def test_packed_fma_variants_are_bit_identical(pkg, orc, weights_file, monkeypatch, config, ftype):
    """BARK_B200_FFMA2 (default on; 0 = scalar FMA): the tiled mat-mul / scores / P.V kernels with the 64 FMAs of a chain step issued as 32 packed FFMA2
    (fma.rn.f32x2).  Per component the arithmetic is __fmaf_rn's, so prefill logits, fine passes and a whole generation must not
    move by a bit — against the default kernels and against the oracle."""
    path = weights_file(config, ftype)
    o = orc.Oracle(path, seed=0, n_steps=24)
    rng = np.random.default_rng(29)
    toks = np.concatenate([rng.integers(0, 10000, 256), [12050], rng.integers(10000, 12048, 53)]).astype(np.int32)
    buf = rng.integers(0, 1024, (8, 1024)).astype(np.int32); buf[:, 640:] = 1024; buf[5:, :] = 1024
    res = {}
    for f2 in ("0", "1"):
        monkeypatch.setenv("BARK_B200_FFMA2", f2)
        with pkg.Bark(path, seed=0, n_steps_text_encoder=24) as b:
            lg, _ = b.gpt_eval(1, toks, 0, False)
            sem, _ = b.gpt_eval(0, o.tokenize("packed"), 0, True)
            fl = b.fine_eval(buf, 5)
            audio = b.generate("hello world")
            res[f2] = (lg, sem, fl, audio, [b.tokens(i).copy() for i in range(3)])
    for a, c in zip(res["0"][:4], res["1"][:4]):
        assert np.array_equal(bits(a), bits(c))
    for a, c in zip(res["0"][4], res["1"][4]):
        assert np.array_equal(a, c)
    lo, _ = o.gpt_eval(1, toks, 0, False)
    assert np.array_equal(bits(res["1"][0]), bits(lo))
    assert np.array_equal(bits(res["1"][2]), bits(o.fine_eval(buf, 5)))


@pytest.mark.parametrize("qname,ftype_id", [("q4_1", 3), ("q5_0", 8), ("q5_1", 9), ("q8_0", 7)])
@pytest.mark.parametrize("config,src_ftype,n_steps", [("tiny", "f16", 16), ("mini", "f32", 24)])
def test_experimental_quant_types(pkg, orc, weights_file, tmp_path, monkeypatch, config, src_ftype, n_steps, qname, ftype_id):
    """q4_1 / q5_0 / q5_1 / q8_0 GPT weights (qx_kernels.cu) against the oracle,
    whose arithmetic for these types is pinned bit-exactly against the unmodified reference (tests/test_quantize.py)."""
    src = weights_file(config, src_ftype)
    path = str(tmp_path / f"{qname}.bin")
    assert pkg.lib().bark_model_quantize(src.encode(), path.encode(), ftype_id)
    o = orc.Oracle(path, seed=0, n_steps=n_steps)
    rng = np.random.default_rng(31)
    with pkg.Bark(path, seed=0, n_steps_text_encoder=n_steps) as b:
        assert int(b.hparams(0)[9]) % 1000 == ftype_id
        toks, pg, po = o.tokenize("Hello, world"), 0, 0
        for step in range(5):
            lg, pg = b.gpt_eval(0, toks, pg, True)
            lo, po = o.gpt_eval(0, toks, po, True)
            assert np.array_equal(bits(lg), bits(lo)), f"semantic step {step}: {int((lg != lo).sum())} logits differ, max {np.abs(lg - lo).max():.3e}"
            toks = np.array([int(np.argmax(lo[:10000]))], np.int32)
        toks = np.concatenate([rng.integers(0, 10000, 256), [12050], rng.integers(10000, 12048, 29)]).astype(np.int32)
        pg = po = 0
        for step in range(5):
            lg, pg = b.gpt_eval(1, toks, pg, False)
            lo, po = o.gpt_eval(1, toks, po, False)
            assert np.array_equal(bits(lg), bits(lo)), f"coarse step {step}: {int((lg != lo).sum())} logits differ"
            toks = np.array([10000 + int(np.argmax(lo[10000:12048]))], np.int32)
        buf = rng.integers(0, 1024, (8, 1024)).astype(np.int32); buf[:, 400:] = 1024; buf[4:, :] = 1024
        assert np.array_equal(bits(b.fine_eval(buf, 4)), bits(o.fine_eval(buf, 4)))
        ref = o.generate("hello world")
        audio = b.generate("hello world")
        assert np.array_equal(b.tokens(0), ref["semantic"])
        assert np.array_equal(b.tokens(1), ref["coarse"])
        assert np.array_equal(b.tokens(2), ref["fine"])
        assert wav_rel(audio, ref["audio"]) < WAV_RTOL


def _generate_in_thread(pkg, path, device, seed, prompt, out, key):
    try:
        with pkg.Bark(path, seed=seed, n_steps_text_encoder=20, device=device) as b:
            audio = b.generate(prompt)
            out[key] = (b.tokens(0).copy(), b.tokens(1).copy(), b.tokens(2).copy(), audio)
    except Exception as e:                                         # surfaces in the asserting thread
        out[key] = e


@pytest.mark.parametrize("two_devices", [False, True])
def test_one_host_thread_per_context_in_one_process(pkg, weights_file, two_devices):
    """SURVEY §5 / bark.h threading contract as this library states it (INTEGRATION.md §4): one host thread per context, several
    contexts per process — on one GPU, and on two GPUs (kernel attributes are configured per device, launch annotations are
    thread-local, counters atomic).  Each thread's tokens and waveform equal the single-threaded run of the same (seed, prompt)."""
    import threading
    from conftest import cuda_device_count
    if two_devices and cuda_device_count() < 2:
        pytest.skip("needs two GPUs")
    path = weights_file("mini", "f16")
    jobs = [(0, 3, "hello world"), (1 if two_devices else 0, 4, "The quick brown fox")]
    ref = {}
    for i, (dev, seed, prompt) in enumerate(jobs):
        _generate_in_thread(pkg, path, dev, seed, prompt, ref, i)
        assert not isinstance(ref[i], Exception), ref[i]
    got = {}
    threads = [threading.Thread(target=_generate_in_thread, args=(pkg, path, dev, seed, prompt, got, i)) for i, (dev, seed, prompt) in enumerate(jobs)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(300)
    for i in range(len(jobs)):
        assert not isinstance(got[i], Exception), got[i]
        for a, c in zip(ref[i][:3], got[i][:3]):
            assert np.array_equal(a, c)
        assert np.array_equal(bits(ref[i][3]), bits(got[i][3]))


def test_exchange_epochs_survive_the_32_bit_wrap(pkg, weights_file, monkeypatch):
    """The decode kernel's tagged exchanges use a 32-bit epoch that advances 6 * n_layer per token; just before it would wrap the host
    drains the stream, clears the exchange words and restarts at 0 (gpt_forward.cu decode_step).  Start 40 tokens before the wrap."""
    path = weights_file("tiny", "f16")
    with pkg.Bark(path, seed=0, n_steps_text_encoder=20) as b:
        a0 = b.generate("hello world"); t0 = [b.tokens(i).copy() for i in range(3)]
    monkeypatch.setenv("BARK_B200_TAG_BASE", str(2 ** 32 - 40 * 12))
    with pkg.Bark(path, seed=0, n_steps_text_encoder=20) as b:
        a1 = b.generate("hello world"); t1 = [b.tokens(i).copy() for i in range(3)]
    for x, y in zip(t0, t1):
        assert np.array_equal(x, y)
    assert np.array_equal(bits(a0), bits(a1))
