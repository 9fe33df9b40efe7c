"""GPU: batched generation (bark_b200_generate_audio_batch, csrc/batch.cu).  Every item of a batch must be bit-identical — semantic,
coarse and fine ids and the waveform's bits — to a fresh single-prompt context with the item's seed generating the item's prompt."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import FIXTURE_DIR, bits

pytestmark = pytest.mark.gpu


def prompts(n):
    return ["hello world" if i == 0 else f"hello world {i}" for i in range(n)]


def single_run(pkg, path, seed, text, **kw):
    with pkg.Bark(path, seed=seed, **kw) as b:
        audio = b.generate(text)
        return audio, [b.tokens(i).copy() for i in range(3)]


def assert_same(item, ref, what=""):
    (a, t), (ra, rt) = item, ref
    for stage in range(3):
        assert np.array_equal(t[stage], rt[stage]), f"{what}: stage {stage} ids differ ({t[stage].shape} vs {rt[stage].shape})"
    assert a.shape == ra.shape and np.array_equal(bits(a), bits(ra)), f"{what}: waveform differs"


def check_batch(pkg, path, n, seeds=None, **kw):
    seeds = list(range(n)) if seeds is None else seeds
    texts = prompts(n)
    with pkg.Bark(path, seed=99, **kw) as b:
        got = b.generate_batch(texts, seeds)
        stats = b.batch_stats()
    for i in range(n):
        assert_same(got[i], single_run(pkg, path, seeds[i], texts[i], **kw), f"item {i} of {n}")
    return got, stats


def quantized(pkg, weights_file, config, src_ftype, qname):
    ftype_id = {"q4_0": 2, "q4_1": 3, "q5_0": 8, "q5_1": 9, "q8_0": 7}[qname]
    src = weights_file(config, src_ftype)
    dst = os.path.join(FIXTURE_DIR, f"{config}_{src_ftype}_1234_{qname}.bin")
    if not os.path.exists(dst):
        assert pkg.lib().bark_model_quantize(src.encode(), (dst + ".tmp").encode(), ftype_id)
        os.replace(dst + ".tmp", dst)
    return dst


@pytest.mark.parametrize("config,ftype,n", [("tiny", "f16", 1), ("tiny", "f16", 3), ("tiny", "f16", 17), ("mini", "f32", 3), ("mini", "f16", 17),
                                            ("tiny", "q4_0", 3), ("tiny", "q8_0", 17), ("tiny", "q5_1", 3), ("wide", "f16", 3)])
def test_batch_items_equal_single_prompt_runs(pkg, weights_file, config, ftype, n):
    """B = 1, B < 16 (few-row mat-mul) and B >= 16 (tiled mat-mul), f32 / f16 / quantised weights, bark-large widths."""
    path = quantized(pkg, weights_file, config, "f16", ftype) if ftype.startswith("q") else weights_file(config, ftype)
    _, stats = check_batch(pkg, path, n, n_steps_text_encoder=24)
    assert stats["batched_steps"] > 0


def test_batch_against_the_oracle(pkg, orc, weights_file):
    path = weights_file("tiny", "f16")
    texts, seeds = prompts(3), [5, 6, 7]
    with pkg.Bark(path, seed=0, n_steps_text_encoder=20) as b:
        got = b.generate_batch(texts, seeds)
    for i in range(3):
        ref = orc.Oracle(path, seed=seeds[i], n_steps=20).generate(texts[i])
        audio, toks = got[i]
        for stage, key in enumerate(("semantic", "coarse", "fine")):
            assert np.array_equal(toks[stage], ref[key]), f"item {i}: {key} ids differ from the oracle"
        assert audio.shape == ref["audio"].shape and np.array_equal(bits(audio), bits(ref["audio"]))


@pytest.mark.parametrize("config,ftype,n", [("tiny", "f16", 3), ("mini", "f32", 3), ("mini", "f16", 17)])
def test_teacher_forced_batched_logits(pkg, weights_file, config, ftype, n):
    """Distinct prompts per item, 250 prompt ids + 40 batched steps: n_kv crosses multiples of 8 and 32 (soft_max tail, P.V leftovers).
    Each item's logits equal the single-context evaluation (the persistent decode kernel) bit for bit, for both causal models."""
    path = weights_file(config, ftype)
    rng = np.random.default_rng(41)
    ln, steps = 250, 40
    with pkg.Bark(path, seed=0) as b:
        for which, hi in ((0, 10000), (1, 12048)):
            p = rng.integers(0, hi, (n, ln)).astype(np.int32)
            x = rng.integers(0, hi, (n, steps)).astype(np.int32)
            got = b.batch_eval(which, p, x)
            for i in range(n):
                lg, pg = b.gpt_eval(which, p[i], 0, False)
                for j in range(steps):
                    lg, pg = b.gpt_eval(which, x[i, j:j + 1], pg, False)
                    assert np.array_equal(bits(got[i, j]), bits(lg)), \
                        f"model {which} item {i} step {j} (n_kv {ln + j + 1}): {int((got[i, j] != lg).sum())} logits differ"


def test_ragged_batch(pkg, weights_file):
    """min_eos_p low enough that items stop the semantic stage at different steps (the batch compacts); coarse windows then differ too."""
    path = weights_file("tiny", "f16")
    got, _ = check_batch(pkg, path, 6, n_steps_text_encoder=150, min_eos_p=1.2e-5)
    lengths = [t[0].size for _, t in got]
    assert len(set(lengths)) > 1 and min(lengths) < 150, f"no ragged stop: semantic lengths {lengths}; adjust min_eos_p in this test"


def test_long_clip_batch(pkg, weights_file):
    """230 semantic steps: 12 coarse windows, saturated history, prefix reuse inside every item's own cache."""
    path = weights_file("tiny", "f16")
    got, _ = check_batch(pkg, path, 3, n_steps_text_encoder=230)
    assert all(t[1].shape[0] == 345 for _, t in got)


def test_forced_host_replays_inside_a_batch(pkg, weights_file, monkeypatch):
    path = weights_file("mini", "f16")
    monkeypatch.setenv("BARK_B200_SAMPLE_FLAG_EVERY", "3")
    with pkg.Bark(path, seed=0, n_steps_text_encoder=30) as b:
        got = b.generate_batch(prompts(4), [0, 1, 2, 3])
        assert b.batch_stats()["host_replays"] > 0
    monkeypatch.delenv("BARK_B200_SAMPLE_FLAG_EVERY")
    for i in range(4):
        assert_same(got[i], single_run(pkg, path, i, prompts(4)[i], n_steps_text_encoder=30), f"item {i}")


def ctx_audio(pkg, b):
    n = pkg.lib().bark_get_audio_data_size(b.ctx)
    return np.ctypeslib.as_array(pkg.lib().bark_get_audio_data(b.ctx), shape=(n,)).copy()


def test_batch_leaves_single_prompt_state_alone(pkg, weights_file):
    """generate -> batch -> generate gives the same second result as generate -> generate (RNG, tokens, audio, statistics)."""
    path = weights_file("tiny", "f16")
    runs = []
    for with_batch in (False, True):
        with pkg.Bark(path, seed=4, n_steps_text_encoder=20) as b:
            b.generate("first prompt")
            if with_batch:
                a_before = ctx_audio(pkg, b)
                t_before = [b.tokens(i).copy() for i in range(3)]
                s_before = b.stats()[1].copy()
                b.generate_batch(prompts(3), [1, 2, 3])
                assert np.array_equal(bits(a_before), bits(ctx_audio(pkg, b)))
                for i in range(3):
                    assert np.array_equal(t_before[i], b.tokens(i))
                assert np.array_equal(s_before, b.stats()[1])
            a = b.generate("second prompt")
            runs.append((a, [b.tokens(i).copy() for i in range(3)]))
    assert_same(runs[1], runs[0], "second generate")


def test_bad_batch_input_fails_cleanly(pkg, weights_file):
    L = pkg.lib()
    path = weights_file("tiny", "f16")
    with pkg.Bark(path, seed=0, n_steps_text_encoder=12) as b:
        texts = (C.c_char_p * 33)(*[b"hi"] * 33)
        seeds = (C.c_uint32 * 33)(*range(33))
        assert L.bark_b200_generate_audio_batch(b.ctx, texts, seeds, 0) is False
        assert L.bark_b200_generate_audio_batch(b.ctx, texts, seeds, 33) is False
        with_null = (C.c_char_p * 2)(b"hi", None)
        assert L.bark_b200_generate_audio_batch(b.ctx, with_null, seeds, 2) is False
        assert L.bark_b200_generate_audio_batch(b.ctx, None, seeds, 1) is False
        assert L.bark_b200_generate_audio_batch(None, texts, seeds, 1) is False
        assert L.bark_b200_batch_audio(b.ctx, 0, None, 0) == -1                 # nothing generated yet
        got = b.generate_batch(["hello world", "again"], [0, 1])
        assert L.bark_b200_batch_audio(b.ctx, 2, None, 0) == -1
        assert L.bark_b200_batch_audio(b.ctx, -1, None, 0) == -1
        assert L.bark_b200_batch_tokens(b.ctx, 0, 3, None, 0) == -1
        assert L.bark_b200_batch_tokens(b.ctx, 5, 0, None, 0) == -1
        assert L.bark_b200_batch_audio(b.ctx, 1, None, 0) == got[1][0].size
        # the context still works after the refusals
        assert_same(b.generate_batch(["hello world"], [0])[0], got[0], "after bad input")


def test_fast_mode_batch(pkg, weights_file, monkeypatch):
    """BARK_B200_MODE=fast: the batch's fine stage is the same fast-mode fine_eval, so each item equals its own fast-mode run."""
    monkeypatch.setenv("BARK_B200_MODE", "fast")
    path = weights_file("mini", "f16")
    with pkg.Bark(path, seed=0) as b:
        assert b.fast_mode
    check_batch(pkg, path, 3, n_steps_text_encoder=24)


def test_bench_size_batch(pkg):
    """bark-small f16, n_steps_text_encoder = 138, eight items of the bench workload (seed i, "hello world" / "hello world {i}")."""
    import bench
    path = bench.weights_path()
    n = bench.N_STEPS_TEXT
    seeds = [bench.rank_workload(i)["seed"] for i in range(8)]
    texts = [bench.rank_workload(i)["prompt"] for i in range(8)]
    with pkg.Bark(path, seed=0, n_steps_text_encoder=n) as b:
        got = b.generate_batch(texts, seeds)
    for i in range(8):
        assert_same(got[i], single_run(pkg, path, seeds[i], texts[i], n_steps_text_encoder=n), f"bench item {i}")
