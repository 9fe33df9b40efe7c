"""Regenerates tests/golden/ref_checks.npz: what the unmodified reference (oracle/_ref/libbark_ref.so, built by oracle/Makefile)
returns for the inputs of the tests that compare against it, so that those tests run where the reference is not available:

  tests/test_oracle_vs_ref.py      tiny f16: tokenizer, teacher-forced causal / fine passes, sampler, EnCodec, a whole generation
  tests/test_prefix_rows.py        mini f32 / f16: the from-scratch coarse logits the canonical-row tails must equal
  tests/test_quantize.py           the reference tool's quantised files (sha1) and the reference on those files
  tests/test_parity_gpu.py         bark-small f16: teacher-forced semantic logits and a 12-step generation

Float arrays are stored as the sha1 of their bits (plus a short head for diagnostics), token ids and short waveforms in full.
Each test feeds the oracle (or the CUDA path) the same inputs as below, so the two files must be kept in step.

    python tests/golden/make_golden_ref_checks.py          (needs oracle/_ref, i.e. `make -C oracle ref` with the reference tree)
"""
import ctypes as C
import hashlib
import importlib
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
os.environ.setdefault("BARK_B200_QUIET", "1")
import __graft_entry__ as graft  # noqa: E402

TOKENIZER_TEXTS = ["hello world", "", "Hello, world! 123 café zz", "ÀÉÎõü ñ ç", "a" * 600, "x,y;z...", "日本語 text", "tab\there"]
QUANT_FTYPES = {"q4_0": 2, "q4_1": 3, "q8_0": 7, "q5_0": 8, "q5_1": 9}
QUANT_CONFIGS = [("tiny", "f16"), ("mini", "f32")]
HEAD = 32


def sha(a):
    return hashlib.sha1(np.ascontiguousarray(a, np.float32).tobytes()).hexdigest()


def main():
    pkg = graft.load_package()
    weights = importlib.import_module("bark_cpp_b200.weights")
    orc = graft.load_oracle_bindings()
    assert orc.have_ref(), "oracle/_ref/libbark_ref.so is not built"
    fixtures = os.environ.get("BARK_B200_FIXTURES") or os.path.join(tempfile.gettempdir(), f"bark_b200_fixtures_{os.getuid()}")
    os.makedirs(fixtures, exist_ok=True)
    out = {}

    def wfile(config, ftype):
        path = os.path.join(fixtures, f"{config}_{ftype}_1234.bin")
        if not os.path.exists(path):
            weights.write_weights(path + ".tmp", weights.CONFIGS[config](weights.F16 if ftype == "f16" else weights.F32), 1234)
            os.replace(path + ".tmp", path)
        return path

    # ---- tests/test_oracle_vs_ref.py: tiny f16, seed 0, n_steps 16
    r = orc.Ref(wfile("tiny", "f16"), seed=0, n_steps=16)
    out["vs_ref_tokenize"] = np.stack([r.tokenize(t) for t in TOKENIZER_TEXTS])
    rng = np.random.default_rng(1)
    for which, first, merge in ((0, None, True), (1, np.concatenate([rng.integers(0, 10000, 256), [12050], rng.integers(10000, 12048, 37)]).astype(np.int32), False)):
        toks = r.tokenize("hello world") if first is None else first
        n_past, shas, heads, pasts = 0, [], [], []
        for _ in range(40):
            lg, n_past = r.gpt_eval(which, toks, n_past, merge)
            shas.append(sha(lg)); heads.append(lg[:HEAD]); pasts.append(n_past)
            toks = np.array([int(np.argmax(lg[:10000])) if which == 0 else 10000 + int(np.argmax(lg[10000:12048]))], np.int32)
        out[f"vs_ref_causal{which}_sha1"], out[f"vs_ref_causal{which}_head"], out[f"vs_ref_causal{which}_n_past"] = np.array(shas), np.stack(heads), np.array(pasts, np.int32)
    rng = np.random.default_rng(2)
    buf = rng.integers(0, 1024, (8, 1024)).astype(np.int32)
    for nn in (2, 7):
        x = buf.copy(); x[nn:, :] = 1024
        out[f"vs_ref_fine{nn}_sha1"] = np.array(sha(r.fine_eval(x, nn)))
    rng = np.random.default_rng(3)
    r.reseed(9)
    tok, eos = [], []
    for i in range(150):
        lg = (rng.standard_normal((10048, 1024)[i % 2]) * 4).astype(np.float32)
        t, e = r.sample(lg, (0.7, 0.5, 0.0)[i % 3])
        tok.append(t); eos.append(e)
    out["vs_ref_sample_token"], out["vs_ref_sample_eos"] = np.array(tok, np.int32), np.array(eos, np.float32)
    rng = np.random.default_rng(4)
    for T in (7, 40):
        a = r.encodec_decode(rng.integers(0, 1024, (8, T)).astype(np.int32))
        out[f"vs_ref_encodec{T}_sha1"], out[f"vs_ref_encodec{T}_size"] = np.array(sha(a)), np.array(a.size)
    r.reseed(0)
    g = r.generate("hello world")
    for k in ("semantic", "coarse", "fine"):
        out[f"vs_ref_generate_{k}"] = g[k]
    out["vs_ref_generate_audio"] = g["audio"]
    o_tab, r_tab = orc.gelu_tables()
    out["vs_ref_gelu_sha1"] = np.array(hashlib.sha1(r_tab.tobytes()).hexdigest())
    r.close()

    # ---- tests/test_prefix_rows.py: the reference's from-scratch coarse logits, whose tails on canonical rows are equal to them
    for ftype in ("f32", "f16"):
        r = orc.Ref(wfile("mini", ftype))
        rng = np.random.default_rng(21)
        full = np.concatenate([rng.integers(0, 10000, 256), [12050], rng.integers(10000, 12048, 75)]).astype(np.int32)
        scratch, _ = r.gpt_eval(1, full, 0, False)
        for cut in (256, 288, 320):
            r.gpt_eval(1, full[:cut + 5], 0, False)
            tail, _ = r.gpt_eval(1, full[cut:], cut, False)
            assert np.array_equal(tail.view(np.uint32), scratch.view(np.uint32)), (ftype, cut)
        out[f"prefix_rows_{ftype}_sha1"] = np.array(sha(scratch))
        r.close()

    # ---- tests/test_quantize.py
    keep = orc.Ref(wfile("tiny", "f16"))            # ggml_init fills the f16 tables the reference's quantizer relies on
    R = C.CDLL(orc.REF_SO)
    R.bark_model_quantize.restype = C.c_bool
    R.bark_model_quantize.argtypes = [C.c_char_p, C.c_char_p, C.c_int]
    with tempfile.TemporaryDirectory() as d:
        for config, src_ftype in QUANT_CONFIGS:
            src = wfile(config, src_ftype)
            for qname, ftype_id in sorted(QUANT_FTYPES.items()):
                key = f"quant_{config}_{src_ftype}_{qname}"
                ref_out = os.path.join(d, "ref.bin")
                devnull, saved = os.open(os.devnull, os.O_WRONLY), os.dup(1)
                os.dup2(devnull, 1)                              # the reference prints one line per tensor
                try:
                    assert R.bark_model_quantize(src.encode(), ref_out.encode(), ftype_id)
                finally:
                    os.dup2(saved, 1); os.close(devnull); os.close(saved)
                data = open(ref_out, "rb").read()
                out[f"{key}_file_sha1"], out[f"{key}_file_size"] = np.array(hashlib.sha1(data).hexdigest()), np.array(len(data))
                # the oracle test runs on the library's quantised file; it must be the reference tool's byte for byte
                path = os.path.join(d, f"{qname}.bin")
                assert pkg.lib().bark_model_quantize(src.encode(), path.encode(), ftype_id)
                assert open(path, "rb").read() == data, key
                r = orc.Ref(path, seed=0, n_steps=10)
                rng = np.random.default_rng(17)
                toks, n_past, shas = r.tokenize("Hello, world"), 0, []
                for _ in range(4):
                    lg, n_past = r.gpt_eval(0, toks, n_past, True)
                    shas.append(sha(lg))
                    toks = np.array([int(np.argmax(lg[:10000]))], np.int32)
                out[f"{key}_semantic_sha1"] = np.array(shas)
                toks = np.concatenate([rng.integers(0, 10000, 256), [12050], rng.integers(10000, 12048, 21)]).astype(np.int32)
                n_past, shas = 0, []
                for _ in range(3):
                    lg, n_past = r.gpt_eval(1, toks, n_past, False)
                    shas.append(sha(lg))
                    toks = np.array([10000 + int(np.argmax(lg[10000:12048]))], np.int32)
                out[f"{key}_coarse_sha1"] = np.array(shas)
                buf = rng.integers(0, 1024, (8, 1024)).astype(np.int32); buf[:, 300:] = 1024; buf[4:, :] = 1024
                out[f"{key}_fine_sha1"] = np.array(sha(r.fine_eval(buf, 4)))
                g = r.generate("hello world")
                for k in ("semantic", "coarse", "fine"):
                    out[f"{key}_generate_{k}"] = g[k]
                out[f"{key}_generate_audio_sha1"] = np.array(sha(g["audio"]))
                r.close()
                print(key, "semantic", g["semantic"].size, "frames", g["coarse"].shape[0], flush=True)
    keep.close()

    # ---- tests/test_parity_gpu.py::test_full_size_against_the_reference_itself: bark-small f16, seed 0, n_steps 12
    r = orc.Ref(wfile("small", "f16"), seed=0, n_steps=12)
    prompt = r.tokenize("hello world")
    out["small_prompt_ids"] = prompt
    toks, n_past, shas, heads = prompt, 0, [], []
    for _ in range(6):
        lg, n_past = r.gpt_eval(0, toks, n_past, True, n_threads=8)
        shas.append(sha(lg)); heads.append(lg[:HEAD])
        toks = np.array([int(np.argmax(lg[:10000]))], np.int32)
    out["small_semantic_sha1"], out["small_semantic_head"] = np.array(shas), np.stack(heads)
    g = r.generate("hello world", n_threads=8)
    for k in ("semantic", "coarse", "fine", "audio"):
        out[f"small_generate_{k}"] = g[k]
    out["reference_build"] = np.array(r.build_info())
    r.close()

    dst = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_checks.npz")
    np.savez_compressed(dst, **out)
    print(dst, os.path.getsize(dst), "bytes", len(out), "arrays")


if __name__ == "__main__":
    main()
