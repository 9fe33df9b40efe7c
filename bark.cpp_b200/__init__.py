"""ctypes binding of libbark_b200.so — the B200-native drop-in for bark.cpp's hot path.

The product is the C-ABI shared library (include/bark.h, include/bark_b200.h); this module only
loads it and mirrors the reference's call sequence (bark_context_default_params -> bark_load_model
-> bark_generate_audio -> bark_get_audio_data -> bark_free, examples/main/main.cpp:49-91) for the
Python-side tests and the benchmark.  There is no CPU path: loading fails loudly when the CUDA
extension has not been built, and bark_load_model fails when no sm_100 device is present.

The directory name contains a dot, so import it through `__graft_entry__.load_package()`.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbark_b200.so")

PROGRESS_CB = C.CFUNCTYPE(None, C.c_void_p, C.c_int, C.c_int, C.c_void_p)


class BarkContextParams(C.Structure):
    """struct bark_context_params (include/bark.h; reference bark.h:81-141) — passed by value."""
    _fields_ = [
        ("verbosity", C.c_int), ("temp", C.c_float), ("fine_temp", C.c_float), ("min_eos_p", C.c_float),
        ("sliding_window_size", C.c_int32), ("max_coarse_history", C.c_int32), ("sample_rate", C.c_int32),
        ("target_bandwidth", C.c_int32), ("cls_token_id", C.c_int32), ("sep_token_id", C.c_int32),
        ("n_steps_text_encoder", C.c_int32), ("text_pad_token", C.c_int32), ("text_encoding_offset", C.c_int32),
        ("semantic_rate_hz", C.c_float), ("semantic_pad_token", C.c_int32), ("semantic_vocab_size", C.c_int32),
        ("semantic_infer_token", C.c_int32), ("coarse_rate_hz", C.c_float), ("coarse_infer_token", C.c_int32),
        ("coarse_semantic_pad_token", C.c_int32), ("n_coarse_codebooks", C.c_int32), ("n_fine_codebooks", C.c_int32),
        ("codebook_size", C.c_int32), ("progress_callback", PROGRESS_CB), ("progress_callback_user_data", C.c_void_p),
    ]


class BarkStatistics(C.Structure):
    _fields_ = [("t_load_us", C.c_int64), ("t_eval_us", C.c_int64), ("t_semantic_us", C.c_int64), ("t_coarse_us", C.c_int64),
                ("t_fine_us", C.c_int64), ("n_sample_semantic", C.c_int32), ("n_sample_coarse", C.c_int32), ("n_sample_fine", C.c_int32)]


# every symbol the two public headers declare (tests check the library exports exactly these)
EXPORTS = [
    "bark_context_default_params", "bark_load_model", "bark_generate_audio", "bark_get_audio_data", "bark_get_audio_data_size",
    "bark_get_load_time", "bark_get_eval_time", "bark_reset_statistics", "bark_model_quantize", "bark_free",
    "bark_b200_set_device", "bark_b200_version", "bark_b200_gpt_eval", "bark_b200_fine_eval", "bark_b200_encodec_decode",
    "bark_b200_sample", "bark_b200_sample_rows", "bark_b200_reseed", "bark_b200_tokenize", "bark_b200_forward_text_encoder",
    "bark_b200_forward_coarse_encoder", "bark_b200_forward_fine_encoder", "bark_b200_get_tokens", "bark_b200_set_tokens",
    "bark_b200_get_stats", "bark_b200_get_hparams", "bark_b200_kernel_launches", "bark_b200_layernorm_fallbacks",
    "bark_b200_profile_enable", "bark_b200_profile_report", "bark_b200_io_counters", "bark_b200_decode_timing", "bark_b200_decode_adapt",
    "bark_b200_shard_init", "bark_b200_shard_connect", "bark_b200_shard_nvlink_bytes",
    "bark_b200_fast_mode", "bark_b200_fast_gemm", "bark_b200_fast_attention",
    "bark_b200_generate_audio_batch", "bark_b200_batch_audio", "bark_b200_batch_tokens", "bark_b200_batch_eval", "bark_b200_batch_stats",
    "ggml_time_init", "ggml_time_us", "ggml_time_ms", "ggml_init", "ggml_free",
]

_lib = None


def lib() -> C.CDLL:
    """Load libbark_b200.so (built by `make -C bark.cpp_b200` / __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: build the CUDA extension first (python -c 'import __graft_entry__ as g; g.build()'). "
                           "There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i32p, f32p = C.c_void_p, C.c_void_p, C.c_void_p
    L.bark_context_default_params.restype = BarkContextParams
    L.bark_load_model.restype = vp
    L.bark_load_model.argtypes = [C.c_char_p, BarkContextParams, C.c_uint32]
    L.bark_generate_audio.restype = C.c_bool
    L.bark_generate_audio.argtypes = [vp, C.c_char_p, C.c_int]
    L.bark_get_audio_data.restype = C.POINTER(C.c_float)
    L.bark_get_audio_data.argtypes = [vp]
    L.bark_get_audio_data_size.restype = C.c_int
    L.bark_get_audio_data_size.argtypes = [vp]
    for n in ("bark_get_load_time", "bark_get_eval_time"):
        getattr(L, n).restype = C.c_int64
        getattr(L, n).argtypes = [vp]
    L.bark_reset_statistics.argtypes = [vp]
    L.bark_model_quantize.restype = C.c_bool
    L.bark_model_quantize.argtypes = [C.c_char_p, C.c_char_p, C.c_int]
    L.bark_free.argtypes = [vp]
    L.bark_b200_set_device.argtypes = [C.c_int]
    L.bark_b200_version.restype = C.c_char_p
    L.bark_b200_gpt_eval.restype = C.c_int
    L.bark_b200_gpt_eval.argtypes = [vp, C.c_int, i32p, C.c_int, C.POINTER(C.c_int), C.c_int, f32p]
    L.bark_b200_fine_eval.restype = C.c_int
    L.bark_b200_fine_eval.argtypes = [vp, i32p, C.c_int, f32p]
    L.bark_b200_encodec_decode.restype = C.c_int
    L.bark_b200_encodec_decode.argtypes = [vp, i32p, C.c_int, f32p, C.c_int]
    L.bark_b200_sample.restype = C.c_int
    L.bark_b200_sample.argtypes = [vp, C.c_int, f32p, C.c_int, C.c_float, C.POINTER(C.c_float)]
    L.bark_b200_sample_rows.restype = C.c_int
    L.bark_b200_sample_rows.argtypes = [vp, f32p, C.c_int, C.c_int, C.c_float, i32p, f32p]
    L.bark_b200_reseed.argtypes = [vp, C.c_uint32]
    L.bark_b200_tokenize.argtypes = [vp, C.c_char_p, i32p]
    for n in ("bark_b200_forward_text_encoder", "bark_b200_forward_coarse_encoder", "bark_b200_forward_fine_encoder"):
        getattr(L, n).restype = C.c_bool
        getattr(L, n).argtypes = [vp, C.c_int]
    L.bark_b200_get_tokens.restype = C.c_int
    L.bark_b200_get_tokens.argtypes = [vp, C.c_int, i32p, C.c_int]
    L.bark_b200_set_tokens.argtypes = [vp, C.c_int, i32p, C.c_int]
    L.bark_b200_get_stats.argtypes = [vp, C.POINTER(BarkStatistics), C.c_void_p]
    L.bark_b200_get_hparams.argtypes = [vp, C.c_int, i32p]
    L.bark_b200_kernel_launches.restype = C.c_ulonglong
    L.bark_b200_layernorm_fallbacks.restype = C.c_uint
    L.bark_b200_layernorm_fallbacks.argtypes = [vp]
    L.bark_b200_profile_enable.argtypes = [C.c_int]
    L.bark_b200_profile_report.restype = C.c_int
    L.bark_b200_profile_report.argtypes = [C.c_char_p, C.c_int]
    L.bark_b200_io_counters.argtypes = [C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong), C.c_int]
    L.bark_b200_decode_timing.restype = C.c_int
    L.bark_b200_decode_timing.argtypes = [vp, C.c_void_p, C.c_int]
    L.bark_b200_decode_adapt.restype = C.c_int
    L.bark_b200_decode_adapt.argtypes = [vp, C.c_int, C.c_void_p, C.c_int]
    L.bark_b200_shard_init.restype = C.c_int
    L.bark_b200_shard_init.argtypes = [vp, C.c_int, C.c_int, vp]
    L.bark_b200_shard_connect.restype = C.c_int
    L.bark_b200_shard_connect.argtypes = [vp, vp]
    L.bark_b200_shard_nvlink_bytes.restype = C.c_ulonglong
    L.bark_b200_shard_nvlink_bytes.argtypes = [vp, C.c_int]
    L.bark_b200_fast_mode.restype = C.c_int
    L.bark_b200_fast_mode.argtypes = [vp]
    L.bark_b200_fast_gemm.restype = C.c_int
    L.bark_b200_fast_gemm.argtypes = [vp, vp, vp, C.c_int, C.c_int, C.c_int]
    L.bark_b200_fast_attention.restype = C.c_int
    L.bark_b200_fast_attention.argtypes = [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int]
    L.bark_b200_generate_audio_batch.restype = C.c_bool
    L.bark_b200_generate_audio_batch.argtypes = [vp, C.POINTER(C.c_char_p), C.POINTER(C.c_uint32), C.c_int]
    L.bark_b200_batch_audio.restype = C.c_int
    L.bark_b200_batch_audio.argtypes = [vp, C.c_int, f32p, C.c_int]
    L.bark_b200_batch_tokens.restype = C.c_int
    L.bark_b200_batch_tokens.argtypes = [vp, C.c_int, C.c_int, i32p, C.c_int]
    L.bark_b200_batch_eval.restype = C.c_int
    L.bark_b200_batch_eval.argtypes = [vp, C.c_int, C.c_int, i32p, C.c_int, i32p, C.c_int, f32p]
    L.bark_b200_batch_stats.restype = C.c_int
    L.bark_b200_batch_stats.argtypes = [vp, C.c_void_p]
    L.ggml_time_us.restype = C.c_int64
    _lib = L
    return L


def _p(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


class Bark:
    """One bark_context on one GPU.  Mirrors how examples/main/main.cpp uses bark.h."""

    def __init__(self, model_path: str, seed: int = 0, n_steps_text_encoder: int | None = None, temp=None, fine_temp=None,
                 min_eos_p=None, device: int | None = None, progress=None):
        L = lib()
        p = L.bark_context_default_params()
        if n_steps_text_encoder is not None:
            p.n_steps_text_encoder = n_steps_text_encoder
        if temp is not None:
            p.temp = temp
        if fine_temp is not None:
            p.fine_temp = fine_temp
        if min_eos_p is not None:
            p.min_eos_p = min_eos_p
        self._cb = PROGRESS_CB(progress) if progress else PROGRESS_CB()
        p.progress_callback = self._cb
        if device is not None:
            L.bark_b200_set_device(device)
        self.params = p
        self.ctx = L.bark_load_model(os.fsencode(model_path), p, seed)
        if not self.ctx:
            raise RuntimeError(f"bark_load_model failed for {model_path} (see stderr); no CPU fallback exists")
        self.ctx = C.c_void_p(self.ctx)

    def close(self):
        if getattr(self, "ctx", None):
            lib().bark_free(self.ctx)
            self.ctx = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- bark.h ----
    def generate(self, text: str, n_threads: int = 1) -> np.ndarray:
        if not lib().bark_generate_audio(self.ctx, text.encode(), n_threads):
            raise RuntimeError("bark_generate_audio failed")
        n = lib().bark_get_audio_data_size(self.ctx)
        return np.ctypeslib.as_array(lib().bark_get_audio_data(self.ctx), shape=(n,)).copy()

    @property
    def load_time_us(self):
        return lib().bark_get_load_time(self.ctx)

    @property
    def eval_time_us(self):
        return lib().bark_get_eval_time(self.ctx)

    # ---- bark_b200.h ----
    def hparams(self, which: int) -> np.ndarray:
        a = np.zeros(10, np.int32)
        lib().bark_b200_get_hparams(self.ctx, which, _p(a))
        return a

    def tokens(self, stage: int) -> np.ndarray:
        n = lib().bark_b200_get_tokens(self.ctx, stage, None, 0)
        a = np.zeros(max(n, 1), np.int32)
        lib().bark_b200_get_tokens(self.ctx, stage, _p(a), n)
        a = a[:n]
        return a.reshape(-1, 2) if stage == 1 else a.reshape(-1, 8) if stage == 2 else a

    def set_tokens(self, stage: int, arr):
        a = np.ascontiguousarray(arr, np.int32).ravel()
        lib().bark_b200_set_tokens(self.ctx, stage, _p(a), a.size)

    def tokenize(self, text: str) -> np.ndarray:
        a = np.zeros(513, np.int32)
        lib().bark_b200_tokenize(self.ctx, text.encode(), _p(a))
        return a

    def gpt_eval(self, which: int, tokens, n_past: int, merge_ctx: bool):
        t = np.ascontiguousarray(tokens, np.int32)
        out = np.zeros(int(self.hparams(which)[6]), np.float32)
        np_ = C.c_int(n_past)
        if not lib().bark_b200_gpt_eval(self.ctx, which, _p(t), t.size, C.byref(np_), int(merge_ctx), _p(out)):
            raise RuntimeError("bark_b200_gpt_eval failed")
        return out, np_.value

    def fine_eval(self, in_buffer, nn: int) -> np.ndarray:
        t = np.ascontiguousarray(in_buffer, np.int32)
        assert t.size == 8 * 1024
        out = np.zeros((1024, int(self.hparams(2)[6])), np.float32)
        if not lib().bark_b200_fine_eval(self.ctx, _p(t), nn, _p(out)):
            raise RuntimeError("bark_b200_fine_eval failed")
        return out

    def encodec_decode(self, codes_8xT) -> np.ndarray:
        c = np.ascontiguousarray(codes_8xT, np.int32)
        T = c.shape[1]
        out = np.zeros(320 * T, np.float32)
        n = lib().bark_b200_encodec_decode(self.ctx, _p(c), T, _p(out), out.size)
        if n < 0:
            raise RuntimeError("bark_b200_encodec_decode failed")
        return out[:n]

    def sample(self, which: int, logits, temp: float):
        l = np.ascontiguousarray(logits, np.float32)
        e = C.c_float(0)
        return lib().bark_b200_sample(self.ctx, which, _p(l), l.size, temp, C.byref(e)), e.value

    def sample_rows(self, logits_rows, temp: float):
        """Device sampler over [rows][n] logits; returns (tokens, eos_p, n_rows_replayed_on_host)."""
        l = np.ascontiguousarray(logits_rows, np.float32)
        rows, n = l.shape
        tok = np.zeros(rows, np.int32); eos = np.zeros(rows, np.float32)
        r = lib().bark_b200_sample_rows(self.ctx, _p(l), n, rows, temp, _p(tok), _p(eos))
        if r < 0:
            raise RuntimeError("bark_b200_sample_rows failed")
        return tok, eos, r

    def reseed(self, seed: int):
        lib().bark_b200_reseed(self.ctx, seed)

    def forward(self, stage: int):
        f = [lib().bark_b200_forward_text_encoder, lib().bark_b200_forward_coarse_encoder, lib().bark_b200_forward_fine_encoder][stage]
        if not f(self.ctx, 1):
            raise RuntimeError("stage failed")

    def stats(self):
        s = BarkStatistics()
        pm = np.zeros(9, np.int64)
        lib().bark_b200_get_stats(self.ctx, C.byref(s), _p(pm))
        return s, pm.reshape(3, 3)

    def shard_init(self, rank: int, world: int) -> bytes:
        """Row-sharded fine stage, step 1: returns this rank's 64-byte CUDA IPC handle."""
        h = C.create_string_buffer(64)
        if not lib().bark_b200_shard_init(self.ctx, rank, world, C.cast(h, C.c_void_p)):
            raise RuntimeError("bark_b200_shard_init failed")
        return h.raw

    def shard_connect(self, all_handles: bytes):
        """step 2: all ranks' handles, rank order (world * 64 bytes)."""
        buf = C.create_string_buffer(all_handles, len(all_handles))
        if not lib().bark_b200_shard_connect(self.ctx, C.cast(buf, C.c_void_p)):
            raise RuntimeError("bark_b200_shard_connect failed")

    def shard_nvlink_bytes(self, reset: bool = False) -> int:
        return int(lib().bark_b200_shard_nvlink_bytes(self.ctx, int(reset)))

    @property
    def fast_mode(self) -> bool:
        return bool(lib().bark_b200_fast_mode(self.ctx))

    def layernorm_fallbacks(self) -> int:
        return int(lib().bark_b200_layernorm_fallbacks(self.ctx))

    # ---- batched generation ----
    def generate_batch(self, texts, seeds):
        """Several prompts on this context's GPU in one call; item i equals a fresh context with seed seeds[i] generating texts[i].
        Returns [(audio, [semantic, coarse, fine]), ...]; the context's own RNG and outputs are left as they were."""
        n = len(texts)
        if len(seeds) != n:
            raise ValueError("one seed per prompt")
        t = (C.c_char_p * n)(*[s.encode() for s in texts])
        sd = (C.c_uint32 * n)(*seeds)
        if not lib().bark_b200_generate_audio_batch(self.ctx, t, sd, n):
            raise RuntimeError("bark_b200_generate_audio_batch failed (see stderr)")
        out = []
        for i in range(n):
            m = lib().bark_b200_batch_audio(self.ctx, i, None, 0)
            audio = np.zeros(m, np.float32)
            lib().bark_b200_batch_audio(self.ctx, i, _p(audio), m)
            toks = []
            for stage in range(3):
                k = lib().bark_b200_batch_tokens(self.ctx, i, stage, None, 0)
                a = np.zeros(max(k, 1), np.int32)
                lib().bark_b200_batch_tokens(self.ctx, i, stage, _p(a), k)
                a = a[:k]
                toks.append(a.reshape(-1, 2) if stage == 1 else a.reshape(-1, 8) if stage == 2 else a)
            out.append((audio, toks))
        return out

    def batch_eval(self, which: int, prompts, next_ids) -> np.ndarray:
        """Teacher-forced batched decode: prompts [n][len] into per-item caches, then next_ids [n][steps] as batched steps;
        returns logits [n][steps][n_out_vocab]."""
        p = np.ascontiguousarray(prompts, np.int32); x = np.ascontiguousarray(next_ids, np.int32)
        n, ln = p.shape; steps = x.shape[1]
        out = np.zeros((n, steps, int(self.hparams(which)[6])), np.float32)
        if not lib().bark_b200_batch_eval(self.ctx, which, n, _p(p), ln, _p(x), steps, _p(out)):
            raise RuntimeError("bark_b200_batch_eval failed")
        return out

    def batch_stats(self) -> dict:
        """The last batch call: per-stage microseconds, batched decode steps, sampled rows replayed on the host."""
        a = np.zeros(6, np.int64)
        lib().bark_b200_batch_stats(self.ctx, _p(a))
        return dict(zip(("semantic_us", "coarse_us", "fine_us", "codec_us", "batched_steps", "host_replays"), (int(v) for v in a)))


def fast_gemm(A: np.ndarray, W: np.ndarray) -> np.ndarray:
    """C = A W^T on the tcgen05 path; A [M][K], W [N][K] float16."""
    A = np.ascontiguousarray(A, np.float16); W = np.ascontiguousarray(W, np.float16)
    M, K = A.shape; N = W.shape[0]
    out = np.zeros((M, N), np.float32)
    if not lib().bark_b200_fast_gemm(_p(A), _p(W), _p(out), M, N, K):
        raise RuntimeError("bark_b200_fast_gemm failed")
    return out


def fast_attention(q: np.ndarray, k: np.ndarray, v: np.ndarray, n_head: int) -> np.ndarray:
    """Non-causal attention on the tcgen05 path; q, k, v [n][E] float16 -> [n][E] float16."""
    q, k, v = (np.ascontiguousarray(a, np.float16) for a in (q, k, v))
    n, E = q.shape
    out = np.zeros((n, E), np.float16)
    if not lib().bark_b200_fast_attention(_p(q), _p(k), _p(v), _p(out), n, E, n_head):
        raise RuntimeError("bark_b200_fast_attention failed")
    return out


def kernel_launches() -> int:
    return int(lib().bark_b200_kernel_launches())


def profile_enable(on: bool):
    lib().bark_b200_profile_enable(int(on))


def profile_report() -> dict:
    import json
    n = lib().bark_b200_profile_report(None, 0)
    buf = C.create_string_buffer(n + 16)
    lib().bark_b200_profile_report(buf, n + 16)
    return json.loads(buf.value.decode())


def io_counters(reset: bool = False):
    a, b = C.c_ulonglong(0), C.c_ulonglong(0)
    lib().bark_b200_io_counters(C.byref(a), C.byref(b), int(reset))
    return a.value, b.value
