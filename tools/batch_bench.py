#!/usr/bin/env python3
"""Batched generation (bark_b200_generate_audio_batch) against the same items generated one after another, on one GPU.

Workload: the bench's (bark-small f16 synthetic weights, n_steps_text_encoder = 138; item i = seed i with "hello world" /
"hello world {i}", bench.py rank_workload).  For each batch size B: one warm-up batch call, then `--rounds` rounds that alternate
one timed batch call (host clock around the C call, which ends in a synchronise) with the same B items generated one after another
on a single-prompt context (reseeded per item: the seed is the only state a generation carries).  Every item is asserted
bit-identical between the two.  Reported per B: aggregate audio s/s of both, the per-stage split, launches per batched decode step,
and — from a separate profiled batch call — the device time of batch_decode_attention and its achieved GB/s.  Then the same for the
fast-mode fine stage (BARK_B200_MODE=fast).  Prints one JSON document (and writes it to --out when given).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("BARK_B200_QUIET", "1")

import numpy as np  # noqa: E402

import __graft_entry__ as graft  # noqa: E402
import bench  # noqa: E402

SR = 24000


def gpu_info():
    try:
        q = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,power.max_limit", "--format=csv,noheader", "-i", "0"], text=True, timeout=30)
        name, limit, max_limit = [s.strip() for s in q.strip().split(",")]
        return dict(name=name, power_limit=limit, power_max_limit=max_limit)
    except Exception as e:  # the measurement stands without it, but says so
        return dict(error=str(e))


def launches_per_step(pkg, b, B):
    """kernel launches of one batched decode step (teacher-forced coarse steps at n_kv ~ 300), from two step counts"""
    rng = np.random.default_rng(0)
    p = rng.integers(0, 12048, (B, 300)).astype(np.int32)
    counts = []
    for steps in (2, 6):
        x = rng.integers(10000, 12048, (B, steps)).astype(np.int32)
        l0 = pkg.kernel_launches()
        b.batch_eval(1, p, x)
        counts.append(pkg.kernel_launches() - l0)
    return (counts[1] - counts[0]) / 4


def run_mode(pkg, path, n_steps, sizes, rounds):
    L = pkg.lib()
    bb = pkg.Bark(path, seed=0, n_steps_text_encoder=n_steps)
    single = pkg.Bark(path, seed=0, n_steps_text_encoder=n_steps)
    rows = []
    try:
        for B in sizes:
            wl = [bench.rank_workload(i) for i in range(B)]
            texts, seeds = [w["prompt"] for w in wl], [w["seed"] for w in wl]
            bb.generate_batch(texts, seeds)                         # warm-up (allocates the per-item caches)
            t_batch, t_seq, stages_b, stages_s = [], [], [], []
            for _ in range(rounds):
                ct = (C.c_char_p * B)(*[t.encode() for t in texts]); cs = (C.c_uint32 * B)(*seeds)
                t0 = time.perf_counter()
                ok = L.bark_b200_generate_audio_batch(bb.ctx, ct, cs, B)
                t_batch.append(time.perf_counter() - t0)
                assert ok
                stages_b.append(bb.batch_stats())
                got = [None] * B
                t0 = time.perf_counter()
                for i in range(B):
                    single.reseed(seeds[i])
                    a = single.generate(texts[i])
                    got[i] = (a, [single.tokens(k).copy() for k in range(3)])
                t_seq.append(time.perf_counter() - t0)
                s, _ = single.stats()
                stages_s.append(dict(semantic_us=s.t_semantic_us, coarse_us=s.t_coarse_us, fine_us=s.t_fine_us))
                for i in range(B):
                    n = L.bark_b200_batch_audio(bb.ctx, i, None, 0)
                    ab = np.zeros(n, np.float32); L.bark_b200_batch_audio(bb.ctx, i, ab.ctypes.data_as(C.c_void_p), n)
                    assert ab.shape == got[i][0].shape and np.array_equal(ab.view(np.uint32), got[i][0].view(np.uint32)), f"B={B} item {i}: waveform differs"
                    for k in range(3):
                        m = L.bark_b200_batch_tokens(bb.ctx, i, k, None, 0)
                        tb = np.zeros(max(m, 1), np.int32); L.bark_b200_batch_tokens(bb.ctx, i, k, tb.ctypes.data_as(C.c_void_p), m)
                        assert np.array_equal(tb[:m], got[i][1][k].ravel()), f"B={B} item {i}: stage {k} ids differ"
            audio_s = sum(g[0].size for g in got) / SR
            pkg.profile_enable(True)
            bb.generate_batch(texts, seeds)
            prof = pkg.profile_report()
            pkg.profile_enable(False)
            att = {k: v for k, v in prof.items() if k.startswith("batch_decode_attention")}
            att_ms = sum(v["ms"] for v in att.values()); att_bytes = sum(v["bytes"] for v in att.values()); att_n = sum(v["launches"] for v in att.values())
            st = stages_b[-1]
            rows.append(dict(
                B=B, audio_s=round(audio_s, 3), identical=True,
                batch_s=[round(t, 4) for t in t_batch], sequential_s=[round(t, 4) for t in t_seq],
                batch_audio_s_per_s=round(audio_s / min(t_batch), 2), sequential_audio_s_per_s=round(audio_s / min(t_seq), 2),
                speedup=round(min(t_seq) / min(t_batch), 3),
                batch_stage_ms={k[:-3]: round(st[k] / 1e3, 1) for k in ("semantic_us", "coarse_us", "fine_us", "codec_us")},
                batched_steps=st["batched_steps"], host_replays=st["host_replays"],
                batch_decode_ms_per_step=round((st["semantic_us"] + st["coarse_us"]) / 1e3 / max(st["batched_steps"], 1), 3),
                sequential_last_item_stage_ms={k[:-3]: round(v / 1e3, 1) for k, v in stages_s[-1].items()},
                launches_per_batched_step=launches_per_step(pkg, bb, B),
                batch_decode_attention=dict(launches=att_n, device_ms=round(att_ms, 3), us_per_launch=round(1e3 * att_ms / max(att_n, 1), 2),
                                            gb_per_s=round(att_bytes / (att_ms * 1e-3) / 1e9, 1) if att_ms else None),
                profiled_total_device_ms=round(sum(v["ms"] for v in prof.values()), 2),
            ))
            print(json.dumps(rows[-1]), file=sys.stderr, flush=True)
    finally:
        bb.close(); single.close()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1,2,4,8,16,32")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--fast-sizes", default="1,8,32")
    ap.add_argument("--out")
    a = ap.parse_args()
    pkg = graft.load_package()
    path = bench.weights_path()
    n_steps = bench.N_STEPS_TEXT
    res = dict(workload=f"{bench.BENCH_CONFIG} f16 synthetic weights, n_steps_text_encoder={n_steps}, item i = seed i / bench prompt i",
               gpu=gpu_info())
    os.environ.pop("BARK_B200_MODE", None)
    res["parity"] = run_mode(pkg, path, n_steps, [int(s) for s in a.sizes.split(",")], a.rounds)
    os.environ["BARK_B200_MODE"] = "fast"                      # read at bark_load_model
    res["fast"] = run_mode(pkg, path, n_steps, [int(s) for s in a.fast_sizes.split(",")], a.rounds)
    os.environ.pop("BARK_B200_MODE", None)
    res["gpu_after"] = gpu_info()
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
