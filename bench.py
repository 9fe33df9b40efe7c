#!/usr/bin/env python
"""bench.py — throughput of the bark.cpp hot path on B200 (driver contract: one JSON line from rank 0).

  python bench.py --gpus N --steps K --warmup W            our CUDA path through the C-ABI (libbark_b200.so)
  python bench.py --impl reference --gpus N --steps K ...  the reference's own CPU path (oracle/_ref) on the host cores
  --dump-outputs DIR                                         also write what the last timed step returned as DIR/<name>.npy

Workload (BASELINE.json configs[1]): bark-small dimensions, f16 GPT + f16 codec, batch 1 per GPU, full
semantic -> coarse -> fine -> EnCodec, synthetic seeded weights (no checkpoint is reachable offline), prompt
"hello world", seed 0, n_steps_text_encoder = 138 -> 138 semantic / 414 coarse / 6144 fine samples, 207 frames,
66 240 samples = 2.76 s of 24 kHz audio (the README-sized clip of BASELINE.md).  One "step" = one
bark_generate_audio call.  metric = audio seconds produced per wall second (inverse RTF); per-stage tokens/s
ride along.  N > 1: one context per GPU, distinct prompt seeds, no collective on the data path (SURVEY §8e:
prompts are independent units) -> weak scaling, value = N clips / max-over-ranks time.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("BARK_B200_QUIET", "1")

import numpy as np  # noqa: E402

import __graft_entry__ as graft  # noqa: E402

UNIT = "audio_s/s"
# --config: which BASELINE.json config the line measures (metric text and workload name follow it)
BENCH_CONFIGS = {
    "small":      dict(dims="small", ftype="f16", quant=None,   label="bark-small f16",                          baseline="BASELINE configs[1]"),
    "large":      dict(dims="large", ftype="f16", quant=None,   label="bark-large f16",                          baseline="BASELINE configs[2] (one prompt per GPU)"),
    "small_q4_0": dict(dims="small", ftype="f16", quant="q4_0", label="bark-small q4_0 GPT weights + f16 codec", baseline="BASELINE configs[3]"),
    "fine_only":  dict(dims="small", ftype="f16", quant=None,   label="fine encoder only, bark-small f16, 6144 sampled tokens (one 1024-frame window x 6 codebook passes), rows of the window sharded over the GPUs",
                       baseline="BASELINE configs[4]"),
    "tiny":       dict(dims="tiny",  ftype="f16", quant=None,   label="tiny test config f16",                    baseline="test plumbing only"),
}
def metric_name(cfg):
    return f"audio sec/sec (inverse RTF), {BENCH_CONFIGS[cfg]['label']}, batch 1 per GPU, semantic->coarse->fine->encodec"
PROMPT = "hello world"
N_STEPS_TEXT = 138
# the C oracle's bounded sample: 6 semantic steps -> 9 frames; 4 steps would give 6 frames, no more than the reflect padding of
# the codec's first convolution (kernel 7), which the reference (ggml_pad_reflect_1d) and the oracle both reject
PORT_STEPS = 6
SAMPLE_RATE = 24000
# generated weight files, cached between runs; per user, since another user's directory of the same name is not writable
FIXTURE_DIR = os.environ.get("BARK_B200_FIXTURES") or os.path.join(tempfile.gettempdir(), f"bark_b200_fixtures_{os.getuid()}")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], tflops=d.get("bf16_tflops_sustained", d["bf16_tflops"]), tflops_burst=d["bf16_tflops"], source="measured")
    return dict(hbm_gbs=6650.0, tflops=1400.0, tflops_burst=1590.0, source="fallback")


def measured_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed `ncu --set full` capture (profiles/, tools/summarize_ncu.py traffic); None if not captured"""
    p = os.path.join(ROOT, "profiles", "r02_decode_traffic.json")
    if not os.path.exists(p):
        p = os.path.join(ROOT, "profiles", "r01_decode_traffic.json")
    if os.path.exists(p):
        d = json.load(open(p))
        if d.get("kernel", "").split("<")[0] == kernel.split("<")[0]:
            return int(d["traffic_bytes"])
    return None


# tests/test_bench_contract.py sets this to "tiny" to exercise the reference arm's plumbing in seconds; every real run uses bark-small
BENCH_CONFIG = os.environ.get("BARK_B200_BENCH_CONFIG", "small")


def weights_path(config=None, ftype="f16", seed=1234):
    """Synthetic ggml_weights.bin of a bench config (written once per box).  Quantised configs are made from the f16 file by the
    library's own bark_model_quantize, which is byte-identical to the reference tool (tests/test_quantize.py)."""
    config = config or BENCH_CONFIG
    spec = BENCH_CONFIGS.get(config, dict(dims=config, ftype=ftype, quant=None))
    import importlib
    pkg = graft.load_package()
    weights = importlib.import_module("bark_cpp_b200.weights")
    os.makedirs(FIXTURE_DIR, exist_ok=True)
    path = os.path.join(FIXTURE_DIR, f"{spec['dims']}_{spec['ftype']}_{seed}.bin")
    if not os.path.exists(path):
        tmp = path + f".tmp{os.getpid()}"
        weights.write_weights(tmp, weights.CONFIGS[spec["dims"]](weights.F16 if spec["ftype"] == "f16" else weights.F32), seed)
        os.replace(tmp, path)
    if spec.get("quant"):
        qpath = os.path.join(FIXTURE_DIR, f"{spec['dims']}_{spec['quant']}_{seed}.bin")
        if not os.path.exists(qpath):
            tmp = qpath + f".tmp{os.getpid()}"
            ftype_id = {"q4_0": 2, "q4_1": 3, "q5_0": 8, "q5_1": 9, "q8_0": 7}[spec["quant"]]      # enum ggml_ftype (include/ggml.h)
            if not pkg.lib().bark_model_quantize(os.fsencode(path), os.fsencode(tmp), ftype_id):
                raise RuntimeError("bark_model_quantize failed")
            os.replace(tmp, qpath)
        path = qpath
    return path


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, device=0):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


def dist_env():
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def pin_to_gpu_numa(device):
    """Bind this process to the CPUs local to its GPU (sysfs local_cpulist of the GPU's PCI function).  At N = 8 each rank issues
    ~3 k launches per clip; ranks scheduled on the far socket paid ~4 % (SCALE_r01).  Returns the CPU list string or None."""
    try:
        bus = subprocess.run(["nvidia-smi", f"--id={device}", "--query-gpu=pci.bus_id", "--format=csv,noheader"], capture_output=True, text=True, timeout=20).stdout.strip()
        if not bus:
            return None
        dom, rest = bus.split(":", 1)
        sysfs = f"/sys/bus/pci/devices/{dom[-4:].lower()}:{rest.lower()}/local_cpulist"
        cpus = set()
        txt = open(sysfs).read().strip()
        for part in txt.split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return txt
    except Exception:
        pass
    return None


def rank_workload(rank):
    """The path shards by prompt (SURVEY §8e): every rank owns one independent clip, its own seed and prompt; no data-path collective."""
    return dict(seed=rank, prompt=PROMPT if rank == 0 else f"{PROMPT} {rank}")


def reduce_over_ranks(dist, elapsed, n_audio, device):
    """Whole-job figures: time = MAX over ranks, audio = SUM over ranks (works on nccl/cuda and gloo/cpu alike)."""
    if dist is None:
        return float(elapsed), float(n_audio)
    import torch
    t = torch.tensor([elapsed], device=device, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    tot = torch.tensor([float(n_audio)], device=device, dtype=torch.float64)
    dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    return float(t.item()), float(tot.item())


def algorithmic_work(pkg_bark):
    """Per-clip algorithmic bytes / flops of the two roofline regimes (SURVEY §8d formulas), from the loaded header."""
    out = {}
    for which, name in ((0, "semantic"), (1, "coarse"), (2, "fine")):
        L, H, E, ctx, bias, n_in, n_out, n_heads, n_wtes, ftype = [int(v) for v in pkg_bark.hparams(which)]
        bpw = {0: 4, 1: 2, 2: 18 / 32}[ftype % 1000]
        out[name] = dict(L=L, E=E, n_out=n_out, bpw=bpw,
                         decode_weight_bytes=(12 * L * E * E + n_out * E) * bpw,
                         dense_flops=lambda N, rows_out, L=L, E=E, n_out=n_out: 2 * N * 12 * L * E * E + 4 * N * N * E * L + 2 * rows_out * E * n_out)
    return out


def run_ours(args):
    rank, world, local = dist_env()
    pkg = graft.load_package()
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod
        torch.cuda.set_device(local)
        dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist = dist_mod
    if rank == 0:
        weights_path()                                        # one writer; the other ranks find the file after the barrier
    if dist:
        dist.barrier()
    path = weights_path()
    device = local if world > 1 else int(os.environ.get("BARK_B200_DEVICE", "0"))
    pinned = pin_to_gpu_numa(device) if world > 1 else None
    wl = rank_workload(rank)
    b = pkg.Bark(path, seed=wl["seed"], n_steps_text_encoder=N_STEPS_TEXT, device=device)
    prompt = wl["prompt"]

    def sync_all():
        if dist:
            dist.barrier()

    for _ in range(args.warmup):
        audio = b.generate(prompt)
    n_audio = audio.size if args.warmup else None

    # ---- timed region: EXACTLY K steps, barrier + sync on both sides, wall clock around the public C-ABI call with
    # host buffers (prompt text in, waveform copied out) = the e2e figure; the device-event figure is taken per kernel below
    sampler = ClockSampler(device)
    pkg.io_counters(reset=True)
    launches0 = pkg.kernel_launches()
    sync_all()
    sampler.start()
    t0 = time.perf_counter()
    stage_us = np.zeros(3); n_samples = np.zeros(3)
    for _ in range(args.steps):
        audio = b.generate(prompt)
        s, pm = b.stats()
        stage_us += [s.t_semantic_us, s.t_coarse_us, s.t_fine_us]
    sync_all()
    elapsed = time.perf_counter() - t0
    clocks = sampler.stop()
    launches = pkg.kernel_launches() - launches0
    h2d, d2h = pkg.io_counters()
    n_audio = audio.size
    last_outputs = dict(audio=audio, semantic_tokens=b.tokens(0), coarse_tokens=b.tokens(1), fine_tokens=b.tokens(2))
    s, pm = b.stats()
    n_samples = [pm[0][2], pm[1][2], pm[2][2]]        # cumulative since load (reference semantics, bark.cpp:1698)
    n_calls = args.warmup + args.steps

    elapsed_max, total_audio_samples = reduce_over_ranks(dist, elapsed, n_audio, "cuda")
    audio_s_per_step = total_audio_samples / SAMPLE_RATE
    e2e_value = audio_s_per_step * args.steps / elapsed_max

    # ---- per-kernel device time (CUDA events on the launching stream) for the roofline: one extra profiled step on EVERY rank.
    # The profiled step starts from the load-time RNG state (reseed), so rank 0's tokens are the ones the reference produces
    # for (file, prompt, seed 0, 138 steps): the parity leg below compares them with the cpu_baseline run of the same clip.
    pkg.profile_enable(True)
    b.reseed(wl["seed"])
    audio_prof = b.generate(prompt)
    ours_tokens = dict(semantic=b.tokens(0).copy(), coarse=b.tokens(1).copy(), fine=b.tokens(2).copy(), audio=audio_prof)
    rep = pkg.profile_report()
    pkg.profile_enable(False)
    tot_ms = sum(v["ms"] for v in rep.values()) or 1.0
    # value = whole-job throughput with inputs resident: all ranks' audio / MAX over ranks of the summed device kernel time of one clip
    dev_s_max, _ = reduce_over_ranks(dist, tot_ms * 1e-3, n_audio, "cuda")
    value = audio_s_per_step / dev_s_max

    roofline, roofline_all, kernels = None, None, None
    if rank == 0:
        P = peaks()
        kernels = {k: dict(launches=v["launches"], ms=round(v["ms"], 3), share=round(v["ms"] / tot_ms, 4)) for k, v in sorted(rep.items(), key=lambda kv: -kv[1]["ms"])}
        def roof(name, v):
            """achieved vs the measured peak of the roof that bounds this kernel: dense passes (mat-mul / attention of the prefill and
            fine passes) on the tensor roof by themselves (SURVEY §8d), everything else on HBM bytes"""
            sec = v["ms"] * 1e-3
            gbs = v["bytes"] / sec / 1e9 if sec else 0.0
            tfs = v["flops"] / sec / 1e12 if sec else 0.0
            f_h, f_t = gbs / P["hbm_gbs"], tfs / P["tflops"]
            common = dict(kernel=name, launches=v["launches"], avg_launch_us=round(sec * 1e6 / max(v["launches"], 1), 2), share=round(v["ms"] / tot_ms, 4),
                          traffic=measured_traffic(name), algorithmic_bytes_per_launch=int(v["bytes"] / max(v["launches"], 1)), peak_source=P["source"])
            dense = any(t in name for t in ("gemm", "attn_", "flash", "umma"))
            if v["bytes"] > 0 and not (dense and v["flops"] > 0):
                return dict(bound="hbm", achieved=round(gbs, 1), peak=P["hbm_gbs"], unit="GB/s", frac=round(f_h, 4), **common)
            return dict(bound="tensor", achieved=round(tfs, 2), peak=P["tflops"], unit="TFLOP/s", frac=round(f_t, 4),
                        note="dense contraction against the measured bf16 tensor peak; in parity mode it runs as fp32 FMA chains in the reference's lane order on CUDA cores (ceiling ~74 TFLOP/s)", **common)
        ranked = sorted(rep.items(), key=lambda kv: -kv[1]["ms"])
        roofline = roof(*ranked[0])
        roofline_all = [roof(n, v) for n, v in ranked[:8]]

    if rank != 0:
        b.close()
        if dist:
            dist.destroy_process_group()
        return
    spec = BENCH_CONFIGS[BENCH_CONFIG]
    result = {
        "metric": metric_name(BENCH_CONFIG), "value": round(value, 4), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(elapsed_max / args.steps * 1e3, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": ("q4_0 weights / q8_0 activation blocks, " if spec["quant"] else "f16 weights/operands, ") + "f32 accumulate (reference arithmetic)",
        "data": "synthetic (seeded random weights in ggml_weights.bin format, prompt 'hello world')",
        "config": {"workload": f"{spec['label']}, batch=1 per GPU, n_steps_text_encoder={N_STEPS_TEXT} -> {audio_s_per_step / world:.2f} s clip ({spec['baseline']})", "parallelism": f"replica x{world} (one prompt per GPU, no collective" + (f"; each rank pinned to its GPU's local CPUs, rank 0: {pinned}" if pinned else "") + ")",
                   "mode": os.environ.get("BARK_B200_MODE", "parity") + " (parity = token ids bit-identical to the CPU reference; coarse windows start from the cached canonical K/V rows, exact, DESIGN.md §6)",
                   "l2": "inputs larger than L2: the weights streamed per clip exceed the 126 MB L2 many times over; no flush needed"},
        "value_note": "all ranks' audio / MAX over ranks of the summed CUDA-event kernel time of one clip (inputs resident, no host gaps)",
        "e2e": {"value": round(e2e_value, 4), "unit": UNIT, "h2d_bytes_per_step": int(h2d / args.steps), "d2h_bytes_per_step": int(d2h / args.steps),
                "note": "wall clock around bark_generate_audio (C-ABI, host text in / host waveform out): prompt ids, uniforms and codes H2D, sampled tokens and waveform D2H inside the timed region"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "stages": {n: {"tokens_per_s": round(float(ns) / n_calls / (us / args.steps * 1e-6), 1) if us else None, "ms": round(us / args.steps / 1e3, 2)}
                   for n, ns, us in zip(("semantic", "coarse", "fine"), n_samples, stage_us)},
        "audio_seconds_per_step": round(audio_s_per_step, 4),
        "roofline": roofline, "roofline_top": roofline_all, "kernels": kernels,
    }
    ok = True
    if world == 1 and not args.no_cpu_baseline:
        base, ref_out = cpu_baseline(path, budget_s=args.cpu_budget, want_outputs=True)
        result["cpu_baseline"] = base
        if ref_out is not None:
            par = {k: bool(np.array_equal(ours_tokens[k], ref_out[k])) for k in ("semantic", "coarse", "fine")}
            same_len = ours_tokens["audio"].shape == ref_out["audio"].shape
            par["wav_rel"] = float(np.abs(ours_tokens["audio"] - ref_out["audio"]).max() / max(np.abs(ref_out["audio"]).max(), 1e-30)) if same_len else None
            par["against"] = f"{base['kind']} CPU run of the same file / prompt / seed 0 / n_steps_text_encoder={N_STEPS_TEXT} inside this job"
            fast = os.environ.get("BARK_B200_MODE", "parity") != "parity"
            ok = fast or (par["semantic"] and par["coarse"] and par["fine"] and same_len and par["wav_rel"] < 1e-3)
            par["ok"] = bool(ok)
            result["parity"] = par
    b.close()
    if world == 1 and not args.no_fast and BENCH_CONFIGS[BENCH_CONFIG]["quant"] is None and os.environ.get("BARK_B200_MODE", "parity") == "parity":
        result["fast_mode"] = fast_mode_leg(pkg, path, device, prompt, args, ours_tokens)
    if dist:
        dist.destroy_process_group()
    emit(result)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_outputs)
    if not ok:
        sys.stderr.write("bench.py: PARITY FAILURE against the CPU reference on the benchmarked clip\n")
        sys.exit(3)


def fast_mode_leg(pkg, path, device, prompt, args, parity_out):
    """The same clip with BARK_B200_MODE=fast (fine passes on the tensor cores: tcgen05 GEMMs + flash-style attention,
    csrc/fast_kernels.cu).  NOT the contract path: fine ids are not bit-identical; reported next to the parity numbers."""
    os.environ["BARK_B200_MODE"] = "fast"
    try:
        b = pkg.Bark(path, seed=0, n_steps_text_encoder=N_STEPS_TEXT, device=device)
        if not b.fast_mode:
            b.close()
            return {"available": False}
        for _ in range(2):
            b.generate(prompt)
        t0 = time.perf_counter(); fine_us = 0
        for _ in range(args.steps):
            audio = b.generate(prompt)
            fine_us += b.stats()[0].t_fine_us
        dt = (time.perf_counter() - t0) / args.steps
        pkg.profile_enable(True)
        b.reseed(0)
        audio = b.generate(prompt)
        rep = pkg.profile_report()
        pkg.profile_enable(False)
        fine = b.tokens(2)
        same_front = bool(np.array_equal(b.tokens(0), parity_out["semantic"]) and np.array_equal(b.tokens(1), parity_out["coarse"]))
        P = peaks()
        dense = {k: v for k, v in rep.items() if "umma" in k or "flash" in k}
        d_ms = sum(v["ms"] for v in dense.values()); d_fl = sum(v["flops"] for v in dense.values())
        out = {"available": True, "e2e": {"value": round(audio.size / SAMPLE_RATE / dt, 4), "unit": UNIT}, "ms_per_step": round(dt * 1e3, 3), "fine_stage_ms": round(fine_us / args.steps / 1e3, 3),
               "fine_pass_ms": round(fine_us / args.steps / 1e3 / 6, 3),
               "semantic_coarse_ids_identical_to_parity": same_front, "fine_ids_equal_to_parity": round(float((fine == parity_out["fine"]).mean()), 4) if fine.shape == parity_out["fine"].shape else None,
               "wav_rel_vs_parity": round(float(np.abs(audio - parity_out["audio"]).max() / max(np.abs(parity_out["audio"]).max(), 1e-30)), 4) if audio.shape == parity_out["audio"].shape else None,
               "tensor_kernels": {k: dict(launches=v["launches"], ms=round(v["ms"], 3), tflops=round(v["flops"] / (v["ms"] * 1e-3) / 1e12, 1) if v["ms"] else None) for k, v in dense.items()},
               "roofline": {"bound": "tensor", "achieved": round(d_fl / (d_ms * 1e-3) / 1e12, 1) if d_ms else None, "peak": P["tflops"], "unit": "TFLOP/s",
                            "frac": round(d_fl / (d_ms * 1e-3) / 1e12 / P["tflops"], 4) if d_ms else None, "kernels": "umma_gemm_kernel + flash_attn_kernel of one clip (CUDA events)", "peak_source": P["source"]},
               "note": "opt-in BARK_B200_MODE=fast; validated by teacher forcing (tests/test_fast_mode.py), not bit-identical"}
        b.close()
        return out
    finally:
        os.environ.pop("BARK_B200_MODE", None)


def run_fine_only(args):
    """BASELINE configs[4]: the fine stage alone on a synthetic 1024-frame window (coarse codes uniform in [0, 1024)), STRONG scaling:
    the 1024 rows of every pass are split over the N GPUs (csrc/shard.cu: K / V rows stored into the peers' buffers over NVLink from
    the QKV mat-mul's epilogue, one flag barrier per layer, sampled ids published the same way).  Every rank must end with the fine
    tokens of the unsharded run, bit for bit; the line says so (`parity`) and the run fails otherwise."""
    rank, world, local = dist_env()
    pkg = graft.load_package()
    dist = None
    import torch
    if world > 1:
        import torch.distributed as dist_mod
        torch.cuda.set_device(local)
        dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist = dist_mod
    if rank == 0:
        path = weights_path()
    if dist:
        dist.barrier()
    path = weights_path()
    device = local if world > 1 else int(os.environ.get("BARK_B200_DEVICE", "0"))
    pinned = pin_to_gpu_numa(device) if world > 1 else None
    b = pkg.Bark(path, seed=0, n_steps_text_encoder=N_STEPS_TEXT, device=device)
    coarse = np.random.default_rng(11).integers(0, 1024, (1024, 2)).astype(np.int32)

    def one_pass():
        b.reseed(0)
        b.set_tokens(1, coarse)
        b.forward(2)
        return b.tokens(2).copy()

    ref_tokens = one_pass()                                   # unsharded: the N = 1 answer, on every rank
    if world > 1:
        h = b.shard_init(rank, world)
        t = torch.frombuffer(bytearray(h), dtype=torch.uint8).cuda()
        allh = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(allh, t)
        b.shard_connect(b"".join(bytes(x.cpu().numpy().tobytes()) for x in allh))
        dist.barrier()
    for _ in range(args.warmup):
        tokens = one_pass()
    sampler = ClockSampler(device)
    launches0 = pkg.kernel_launches()
    pkg.io_counters(reset=True)
    b.shard_nvlink_bytes(reset=True)
    if dist:
        dist.barrier()
    torch.cuda.synchronize()
    sampler.start()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        tokens = one_pass()
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    elapsed = time.perf_counter() - t0
    clocks = sampler.stop()
    launches = pkg.kernel_launches() - launches0
    h2d, d2h = pkg.io_counters()
    nvl = b.shard_nvlink_bytes()
    same = bool(np.array_equal(tokens, ref_tokens))
    elapsed_max, n_same = reduce_over_ranks(dist, elapsed, 1.0 if same else 0.0, "cuda")
    # device-time figure: summed CUDA-event kernel time of one profiled window, MAX over ranks
    pkg.profile_enable(True)
    one_pass()
    rep = pkg.profile_report()
    pkg.profile_enable(False)
    tot_ms = sum(v["ms"] for v in rep.values()) or 1.0
    dev_s_max, _ = reduce_over_ranks(dist, tot_ms * 1e-3, 0, "cuda")
    b.close()
    if dist:
        dist.destroy_process_group()
    if rank != 0:
        return
    ok = n_same == world
    P = peaks()
    ranked = sorted(rep.items(), key=lambda kv: -kv[1]["ms"])
    top, tv = ranked[0]
    tfs = tv["flops"] / (tv["ms"] * 1e-3) / 1e12 if tv["ms"] else 0.0
    e2e = 6144 * args.steps / elapsed_max
    emit({
        "metric": "fine-stage tokens/s, " + BENCH_CONFIGS["fine_only"]["label"], "value": round(6144 / dev_s_max, 1), "unit": "tokens/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(elapsed_max / args.steps * 1e3, 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f16 weights/operands, f32 accumulate (reference arithmetic)", "data": "synthetic (seeded random weights; coarse codes uniform in [0, 1024), seed 11)",
        "config": {"workload": "fine-only, 6144 tokens: one 1024-frame window, 6 codebook passes (BASELINE configs[4])", "parallelism": f"rows of the window sharded x{world}" + (f" (pinned: {pinned})" if pinned else ""),
                   "collective": "K/V all-gather fused into the QKV mat-mul epilogue (peer stores over NVLink, CUDA IPC) + one flag barrier per layer; no NCCL on the data path" if world > 1 else "none",
                   "l2": "weights (0.17 GB per pass) exceed the L2"},
        "value_note": "6144 tokens / MAX over ranks of the summed CUDA-event kernel time of one window",
        "e2e": {"value": round(e2e, 1), "unit": "tokens/s", "h2d_bytes_per_step": int(h2d / args.steps), "d2h_bytes_per_step": int(d2h / args.steps),
                "note": "wall clock around bark_forward_fine_encoder (C-ABI; codes in, sampled ids out) incl. host sampling control, max over ranks"},
        "gpu_launches": int(launches), "clocks": clocks,
        "parity": {"fine_ids_identical_to_unsharded_on_all_ranks": ok, "ok": ok},
        "nvlink": {"bytes_stored_to_peers_per_step_rank0": int(nvl / args.steps), "achieved_GBps_rank0_out": round(nvl / elapsed / 1e9, 2) if world > 1 else 0.0,
                   "note": "payload is small (K/V rows of 1024/N positions per layer); the stage is bounded by the parity-mode mat-muls, not by the link"},
        "roofline": {"bound": "tensor", "kernel": top, "achieved": round(tfs, 2), "peak": P["tflops"], "unit": "TFLOP/s", "frac": round(tfs / P["tflops"], 4), "launches": tv["launches"],
                     "avg_launch_us": round(tv["ms"] * 1e3 / max(tv["launches"], 1), 2), "traffic": None, "peak_source": P["source"]},
        "kernels": {k: dict(launches=v["launches"], ms=round(v["ms"], 3)) for k, v in ranked[:8]},
    })
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(fine_tokens=tokens))
    if not ok:
        sys.stderr.write("bench.py: sharded fine tokens differ from the unsharded run\n")
        sys.exit(3)


def usable_cpus():
    """CPUs this container may really use: affinity mask capped by the cgroup CPU quota (nproc alone over-reports on shared hosts)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


REF_2GIB_NOTE = " (the unmodified reference cannot load this file: it is >= 2 GiB and bark.cpp:1150 keeps the codec offset in an int)"


def ref_can_load(orc, path):
    return orc.have_ref() and os.path.getsize(path) < 2 ** 31


def best_threads(orc, path):
    """ggml's thread pool spins on a barrier per graph node, so "all cores" is not its fastest setting on a big host:
    try a few thread counts on a short clip and keep the best (reported as `cores`)."""
    usable = usable_cpus()
    cands = sorted({c for c in (4, 8, 16, 32, usable) if c <= usable})
    best = None
    for c in cands:                                          # ascending; stop as soon as more threads stop helping
        r = orc.Ref(path, seed=0, n_steps=8)
        t0 = time.perf_counter(); r.generate(PROMPT, n_threads=c); dt = time.perf_counter() - t0
        r.close()
        if best is not None and dt > best[1]:
            break
        best = (c, dt)
    return best[0], cands


def cpu_baseline(path, budget_s=30.0, steps=1, want_outputs=False):
    """The reference's CPU path on this box's host cores, on the SAME clip the CUDA arm times (same file, prompt, seed,
    n_steps_text_encoder): oracle/_ref (the unmodified reference) when it travelled with the snapshot, else the C oracle port
    on a bounded sample.  One full clip is ~8 s at the best thread count on the GPU box's host."""
    orc = graft.load_oracle_bindings()
    cores = os.cpu_count() or 1
    if ref_can_load(orc, path):
        threads, cands = best_threads(orc, path)
        r = orc.Ref(path, seed=0, n_steps=N_STEPS_TEXT)
        t0 = time.perf_counter()
        for _ in range(steps):
            g = r.generate(PROMPT, n_threads=threads)
        dt = (time.perf_counter() - t0) / steps
        st = r.stats()
        base = {"value": round(g["audio"].size / SAMPLE_RATE / dt, 5), "unit": UNIT, "cores": threads, "host_cores": cores, "kind": "reference",
                "sample": f"same weights/prompt/seed, n_steps_text_encoder={N_STEPS_TEXT} -> {g['audio'].size / SAMPLE_RATE:.2f} s clip (the whole bench clip), one bark_generate_audio at -t {threads} "
                          f"(best of {cands} on a short clip): {dt:.2f} s (semantic {st[2] / 1e3:.0f} ms, coarse {st[3] / 1e3:.0f} ms, fine {st[4] / 1e3:.0f} ms)",
                "build": r.build_info(), "seconds": round(dt, 3)}
        return (base, g) if want_outputs else base
    orc.build_oracle()
    o = orc.Oracle(path, seed=0, n_steps=PORT_STEPS)
    t0 = time.perf_counter(); g = o.generate(PROMPT); dt = time.perf_counter() - t0
    base = {"value": round(g["audio"].size / SAMPLE_RATE / dt, 5), "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"C oracle (OpenMP), bounded sample n_steps_text_encoder={PORT_STEPS} -> {g['audio'].size / SAMPLE_RATE:.2f} s clip in {dt:.2f} s" + REF_2GIB_NOTE * (os.path.getsize(path) >= 2 ** 31),
            "seconds": round(dt, 3)}
    return (base, None) if want_outputs else base


def run_reference(args):
    """The reference's own CPU implementation on the host cores, SAME config as the CUDA arm: same file, prompt, seed and
    n_steps_text_encoder (one step = one whole clip, ~8 s on the GPU box's host)."""
    rank, world, _ = dist_env()
    if rank != 0:
        return
    path = weights_path()
    orc = graft.load_oracle_bindings()
    times, audio_s = [], None
    spec = BENCH_CONFIGS[BENCH_CONFIG]
    if ref_can_load(orc, path):
        cores, cands = best_threads(orc, path)
        r = orc.Ref(path, seed=0, n_steps=N_STEPS_TEXT)
        st = None
        for i in range(args.warmup + args.steps):
            r.reseed(0)
            t0 = time.perf_counter(); g = r.generate(PROMPT, n_threads=cores); dt = time.perf_counter() - t0
            if i >= args.warmup:
                times.append(dt)
            audio_s = g["audio"].size / SAMPLE_RATE
            st = r.stats()
        kind, n = "reference", N_STEPS_TEXT
        sample = (f"same weights/prompt/seed as the CUDA arm, n_steps_text_encoder={n} -> {audio_s:.2f} s clip per step, -t {cores} (best of {cands} on a short clip); "
                  f"last step: semantic {st[2] / 1e3:.0f} ms, coarse {st[3] / 1e3:.0f} ms, fine {st[4] / 1e3:.0f} ms")
        build = r.build_info()
    else:
        cores, n = os.cpu_count() or 1, PORT_STEPS
        orc.build_oracle()
        o = orc.Oracle(path, seed=0, n_steps=n)
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter(); g = o.generate(PROMPT); dt = time.perf_counter() - t0
            if i >= args.warmup:
                times.append(dt)
            audio_s = g["audio"].size / SAMPLE_RATE
        kind, sample, build = "port", f"C oracle (OpenMP), bounded sample n_steps_text_encoder={n} -> {audio_s:.2f} s clip per step" + REF_2GIB_NOTE * (os.path.getsize(path) >= 2 ** 31), "oracle/bark_oracle.c"
    total = sum(times)
    value = audio_s * len(times) / total
    base = {"value": round(value, 5), "unit": UNIT, "cores": cores, "host_cores": os.cpu_count() or 1, "kind": kind, "sample": sample, "build": build, "seconds": round(total / len(times), 3)}
    emit({
        "impl": "reference", "metric": metric_name(BENCH_CONFIG), "value": round(value, 5), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(total / len(times) * 1e3, 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16 weights/operands, f32 accumulate" if not spec["quant"] else "q4_0 weights / q8_0 activation blocks, f32 accumulate", "data": "synthetic (same file as the CUDA arm)",
        "config": {"workload": f"{spec['label']}, batch=1, n_steps_text_encoder={n} -> {audio_s:.2f} s clip ({spec['baseline']})", "parallelism": f"host CPU, {cores} threads"},
        "cpu_baseline": base, "e2e": {"value": round(value, 5), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(audio=g["audio"], semantic_tokens=g["semantic"], coarse_tokens=g["coarse"], fine_tokens=g["fine"]))


def dump_outputs(out_dir, arrays):
    """What the timed path returned in its last step, as out_dir/<name>.npy in float32 (token ids < 2^24 are exact), so that two
    builds run with the same arguments (same seeded weights, prompt and seed) can be compared output for output.  Every
    array is the whole output: a waveform of a clip and its token ids stay far below 64 MB."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(a, np.float32))


_REAL_STDOUT = None


def emit(obj):
    """The one JSON line of the contract goes to the real stdout; everything else (C-level prints of the reference
    harness, library banners) was redirected to stderr in main()."""
    os.write(_REAL_STDOUT, (json.dumps(obj) + "\n").encode())


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-fast", action="store_true", help="skip the extra fast-mode (tensor-core fine passes) leg")
    ap.add_argument("--cpu-budget", type=float, default=30.0)
    ap.add_argument("--config", default=None, choices=sorted(BENCH_CONFIGS), help="which BASELINE config to measure (default: bark-small f16 = configs[1])")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the waveform and token ids of the last timed step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    global BENCH_CONFIG
    if args.config:
        BENCH_CONFIG = args.config
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    elif BENCH_CONFIG == "fine_only":
        run_fine_only(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
