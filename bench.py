"""bench.py -- headline metric of BASELINE.json on B200: whisper-large-v3 tokens/sec (and RTF) on 30 s chunks.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes what the last timed step computed (rank 0's chunks) as DIR/<name>.npy; the inputs are seeded, so two
builds run with the same arguments can be compared output for output.

A "step" is one pass of the hot path over one batch of synthetic 30 s chunks on every rank:
PCM -> log-mel -> 32-layer encoder -> cross K/V -> `new_tokens` greedy decoder steps -> token ids.
  value : whole-job tokens/s with the PCM already resident in HBM (device-timed, max over ranks)
  e2e   : the same through the public API (thestage-style ASRPipeline call) with HOST buffers: pinned H2D of the PCM
          and D2H of the token ids inside the timed region
Workload = BASELINE.json configs[1]: whisper-large-v3 dims, random weights (no checkpoint offline), one synthetic
30 s chunk per GPU, greedy, EOS suppressed so exactly `new_tokens` tokens are produced (SURVEY.md §8d).
Independent chunks shard across ranks with no data-path collective (weak scaling); the only collective is the weight
broadcast at init.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("TRANSFORMERS_OFFLINE", "1")
os.environ.setdefault("HF_HUB_OFFLINE", "1")
os.environ.setdefault("TOKENIZERS_PARALLELISM", "false")

NEW_TOKENS = 128
PRESET = os.environ.get("BW_BENCH_PRESET", "large-v3")
CHUNK_S = 30


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d.get("hbm_gbs", 6650.0)), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.strip().split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def ncu_traffic_bytes():
    """DRAM bytes of one decoder-step kernel launch from the committed `ncu --set full` capture (profiles/*_mega_ncu_raw.csv:
    dram__bytes_read.sum + dram__bytes_write.sum) -- a measurement taken under the profiler, reported beside the live
    CUDA-event numbers, never instead of them.  None when no capture is committed."""
    import csv
    import glob

    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_mega_ncu_raw.csv")))
    if not files:
        return None, None
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    tot = 0.0
    for row in csv.reader(open(files[-1])):
        if len(row) == 3 and row[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            tot += float(row[2]) * scale.get(row[1], 1.0)
    return (tot or None), os.path.relpath(files[-1], ROOT)


def decode_bytes_per_step(dims, S: int, A: int, t_mean: float) -> float:
    """Algorithmic HBM bytes of one decoder step (SURVEY.md §8d): weights + A * cross-KV + A * self-KV(t)."""
    d, L, V, ffn = dims.d_model, dims.dec_layers, dims.vocab, dims.ffn
    # per layer: self q/k/v/out (4 d^2) + cross q/out (2 d^2) + fc1/fc2 (2 d ffn) = 14 d^2 at ffn = 4 d; the cross K/V projection
    # weights belong to the encoder pass (their product, the cross K/V cache, is what a step streams)
    w = 2.0 * (L * (6 * d * d + 2 * d * ffn) + V * d)
    xkv = 2.0 * L * 2 * S * d
    skv = 2.0 * L * 2 * t_mean * d
    return w + A * xkv + A * skv


def workload_config(A: int, world: int) -> dict:
    """The `config` block both arms print: identical keys and values, so the driver's same-config check compares like with like
    (round 1 timed the CPU arm on 16 tokens and the GPU arm on 128: VERDICT.md weak #7)."""
    return {"workload": f"whisper-{PRESET} dims (random weights), {A} x {CHUNK_S}s synthetic chunk per GPU, greedy, "
                        f"{NEW_TOKENS} new tokens (EOS and timestamp ids suppressed: fixed length)",
            "chunks_per_gpu": A, "new_tokens": NEW_TOKENS, "parallelism": f"dp{world} (independent chunks, no data-path collective)",
            "l2": "b200 arm: 256 MB flush write between timed iterations; reference arm: host CPU, not applicable"}


def _cpu_pipe():
    import torch

    from oracle import hf_ref
    from thewhisper_b200 import synthetic as S

    cores = min(os.cpu_count() or 1, 32)  # HF/oneDNN on 128 threads is several times slower than on 32 (oversubscription)
    torch.set_num_threads(cores)
    model = S.make_hf_model(PRESET, seed=0)
    model.generation_config = S.make_generation_config(PRESET, eos_suppressed=True, suppress_timestamps=True)
    pipe = hf_ref.make_ref_pipeline(model, S.make_feature_extractor(CHUNK_S), S.make_tokenizer(), chunk_length_s=CHUNK_S, device="cpu")
    gk = {"num_beams": 1, "do_sample": False, "language": "en", "task": "transcribe", "max_new_tokens": NEW_TOKENS}
    return pipe, gk, cores


def run_reference(args, rank: int, world: int):
    """--impl reference: the reference's own CPU path (HF transformers driven by the restated reference glue in
    oracle/hf_ref.py -- the reference package itself cannot travel to the GPU box) on the host cores, on the SAME workload as
    the b200 arm: one 30 s chunk, 128 greedy tokens per step.  Each step is one such call (~10-20 s on 32 threads)."""
    if rank != 0:
        return
    from thewhisper_b200 import synthetic as S

    pipe, gk, cores = _cpu_pipe()
    audio = S.synth_audio(CHUNK_S, seed=1000)
    times = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        pipe(audio.copy(), generate_kwargs=dict(gk))
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            times.append(dt)
    ms = 1e3 * float(np.mean(times))
    value = NEW_TOKENS / (ms / 1e3)
    line = {
        "impl": "reference", "metric": "tokens_per_sec", "value": value, "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(1, world),
        "derived": {"rtf": (ms / 1e3) / CHUNK_S, "rtfx": CHUNK_S / (ms / 1e3)},
        "cpu_baseline": {"value": value, "unit": "tokens/s", "cores": cores, "kind": "port",
                         "sample": f"{args.steps} timed calls of 1 x {CHUNK_S}s chunk x {NEW_TOKENS} greedy tokens, HF transformers fp32 via oracle/hf_ref.py"},
        "e2e": {"value": value, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="b200 arm: write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch
    import torch.distributed as dist

    from thewhisper_b200 import synthetic as S
    from thewhisper_b200.engine import DecodeOptions, ModelDims, pack_weights

    args.warmup = max(args.warmup, 3)
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    # ---- weights: rank 0 builds the random checkpoint, ONE NCCL broadcast at init, nothing per step
    from thewhisper_b200.nvidia import ASRPipeline
    from thewhisper_b200.parallel import broadcast_weights

    cfg = S.make_hf_config(PRESET)
    dims = ModelDims.from_hf_config(cfg)
    gcfg = S.make_generation_config(PRESET, eos_suppressed=True, suppress_timestamps=True)
    t0 = time.time()
    if rank == 0:
        model = S.make_hf_model(PRESET, seed=0)
        sd = model.state_dict()
        weights = pack_weights(sd, dims, sd["model.encoder.embed_positions.weight"].float(), dev)
        del sd
    else:
        from transformers import WhisperForConditionalGeneration

        with torch.device("meta"):
            model = WhisperForConditionalGeneration(cfg)  # shapes/config only; the weights arrive over NCCL
        weights = None
    model.generation_config = gcfg
    weights = broadcast_weights(weights, dev)
    torch.cuda.synchronize()
    t_weights = time.time() - t0

    A = 1  # chunks per GPU per step (BASELINE.json configs[1])
    pipe = ASRPipeline(model, feature_extractor=S.make_feature_extractor(CHUNK_S), tokenizer=S.make_tokenizer(),
                       chunk_length_s=CHUNK_S, device=str(dev), batch_size=A, max_beams=1, weights=weights)
    eng = pipe.engine
    opts = DecodeOptions(eos_token=S.EOS, pad_token=S.EOS, suppress_tokens=list(gcfg.suppress_tokens),
                         begin_suppress_tokens=list(gcfg.begin_suppress_tokens))
    prompt = np.array([[S.SOT, S.LANG_EN, S.TRANSCRIBE, S.NOTIMESTAMPS]] * A, dtype=np.int32)
    pcm = np.stack([S.synth_audio(CHUNK_S, seed=1000 + rank * A + i) for i in range(A)])
    pcm_dev = torch.from_numpy(pcm).to(dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2
    gk = {"num_beams": 1, "do_sample": False, "language": "en", "task": "transcribe", "max_new_tokens": NEW_TOKENS}

    def step_resident():
        eng.logmel_device(pcm_dev, A)
        eng.encode(A)
        eng.decode_begin(prompt, A, 1, opts)
        eng.decode_run(prompt.shape[1] - 1 + NEW_TOKENS)

    def step_e2e():
        # the call a user of the reference makes: host PCM in, text out (pinned H2D, D2H of ids, detokenisation inside)
        out = pipe([pcm[i] for i in range(A)], batch_size=A, generate_kwargs=dict(gk))
        return out

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        evs = []
        for _ in range(steps):
            flush.fill_(1)  # evict L2 between iterations
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            evs.append((e0, e1))
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = sum(a.elapsed_time(b) for a, b in evs)
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / steps

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_res = timed(step_resident, args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng, A, prompt.shape[1])
    k0 = eng.decode_kernel_launches()
    ms_e2e = timed(step_e2e, args.steps, args.warmup)
    # decoder kernels of ONE e2e step, counted from the captured step graphs (warm-up steps included in the delta)
    dec_kernels_per_step = (eng.decode_kernel_launches() - k0) // (args.steps + args.warmup)

    # ---- roofline of the dominant kernel family: the decoder step (HBM stream), timed alone on its stream
    def decode_only():
        eng.decode_begin(prompt, A, 1, opts)
        eng.decode_run(prompt.shape[1] - 1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        eng.decode_run(NEW_TOKENS)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / NEW_TOKENS

    step_ms = float(np.median([decode_only() for _ in range(5)]))

    # ---- the tensor-bound part beside it: one encoder pass (32 layers + the 64 cross-K/V projections) of these A chunks, CUDA events
    def encode_only():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        eng.encode(A)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    try:
        enc_ms = float(np.median([encode_only() for _ in range(5)]))
    except Exception:  # informational: never at the cost of the line
        enc_ms = None
    clocks = sampler.stop() if rank == 0 else None
    outs = step_e2e()
    n_words = [len(o["text"].split()) for o in outs]
    assert len(outs) == A and min(n_words) >= 1, n_words

    # ---- the other BASELINE.json configurations (C3 / C5 / C4), every rank its own shard, same public API with host buffers
    configs = extra_configs(model, weights, dev, rank, world, dist) if os.environ.get("BW_BENCH_CONFIGS", "C3,C5,C4") not in ("", "0") else {}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    hbm, how = _peaks()
    bytes_step = decode_bytes_per_step(dims, eng.S, A, 4 + NEW_TOKENS / 2)
    traffic, traffic_src = ncu_traffic_bytes() if (A == 1 and PRESET == "large-v3") else (None, None)
    achieved = bytes_step / (step_ms * 1e-3) / 1e9
    tokens = A * NEW_TOKENS * world
    # log-mel (2) + conv stem (2) + 7 per encoder layer (2 LayerNorm, 4 GEMMs, attention) + final LayerNorm + cross K/V projections (2 per decoder layer)
    n_enc_kernels = 2 + 2 + dims.enc_layers * 7 + 1 + 2 * dims.dec_layers
    mega = dec_kernels_per_step <= 2 * (3 + NEW_TOKENS)
    line = {
        "metric": "tokens_per_sec", "value": tokens / (ms_res / 1e3), "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_res, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": workload_config(A, world),
        "derived": {"rtf": (ms_res / 1e3) / (CHUNK_S * A), "rtfx": (CHUNK_S * A) / (ms_res / 1e3), "decode_only_tokens_per_sec": A * 1e3 / step_ms,
                    "weights_broadcast_s": t_weights, "published_reference_headline": "220 tok/s on L40s (README.md:19), other hardware"},
        "e2e": {"value": tokens / (ms_e2e / 1e3), "unit": "tokens/s", "h2d_bytes_per_step": int(pcm.nbytes + prompt.nbytes),
                "d2h_bytes_per_step": int((NEW_TOKENS // 32) * (A * dims.max_target_positions * 4 + A * 4 + 4)), "ms_per_step": ms_e2e,
                "api": "thewhisper_b200.nvidia.ASRPipeline.__call__(list of host float32 arrays) -> text",
                "rtf": (ms_e2e / 1e3) / (CHUNK_S * A)},
        "gpu_launches": args.steps * (n_enc_kernels + dec_kernels_per_step),
        "gpu_launches_detail": {"per_step_encoder_side": n_enc_kernels, "per_step_decoder": dec_kernels_per_step,
                                "decoder_steps_per_step": 3 + NEW_TOKENS,
                                "note": "decoder kernels counted from the captured CUDA graphs (bw_decode_kernel_launches)"},
        "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": ("decode_mega_kernel (one persistent kernel per decoder step: 32 layers + LM head + greedy select)"
                                                 if mega else "decoder step (per-op gemv/attention/select kernels, one CUDA graph)"), "achieved": achieved,
                     "peak": hbm, "unit": "GB/s", "frac": achieved / hbm, "peak_source": how, "traffic": traffic,
                     "traffic_source": traffic_src,
                     "bytes_per_step": bytes_step, "ms_per_decoder_step": step_ms},
    }
    try:
        if enc_ms:
            d, S_enc, ffn = dims.d_model, eng.S, dims.ffn
            flop = A * (dims.enc_layers * (2.0 * S_enc * (4 * d * d + 2 * d * ffn) + 4.0 * S_enc * S_enc * d) + dims.dec_layers * 2 * 2.0 * S_enc * d * d)
            pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
            tf = flop / (enc_ms * 1e-3) / 1e12
            line["encoder"] = {"bound": "tensor", "kernel": "encoder pass: gemm_tc2_kernel (tcgen05 CTA pairs) + attn_enc_tc2_kernel, one CUDA graph", "chunks": A,
                               "ms_per_pass": enc_ms, "flop_per_pass": flop, "achieved": tf, "unit": "TFLOP/s",
                               "peak_sustained": pk.get("bf16_tflops_sustained"), "peak_burst": pk.get("bf16_tflops"),
                               "frac_sustained": tf / pk["bf16_tflops_sustained"] if pk.get("bf16_tflops_sustained") else None,
                               "note": "informational; B = 1 is the latency-bound case (profiles/r2jn_summary.md: 0.65 of sustained at 64 chunks)"}
    except Exception as ex:  # informational entry: never at the cost of the line
        line["encoder"] = {"error": repr(ex)}
    line["configs"] = configs
    if not args.no_cpu_baseline:
        try:
            line["cpu_baseline"] = cpu_baseline()
        except Exception as ex:  # the GPU numbers stand on their own
            line["cpu_baseline"] = {"value": None, "unit": "tokens/s", "error": repr(ex)}
        if world == 1 and not os.environ.get("BW_NO_HF_CUDA"):
            del pipe, eng, weights
            torch.cuda.empty_cache()
            line["hf_cuda"] = hf_cuda_leg(dev)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir: str, eng, A: int, plen: int) -> None:
    """What the last resident step left in the engine, read back the way a caller of that path reads it: the generated token
    ids (float64, exact), the logits of the last decoder step and the encoder output (float32).  About 8 MB at large-v3 dims."""
    toks, _, _ = eng.decode_read()
    arrays = {"tokens": toks[:A, plen:plen + NEW_TOKENS].astype(np.float64),
              "logits": eng.logits()[:A].cpu().numpy(),
              "encoder_out": eng.encoder_output(A).cpu().numpy()}
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def extra_configs(model, weights, dev, rank, world, dist):
    """BASELINE.json configs[2..4] beside the headline: C3 (64 x 30 s, greedy + word timestamps), C5 (64 x 30 s, beam 5) and C4
    (32 streams, 15 s window) PER GPU -- at N GPUs the job is N x that (64 x 8 = 512 chunks, 32 x 8 = 256 streams: the sizes
    BASELINE.json quotes).  Whole-job value = units of all ranks / max-over-ranks time; each entry carries its own decoder-step roofline."""
    import torch

    from thewhisper_b200 import synthetic as S
    from thewhisper_b200.engine import interpolate_positions
    from tools.bench_configs import run_batch, run_streaming

    want = [c for c in os.environ.get("BW_BENCH_CONFIGS", "C3,C5,C4").split(",") if c]
    out = {}

    def agg(key_s):
        t = torch.tensor([key_s], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for c in want:
        try:
            if c in ("C3", "C5"):
                beams, wts = (1, True) if c == "C3" else (5, False)
                model.generation_config = S.make_generation_config(PRESET, eos_suppressed=True, suppress_timestamps=not wts)
                r = run_batch(c, 64, beams, wts, NEW_TOKENS, 2, PRESET, False, model=model, weights=weights, device=str(dev))
                dt = agg(r["seconds_per_batch"])
                r.update({"n_gpus": world, "chunks_total": 64 * world, "seconds_per_batch_max_over_ranks": dt,
                          "tokens_per_sec": 64 * world * NEW_TOKENS / dt, "rtfx": 64 * world * CHUNK_S / dt})
            elif c == "C4":
                model.generation_config = S.make_generation_config(PRESET, eos_suppressed=True, suppress_timestamps=False)
                w15 = dict(weights)
                w15["enc.pos"] = interpolate_positions(weights["enc.pos"], 15).to(dev)
                r = run_streaming(32, 24, PRESET, False, model=model, weights15=w15, device=str(dev))
                tick = agg(r["median_tick_s"])
                r.update({"n_gpus": world, "streams_total": 32 * world, "median_tick_s_max_over_ranks": tick,
                          "realtime_streams_sustained": 32 * world * 0.5 / tick})
            else:
                continue
            out[c] = r
        except Exception as ex:  # a config that fails must not take the headline down with it
            out[c] = {"error": repr(ex)[:300]}
        torch.cuda.empty_cache()
    return out


def cpu_baseline():
    """Bounded CPU sample of the same workload (one 30 s chunk, 128 greedy tokens) through the oracle (kind "port": restated
    reference glue over the installed transformers), on this box's host cores: one warm-up call of 8 tokens (oneDNN primitive
    caches), one timed full call."""
    from thewhisper_b200 import synthetic as S

    pipe, gk, cores = _cpu_pipe()
    audio = S.synth_audio(CHUNK_S, seed=1000)
    pipe(audio.copy(), generate_kwargs=dict(gk, max_new_tokens=8))
    t0 = time.perf_counter()
    pipe(audio.copy(), generate_kwargs=dict(gk))
    dt = time.perf_counter() - t0
    return {"value": NEW_TOKENS / dt, "unit": "tokens/s", "cores": cores, "kind": "port",
            "sample": f"1 x {CHUNK_S}s chunk, {NEW_TOKENS} greedy tokens (the bench workload), fp32 HF transformers on CPU, 1 short warm-up + 1 timed call ({dt:.1f}s)"}


def hf_cuda_leg(dev):
    """Informational (BASELINE.md section 3): the reference's HF class with device='cuda' on the same B200, same workload, fp16 and
    bf16 (sdpa attention), outside every timed region of the b200 arm.  Not the parity oracle and not the reference arm."""
    import torch

    from oracle import hf_ref
    from thewhisper_b200 import synthetic as S

    out = {}
    audio = S.synth_audio(CHUNK_S, seed=1000)
    gk = {"num_beams": 1, "do_sample": False, "language": "en", "task": "transcribe", "max_new_tokens": NEW_TOKENS}
    for name, dt in (("fp16", torch.float16), ("bf16", torch.bfloat16)):
        try:
            model = S.make_hf_model(PRESET, seed=0, dtype=dt)
            model.generation_config = S.make_generation_config(PRESET, eos_suppressed=True, suppress_timestamps=True)
            pipe = hf_ref.make_ref_pipeline(model, S.make_feature_extractor(CHUNK_S), S.make_tokenizer(), chunk_length_s=CHUNK_S,
                                            device=str(dev), torch_dtype=dt)
            for _ in range(2):
                pipe(audio.copy(), generate_kwargs=dict(gk))
            torch.cuda.synchronize()
            ts = []
            for _ in range(3):
                t0 = time.perf_counter()
                pipe(audio.copy(), generate_kwargs=dict(gk))
                torch.cuda.synchronize()
                ts.append(time.perf_counter() - t0)
            out[name] = {"tokens_per_sec": NEW_TOKENS / float(np.median(ts)), "ms_per_step": 1e3 * float(np.median(ts))}
            del pipe, model
            torch.cuda.empty_cache()
        except Exception as ex:
            out[name] = {"error": repr(ex)[:200]}
    out["what"] = "HF transformers WhisperForConditionalGeneration via the reference's ASRPipeline glue, device=cuda (eager torch ops), wall clock, median of 3"
    return out


if __name__ == "__main__":
    main()
