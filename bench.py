#!/usr/bin/env python
"""bench.py -- VibeVoice generation hot path on B200: audio-seconds generated per wall-second.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU path (oracle port) on host cores
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR  # also write the last timed step's outputs to DIR/*.npy

Workload (BASELINE.json configs[1], SURVEY 8d-2): VibeVoice-1.5B, 1 speaker, 64K context = 63,488-token synthetic prompt +
2,047 generated speech frames (context ends at 65,535 = max_position_embeddings - 1; 273 s of audio per step), 30 diffusion
steps, cfg 1.3, random-init weights, one prompt per GPU.  (`--prompt-len 61440 --frames 4095` gives SURVEY's variant.)
A "step" is one complete pass of the hot path over that prompt:
  value : K steps of the steady-state frame loop (LM decode pos+neg -> CFG diffusion sampler -> codec decode -> semantic
          encode -> connectors) with the prompt KV already resident in HBM; device-timed with CUDA events.
  e2e   : K calls of the public API `VibeVoiceForConditionalGenerationInference.generate()` with HOST input_ids: prompt
          prefill, per-frame token read-back and noise upload, and the waveform copied back to the host are all inside the
          timed region.
With N > 1 every rank runs the same workload on its own prompt (weak scaling; prompts shard by batch, SURVEY 8e); the only
collective is the final NCCL gather of the waveforms to rank 0.  Frames stream ~13 GB of weights+KV each (>> 126 MB L2), so no
explicit L2 flush is needed between iterations ("inputs larger than L2").
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

AUDIO_S_PER_FRAME = 3200.0 / 24000.0
DUMP_BYTES = 64 * 10**6          # --dump-outputs: size of everything it writes, at most
# DRAM traffic of one frame / one LM step from an ncu pass (dram__bytes_read.sum + dram__bytes_write.sum over every kernel of the frame),
# see profiles/ (filled in by the profiling run of this round; None = not captured for that model)
TRAFFIC_NOTE = {
    "1.5b": "10.96 GB DRAM (read + write) per frame for 12.98 GB algorithmic at ctx 61440: the four stream_kernel launches move 4.39 (LM stack: "
            "4.40 algorithmic) + 5.02 (30-step sampler: 7.09 algorithmic, the rest of the head's re-reads hit the 126 MB L2) + 0.66 + 0.67 GB "
            "(codec front / back), every other kernel 0.23 GB (ncu --set full + launch list of the final kernels, profiles/r02_prof_stream3_raw.csv, "
            "profiles/r02_launches_15b_ctx61440_frame_final.txt)",
    "1.5b:lm": "4.387 GB dram read + 0.012 GB written for 4.40 GB algorithmic (ncu --set full, profiles/r02_prof_stream3_raw.csv, launch 0)",
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--model", default="1.5b", choices=["1.5b", "7b", "1.5b-l2", "tiny", "small", "streaming-0.5b"])
    ap.add_argument("--runs", type=int, default=100, help="streaming-0.5b: generate() calls the latency percentiles are taken over")
    ap.add_argument("--prompt-len", type=int, default=None)
    ap.add_argument("--frames", type=int, default=None, help="speech frames generated per step")
    ap.add_argument("--diffusion-steps", type=int, default=30)
    ap.add_argument("--cfg-scale", type=float, default=1.3)
    ap.add_argument("--batch", type=int, default=1, help="prompts per GPU")
    ap.add_argument("--cpu-frames", type=int, default=None, help="frames in the CPU sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-7b", action="store_true", help="skip the VibeVoice-7B sub-configs appended to the 1.5B line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32, %d MB at most in "
                         "all: a fixed, seeded sample of each array beyond that)" % (DUMP_BYTES // 10**6))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and (args.impl != "b200" or args.model == "streaming-0.5b"):
        ap.error("--dump-outputs writes the outputs of the CUDA frame loop (--impl b200, not --model streaming-0.5b)")
    return args


def dump_outputs(out_dir, arrays):
    """Write {name: array} as out_dir/<name>.npy in float32.  When the arrays hold more than DUMP_BYTES, every array keeps the same
    fraction of its elements, at positions drawn from a generator seeded by 0 (sorted, flattened), so that two runs with the same
    arguments write the same elements.  Their values agree to about 1e-4 rel-L2, not bit for bit: the stream kernel accumulates
    with fp32 atomics."""
    arrays = {k: np.ascontiguousarray(v, dtype=np.float32) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    budget = DUMP_BYTES - 1024 * len(arrays)                     # room for the .npy headers
    frac = min(1.0, budget / total) if total else 1.0
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if frac < 1.0:
            a = a.reshape(-1)[np.unique(np.random.default_rng(0).integers(0, a.size, int(a.size * frac)))]
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log("outputs written to %s: %s%s" % (out_dir, ", ".join("%s %s" % (k, tuple(v.shape)) for k, v in arrays.items()),
                                           "" if frac == 1.0 else " (seeded %.3f sample of each)" % frac))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


_T0 = time.time()


def log(msg):
    sys.stderr.write("[bench %7.1fs] %s\n" % (time.time() - _T0, msg))
    sys.stderr.flush()


def usable_cores() -> int:
    """Cores this process may actually use: scheduler affinity capped by the cgroup CPU quota (os.cpu_count() reports the
    host's cores inside a container and oversubscribing them makes the CPU baseline pathologically slow)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if q > 0:
                    n = min(n, max(1, int(q / per + 0.5)))
            break
        except Exception:
            continue
    return max(1, n)


def dist_env():
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    return rank, world, local


def workload(args):
    from vibevoice_b200.configuration import preset_config
    cfg = preset_config(args.model)
    maxpos = cfg.decoder_config.max_position_embeddings
    if args.model in ("1.5b", "7b"):
        L0 = args.prompt_len if args.prompt_len is not None else (63488 if args.model == "1.5b" else 30720)
        F = args.frames if args.frames is not None else maxpos - 1 - L0
    else:
        L0 = args.prompt_len or 64
        F = args.frames or 32
    assert L0 + F + 1 <= maxpos, "prompt + frames exceed max_position_embeddings"
    return cfg, L0, F


def algorithmic_bytes_per_frame(wb, cfg, ctx_pos, ctx_neg, n_steps, B):
    """SURVEY 8d: W_lm + N*W_head_step + W_condproj + W_dec + W_sem + W_conn + sum_rows kvB*(ctx_pos+ctx_neg) + 5*H*2 (bf16)."""
    dc = cfg.decoder_config
    kvB = dc.num_hidden_layers * 2 * dc.num_key_value_heads * dc.head_dim * 2
    return (wb["lm"] + n_steps * wb["head_step"] + wb["cond_proj"] + wb["decoder"] + wb["semantic"] + wb["connectors"]
            + B * kvB * (ctx_pos + ctx_neg))


# ------------------------------------------------------------------------------------------------------------------
def run_reference(args):
    """The reference's own CPU implementation of the path (oracle port: reference modules' arithmetic restated in
    PyTorch fp32 + installed-transformers-equivalent Qwen2, SURVEY 8c) timed on the host cores with all threads."""
    rank, world, local = dist_env()
    if rank != 0:
        return
    from oracle import vv_oracle as O
    from vibevoice_b200.synth import SynthTokenizer, synth_state_dict
    cfg, L0, F = workload(args)
    torch.set_num_threads(usable_cores())
    tok = SynthTokenizer(cfg.decoder_config.vocab_size)
    t0 = time.time()
    w = {k: v.float() for k, v in synth_state_dict(cfg, 1234, torch.bfloat16, parts=("lm", "head", "acoustic_decoder", "semantic",
                                                                                      "connectors", "lm_head")).items()}
    frames = args.cpu_frames or 4
    res = cpu_sample(O, w, cfg, tok, L0, frames, args, steps=args.steps, warmup=args.warmup)
    line = {"metric": "audio_seconds_per_second", "value": res["value"], "unit": "audio-s/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": config_dict(args, cfg, L0, F),
            "cpu_baseline": {"value": res["value"], "unit": "audio-s/s", "cores": res["cores"], "kind": "port", "sample": res["sample"]},
            "e2e": {"value": res["value"], "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "setup_s": round(time.time() - t0, 1)}
    print(json.dumps(line), flush=True)


def cpu_sample(O, w, cfg, tok, L0, frames, args, steps=1, warmup=1, budget_s=25.0):
    """Bounded sample of the same workload on the CPU: steady-state frames at context L0 (synthetic KV prefix of the right
    size -- a 64K-token CPU prefill alone would take minutes), 30 diffusion steps, cfg 1.3.  Each step is `frames` frames; if
    the first warm-up frame shows that the whole sample would exceed `budget_s`, frames/step drops to 1."""
    dc = cfg.decoder_config
    torch.manual_seed(0)
    cap = L0 + (warmup + steps) * frames + 16
    pos, neg = O.KVCache(dc.num_hidden_layers, capacity=cap), O.KVCache(dc.num_hidden_layers, capacity=cap)
    for l in range(dc.num_hidden_layers):
        pos.preload(l, torch.randn(dc.num_key_value_heads, L0, dc.head_dim) * 0.5, torch.randn(dc.num_key_value_heads, L0, dc.head_dim) * 0.5)
    e0 = w["model.language_model.embed_tokens.weight"][tok.speech_start_id]
    a, s = O.StreamState(1), O.StreamState(1)
    t = time.time()
    O.steady_frames(w, cfg, tok, pos, neg, e0, 1, args.cfg_scale, args.diffusion_steps, a, s)      # untimed first-touch frame
    t_frame = time.time() - t
    if t_frame * frames * (warmup + steps) > budget_s:
        frames = 1
    if t_frame * (warmup + steps) > 4 * budget_s:
        warmup = min(warmup, 1)
    times = []
    for it in range(warmup + steps):
        t = time.time()
        O.steady_frames(w, cfg, tok, pos, neg, e0, frames, args.cfg_scale, args.diffusion_steps, a, s)
        times.append(time.time() - t)
    el = sum(times[warmup:])
    return {"value": steps * frames * AUDIO_S_PER_FRAME / el, "ms_per_step": 1e3 * el / steps, "cores": torch.get_num_threads(),
            "sample": "%d steady-state frame(s)/step at ctx %d (synthetic KV prefix), %d diffusion steps, fp32, torch %d threads "
                      "(os.cpu_count %d); %d timed step(s) after %d warm-up" % (frames, L0, args.diffusion_steps, torch.get_num_threads(),
                                                                                os.cpu_count() or 0, steps, warmup)}


def config_dict(args, cfg, L0, F):
    return {"workload": "VibeVoice-%s random-init, %d prompt(s)/GPU, %d-token synthetic prompt, %d speech frames/step, %d diffusion steps, "
                        "cfg %.2f" % (args.model, args.batch, L0, F, args.diffusion_steps, args.cfg_scale),
            "prompt_len": L0, "frames_per_step": F, "diffusion_steps": args.diffusion_steps, "batch_per_gpu": args.batch,
            "parallelism": "replicas x%d (prompts sharded by batch, no data-path collective)" % args.gpus,
            "l2": "inputs larger than L2 (each frame streams GBs of weights + KV)"}


# ------------------------------------------------------------------------------------------------------------------
def run_extra_config(tag, preset, B, L0, F, args, rank, world, local, dev, peak):
    """Steady-state loop of another BASELINE configuration (same method as `value`): 1 warm-up + `--steps` timed steps of F frames.
    Every rank executes the same sequence of collectives whether or not its own part failed (a Python-level failure on one rank must
    not leave the others waiting in a barrier): failures are agreed on with a MIN all-reduce after each phase."""
    import torch.distributed as dist
    from vibevoice_b200.configuration import preset_config
    from vibevoice_b200.modeling import VibeVoiceForConditionalGenerationInference
    from vibevoice_b200.synth import SynthTokenizer, iter_synth_state_dict_fast

    def agree(ok):
        if world == 1:
            return ok
        t = torch.tensor([1.0 if ok else 0.0], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return bool(t.item() > 0.5)

    err, model, eng, step, wb, cfg = None, None, None, None, None, None
    try:
        cfg = preset_config(preset)
        tok = SynthTokenizer(cfg.decoder_config.vocab_size)
        model = VibeVoiceForConditionalGenerationInference(cfg, tok, max_batch=B, device=local, torch_prefill=True)
        parts = ("lm", "head", "acoustic_decoder", "semantic", "connectors", "lm_head")
        model.load_state_dict(iter_synth_state_dict_fast(cfg, 4321 + rank, device=dev, parts=parts), tok)
        model.set_ddpm_inference_steps(args.diffusion_steps)
        eng = model.engine
        wb = eng.weight_bytes()
        eng.kv_init(B * (L0 + F + 8) + B * (F + 8))
        eng.set_diffusion_steps(args.diffusion_steps)
        g = torch.Generator().manual_seed(200 + rank)
        ids = torch.randint(0, 151643, (B, L0), generator=g)
        ids[:, -1] = tok.speech_start_id
        embw = model._lm_sd["model.language_model.embed_tokens.weight"]
        with torch.cuda.stream(eng.stream):
            for r in range(B):
                model._prefill.run(eng, r, embw[ids[r].to(dev)])
        eng.sync()
        noise_tab = torch.randn(F, B, 64, device=dev)
        ones = [1] * (2 * B)

        def step():
            eng.codec_state_reset()
            for r in range(B):
                eng.kv_set_len(r, L0); eng.kv_set_len(B + r, 0)
            eng.embed_tokens([tok.speech_start_id] * (2 * B), eng.embeds)
            with torch.cuda.stream(eng.stream):
                eng.active.fill_(1)
            for f in range(F):
                eng.lm_decode()
                eng.kv_commit(ones)
                with torch.cuda.stream(eng.stream):
                    eng.noise.copy_(noise_tab[f])
                eng.frame_tail(args.cfg_scale)
        step()                                                  # warm-up
    except Exception as e:
        err = "%s: %s" % (type(e).__name__, str(e)[:300])

    def cleanup():
        try:
            if eng is not None:
                eng.close()
        except Exception:
            pass
        torch.cuda.empty_cache()

    if not agree(err is None):
        cleanup()
        return {"config": tag, "error": err or "failed on another rank"}
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    K = args.steps
    ms = 0.0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    try:
        e0.record(eng.stream)
        for _ in range(K):
            step()
        e1.record(eng.stream)
    except Exception as e:
        err = "%s: %s" % (type(e).__name__, str(e)[:300])
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    if err is None:
        ms = e0.elapsed_time(e1)
    if not agree(err is None):
        cleanup()
        return {"config": tag, "error": err or "failed on another rank"}
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ms_frame = ms / (K * F)
    abytes = algorithmic_bytes_per_frame(wb, cfg, L0 + (F - 1) / 2.0 + 1, (F - 1) / 2.0 + 1, args.diffusion_steps, B)
    ach = abytes / (ms_frame * 1e-3) / 1e9
    out = {"config": tag, "model": preset, "batch_per_gpu": B, "prompt_len": L0, "frames_per_step": F, "steps": K, "warmup": 1,
           "value": round(K * F * B * world * AUDIO_S_PER_FRAME / (ms / 1e3), 3), "unit": "audio-s/s", "n_gpus": world,
           "ms_per_frame": round(ms_frame, 4), "algorithmic_bytes_per_frame": int(abytes),
           "roofline": {"bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4)}}
    cleanup()
    del model, eng
    return out


def run_b200(args):
    rank, world, local = dist_env()
    import torch.distributed as dist
    if world > 1:
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    from vibevoice_b200.modeling import ForcedTokenScript, VibeVoiceForConditionalGenerationInference
    from vibevoice_b200.synth import SynthTokenizer, iter_synth_state_dict_fast
    cfg, L0, F = workload(args)
    B = args.batch
    tok = SynthTokenizer(cfg.decoder_config.vocab_size)
    t_setup = time.time()
    model = VibeVoiceForConditionalGenerationInference(cfg, tok, max_batch=B, device=local, torch_prefill=True)
    parts = ("lm", "head", "acoustic_decoder", "semantic", "connectors", "lm_head")
    model.load_state_dict(iter_synth_state_dict_fast(cfg, 1234 + rank, device=dev, parts=parts), tok)
    model.set_ddpm_inference_steps(args.diffusion_steps)
    eng = model.engine
    wb = eng.weight_bytes()
    eng.kv_init(B * (L0 + F + 8) + B * (F + 8))
    eng.set_diffusion_steps(args.diffusion_steps)
    g = torch.Generator().manual_seed(100 + rank)
    ids = torch.randint(0, min(cfg.decoder_config.vocab_size, 151643), (B, L0), generator=g)
    ids[:, -1] = tok.speech_start_id
    K, W = args.steps, args.warmup

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---------------- value: steady-state loop, prompt KV resident ----------------
    embw = model._lm_sd["model.language_model.embed_tokens.weight"]
    with torch.cuda.stream(eng.stream):
        for r in range(B):
            model._prefill.run(eng, r, embw[ids[r].to(dev)])
    eng.sync()
    log("weights + prefill(%d tokens) done" % L0)
    noise_tab = torch.randn(F, B, 64, device=dev, generator=torch.Generator(device=dev).manual_seed(300 + rank))
    ones = [1] * (2 * B)
    dump = args.dump_outputs is not None and rank == 0
    if dump:     # per-frame audio and token logits of the last timed step (device-to-device copies on the engine stream)
        audio_out = torch.empty(F, B, 3200, device=dev)
        logits_out = torch.empty(F, *eng.logits.shape, device=dev)

    def value_step(capture=False):
        eng.codec_state_reset()
        for r in range(B):
            eng.kv_set_len(r, L0); eng.kv_set_len(B + r, 0)
        eng.embed_tokens([tok.speech_start_id] * (2 * B), eng.embeds)
        with torch.cuda.stream(eng.stream):
            eng.active.fill_(1)
        for f in range(F):
            eng.lm_decode()
            eng.kv_commit(ones)
            with torch.cuda.stream(eng.stream):
                eng.noise.copy_(noise_tab[f])
            eng.frame_tail(args.cfg_scale)
            if capture:
                with torch.cuda.stream(eng.stream):
                    audio_out[f].copy_(eng.audio)
                    logits_out[f].copy_(eng.logits)

    for _ in range(W):
        value_step()
    barrier()
    log("value warm-up done")
    clocks = ClockSampler(local)
    clocks.start()
    launches0 = eng.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(eng.stream)
    for k in range(K):
        value_step(capture=dump and k == K - 1)
    ev1.record(eng.stream)
    barrier()
    ms_value = ev0.elapsed_time(ev1)
    log("value timed: %.1f ms for %d steps" % (ms_value, K))
    launches = eng.launch_count() - launches0
    clk = clocks.stop()
    if world > 1:
        t = torch.tensor([ms_value], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_value = float(t.item())
    frames_total = K * F * B * world
    value = frames_total * AUDIO_S_PER_FRAME / (ms_value / 1e3)
    ms_frame = ms_value / (K * F)
    # roofline of the frame program (2 CUDA-graph launches per frame): algorithmic bytes / measured frame time
    ctx_pos = L0 + (F - 1) / 2.0 + 1
    ctx_neg = (F - 1) / 2.0 + 1
    abytes = algorithmic_bytes_per_frame(wb, cfg, ctx_pos, ctx_neg, args.diffusion_steps, B)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = abytes / (ms_frame * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                "traffic": None, "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)",
                "unit_of_work": "one speech frame = lm_decode graph + frame_tail graph",
                "algorithmic_bytes_per_frame": int(abytes), "ms_per_frame": round(ms_frame, 4)}

    # ---------------- per-segment rooflines at this context (each C-ABI entry point alone, CUDA events on the engine stream) ----------------
    def segment_rooflines():
        dc = cfg.decoder_config
        kvB = dc.num_hidden_layers * 2 * dc.num_key_value_heads * dc.head_dim * 2
        for r in range(B):
            eng.kv_set_len(r, L0); eng.kv_set_len(B + r, 0)
        eng.embed_tokens([tok.speech_start_id] * (2 * B), eng.embeds)

        def lm():
            eng.lm_decode()
            eng.kv_commit(ones)
        segs = [("lm_decode", lm, wb["lm"] + B * kvB * (L0 + 8)),
                ("diffusion_sample", lambda: eng.diffusion_sample(args.cfg_scale), args.diffusion_steps * wb["head_step"] + wb["cond_proj"]),
                ("codec_decode", eng.codec_decode, wb["decoder"]),
                ("semantic_encode", eng.semantic_encode, wb["semantic"]),
                ("connect", eng.connect, wb["connectors"])]
        out = {}
        for name, fn, nbytes in segs:
            for _ in range(3):
                fn()
            eng.sync()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n = 16
            e0.record(eng.stream)
            for _ in range(n):
                fn()
            e1.record(eng.stream)
            eng.sync()
            us = e0.elapsed_time(e1) * 1e3 / n
            out[name] = {"us": round(us, 1), "algorithmic_bytes": int(nbytes), "achieved_GBps": round(nbytes / us / 1e3, 1),
                         "frac": round(nbytes / us / 1e3 / peak, 4)}
        return out
    segs = segment_rooflines()
    roofline["segments"] = segs
    roofline["traffic"] = TRAFFIC_NOTE.get(args.model)
    lm_seg = segs["lm_decode"]
    roofline["dominant_kernel"] = {
        "kernel": "stream_kernel (vv_stream.cuh): the whole %d-layer decoder stack of one step as ONE persistent launch -- tcgen05.mma + TMEM, "
                  "weight tiles and K/V pages by TMA through one ring" % cfg.decoder_config.num_hidden_layers,
        "bound": "hbm", "achieved": lm_seg["achieved_GBps"], "peak": peak, "unit": "GB/s", "frac": lm_seg["frac"],
        "algorithmic_bytes_per_launch": lm_seg["algorithmic_bytes"], "us_per_launch": lm_seg["us"],
        "traffic": TRAFFIC_NOTE.get(args.model + ":lm"),
        "note": "vv_lm_decode timed alone (copy-in, the stream launch, final norm, 4-row lm_head); weights + KV of one step >> L2"}
    head_step_us = segs["diffusion_sample"]["us"] / args.diffusion_steps
    log("segment rooflines done")

    # ---------------- e2e: public generate() with host buffers ----------------
    e2e = None
    if not args.no_e2e:
        script = [[tok.speech_diffusion_id] * F + [tok.eos_token_id]] * B

        def e2e_step():
            torch.manual_seed(0)
            out = model.generate(input_ids=ids, tokenizer=tok, cfg_scale=args.cfg_scale, is_prefill=False,
                                 logits_processor=[ForcedTokenScript(script)], max_new_tokens=F + 1, max_length_times=1e9,
                                 show_progress_bar=False)
            with torch.cuda.stream(eng.stream):
                wav = [o.to("cpu", non_blocking=False) for o in out.speech_outputs]
            return wav
        for _ in range(min(W, 3)):
            wav = e2e_step()
            log("e2e warm-up step done")
        barrier()
        ev0.record(eng.stream)
        t0 = time.time()
        for _ in range(K):
            wav = e2e_step()
        if world > 1:   # the trivial result gather (SURVEY 8e): waveforms to rank 0 over NCCL
            from vibevoice_b200.distributed import gather_waveforms
            gathered = gather_waveforms([w_.to(dev) for w_ in wav], device=dev, dst=0)
            if rank == 0:
                assert sum(len(r_) for r_ in gathered) == B * world
        ev1.record(eng.stream)
        barrier()
        ms_e2e = max(ev0.elapsed_time(ev1), (time.time() - t0) * 1e3 if world == 1 else 0.0)
        if world > 1:
            t = torch.tensor([ms_e2e], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_e2e = float(t.item())
        log("e2e timed: %.1f ms" % ms_e2e)
        assert wav[0].shape == (1, F * 3200)
        h2d = B * L0 * 8 + F * (B * 64 * 4 + B * 4)
        d2h = B * F * 3200 * 4 + F * (B * 4 + B * len(eng.valid_ids) * 4)
        e2e = {"value": round(frames_total * AUDIO_S_PER_FRAME / (ms_e2e / 1e3), 3), "unit": "audio-s/s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "ms_per_step": round(ms_e2e / K, 2), "includes": "prompt prefill (PyTorch library kernels), "
               "per-frame token read-back + noise upload, waveform D2H" + (", NCCL gather to rank 0" if world > 1 else "")}

    # ---------------- CPU baseline beside it (rank 0, N=1) ----------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import vv_oracle as O
        torch.set_num_threads(usable_cores())
        names = [n for n, _, _ in __import__("vibevoice_b200.synth", fromlist=["param_specs"]).param_specs(cfg, parts)]
        w = {}
        for name, t in iter_synth_state_dict_fast(cfg, 1234 + rank, device=dev, parts=parts):
            w[name] = t.float().cpu()
        log("cpu weights copied")
        cpu = cpu_sample(O, w, cfg, tok, L0, args.cpu_frames or 4, args, steps=1, warmup=1)
        log("cpu sample done")
        cpu = {"value": round(cpu["value"], 4), "unit": "audio-s/s", "cores": cpu["cores"], "kind": "port", "sample": cpu["sample"]}

    # ---------------- BASELINE configs #3 / #4 on the same clock: VibeVoice-7B, short frame counts (the headline stays on config #2) ----
    extra_configs = []
    if dump:
        outputs = {"audio": audio_out.permute(1, 0, 2).reshape(B, F * 3200).cpu().numpy(),
                   "token_logits": logits_out.permute(1, 0, 2).cpu().numpy()}
        if e2e is not None:
            outputs["e2e_audio"] = torch.cat(wav).numpy()
        dump_outputs(args.dump_outputs, outputs)

    if args.model == "1.5b" and not args.no_7b:
        model.engine.close()
        del model, eng
        torch.cuda.empty_cache()
        for (tag, b7, L7, F7) in (("7b ctx 30720, 1 prompt/GPU (BASELINE config #3 shape)", 1, 30720, 48),
                                  ("7b 4 prompts/GPU, 256-token prompts (BASELINE config #4 per-GPU share)", 4, 256, 48)):
            # (a sub-config must never take the headline line down with it: run_extra_config reports its own failures)
            extra_configs.append(run_extra_config(tag, "7b", b7, L7, F7, args, rank, world, local, dev, peak))
            log("extra config done: %s" % tag)

    if rank == 0:
        line = {"metric": "audio_seconds_per_second", "value": round(value, 3), "unit": "audio-s/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": round(ms_value / K, 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
                "data": "synthetic", "config": config_dict(args, cfg, L0, F), "rtf": round(1.0 / (value / world), 5),
                "roofline": roofline, "diffusion_head_step_us": round(head_step_us, 2),
                "diffusion_head_step_floor_us": round(wb["head_step"] / peak / 1e3, 2),
                "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clk, "configs": extra_configs,
                "weight_bytes": wb, "setup_s": round(time.time() - t_setup, 1)}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------------------
def run_streaming_latency(args):
    """BASELINE config #5: VibeVoice-Streaming-0.5B, 8K-token cached prompt, 5 diffusion steps, cfg 1.5, text / speech windows 5 / 6 --
    p50 of the time from generate() entry to the first [1, 3200] chunk handed to AudioStreamer.put, over `--runs` calls
    (demo/streaming_inference_from_file.py:170, 291: the prompt state comes from a cached `all_prefilled_outputs`, as here)."""
    from types import SimpleNamespace
    from vibevoice_b200 import streaming as S
    from vibevoice_b200.configuration import preset_config
    from vibevoice_b200.streamer import AudioStreamer
    from vibevoice_b200.synth import iter_synth_state_dict_fast
    dev = torch.device("cuda", 0)
    cfg = preset_config("streaming-0.5b")
    dc = cfg.decoder_config
    H, tts_layers = dc.hidden_size, 20
    low = dc.num_hidden_layers - tts_layers
    L0 = args.prompt_len or 8192
    steps = 5 if args.diffusion_steps == 30 else args.diffusion_steps
    g = torch.Generator(device=dev).manual_seed(7)

    def items():
        for name, t in iter_synth_state_dict_fast(cfg, 1234, device=dev, parts=("lm", "head", "acoustic_decoder", "connectors")):
            if not name.startswith("model.semantic"):          # the streaming model has no semantic branch (zero-filled by the loader)
                yield name, t
        yield "model.tts_input_types.weight", torch.randn(2, H, device=dev, generator=g) * 0.05
        yield "tts_eos_classifier.fc1.weight", torch.randn(H, H, device=dev, generator=g) * 0.05
        yield "tts_eos_classifier.fc1.bias", torch.zeros(H, device=dev)
        yield "tts_eos_classifier.fc2.weight", torch.randn(1, H, device=dev, generator=g) * 0.05
        yield "tts_eos_classifier.fc2.bias", torch.full((1,), -8.0, device=dev)       # never stops inside the measured window
    t_setup = time.time()
    m = S.VibeVoiceStreamingForConditionalGenerationInference(cfg, tts_backbone_num_hidden_layers=tts_layers)
    m.load_state_dict(items())
    m.set_ddpm_inference_steps(steps)
    eng = m.engine

    def cache(n_layers, L):          # the reference's cached-prompt format: per-layer (key, value) [1, kv_heads, L, head_dim], bf16, rotated keys
        return tuple((torch.randn(1, dc.num_key_value_heads, L, dc.head_dim, device=dev, generator=g).to(torch.bfloat16) * 0.5,
                      torch.randn(1, dc.num_key_value_heads, L, dc.head_dim, device=dev, generator=g).to(torch.bfloat16) * 0.5) for _ in range(n_layers))
    out = lambda n, L: SimpleNamespace(past_key_values=cache(n, L), last_hidden_state=torch.randn(1, L, H, device=dev, generator=g) * 0.1)
    prefilled = {"lm": out(low, L0), "tts_lm": out(tts_layers, L0), "neg_lm": out(low, 1), "neg_tts_lm": out(tts_layers, 1)}
    prompt = torch.randint(0, 150000, (L0,))
    text = torch.randint(0, 150000, (40,))
    log("streaming model ready (%d-token cached prompt)" % L0)

    class FirstChunk(AudioStreamer):
        def __init__(self):
            super().__init__(batch_size=1)
            self.t_first = None

        def put(self, audio_chunks, sample_indices):
            if self.t_first is None:
                self.t_first = time.perf_counter()
            super().put(audio_chunks, sample_indices)
    lat = []
    clocks = ClockSampler(0)
    for it in range(args.warmup + args.runs):
        if it == args.warmup:
            clocks.start()
        st = FirstChunk()
        torch.manual_seed(it)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        res = m.generate(input_ids=prompt[None], tts_lm_input_ids=prompt[None], tts_text_ids=text[None], neg_text_input_id=151655,
                         cfg_scale=1.5 if args.cfg_scale == 1.3 else args.cfg_scale, max_new_tokens=5 + 6, all_prefilled_outputs=prefilled,
                         audio_streamer=st)
        if it >= args.warmup:
            lat.append((st.t_first - t0) * 1e3)
        assert res.speech_outputs[0] is not None and res.speech_outputs[0].shape[-1] >= 3200
    clk = clocks.stop()
    lat = np.asarray(lat)
    line = {"metric": "first_audio_latency_ms_p50", "value": round(float(np.percentile(lat, 50)), 3), "unit": "ms", "n_gpus": 1, "steps": args.runs,
            "warmup": args.warmup, "ms_per_step": round(float(lat.mean()), 3), "higher_is_better": False, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "VibeVoice-Streaming-0.5B random-init (24 layers = 4 text + 20 TTS, H 896, 14/2 heads of 64), %d-token cached prompt "
                                   "imported through vv_kv_write, first text window of 5 tokens, %d diffusion steps, cfg 1.5: generate() entry -> "
                                   "first [1,3200] chunk at AudioStreamer.put" % (L0, steps), "prompt_len": L0, "diffusion_steps": steps},
            "p90_ms": round(float(np.percentile(lat, 90)), 3), "min_ms": round(float(lat.min()), 3), "clocks": clk,
            "gpu_launches": int(eng.launch_count()), "setup_s": round(time.time() - t_setup, 1)}
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    if args.model == "streaming-0.5b":
        return run_streaming_latency(args)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
