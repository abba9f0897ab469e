#!/usr/bin/env python
"""Benchmark of the VisualCLA hot path on B200 (contract: see the task's section (4) and DESIGN.md "Measurement").

A "step" = one pass of the whole path over one batch of synthetic requests:
    B images (224x224) + 64-token prompts -> ViT-L/14 -> Resampler -> projector -> LLaMA-7B prefill (S = 128)
    -> 256 greedy tokens (KV-cached decode, CUDA graph), i.e. BASELINE.json configs[1] (batch 8 per GPU).
metric = images+256-token generations per second (whole job, all GPUs).

  python bench.py --gpus 1 --steps 5 --warmup 3            # this repo's CUDA path
  python bench.py --impl reference ...                      # reference algorithm on the host cores (CPU oracle port)
  torchrun --nproc-per-node N bench.py --gpus N ...         # data parallel, one rank per GPU, weak scaling
  python bench.py ... --dump-outputs DIR                    # also write the last timed step's tokens as DIR/tokens.npy
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "visual-chinese-llama-alpaca_b200"))

METRIC = "image+64-token-prompt -> 256-token generations per second (VisualCLA-7B path)"
UNIT = "gens/s"
T_TEXT, N_NEW, NQ = 64, 256, 64
S_PREFILL = T_TEXT + NQ


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference", "hf-cuda"])
    ap.add_argument("--hf-dtype", default="float16", choices=["float16", "bfloat16"], help="hf-cuda arm: the reference ships fp16 (inference.py:47)")
    ap.add_argument("--batch-per-gpu", type=int, default=8)
    ap.add_argument("--new-tokens", type=int, default=N_NEW)
    ap.add_argument("--prompt-tokens", type=int, default=T_TEXT, help="text tokens per prompt (64 = configs[1]; 128 = configs[2])")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --batch-per-gpu requests on every GPU; strong: a fixed global batch of 64 (SURVEY 8d config 4: B_local = 64/N)")
    ap.add_argument("--no-extras", action="store_true", help="skip the configs[2] / configs[4] / strong-scaling / HF-CUDA blocks of the default line")
    ap.add_argument("--pdl", type=int, default=int(os.environ.get("VCLA_PDL", "1")))
    ap.add_argument("--dump-outputs", metavar="DIR", help="native arm: after the timed steps, write the (global batch, new tokens) greedy "
                                                          "tokens of the last timed step to DIR/tokens.npy (float64), to compare builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes the native arm's outputs; use it with --impl native")
    return args


def dump_outputs(out_dir, tokens):
    """Write what one timed step returned to its caller: the greedy tokens, exact in float64."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "tokens.npy"), tokens.cpu().numpy().astype(np.float64))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sus=d.get("bf16_tflops_sustained", d["bf16_tflops"]), source="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sus=1400.0, source="fallback")


# ----------------------------------------------------------------------------------------------------------------
# algorithmic work (SURVEY.md section 8d / BASELINE.md section 3)
# ----------------------------------------------------------------------------------------------------------------
BODY_PARAMS, LM_PARAMS = 6.476e9, 0.2046e9
VISION_FLOP_PER_IMAGE = 179.2e9
KV_BYTES_PER_TOKEN = 524288


def decode_step_bytes(B, ctx):
    return (BODY_PARAMS + LM_PARAMS) * 2 + B * (ctx + 1) * KV_BYTES_PER_TOKEN


def prefill_flops(B, S):
    per_tok = 2 * BODY_PARAMS + 4 * 4096 * 32 * (S + 1) / 2
    return B * (VISION_FLOP_PER_IMAGE + S * per_tok + 2 * LM_PARAMS)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (profiling recipe's clocks line)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self._stop = index, [], threading.Event()
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self.t.join(timeout=6)

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for n, v in zip(names, r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def synth_inputs(B, seed=1234, T=T_TEXT):
    """SURVEY 8(d): randn pixels (CLIP-normalised scale), ids = [BOS, <img>, </img>, uniform random...]."""
    import torch
    g = torch.Generator().manual_seed(seed)
    px = torch.randn(B, 3, 224, 224, generator=g).half()
    ids = torch.randint(3, 49954, (B, T), generator=g)
    ids[:, 0], ids[:, 1], ids[:, 2] = 1, 49954, 49955
    return px, ids


# ----------------------------------------------------------------------------------------------------------------
# CPU leg: the oracle port of the reference algorithm on the host cores, bounded sample, extrapolated
# ----------------------------------------------------------------------------------------------------------------
_CPU_STATE = {}


def cpu_reference_sample(B, n_new, sample_B=2, decode_steps=8, threads=None):
    """One bounded CPU sample of the workload with the oracle port (weights are built once per process)."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import visualcla_oracle as O
    # a FIXED thread count (round 1 let a micro-benchmark pick 32 or 64 and the two boxes differed 5x): 32 threads, or every core
    # of a smaller host; os.cpu_count() threads is pathologically slow on the 128-cpu GPU box
    threads = threads or min(32, os.cpu_count() or 1)
    torch.set_num_threads(threads)
    cfg = O.PathConfig()
    if "w" not in _CPU_STATE:
        block = torch.randn(1 << 20)
        w = {}
        for name, shape, std, mean in O.weight_specs(cfg):      # values are irrelevant for timing; finite + non-denormal
            n = 1
            for s in shape:
                n *= s
            reps = (n + block.numel() - 1) // block.numel()
            w[name] = (block.repeat(reps)[:n] * float(std) + float(mean)).reshape(shape)
        _CPU_STATE["w"] = w
    w = _CPU_STATE["w"]
    px, ids = O.make_inputs(cfg, B, T_TEXT, seed=1234)
    sample_B = min(sample_B, B)
    with torch.no_grad():
        t0 = time.perf_counter()
        img = O.vision_encode(w, cfg, px[:sample_B])
        t_vis = (time.perf_counter() - t0) * (B / sample_B)
        s0, s1, _, s3 = O.special_ids(cfg)
        x = O.splice(w, cfg, ids[:sample_B], img, True, s0, s1, s3)
        cache = O.KVCache(cfg.t_layers)
        t0 = time.perf_counter()
        O.llama_forward(w, cfg, x, cache, last_only=True)
        t_pre = (time.perf_counter() - t0) * (B / sample_B)
        # decode at the full batch B (CPU decode is weight-bandwidth bound: time per step ~ independent of B)
        reps = (B + sample_B - 1) // sample_B
        for i in range(cfg.t_layers):
            cache.k[i] = cache.k[i].repeat(reps, 1, 1, 1)[:B]
            cache.v[i] = cache.v[i].repeat(reps, 1, 1, 1)[:B]
        tok = torch.randint(3, 49954, (B,))
        t0 = time.perf_counter()
        for _ in range(decode_steps):
            e = w["text_model.model.embed_tokens.weight"][tok].unsqueeze(1)
            tok = O.llama_forward(w, cfg, e, cache, last_only=True)[:, -1].argmax(-1)
        t_dec = (time.perf_counter() - t0) / decode_steps
    total = t_vis + t_pre + (n_new - 1) * t_dec
    return {"value": B / total, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"oracle/visualcla_oracle.py fp32 on {threads} host threads: vision+prefill measured on {sample_B} of {B} requests "
                      f"(x{B / sample_B:g}), {decode_steps} decode steps at batch {B}; extrapolated to {n_new} tokens "
                      f"(vision {t_vis:.2f}s + prefill {t_pre:.2f}s + {n_new - 1} x {t_dec:.3f}s)",
            "seconds_per_step_extrapolated": total}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    B = args.batch_per_gpu * args.gpus
    vals = []
    for i in range(args.warmup + args.steps):
        r = cpu_reference_sample(B, args.new_tokens)
        if i >= args.warmup:
            vals.append(r)
    value = statistics.mean(v["value"] for v in vals)
    last = vals[-1]
    last["value"] = value
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000.0 * B / value, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": {"workload": f"configs[1]: batch {args.batch_per_gpu}/GPU x {args.gpus} GPU, 224x224 images, "
                                            f"{T_TEXT}-token prompts, {args.new_tokens}-token greedy decode (host CPU, no GPU)"},
            "cpu_baseline": last, "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------
# native arm
# ----------------------------------------------------------------------------------------------------------------
TRACE_TAGS = {1: "gemm_swap", 2: "gemm", 3: "attn_prefill", 4: "attn_decode", 5: "layernorm", 6: "rmsnorm", 7: "rope_cache", 8: "resid_norm",
              9: "silu_mul", 10: "logits1", 11: "logits2", 12: "advance", 13: "embed", 14: "sampler"}
GEMM_BYTES = {"qkv": 3 * 4096 * 4096 * 2, "o_proj": 4096 * 4096 * 2, "gate_up": 2 * 11008 * 4096 * 2, "down_proj": 4096 * 11008 * 2, "lm_head": 49958 * 4096 * 2}


def insitu_decode_kernels(eng, tok, n_layers=32):
    """Per-kernel time INSIDE a graph-replayed decode step, from the in-kernel %globaltimer trace (vcla_trace_*): a kernel's in-situ
    duration = the time between its own dependency resolving and its successor's dependency resolving (= its whole grid, the
    launch gap included), so the durations of one step add up to the step.
    -> ({kernel: mean microseconds}, {kernel: launches counted}, traced span of the step in microseconds)."""
    import torch
    for _ in range(3):
        eng.decode_step(tok, tok, None)          # single-step graph: captured + warm
    torch.cuda.synchronize()
    eng.trace_enable(4096)
    eng.decode_step(tok, tok, None)
    torch.cuda.synchronize()
    ev = eng.trace_read()
    eng.trace_enable(0)
    ev = [e for e in ev if e[2]]                  # kernels that recorded their dependency time
    ev.sort(key=lambda r: r[2])
    names, gi = [], 0
    order = ["qkv", "o_proj", "gate_up", "down_proj"]
    for tag, _a, _b, _c in ev:
        if tag == 1:
            names.append(order[gi % 4] if gi < 4 * n_layers else "lm_head")
            gi += 1
        else:
            names.append(TRACE_TAGS.get(tag, str(tag)))
    dur = {}
    for i in range(len(ev) - 1):
        dur.setdefault(names[i], []).append((ev[i + 1][2] - ev[i][2]) / 1e3)
    return {k: statistics.mean(v) for k, v in dur.items()}, {k: len(v) for k, v in dur.items()}, (ev[-1][2] - ev[0][2]) / 1e3


def run_config(args, world, rank, Bl, T, n_new, steps, warmup, with_e2e, with_trace):
    """Build the 7B model for (batch Bl per GPU, T-token prompts, n_new tokens), time `steps` whole-path steps on the device (inputs
    resident in HBM) and, optionally, end to end from pinned host memory.  Returns a dict of measurements."""
    import torch
    import torch.distributed as dist
    import visualcla
    from visualcla.dp import generate_dp
    B = Bl * world
    S = T + NQ
    max_seq = S + n_new + 1
    model = visualcla.VisualCLAModel.from_synthetic("7b", seed=0, max_batch=Bl, max_seq=max_seq, max_prefill_tokens=Bl * S)
    model.image_at_head = True
    eng = model._engine
    px_h, ids_h = synth_inputs(B, T=T)
    px_h, ids_h = px_h.pin_memory(), ids_h.pin_memory()
    px_d, ids_d = px_h.cuda(non_blocking=True), ids_h.cuda(non_blocking=True)
    torch.cuda.synchronize()
    ev = {}

    def phase_hook(name):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        ev.setdefault(name, []).append(e)

    def step_device():
        return generate_dp(model, ids_d, px_d, n_new, phase_hook=phase_hook)

    def step_e2e():
        out = generate_dp(model, ids_h, px_h, n_new)   # pinned host inputs: each rank copies its slice host -> device inside the timed region
        return out.cpu()                              # device -> host read of the result

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(k):
            out = fn()
        t1.record()
        barrier()
        ms = torch.tensor([t0.elapsed_time(t1)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms), out

    for _ in range(max(warmup, 1)):
        step_device()
    ev.clear()
    eng.kernel_launches(reset=True)
    with ClockSampler(int(os.environ.get("LOCAL_RANK", "0"))) as clocks:
        ms, out = timed(step_device, steps)
    res = {"B_local": Bl, "B": B, "T": T, "S": S, "n_new": n_new, "ms": ms, "steps": steps, "value": B * steps / (ms / 1000.0),
           "launches": eng.kernel_launches(reset=True), "clocks": clocks.summary(), "tokens": out}
    pre_ms = [a.elapsed_time(b) for a, b in zip(ev.get("start", []), ev.get("prefill_done", []))]
    dec_ms = [a.elapsed_time(b) for a, b in zip(ev.get("prefill_done", []), ev.get("done", []))]
    pk = peaks()
    if pre_ms and dec_ms:
        pre, dec = statistics.mean(pre_ms), statistics.mean(dec_ms)
        dec_bytes = sum(decode_step_bytes(Bl, S + i) for i in range(n_new - 1))
        res["phases"] = {
            "prefill_ms": pre, "decode_ms": dec, "decode_ms_per_token": dec / max(1, n_new - 1),
            "prefill": {"bound": "tensor", "achieved": prefill_flops(Bl, S) / (pre / 1e3) / 1e12, "peak": pk["tf_sus"], "unit": "TFLOP/s",
                        "frac": prefill_flops(Bl, S) / (pre / 1e3) / 1e12 / pk["tf_sus"],
                        "note": "vision + LLaMA prefill, algorithmic FLOPs / CUDA-event time, of " + pk["source"] + " sustained bf16 peak"},
            "decode": {"bound": "hbm", "achieved": dec_bytes / (dec / 1e3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                       "frac": dec_bytes / (dec / 1e3) / 1e9 / pk["hbm"],
                       "note": f"{n_new - 1} graph-captured decode steps, algorithmic bytes (13.361 GB weights + KV, mean ctx {S + (n_new - 1) / 2.0:.0f}) / CUDA-event time"}}
    if with_e2e:
        step_e2e()
        ms_e2e, out_e2e = timed(step_e2e, steps)
        assert torch.equal(out_e2e, out.cpu()), "e2e and device-resident runs must produce the same tokens"
        res["e2e"] = {"value": B * steps / (ms_e2e / 1000.0), "unit": UNIT, "h2d_bytes_per_step": int(px_h.numel() * 2 + ids_h.numel() * 8),
                      "d2h_bytes_per_step": int(B * n_new * 8), "ms_per_step": ms_e2e / steps}
    if with_trace and world == 1:
        # chat()'s real default is SAMPLING (ref modeling_utils.py:36-47): the same workload through VisualCLAModel.generate with the
        # reference's DEFAULT_GENERATION_CONFIG -- repetition penalty, no-repeat-ngram, temperature, top-k, top-p and the draw run in
        # one fused kernel per step inside the decode graphs (csrc/sampler.cu)
        try:
            import copy
            from visualcla.modeling_utils import DEFAULT_GENERATION_CONFIG
            gcs = copy.deepcopy(DEFAULT_GENERATION_CONFIG)
            gcs.max_new_tokens, gcs.eos_token_id, gcs.pad_token_id = n_new, None, 0

            def step_sample():
                return model.generate(input_ids=ids_d, pixel_values=px_d, generation_config=gcs)
            step_sample()
            ms_s, out_s = timed(step_sample, 2)
            res["sampling"] = {"value": B * 2 / (ms_s / 1000.0), "unit": UNIT, "ms_per_step": ms_s / 2, "steps": 2,
                               "config": "DEFAULT_GENERATION_CONFIG (do_sample, temperature 0.5, top_k 40, top_p 0.9, repetition_penalty 1.1, no_repeat_ngram_size 15), "
                                         "device-side fused sampler inside the decode CUDA graphs", "shape": list(out_s.shape)}
        except Exception as e:  # noqa: BLE001
            res["sampling"] = {"error": repr(e)}
    if with_trace and rank == 0:
        # the caches now hold S + n_new - 1 tokens: the traced step runs at the END-of-generation context
        tok = eng.token_buffer(Bl)
        mode, rows = model._image_layout(ids_d[:Bl], px_d[:Bl])
        eng.vision_encode(px_d[:Bl])
        _, first, _ = eng.prefill(ids_d[:Bl], mode, rows, all_logits=False, last_logits=False)
        tok.copy_(first)
        eng.decode_many(tok, n_new // 2)            # mid-generation context for the traced step
        try:
            res["insitu_us"], res["insitu_n"], res["insitu_step_us"] = insitu_decode_kernels(eng, tok)
            res["insitu_ctx"] = S + n_new // 2 + 3
        except Exception as e:  # noqa: BLE001
            res["insitu_error"] = repr(e)
        iso = {}
        for i, nm in enumerate(["qkv", "o_proj", "gate_up", "down_proj", "lm_head"]):
            us, nbytes = eng.bench_decode_gemm(i, Bl, reps=3)
            iso[nm] = {"us": us, "GBps": nbytes / us / 1e3, "bytes": nbytes}
        res["isolated"] = iso
    eng.close()
    del model
    torch.cuda.empty_cache()
    return res


def hf_cuda_sample(B, T, n_new, dtype="float16", steps=2):
    """The reference's CUDA path on this GPU (see run_hf_cuda), bounded: 1 warm-up + `steps` timed generations."""
    ns = argparse.Namespace(hf_dtype=dtype, batch_per_gpu=B, new_tokens=n_new, prompt_tokens=T, warmup=1, steps=steps)
    return run_hf_cuda(ns, emit=False)


def run_native(args):
    import torch
    import torch.distributed as dist
    from visualcla import _native

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (native arm) needs a CUDA device: this repo has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    _native.load().vcla_set_pdl(1 if args.pdl else 0)
    if args.scaling == "strong":
        assert 64 % world == 0, "strong scaling uses a global batch of 64"
        args.batch_per_gpu = 64 // world
    Bl, n_new, T = args.batch_per_gpu, args.new_tokens, args.prompt_tokens
    B, S = Bl * world, T + NQ
    main = run_config(args, world, rank, Bl, T, n_new, args.steps, args.warmup, with_e2e=True, with_trace=True)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, main["tokens"])
    pk = peaks()
    cfg_name = {(8, 64, 256): "1", (32, 128, 256): "2", (16, 1024, 512): "4"}.get((Bl, T, n_new), "*")
    line = {"metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": main["ms"] / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic (randn 224x224 pixels, uniform random token ids, hash-normal weights of the VisualCLA-7B architecture)",
            "config": {"workload": f"configs[{cfg_name}]: batch {Bl} per GPU x {world} GPU, 224x224 images, {T}-token prompts (S={S} with 64 image tokens), "
                                   f"{n_new}-token greedy decode, EOS disabled", "global_batch": B, "parallelism": f"dp{world}",
                       "l2": "inputs larger than L2: every decode step streams 13.4 GB of weights (>> 126 MB L2)", "pdl": bool(args.pdl),
                       "token_exchange": "none (1 GPU)" if world == 1 else "NCCL all-gather of the chosen tokens inside the decode CUDA graphs (vcla_nccl_init)"},
            "e2e": main["e2e"], "gpu_launches": int(main["launches"]), "clocks": main["clocks"]}
    if "phases" in main:
        line["phases"] = main["phases"]
    if "sampling" in main:
        line["sampling"] = main["sampling"]
    line["config"]["schedule"] = ("prefill: 5 kernels/layer (deferred RMSNorm + RoPE/KV-append + SwiGLU + residual epilogues in the tcgen05 GEMM, CTA-pair 256x256 "
                                  "tiles, tcgen05 flash attention); decode: 5 kernels/layer (cluster split-K GEMMs with DSMEM reduce and fused consumers), "
                                  "CUDA graphs of 16 steps")
    if rank == 0:
        # ---- roofline of the dominant kernel, IN SITU: the fused gate/up swap-AB tcgen05 GEMM (180.4 MB of weights per launch, the
        #      largest share of a decode step), timed inside a graph-replayed decode step; the isolated micro-benchmark (32 launches
        #      back to back, PDL weight prefetch overlapping neighbours) is reported beside it, not as the headline.
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get("gate_up_dram_bytes_per_launch")
        iso = main.get("isolated", {})
        ins = main.get("insitu_us", {})
        rf = {"bound": "hbm", "peak": pk["hbm"], "unit": "GB/s", "traffic": traffic,
              "kernel": "gemm_tc_kernel<BN,5,swap-AB> fused gate/up projection (22016x4096 bf16 weights, 180.4 MB algorithmic bytes per launch)",
              "of": pk["source"] + " copy bandwidth"}
        if "gate_up" in ins:
            us = ins["gate_up"]
            rf.update({"achieved": GEMM_BYTES["gate_up"] / us / 1e3, "frac": GEMM_BYTES["gate_up"] / us / 1e3 / pk["hbm"], "us": us,
                       "how": "in situ: mean over the 32 layers of one graph-replayed decode step of (successor's dependency-resolved time - own "
                              "dependency-resolved time), %globaltimer trace recorded live by this run (vcla_trace_*)",
                       "in_step_us": {k: round(v, 2) for k, v in ins.items()}, "in_step_launches": main.get("insitu_n"),
                       "in_step_total_us": main.get("insitu_step_us"), "in_step_ctx": main.get("insitu_ctx")})
            floor = {k: GEMM_BYTES[k] / pk["hbm"] / 1e3 for k in GEMM_BYTES}
            rf["in_step_gemm_frac"] = {k: floor[k] / ins[k] for k in floor if k in ins}
        elif "gate_up" in iso:
            rf.update({"achieved": iso["gate_up"]["GBps"], "frac": iso["gate_up"]["GBps"] / pk["hbm"], "how": "isolated (trace unavailable: " + str(main.get("insitu_error")) + ")"})
        if iso:
            rf["isolated"] = {"achieved": iso["gate_up"]["GBps"], "frac": iso["gate_up"]["GBps"] / pk["hbm"], "per_shape": iso,
                              "how": "kernel timed alone with CUDA events over 32 layers' distinct weights, 3 repetitions (burst)"}
        if "phases" in main:
            rf["decode_step_frac"] = main["phases"]["decode"]["frac"]      # what the product delivers: the whole step against the HBM floor
        line["roofline"] = rf
    extras = not args.no_extras and args.scaling == "weak" and (Bl, T, n_new) == (8, 64, 256)
    if extras:
        # ---- the other BASELINE configs and the strong-scaling point, on the same box in the same run (bounded: 1 warm-up + 2 steps)
        blocks = {}
        plan = [("strong_scaling", 64 // world if 64 % world == 0 else None, 64, 256)]
        if world == 1:
            plan = [("configs[2]", 32, 128, 256), ("configs[4]", 16, 1024, 512)] + plan
        for name, b_, t_, n_ in plan:
            if b_ is None:
                continue
            try:
                if name == "strong_scaling" and b_ == Bl:
                    r = main                                   # N = 8: the strong-scaling point IS the main measurement
                else:
                    r = run_config(args, world, rank, b_, t_, n_, 2, 1, with_e2e=False, with_trace=False)
                blk = {"batch_per_gpu": b_, "global_batch": b_ * world, "prompt_tokens": t_, "new_tokens": n_, "value": r["value"], "unit": UNIT,
                       "ms_per_step": r["ms"] / r["steps"], "steps": r["steps"]}
                if "phases" in r:
                    blk.update({"prefill_ms": r["phases"]["prefill_ms"], "prefill_frac": r["phases"]["prefill"]["frac"],
                                "decode_ms_per_token": r["phases"]["decode_ms_per_token"], "decode_frac": r["phases"]["decode"]["frac"]})
                blocks[name] = blk
            except Exception as e:  # noqa: BLE001
                blocks[name] = {"error": repr(e)}
        if "strong_scaling" in blocks:
            blocks["strong_scaling"]["note"] = ("fixed global batch 64 (SURVEY 8d config 4): B_local = 64/N.  Weights are replicated (data parallel), so every GPU "
                                                "still streams the full 13.4 GB per decode step whatever its B_local: expect ~N-independent step time, "
                                                "i.e. poor strong scaling by design of the DP layout north_star prescribes")
        line["configs"] = blocks
    if rank == 0:
        if world == 1 and extras:
            try:
                hf = hf_cuda_sample(Bl, T, n_new, "float16")
                line["hf_cuda_baseline"] = {"value": hf["value"], "unit": UNIT, "dtype": "fp16", "ms_per_step": hf["ms_per_step"], "steps": hf["steps"],
                                            "ratio_e2e": line["e2e"]["value"] / hf["value"], "what": hf["config"]["workload"]}
            except Exception as e:  # noqa: BLE001
                line["hf_cuda_baseline"] = {"error": repr(e)}
        if world == 1 and not args.no_cpu_baseline:
            try:
                line["cpu_baseline"] = cpu_reference_sample(Bl, n_new)
            except Exception as e:  # noqa: BLE001
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {e}"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------------------------
# informational arm: the reference's CUDA path = HF CLIPVisionModel + the Resampler arithmetic in torch + HF
# LlamaForCausalLM.generate(inputs_embeds=...) on the same GPU, same shapes, random weights (north star's 8x denominator).
# /root/reference is not on the GPU box, so the composite module is re-assembled from the very HF classes it calls
# (modeling_visualcla.py:346-391) and the oracle's torch restatement of the in-repo Resampler, run on the device.
# ----------------------------------------------------------------------------------------------------------------
def hf_cuda_step(B, T, n_new, dt):
    """Build the HF composite on cuda:0 with random weights and return step(): one batch of greedy generations, (B, n_new) tokens."""
    import torch
    from transformers import LlamaConfig, LlamaForCausalLM, GenerationConfig
    from transformers.models.clip.modeling_clip import CLIPVisionConfig, CLIPVisionModel
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import visualcla_oracle as O
    cfg = O.PathConfig()
    old = torch.get_default_dtype()
    torch.set_default_dtype(dt)
    with torch.device("cuda"):
        llama = LlamaForCausalLM(LlamaConfig(vocab_size=cfg.t_vocab, hidden_size=cfg.t_hidden, intermediate_size=cfg.t_ffn, num_hidden_layers=cfg.t_layers,
                                             num_attention_heads=cfg.t_heads, num_key_value_heads=cfg.t_heads, rms_norm_eps=cfg.t_eps,
                                             max_position_embeddings=2048, tie_word_embeddings=False, pad_token_id=0, bos_token_id=1, eos_token_id=2)).eval()
        clip = CLIPVisionModel(CLIPVisionConfig(hidden_size=cfg.v_hidden, intermediate_size=cfg.v_ffn, num_hidden_layers=cfg.v_layers,
                                                num_attention_heads=cfg.v_heads, image_size=cfg.v_image, patch_size=cfg.v_patch, hidden_act="quick_gelu")).eval()
        w = {n: torch.randn(*sh) * std + mean for n, sh, std, mean in O.weight_specs(cfg) if n.startswith(("visual_resampler.", "image_projection_layer."))}
    torch.set_default_dtype(old)
    px_h, ids_h = synth_inputs(B, T=T)
    px, ids = px_h.cuda().to(dt), ids_h.cuda()
    gc = GenerationConfig(do_sample=False, max_new_tokens=n_new, min_new_tokens=n_new, eos_token_id=None, pad_token_id=0)

    @torch.no_grad()
    def step():
        emb = llama.get_input_embeddings()(ids)
        vit = clip(pixel_values=px)[0]
        post = clip.vision_model.post_layernorm(vit)
        img = O.project(w, O.resampler_forward(w, cfg, post))
        x = torch.cat([emb[:, :2], img.to(dt), emb[:, 2:]], dim=1)
        mask = torch.ones(x.shape[:2], dtype=torch.long, device="cuda")
        return llama.generate(inputs_embeds=x, attention_mask=mask, generation_config=gc)
    return step


def run_hf_cuda(args, emit=True):
    """Time args.steps generations of the HF composite after max(1, args.warmup) warm-up generations (one is needed to check the shape)."""
    import torch
    if int(os.environ.get("RANK", "0")) != 0:
        return
    B, n_new, T = args.batch_per_gpu, args.new_tokens, args.prompt_tokens
    torch.cuda.set_device(0)
    step = hf_cuda_step(B, T, n_new, getattr(torch, args.hf_dtype))
    warmup = max(1, args.warmup)
    for _ in range(warmup):
        out = step()
    assert out.shape == (B, n_new), out.shape
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(args.steps):
        step()
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / args.steps
    del step, out
    torch.cuda.empty_cache()
    line = ({"impl": "hf-cuda", "metric": METRIC, "value": B / (ms / 1e3), "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": warmup, "ms_per_step": ms,
                      "higher_is_better": True, "dtype": args.hf_dtype, "data": "synthetic, random weights",
                      "config": {"workload": f"batch {B}, {T}-token prompts + 64 image tokens, {n_new} greedy tokens; HF CLIPVisionModel + torch Resampler + "
                                             f"HF LlamaForCausalLM.generate(inputs_embeds) eager/SDPA, transformers {__import__('transformers').__version__}"}})
    if emit:
        print(json.dumps(line), flush=True)
    return line


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "hf-cuda":
        run_hf_cuda(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
