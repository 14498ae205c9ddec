#!/usr/bin/env python
"""GRPO-step throughput of the B200-native BioReason hot path (BASELINE.json metric), plus the CPU reference arm.

  python bench.py --gpus N --steps K --warmup W            # our arm (torchrun launches N ranks for N > 1)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's HF/PyTorch path on the host cores (oracle)

A "step" is one full GRPO optimizer step of config (c) (SURVEY.md §8d): per GPU 1 prompt x G=8 rollouts of C=512 tokens
(EOS suppressed) from a 2 x 668-token-DNA + 512-token-text prompt (P=1848), NT-v2-500M + Qwen3-4B, random-init bf16 weights
(no checkpoints offline), ref-logps forward, policy forward + backward (LoRA r=32 + projector), gradient all-reduce,
AdamW.  value = completion tokens generated-and-trained per second over all ranks.
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
sys.path.insert(0, ROOT)
# one growing VMM segment per size class instead of cudaMalloc/cudaFree round trips (multi-second stalls under multi-process load)
os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:True")


def _positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError("must be at least 1")
    return v


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=_positive_int, default=3, help="timed GRPO steps (each of the resident and the e2e timings runs this many)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--text", default="qwen3-4b")
    ap.add_argument("--dna", default="nt-v2-500m")
    ap.add_argument("--G", type=int, default=8)
    ap.add_argument("--prompts-per-gpu", type=int, default=1)
    ap.add_argument("--dna-len", type=int, default=668)
    ap.add_argument("--text-len", type=int, default=512)
    ap.add_argument("--completion", type=int, default=512)
    ap.add_argument("--micro-rows", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sweep", action="store_true", help="skip the secondary resident-row lines (16 / 32 rows per GPU)")
    ap.add_argument("--cpu-budget-s", type=float, default=25.0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last timed step computed as DIR/<name>.npy")
    return ap.parse_args()


# ----------------------------------------------------------------------------------------------------------------
# clocks sampling during the timed region (B200_PROFILING.md)
# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.idx)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=3)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------
# workload
# ----------------------------------------------------------------------------------------------------------------
def make_prompt_batch(tc, dc, args, seed):
    """`prompts_per_gpu` distinct prompts, each repeated G times consecutively (RepeatRandomSampler layout), on the host."""
    import torch
    from bioreason_b200.synth import synth_batch
    groups = [synth_batch(tc, dc, batch=args.G, n_seq=2, dna_len=args.dna_len, text_len=args.text_len, seed=seed + 17 * i, same_prompt=True)
              for i in range(args.prompts_per_gpu)]
    if len(groups) == 1:
        return groups[0]
    out = dict(input_ids=torch.cat([g["input_ids"] for g in groups]), attention_mask=torch.cat([g["attention_mask"] for g in groups]),
               dna_tokenized={k: torch.cat([g["dna_tokenized"][k] for g in groups]) for k in ("input_ids", "attention_mask")}, batch_idx_map=[])
    for i, g in enumerate(groups):
        out["batch_idx_map"] += [b + i * args.G for b in g["batch_idx_map"]]
    return out


def workload_string(args):
    return ("(c) NT-v2-500M + Qwen3-4B GRPO step: %d prompt x G=%d per GPU, P=%d (2x%d DNA + 4 delimiters + %d text), C=%d, EOS suppressed, "
            "mu=1, beta=0.04, LoRA r=32 + projector, AdamW" % (args.prompts_per_gpu, args.G, args.text_len + 2 * (args.dna_len + 2),
                                                               args.dna_len, args.text_len, args.completion))


def algorithmic_work(tc, dc, args):
    """SURVEY.md §8d A_min: FLOPs of the dense phases and HBM bytes of the decode phase, per GPU per step."""
    d, F, V, nl = tc.hidden_size, tc.intermediate_size, tc.vocab_size, tc.num_hidden_layers
    Hq, Hkv, D = tc.num_attention_heads, tc.num_key_value_heads, tc.head_dim
    body = nl * ((Hq + 2 * Hkv) * D * d + Hq * D * d + 3 * F * d)                  # matmul params / token
    head = V * d
    G, C = args.G, args.completion
    P = args.text_len + 2 * (args.dna_len + 2)
    L = P + C
    npg = args.prompts_per_gpu
    attn = lambda n: nl * 4 * Hq * D * n * n / 2
    enc_body = dc.num_hidden_layers * (4 * dc.hidden_size ** 2 + 3 * dc.intermediate_size * dc.hidden_size)
    enc = 2 * args.dna_len * 2 * enc_body + dc.num_hidden_layers * 4 * dc.hidden_size * args.dna_len ** 2 * 2
    row_fwd = L * 2 * body + C * 2 * head + attn(L)
    dense = npg * (3 * enc + (P * 2 * body + attn(P))                              # encode (rollout/ref/policy) + shared prefill
                   + G * row_fwd * 2                                               # ref fwd + policy fwd
                   + G * (L * 2 * body + C * 4 * head + 2.5 * attn(L)))            # policy bwd: dX only, attn bwd 2.5x, lm_head dlogits+dH
    kv_tok = nl * 2 * Hkv * D * 2
    decode_bytes = (C - 1) * (2 * (body + head) + npg * kv_tok * (P + G * C / 2))
    return dict(dense_flops=dense, decode_bytes=decode_bytes, decode_weight_bytes_per_token_step=2 * (body + head))


DUMP_SAMPLE = 1 << 20          # at most this many of the trainable parameters / gradients are written (there are 68.7 M at config (c))


def dump_outputs(out_dir, trainer, model, loss):
    """What the last training step computed, as out_dir/<name>.npy (float32; the sample indices float64): its loss and metrics, the
    rollout and scores it trained on, and a fixed seeded sample of the trainable parameters after its optimizer step and of the
    gradients that step applied.  Two builds run with the same arguments see the same inputs, so their dumps compare entry by entry."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    step = trainer._buffered_inputs[(trainer._step - 1) % trainer.args.gradient_accumulation_steps]
    out = {"loss": loss}
    for k in ("kl", "clip_ratio"):
        if trainer._metrics.get(k):
            out[k] = trainer._metrics[k][-1]
    for k in ("completion_ids", "completion_mask", "advantages", "ref_per_token_logps", "old_per_token_logps"):
        if step[k] is not None:
            out[k] = step[k]
    ps = model.trainable_parameters()
    params = torch.cat([p.detach().reshape(-1).float() for p in ps])
    grads = torch.cat([p.grad.reshape(-1).float() for p in ps])
    n = params.numel()
    idx = torch.arange(n) if n <= DUMP_SAMPLE else torch.randint(n, (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).unique()
    out["sample_index"] = idx.double()
    out["trainable_params_sample"] = params[idx.to(params.device)]
    out["trainable_grads_sample"] = grads[idx.to(grads.device)]
    for name, v in out.items():
        a = torch.as_tensor(v).detach().cpu()
        np.save(os.path.join(out_dir, name + ".npy"), (a if a.dtype == torch.float64 else a.float()).numpy())


def run_b200(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1)); local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from bioreason_b200.build import ensure_built
    ensure_built()                                                         # the .so normally travels with the tree; build it if it does not
    from bioreason_b200 import ops
    from bioreason_b200.configs import dna_config, text_config
    from bioreason_b200.models import DNALLMModel
    from bioreason_b200.trainer import DNALLMGRPOConfig, DNALLMGRPOTrainer
    tc, dc = text_config(args.text), dna_config(args.dna)
    t_build = time.perf_counter()
    model = DNALLMModel(tc, dc, seed=1234)                               # same seed on every rank -> replicated weights
    B = args.G * args.prompts_per_gpu
    cfg = DNALLMGRPOConfig(num_generations=args.G, max_completion_length=args.completion, per_device_train_batch_size=B,
                           suppress_eos=True, micro_rows=args.micro_rows or None, seed=1234)
    gen = torch.Generator(device="cuda").manual_seed(99 + rank)

    def synthetic_reward(completion_ids, **kw):                          # seeded N(0,1) per row (replaces the CPU regex rewards)
        return torch.randn(completion_ids.shape[0], device="cuda", generator=gen)
    trainer = DNALLMGRPOTrainer(model, [synthetic_reward], cfg)
    torch.cuda.synchronize()
    t_build = time.perf_counter() - t_build

    host = make_prompt_batch(tc, dc, args, seed=1000 + rank)
    pinned = {"input_ids": host["input_ids"].pin_memory(), "attention_mask": host["attention_mask"].pin_memory(),
              "dna_ids": host["dna_tokenized"]["input_ids"].pin_memory(), "dna_mask": host["dna_tokenized"]["attention_mask"].pin_memory()}
    h2d_bytes = sum(t.numel() * t.element_size() for t in pinned.values())

    def to_device():
        return dict(input_ids=pinned["input_ids"].cuda(non_blocking=True), attention_mask=pinned["attention_mask"].cuda(non_blocking=True),
                    dna_tokenized=dict(input_ids=pinned["dna_ids"].cuda(non_blocking=True), attention_mask=pinned["dna_mask"].cuda(non_blocking=True)),
                    batch_idx_map=host["batch_idx_map"])
    resident = to_device()
    tokens_per_step = B * args.completion * world

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    per_step = {}

    def timed(n, fn, tag=None):
        barrier()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(n + 1)]
        evs[0].record()
        for i in range(n):
            fn()
            evs[i + 1].record()
        barrier()
        if tag:
            per_step[tag] = [round(evs[i].elapsed_time(evs[i + 1]), 1) for i in range(n)]
        ms = torch.tensor([evs[0].elapsed_time(evs[n])], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    for _ in range(args.warmup):
        trainer.training_step(resident)
    import gc
    gc.collect(); gc.freeze(); gc.disable()                               # no collector pauses inside the timed regions (host jitter)
    trainer.timings.clear()
    trainer.gpu_phase_ms()
    ops.LAUNCHES[0] = 0
    clocks = ClockSampler(local)
    clocks.start()
    ms = timed(args.steps, lambda: trainer.training_step(resident), tag="resident")
    launches = ops.LAUNCHES[0]
    phase = {k: v / args.steps for k, v in trainer.timings.items()}
    gpu_phase = {k: v / args.steps / 1e3 for k, v in trainer.gpu_phase_ms().items()}      # CUDA-event seconds per step

    loss_host = torch.zeros(1).pin_memory()

    def e2e_step():
        loss = trainer.training_step(to_device())                        # H2D of this step's inputs from pinned memory
        loss_host.copy_(loss.detach().reshape(1), non_blocking=False)    # D2H read of the step's result
    ms_e2e = timed(args.steps, e2e_step, tag="e2e")
    clk = clocks.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, trainer, model, loss_host)

    # ---- roofline of the dominant kernel: the decode weight-streaming GEMM, timed alone with CUDA events (weights of all
    #      layers = 8 GB >> 126 MB L2, so every launch reads HBM)
    work = algorithmic_work(tc, dc, args)
    W = model._rollout_dec or model._dec
    scratch = ops.skinny_scratch(max(tc.vocab_size, 2 * tc.intermediate_size), "cuda")
    x_d = torch.randn(B if B <= 32 else 32, tc.hidden_size, device="cuda").bfloat16()
    x_f = torch.randn(x_d.shape[0], tc.intermediate_size, device="cuda").bfloat16()
    x_a = torch.randn(x_d.shape[0], tc.num_attention_heads * tc.head_dim, device="cuda").bfloat16()

    ssq = torch.ones(32, device="cuda")

    def stream_weights():
        for Lw in W.layers:
            ops.skinny_gemm(x_d, Lw.w_qkv, scratch, sumsq_in=ssq, eps=1e-6); ops.skinny_gemm(x_a, Lw.w_o, scratch)
            ops.skinny_gemm(x_d, Lw.w_gu, scratch, mode=2, sumsq_in=ssq, eps=1e-6); ops.skinny_gemm(x_f, Lw.w_down, scratch)
        ops.skinny_gemm(x_d, W.lm_head, scratch, mode=3)
    stream_weights()
    torch.cuda.synchronize()
    wgraph = torch.cuda.CUDAGraph()                                       # graph replay: no host launch overhead in the timing
    n0 = ops.LAUNCHES[0]
    with torch.cuda.graph(wgraph):
        stream_weights()
    ops.LAUNCHES[0] = n0
    wgraph.replay()
    n_k = 4 * len(W.layers) + 1
    ms_k = timed(5, wgraph.replay) / 5
    bytes_k = work["decode_weight_bytes_per_token_step"]
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    tf_peak = peaks.get("bf16_tflops_sustained", 1400.0)
    ach = bytes_k / (ms_k * 1e-3) / 1e9
    t_step = ms / args.steps / 1e3
    decode_s = gpu_phase.get("rollout", phase.get("rollout", 0.0))
    dense_s = max(t_step - decode_s, 1e-9)
    roofline = {"bound": "hbm", "kernel": "skinny_tc5_kernel (decode weight streaming, %d launches = all GEMMs of one token step for the group, CUDA-graph replay)" % n_k,
                "achieved": round(ach, 1), "peak": hbm_peak, "unit": "GB/s", "frac": round(ach / hbm_peak, 4),
                # dram__bytes_read+write per launch from the committed `ncu --set full` capture: 50.10 MB for the 49.81 MB down_proj launch and
                # dram read+write 31.6 MB for the 31.46 MB qkv launch, 21.1 / 20.97 (o), 102.9 / 99.6 (gate/up incl. 3.2 MB written), 50.1 / 49.8
                # (down): profiles/r02_ncu_targets.txt -> 1.005 .. 1.03 x the algorithmic bytes; the launch-weighted mean is used
                "traffic": int(1.012 * bytes_k / n_k), "traffic_source": "ncu --set full capture, dram bytes / algorithmic bytes = 1.012 (profiles/r02_ncu_targets.txt)",
                "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback",
                "bytes_per_launch_avg": int(bytes_k / n_k), "launch_us_avg": round(ms_k * 1e3 / n_k, 2),
                "phases": {"rollout_s": round(decode_s, 4), "rollout_hbm_frac": round(work["decode_bytes"] / max(decode_s, 1e-9) / 1e9 / hbm_peak, 4),
                           "dense_s": round(dense_s, 4), "dense_tensor_frac": round(work["dense_flops"] / dense_s / 1e12 / tf_peak, 4),
                           "dense_peak_tflops": tf_peak, "gpu_phase_s": {k: round(v, 4) for k, v in gpu_phase.items()},
                           "host_phase_s": {k: round(v, 4) for k, v in phase.items()}}}

    line = {"metric": "GRPO tokens/sec (rollout+update)", "value": round(tokens_per_step / t_step, 2), "unit": "tokens/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": bench_config(args, world), "build_s": round(t_build, 1),
            "e2e": {"value": round(tokens_per_step / (ms_e2e / args.steps / 1e3), 2), "unit": "tokens/s", "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": 4, "ms_per_step": round(ms_e2e / args.steps, 3)},
            "gpu_launches": int(launches), "clocks": clk, "roofline": roofline,
            "step_ms": per_step, "mem_gb": {"max_allocated": round(torch.cuda.max_memory_allocated() / 2 ** 30, 1),
                                            "max_reserved": round(torch.cuda.max_memory_reserved() / 2 ** 30, 1)}}
    # ---- secondary lines: more prompt groups resident per GPU (NOT the benchmark configuration: BASELINE config (c) is one group of
    #      G = 8; the decode weight stream is amortised over more rows).  Row-chunked forward/backward (micro_rows = 8) keeps the
    #      activation footprint of the 8-row step.
    if world == 1 and not args.no_sweep and args.prompts_per_gpu == 1:
        import copy
        sweep = []
        del trainer
        torch.cuda.empty_cache()
        for ppg in (2, 4):
            try:
                a2 = copy.copy(args); a2.prompts_per_gpu = ppg
                B2 = args.G * ppg
                cfg2 = DNALLMGRPOConfig(num_generations=args.G, max_completion_length=args.completion, per_device_train_batch_size=B2,
                                        suppress_eos=True, micro_rows=args.G, seed=1234)
                tr2 = DNALLMGRPOTrainer(model, [synthetic_reward], cfg2)
                hb = make_prompt_batch(tc, dc, a2, seed=1000 + rank)
                res2 = dict(input_ids=hb["input_ids"].cuda(), attention_mask=hb["attention_mask"].cuda(),
                            dna_tokenized={k: v.cuda() for k, v in hb["dna_tokenized"].items()}, batch_idx_map=hb["batch_idx_map"])
                for _ in range(2):
                    tr2.training_step(res2)
                ms2 = timed(2, lambda: tr2.training_step(res2)) / 2
                sweep.append({"rows_per_gpu": B2, "prompts_per_gpu": ppg, "micro_rows": args.G, "value": round(B2 * args.completion / (ms2 / 1e3), 1),
                              "ms_per_step": round(ms2, 1)})
                del tr2, res2
                torch.cuda.empty_cache()
            except Exception as e:                                        # a secondary line must never take the measurement down
                sweep.append({"rows_per_gpu": args.G * ppg, "error": repr(e)[:160]})
        line["secondary_resident_rows"] = sweep
    if rank == 0 and world == 1 and not args.no_cpu_baseline:              # the CPU baseline is timed at N=1 only
        try:
            line["cpu_baseline"] = cpu_reference(args, budget_s=args.cpu_budget_s)
        except Exception as e:                                            # the baseline must never take the measurement down
            line["cpu_baseline"] = {"error": repr(e)[:200]}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------------------------
# CPU reference arm: the reference's HF/PyTorch path (the oracle) on the host cores, bounded sample
# ----------------------------------------------------------------------------------------------------------------
def _fast_init_(module):
    """Fill every parameter with a tiled block of N(0, 0.02) values (a 4 B-parameter normal_() init alone would take the CPU budget)."""
    import torch
    g = torch.Generator().manual_seed(0)
    block = torch.randn(1 << 20, generator=g) * 0.02
    with torch.no_grad():
        for p_ in module.parameters():
            flat = p_.data.view(-1)
            n = flat.numel()
            reps = (n + block.numel() - 1) // block.numel()
            flat.copy_(block.repeat(reps)[:n] if reps > 1 else block[:n])
        for name, p_ in module.named_parameters():
            if name.endswith("norm.weight") or name.endswith("layernorm.weight"):
                p_.data.fill_(1.0)


def cpu_reference(args, budget_s=25.0):
    """The reference's own path (HF Qwen3 / ESM modules, fp32, the oracle's classes) timed on the host cores at the REAL widths AND
    the real depth on a bounded sample, then composed with the reference's schedule for one GRPO step (A_ref of SURVEY.md §8d: the
    reference re-encodes and re-prefills the prompt for each of the G rows and in every pass).  Measured at full depth (36 decoder
    layers): one row of the reference-policy log-prob pass (L = P + C tokens, [L, V] logits included) and cached decode steps for the
    G rows at context P + C/2; measured on one layer and scaled: the backward (a full-depth fwd+bwd row is ~40 s).  The full-depth
    forward also validates the composition (`fwd_measured_over_composed`)."""
    import torch
    from transformers import DynamicCache
    from transformers.models.qwen3.modeling_qwen3 import Qwen3ForCausalLM
    from bioreason_b200.configs import dna_config, text_config
    from oracle.models import build_dna_model
    tc, dc = text_config(args.text), dna_config(args.dna)
    # "all the host threads it can use": oversubscribing a many-core host makes fp32 GEMMs slower, so pick the fastest of a few
    # thread counts on a probe matmul of the layer's shape and report the count actually used
    ncpu = os.cpu_count() or 1
    a_ = torch.randn(2048, tc.hidden_size); b_ = torch.randn(tc.hidden_size, tc.intermediate_size)
    best, cores = None, 1
    for n in sorted({min(ncpu, k) for k in (8, 16, 32, 64, ncpu)}):
        torch.set_num_threads(n)
        a_ @ b_
        t0 = time.perf_counter(); a_ @ b_; dt = time.perf_counter() - t0
        if best is None or dt < best:
            best, cores = dt, n
    torch.set_num_threads(cores)
    del a_, b_
    G, C = args.G, args.completion
    P = args.text_len + 2 * (args.dna_len + 2)
    L = P + C
    nl, nle = tc.num_hidden_layers, dc.num_hidden_layers
    t_build = time.perf_counter()
    with torch.device("meta"):
        lm = Qwen3ForCausalLM(tc)
    lm = lm.to_empty(device="cpu").eval()
    _fast_init_(lm)
    lm.model.rotary_emb = type(lm.model.rotary_emb)(config=tc)                # buffers (inv_freq) do not survive the meta device
    dc1 = dna_config(args.dna); dc1.num_hidden_layers = 1
    with torch.no_grad():
        enc = build_dna_model(dc1, seed=0)
    t_build = time.perf_counter() - t_build
    layer, head = lm.model.layers[0], lm.lm_head

    def t(fn, reps=1, warm=True):
        if warm:
            fn()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        return (time.perf_counter() - t0) / reps

    ids = torch.randint(0, tc.vocab_size - 8, (1, L))
    with torch.no_grad():
        # ---- measured, full depth: one row of the ref-logps pass (grpo_trainer.py:510-520: all-position logits, log_softmax, gather)
        def ref_row():
            logits = lm(input_ids=ids).logits[:, :-1]
            return torch.gather(logits[0].log_softmax(-1), 1, ids[0, 1:, None])
        fwd_row_full = t(ref_row, warm=False)
        # ---- measured, full depth: cached decode steps for the G rows at context P + C/2 (cache pre-filled, 8 real steps)
        ctx = P + C // 2
        cache = DynamicCache(config=tc)
        kv = torch.randn(G, tc.num_key_value_heads, ctx, tc.head_dim) * 0.1
        for li in range(nl):
            cache.update(kv, kv, li)
        nxt = torch.randint(0, tc.vocab_size - 8, (G, 1))
        n_dec = 8
        t0 = time.perf_counter()
        for s_ in range(n_dec):
            pos = torch.full((G, 1), ctx + s_, dtype=torch.long)
            out = lm(input_ids=nxt, past_key_values=cache, position_ids=pos, use_cache=True)
            nxt = out.logits[:, -1].argmax(-1, keepdim=True)
        dec_step_full = (time.perf_counter() - t0) / n_dec
        del cache, kv
        # ---- measured on one layer (scaled by depth): forward at L and at P, encoder layer
        x = torch.randn(1, L, tc.hidden_size)
        pos = torch.arange(L)[None]
        rot = lm.model.rotary_emb(x, pos)
        fwd_layer = t(lambda: layer(x, position_embeddings=rot, attention_mask=None, position_ids=pos))
        hC = torch.randn(1, L, tc.hidden_size)
        fwd_head = t(lambda: head(hC).float().log_softmax(-1))
        enc_fwd1 = t(lambda: enc.esm.encoder.layer[0](torch.randn(2, args.dna_len, dc.hidden_size)))
    xg = x.clone().requires_grad_(True)
    for p_ in layer.parameters():
        p_.requires_grad_(False)

    def fb():
        out = layer(xg, position_embeddings=rot, attention_mask=None, position_ids=pos)
        (out[0] if isinstance(out, tuple) else out).sum().backward()
    fwdbwd_layer = t(fb)
    fwd_composed = nl * fwd_layer + fwd_head
    # compose the reference's schedule (per prompt group of G rows on one device)
    encode = nle * enc_fwd1                                               # 2 sequences of one row
    prefill_row = fwd_row_full * (P / L)                                  # the rollout's prompt pass (HF computes all-position logits there too)
    t_rollout = G * (encode + prefill_row) + C * dec_step_full
    t_ref = G * (encode + fwd_row_full)
    t_policy = G * (encode + nl * fwdbwd_layer + 3 * fwd_head)
    total = (t_rollout + t_ref + t_policy) * args.prompts_per_gpu
    toks = G * C * args.prompts_per_gpu
    return {"value": round(toks / total, 4), "unit": "tokens/s", "cores": cores, "kind": "port",
            "sample": "oracle (HF Qwen3/ESM fp32, real widths). MEASURED at full depth (%d layers): 1 row of the ref-logps pass at L=%d incl. [L,V] "
                      "logits (%.1fs), %d cached decode steps for G=%d rows at ctx %d (%.3fs/step); measured on 1 layer and scaled: fwd+bwd "
                      "(%.2fs/layer), encoder layer (%.3fs); composed with the reference's own schedule (G-fold re-encode/re-prefill, 3 passes): "
                      "est. %.0f s per GRPO step" % (nl, L, fwd_row_full, n_dec, G, ctx, dec_step_full, fwdbwd_layer, enc_fwd1, total),
            "measured": {"fwd_row_full_depth_s": round(fwd_row_full, 2), "decode_step_full_depth_s": round(dec_step_full, 4),
                         "fwd_layer_s": round(fwd_layer, 3), "fwdbwd_layer_s": round(fwdbwd_layer, 3), "lm_head_logsoftmax_s": round(fwd_head, 2),
                         "encoder_layer_s": round(enc_fwd1, 4), "fwd_measured_over_composed": round(fwd_row_full / fwd_composed, 3),
                         "model_build_s": round(t_build, 1)},
            "est_step_s": round(total, 1)}


def bench_config(args, world):
    """The `config` object both arms print (same keys, same values: the driver compares them)."""
    B = args.G * args.prompts_per_gpu
    return {"workload": workload_string(args), "shapes": f"{args.dna}+{args.text}", "rows_per_gpu": B, "parallelism": f"dp{world}",
            "l2": "weights (8 GB) and activations (>60 GB) exceed the 126 MB L2 every step; no flush needed",
            "weights": "seeded random init (no checkpoints offline)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    t0 = time.perf_counter()
    cb = cpu_reference(args)                                              # one bounded-sample measurement (~1 min of host work)
    line = {"impl": "reference", "metric": "GRPO tokens/sec (rollout+update)", "value": cb["value"], "unit": "tokens/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(cb["est_step_s"] * 1e3, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(args, max(1, args.gpus)),
            "how": "host cores via the CPU oracle (one host, whatever --gpus says): bounded sample at real widths and depth, composed with the "
                   "reference schedule; an EXTRAPOLATED estimate of a >20 min step, not a timed step",
            "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "wall_s": round(time.perf_counter() - t0, 1)}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
