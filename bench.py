#!/usr/bin/env python
"""bench.py — BASELINE.json metric: tokens/sec, Llama-3-8B prefill+decode, 32 concurrent sessions x seq 2048
(configs[1]) on N B200s (one engine replica per GPU, weights copied from rank 0 by ONE ncclBroadcast issued inside
libhelixb200.so; weak scaling: 32 sessions per GPU).

One "step" = every session of the workload served once: `sessions` prompts of `seq` random token ids are submitted
through the C ABI (host buffers), prefilled (continuous batching) and each decodes `decode` tokens over the paged KV
cache.  tokens = sessions * (seq + decode).

  value        : tokens / device time of the forward passes (CUDA events on the engine stream, inputs resident)
  e2e          : tokens / wall time through hb_submit/hb_wait/hb_poll with host buffers (H2D + D2H inside)
  roofline / kernels : one extra profiled step (CUDA-event span around every launch, same stream)
  fixed_total  : BASELINE configs[4] framing in the same line: 256 sessions in total, routed from rank 0 with the
                 scheduler's least-active rule (replica.route_least_active == pickBestWarmSlot), 256/N per GPU
  cpu_baseline / --impl reference : CPU stand-in for the reference's llama.cpp CPU path (cannot run offline): the numpy
                 oracle port on all host threads (pinned with threadpoolctl), bounded sample; --cpu-impl hf switches to
                 HF transformers on torch CPU, which measured 30x slower on the GPU box (profiles/r02c_reference_hf.json)

  --dump-outputs DIR : after the timed steps, what the last one returned to the caller as DIR/<name>.npy (float32 /
                 float64, 64 MB in all, a seeded row sample beyond that); inputs are seeded, so two builds compare output
                 for output

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload llama8b|bge|pack] [--dump-outputs DIR]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "tokens/sec Llama-3-8B prefill+decode (32 sessions x seq 2048, continuous batching)"
UNIT = "tokens/s"


def workload_name(args):
    return (f"Llama-3-8B random-init bf16, {args.sessions} sessions/GPU x ({args.seq} prompt + {args.decode} decode) tokens, "
            f"continuous batching, paged KV (page 64), --max-num-seqs {args.max_seqs}")


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def ncu_traffic(family):
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get(family)
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        load = [s for s, p in zip(sm, pw) if p > 300] or sm
        return {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def session_prompt(global_index, seq, vocab):
    return np.random.default_rng(1000003 + global_index).integers(0, vocab, size=seq, dtype=np.int64).astype(np.int32)


def serve_once(e, hb, prompts, decode):
    """All sessions through the public C-ABI path; returns each session's generated token ids."""
    sp = hb.Sampling(max_tokens=decode, temperature=0.0)
    rids = [e.submit(p, sp) for p in prompts]
    outs = []
    for r in rids:
        got, fin = [], 0
        while not fin:
            e.wait(r, 60000)
            toks, fin = e.poll(r)
            got += toks
        e.release(r)
        outs.append(got)
    return outs


DUMP_BYTES = 64 * 10 ** 6   # everything one --dump-outputs writes, .npy headers included


def dump_outputs(path, outputs, budget=DUMP_BYTES):
    """--dump-outputs: each array of `outputs` as path/<name>.npy.  An array over its share of `budget` is cut to a fixed,
    seeded sample of its rows (same rows on every run of the same arguments), whose indices go to path/<name>_rows.npy."""
    os.makedirs(path, exist_ok=True)
    share = budget // len(outputs) - 2 * 128   # room for the array and its row indices, less two .npy headers
    for name, a in outputs.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        if a.nbytes > share:
            keep = share // (a[0].nbytes + 8)
            rows = np.sort(np.random.default_rng(0).choice(len(a), size=keep, replace=False)).astype(np.float64)
            np.save(os.path.join(path, name + "_rows.npy"), rows)
            a = a[rows.astype(np.int64)]
        np.save(os.path.join(path, name + ".npy"), a)


def serve_latency(e, hb, prompts, decode, spread_s=0.0):
    """Untimed extra pass (SURVEY.md §8d config 2): time to first token and inter-token latency as a client polling the C
    ABI sees them.  spread_s = 0: all sessions submitted at t=0; > 0: arrivals spread uniformly over that many seconds
    (the running streams then meet the later prompts' prefill steps)."""
    sp = hb.Sampling(max_tokens=decode, temperature=0.0)
    n = len(prompts)
    t0 = time.perf_counter()
    arrive = [t0 + spread_s * i / max(1, n - 1) for i in range(n)]
    rids, stamps, sub_t, active, nxt = [], {}, {}, [], 0
    while nxt < n or active:
        now = time.perf_counter()
        while nxt < n and now >= arrive[nxt]:
            r = e.submit(prompts[nxt], sp)
            sub_t[r], stamps[r] = time.perf_counter(), []
            active.append(r)
            nxt += 1
        if active:
            e.wait(active[0], 2)
        else:
            time.sleep(max(0.0, arrive[nxt] - time.perf_counter()))
        now = time.perf_counter()
        for r in list(active):
            toks, fin = e.poll(r)
            stamps[r] += [now] * len(toks)
            if fin:
                active.remove(r)
                e.release(r)
    ttft = np.array([s[0] - sub_t[r] for r, s in stamps.items() if s]) * 1e3
    itl = np.concatenate([np.diff(s) for s in stamps.values() if len(s) > 1]) * 1e3
    itl = itl[itl > 0]  # tokens that surfaced in the same poll share a stamp
    q = lambda a, p: float(np.percentile(a, p)) if len(a) else None
    return {"ttft_ms": {"p50": q(ttft, 50), "max": q(ttft, 100)}, "itl_ms": {"p50": q(itl, 50), "p99": q(itl, 99), "max": q(itl, 100)},
            "arrivals": "all at t=0" if spread_s == 0 else f"uniform over {spread_s:.1f} s"}


# ------------------------------------------------------------------ CPU stand-in for the reference's CPU path
def hf_llama_cpu(layers, threads):
    """HF transformers LlamaForCausalLM, Llama-3-8B shape with `layers` layers, fp32 on torch CPU, cheap random init
    (built on the meta device: the default initialiser would spend minutes on 8 B parameters)."""
    os.environ["OMP_NUM_THREADS"] = str(threads)  # torch.distributed.run exports 1
    import torch
    torch.set_num_threads(threads)
    torch.set_grad_enabled(False)
    from transformers import LlamaConfig, LlamaForCausalLM
    from transformers.models.llama.modeling_llama import LlamaRotaryEmbedding
    cfg = LlamaConfig(vocab_size=128256, hidden_size=4096, intermediate_size=14336, num_hidden_layers=layers,
                      num_attention_heads=32, num_key_value_heads=8, head_dim=128, max_position_embeddings=8192,
                      rms_norm_eps=1e-5, tie_word_embeddings=False, rope_parameters={"rope_theta": 500000.0, "rope_type": "default"},
                      attention_bias=False, mlp_bias=False, attn_implementation="sdpa")
    with torch.device("meta"):
        m = LlamaForCausalLM(cfg)
    m = m.to_empty(device="cpu").float().eval()
    g = torch.Generator().manual_seed(0)
    block = torch.randn(1 << 24, generator=g) * 0.02
    for name, p in m.named_parameters():
        flat = p.data.view(-1)
        if "norm" in name:
            flat.fill_(1.0)
            continue
        for i in range(0, flat.numel(), block.numel()):
            k = min(block.numel(), flat.numel() - i)
            flat[i:i + k].copy_(block[:k])
    m.model.rotary_emb = LlamaRotaryEmbedding(config=cfg)  # its inv_freq buffer did not survive to_empty()
    return m, torch


def hf_session(m, torch, prompt_len, decode):
    """One session: prefill + greedy decode through HF's KV cache; returns seconds."""
    ids = torch.from_numpy(np.random.default_rng(7).integers(0, 128256, size=prompt_len)).long()[None]
    t0 = time.perf_counter()
    out = m(ids, use_cache=True)
    past, logits = out.past_key_values, out.logits[0, -1]
    for _ in range(decode):
        t = int(torch.argmax(logits))
        o = m(torch.tensor([[t]]), past_key_values=past, use_cache=True)
        past, logits = o.past_key_values, o.logits[0, -1]
    return time.perf_counter() - t0


def host_threads():
    """All host cores for the BLAS behind numpy / torch, whatever the launcher exported (torch.distributed.run sets
    OMP_NUM_THREADS=1, which made the r01 reference arm single-threaded at N >= 2)."""
    n = os.cpu_count() or 1
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[k] = str(n)
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=n)
        from threadpoolctl import threadpool_info
        got = max([p.get("num_threads", 1) for p in threadpool_info()] or [1])
    except Exception:
        got = n
    return got


def oracle_port(layers, prompt_len):
    """The numpy fp32 oracle (oracle/llama_ref.py) at the Llama-3-8B shape with `layers` of the 32 identical layers:
    returns run(decode) -> seconds for one session (prefill + greedy decode)."""
    from helix_b200 import configs
    from oracle.llama_ref import LlamaOracle
    d = configs.llama3_8b()
    d.layers = layers
    rng = np.random.default_rng(0)
    block = (rng.standard_normal(1 << 22, dtype=np.float32) * 0.02)

    def filled(shape):
        return np.resize(block, int(np.prod(shape))).reshape(shape)
    H, F, V, D = d.hidden, d.ffn, d.vocab, d.head_dim
    sd = {"model.embed_tokens.weight": filled((V, H)), "lm_head.weight": filled((V, H)), "model.norm.weight": np.ones(H, np.float32)}
    for i in range(layers):
        p = f"model.layers.{i}."
        sd[p + "input_layernorm.weight"] = np.ones(H, np.float32)
        sd[p + "post_attention_layernorm.weight"] = np.ones(H, np.float32)
        sd[p + "self_attn.q_proj.weight"] = filled((d.heads * D, H))
        sd[p + "self_attn.k_proj.weight"] = filled((d.kv_heads * D, H))
        sd[p + "self_attn.v_proj.weight"] = filled((d.kv_heads * D, H))
        sd[p + "self_attn.o_proj.weight"] = filled((H, d.heads * D))
        sd[p + "mlp.gate_proj.weight"] = filled((F, H))
        sd[p + "mlp.up_proj.weight"] = filled((F, H))
        sd[p + "mlp.down_proj.weight"] = filled((H, F))
    o = LlamaOracle(d, sd)
    toks = rng.integers(0, V, size=prompt_len).astype(np.int32)

    def run(decode):
        t0 = time.perf_counter()
        o.greedy(toks, decode)
        return time.perf_counter() - t0
    return run


def cpu_stand_in(impl, steps, warmup, budget_s, prompt_len=512, decode=8):
    """`steps` timed sessions after `warmup` on all host threads.  The model is truncated to as many of the 32 identical
    layers (8, 4 or 2) as lets warmup+steps sessions finish inside budget_s on this box; the factor 32/layers is reported
    next to the MEASURED step time, never folded into it."""
    threads = host_threads()
    if impl == "hf":
        m, torch = hf_llama_cpu(8, threads)
        layers, run = 8, (lambda dec: hf_session(m, torch, prompt_len, dec))
        run(2)
    else:
        layers = 8
        run = oracle_port(layers, prompt_len)
        t = run(decode)                      # probe (also warms BLAS threads)
        while layers > 2 and t * (warmup + steps) > budget_s:
            layers //= 2
            run = oracle_port(layers, prompt_len)
            t = run(decode)
    for _ in range(warmup):
        run(decode)
    ts = [run(decode) for _ in range(steps)]
    return {"seconds": ts, "threads": threads, "prompt_len": prompt_len, "decode": decode, "layers": layers, "impl": impl}


def cpu_sample_text(r):
    what = ("the numpy fp32 oracle port (oracle/llama_ref.py)" if r["impl"] == "oracle" else
            "HF transformers LlamaForCausalLM fp32 on torch CPU")
    return (f"{what}, {r['threads']} BLAS threads, Llama-3-8B shape truncated to {r['layers']}/32 layers, ONE session per step: "
            f"{r['prompt_len']}-token prompt + {r['decode']} greedy decode tokens; value = tokens / (measured step time x "
            f"{32 // r['layers']}); stand-in for the reference's llama.cpp CPU path (DEVELOPMENT_CPU_ONLY), which cannot run "
            f"offline.  (HF transformers on torch CPU, the stand-in BASELINE.md names, measured 0.55 tokens/s on this box class "
            f"— 245 s per 136-token session, profiles/r02c_reference_hf.json — so the faster port is the fairer baseline.)")


def reference_arm(args, rank, world):
    """--impl reference: K timed steps after W warm-ups of the CPU stand-in, one session per step, sized to finish in a
    few minutes.  ms_per_step is the measured time of what ran; the depth extrapolation is a separate, stated factor."""
    if rank != 0:
        return
    r = cpu_stand_in(args.cpu_impl, args.steps, args.warmup, budget_s=200.0)
    t = statistics.mean(r["seconds"])
    factor = 32 / r["layers"]
    toks = r["prompt_len"] + r["decode"]
    v = toks / (t * factor)
    sample = cpu_sample_text(r)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args), "sample": sample, "tokens_per_step": toks, "layers_run": r["layers"],
                       "extrapolation_factor": factor},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": r["threads"], "kind": "port", "sample": sample,
                             "measured_step_seconds": r["seconds"], "extrapolation_factor": factor},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def cpu_baseline_field(impl="oracle"):
    """Bounded CPU sample for the native line at N=1 (one probe + one timed session, <= ~30 s)."""
    r = cpu_stand_in(impl, 1, 0, budget_s=25.0)
    t = r["seconds"][0]
    factor = 32 / r["layers"]
    return {"value": (r["prompt_len"] + r["decode"]) / (t * factor), "unit": UNIT, "cores": r["threads"], "kind": "port",
            "measured_seconds": t, "extrapolation_factor": factor, "sample": cpu_sample_text(r)}


# ------------------------------------------------------------------ configs[2]: bge-base batch encode
def bench_bge(args):
    """BASELINE configs[2]: bge-base-en-shaped encoder, batch-encode `--chunks` x 512-token synthetic chunks through
    hb_embed (host token buffers in, fp32 vectors out)."""
    import torch
    import helix_b200 as hb
    from helix_b200 import configs
    desc = configs.bge_base()
    e = hb.Engine(hb.EngineConfig(device=0, max_seqs=64, max_ctx=512, max_batched_tokens=args.max_batched_tokens * 4))
    e.load_random(desc, 2)
    n, L = args.chunks, 512
    rng = np.random.default_rng(2)
    lens = rng.integers(64, L + 1, size=n) if args.ragged else np.full(n, L)  # §8d config 3 varlen variant: U[64, 512]
    offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    total_tokens = int(offs[-1])
    toks = rng.integers(0, desc.vocab, size=total_tokens, dtype=np.int64).astype(np.int32)
    out = np.empty((n, desc.hidden), np.float32)
    warm = min(n, 2048)
    for _ in range(max(1, args.warmup)):
        e.embed_flat(toks[:offs[warm]], offs[:warm + 1], out[:warm])
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    sampler.start()
    s0 = e.stats()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e.embed_flat(toks, offs, out)
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / args.steps
    s1 = e.stats()
    clocks = sampler.stop()
    if args.dump_outputs:   # before the profiled pass below reuses `out`
        dump_outputs(args.dump_outputs, {"embeddings": out})   # the last timed step's fp32 vectors [chunk, hidden]
    dev = (s1["gpu_ms_prefill"] - s0["gpu_ms_prefill"]) / args.steps / 1e3
    e.set_profile(True)
    p0 = e.stats()
    sub = min(n, 8192)
    e.embed_flat(toks[:offs[sub]], offs[:sub + 1], out[:sub])
    p1 = e.stats()
    e.set_profile(False)
    fam, tot_ms = {}, 0.0
    for i, name in ((0, "gemm"), (1, "attention"), (3, "row_kernels")):
        ms = p1["prof_ms"][i] - p0["prof_ms"][i]
        w = p1["prof_work"][i] - p0["prof_work"][i]
        tot_ms += ms
        fam[name] = {"ms": ms, "launches": p1["prof_launches"][i] - p0["prof_launches"][i],
                     "tflops" if i < 2 else "gbs": (w / (ms * 1e-3) / (1e12 if i < 2 else 1e9)) if ms else 0.0}
    # GEMMs 169.9 MFLOP/token + bidirectional attention 4*len*768 FLOP/token (SURVEY.md §8d)
    flops = float(total_tokens) * 169.9e6 + float((lens.astype(np.float64) ** 2).sum()) * 4 * 768
    peaks = measured_peaks()
    g = fam["gemm"]
    line = {"metric": "chunks/sec bge-base-en-shaped batch encode (512-token chunks)", "value": n / dev, "unit": "chunks/s",
            "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"bge-base-en shape random-init, {n} chunks x " + ("U[64,512]" if args.ragged else "512") +
                       " tokens, CLS+L2, fp32 out", "l2": "activations of one engine batch (64k tokens x 3072 x 2 B) > 126 MB L2"},
            "e2e": {"value": n / wall, "unit": "chunks/s", "h2d_bytes_per_step": int(toks.nbytes * 2), "d2h_bytes_per_step": int(out.nbytes),
                    "api": "hb_embed (C ABI, host token buffers in, host fp32 vectors out)"},
            "roofline": {"kernel": "gemm_tn_kernel (tcgen05, encoder GEMMs)", "bound": "tensor", "achieved": g["tflops"],
                         "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s", "frac": g["tflops"] / peaks["bf16_tflops_sustained"],
                         "peak_source": peaks["source"] + " sustained cuBLAS bf16", "share_of_step": g["ms"] / tot_ms if tot_ms else None,
                         "traffic": None},
            "model_tflops": flops / dev / 1e12, "frac_of_measured_sustained": flops / dev / 1e12 / peaks["bf16_tflops_sustained"],
            "gpu_launches": int(s1["kernel_launches"] - s0["kernel_launches"]), "tokens_per_s": total_tokens / dev,
            "kernels_profiled_subset": fam, "clocks": clocks, "finite": bool(np.isfinite(out).all()),
            "unit_norm_err": float(np.abs(np.linalg.norm(out, axis=1) - 1).max())}
    if not args.no_cpu_baseline:
        line["cpu_baseline"] = bge_cpu_baseline()
    print(json.dumps(line), flush=True)
    e.close()


def bge_cpu_baseline(chunks=16):
    """The numpy fp32 oracle (oracle/bert_ref.py) on all host threads over a bounded sample of the same workload."""
    threads = host_threads()
    from helix_b200 import configs
    from oracle.bert_ref import bert_embed
    from oracle import weights
    d = configs.bge_base()
    sd = weights.bert_state_dict(d, 2, 0.02)
    seqs = [np.random.default_rng(30 + i).integers(0, d.vocab, size=512).astype(np.int32) for i in range(chunks)]
    bert_embed(d, sd, seqs[:2])
    t0 = time.perf_counter()
    bert_embed(d, sd, seqs)
    t = time.perf_counter() - t0
    return {"value": chunks / t, "unit": "chunks/s", "cores": threads, "kind": "port", "measured_seconds": t,
            "sample": f"numpy fp32 oracle port (oracle/bert_ref.py), {threads} BLAS threads, {chunks} chunks x 512 tokens, one chunk at a "
                      f"time, CLS + L2 (HF BertModel on torch CPU measured 1.3 chunks/s on this box class)"}


# ------------------------------------------------------------------ configs[3]: multi-model pack on one GPU
def bench_pack(args):
    """BASELINE configs[3]: Llama-3-8B + Llama-3.2-1B + bge-base co-resident on ONE B200 under the scheduler's memory-fit
    rule (global_allocator.go:349-452), mixed chat + embed traffic on three engines/streams.  Each engine owns a share of
    the SMs (hb_engine_cfg.sm_budget; --pack-mode partition = enforced by CUDA green contexts).  Reports each model's
    throughput solo (whole GPU) and packed, and the sum of packed/solo ratios (1.0 = pure time slicing)."""
    import helix_b200 as hb
    from helix_b200 import configs
    from helix_b200.engine import memory_estimate
    GB = 1024 ** 3
    seconds = args.pack_seconds
    shares = {"llama3_8b": args.pack_sms[0], "llama32_1b": args.pack_sms[1], "bge_base": args.pack_sms[2]}

    def specs(mode):
        part = 1 if mode == "partition" else 0
        bud = (lambda k: shares[k]) if mode != "none" else (lambda k: 0)
        return [("llama3_8b", configs.llama3_8b(), hb.EngineConfig(max_seqs=16, max_ctx=2304, max_batched_tokens=8192, use_cuda_graphs=1,
                                                                  sm_budget=bud("llama3_8b"), sm_partition=part)),
                ("llama32_1b", configs.llama32_1b(), hb.EngineConfig(max_seqs=16, max_ctx=2304, max_batched_tokens=8192, use_cuda_graphs=1,
                                                                    sm_budget=bud("llama32_1b"), sm_partition=part, stream_priority=1)),
                ("bge_base", configs.bge_base(), hb.EngineConfig(max_seqs=64, max_ctx=512, max_batched_tokens=32768,
                                                                sm_budget=bud("bge_base"), sm_partition=part, stream_priority=1))]

    def chat_load(e, desc, sessions, prompt, decode, out, key):
        rng = np.random.default_rng(0)
        prompts = [rng.integers(0, desc.vocab, size=prompt).astype(np.int32) for _ in range(sessions)]
        toks, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < seconds:
            toks += sum(map(len, serve_once(e, hb, prompts, decode))) + sessions * prompt
        out[key] = toks / (time.perf_counter() - t0)

    def embed_load(e, desc, chunks, out, key):
        rng = np.random.default_rng(1)
        toks = rng.integers(0, desc.vocab, size=chunks * 512).astype(np.int32)
        offs = (np.arange(chunks + 1) * 512).astype(np.int32)
        n, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < seconds:
            e.embed_flat(toks, offs)
            n += chunks
        out[key] = n / (time.perf_counter() - t0)

    def run(mode, together):
        total = 183359 * 1024 * 1024
        allocated, budgets, engines = 0, {}, {}
        for name, d, cfg in specs(mode):
            need = sum(memory_estimate(d, cfg).values()) + (256 << 20)
            assert total - allocated >= need, "scheduler would not place this slot"   # the reference's single-GPU fit rule
            budgets[name] = need
            allocated += need
            cfg.memory_budget_bytes = need
            e = hb.Engine(cfg)
            e.load_random(d, 1)
            if d.arch == configs.LLAMA:
                e.start()
            engines[name] = (e, d)
        out = {}
        ths = [threading.Thread(target=chat_load, args=(*engines["llama3_8b"], 16, 2048, 64, out, "llama3_8b_tok_s")),
               threading.Thread(target=chat_load, args=(*engines["llama32_1b"], 16, 2048, 64, out, "llama32_1b_tok_s")),
               threading.Thread(target=embed_load, args=(*engines["bge_base"], 4096, out, "bge_chunks_s"))]
        if together:
            [t.start() for t in ths]
            [t.join() for t in ths]
        else:
            for t in ths:
                t.start()
                t.join()
        for name, (e, d) in engines.items():
            st = e.stats()
            assert st["weights_bytes"] + st["kv_bytes"] + st["workspace_bytes"] <= st["budget_bytes"]
            e.close()
        return out, {k: round(v / GB, 2) for k, v in budgets.items()}

    solo, budgets = run("none", together=False)
    res = {"metric": "multi-model pack: sum over models of packed/solo throughput (8B + 1B chat, bge embed; 1.0 = time slicing)",
           "unit": "ratio", "n_gpus": 1, "steps": 1, "warmup": 0, "higher_is_better": True, "dtype": "bf16", "data": "synthetic",
           "config": {"workload": "Llama-3-8B (16 x 2048+64) + Llama-3.2-1B (16 x 2048+64) + bge-base (4096 x 512) on one B200, "
                                  f"{seconds:.0f} s per measurement", "sm_shares": shares, "budgets_gb": budgets},
           "solo": solo, "modes": {}}
    for mode in args.pack_modes:
        try:
            packed, _ = run(mode, together=True)
            ratios = {k: packed[k] / solo[k] for k in solo}
            res["modes"][mode] = {"packed": packed, "packed_over_solo": ratios, "sum": sum(ratios.values())}
        except hb.HBError as ex:
            res["modes"][mode] = {"error": str(ex)}
    ok = [m["sum"] for m in res["modes"].values() if "sum" in m]
    res["value"] = max(ok) if ok else None
    print(json.dumps(res), flush=True)


# ------------------------------------------------------------------ headline
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--sessions", type=int, default=32)
    ap.add_argument("--seq", type=int, default=2048)
    ap.add_argument("--decode", type=int, default=128)
    ap.add_argument("--max-seqs", type=int, default=256, help="--max-num-seqs of the slot (the reference's vLLM default)")
    ap.add_argument("--max-batched-tokens", type=int, default=16384)
    ap.add_argument("--no-graphs", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-impl", default="oracle", choices=["oracle", "hf"], help="CPU stand-in behind cpu_baseline / --impl reference")
    ap.add_argument("--no-fixed-total", action="store_true")
    ap.add_argument("--mixed-step-tokens", type=int, default=512)
    ap.add_argument("--fixed-total-sessions", type=int, default=256)
    ap.add_argument("--layers", type=int, default=0, help="debug: truncate the model (INVALID as a bench number)")
    ap.add_argument("--workload", default="llama8b", choices=["llama8b", "bge", "pack"])
    ap.add_argument("--chunks", type=int, default=100000)
    ap.add_argument("--ragged", action="store_true", help="bge workload: chunk lengths U[64,512] instead of 512")
    ap.add_argument("--pack-seconds", type=float, default=8.0)
    ap.add_argument("--pack-sms", type=int, nargs=3, default=[96, 24, 24], help="SM shares of 8B / 1B / bge")
    ap.add_argument("--pack-modes", nargs="+", default=["none", "budget", "partition"])
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (llama8b: tokens, bge: embeddings)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "native" or args.workload == "pack"):
        ap.error("--dump-outputs: native llama8b and bge workloads only")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return
    if args.workload in ("bge", "pack"):
        if rank == 0:
            (bench_bge if args.workload == "bge" else bench_pack)(args)
        return

    import torch
    import torch.distributed as dist
    import helix_b200 as hb
    from helix_b200 import configs
    from helix_b200.engine import replica_unique_id
    from helix_b200.replica import ArenaView, route_least_active

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    desc = configs.llama3_8b()
    if args.layers:
        desc.layers = args.layers
    max_ctx = ((args.seq + args.decode + 63) // 64 + 1) * 64
    max_seqs = max(args.max_seqs, args.sessions)
    cfg = hb.EngineConfig(device=local_rank, max_seqs=max_seqs, max_ctx=max_ctx,
                          max_batched_tokens=args.max_batched_tokens, use_cuda_graphs=0 if args.no_graphs else 1)
    e = hb.Engine(cfg)
    bcast = None
    if world == 1:
        e.load_random(desc, seed=0)
    else:
        # rank 0 loads; every replica receives its arena by ONE ncclBroadcast issued inside libhelixb200.so
        # (hb_model_load_broadcast, SURVEY.md §8e).  torch.distributed only carries the 128-byte id and the barriers.
        box = [replica_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        if rank == 0:
            e.load_random(desc, seed=0)
        barrier()
        dt = e.load_broadcast(desc, box[0], rank, world)
        ptr, nbytes = e.weights_arena()
        arena = torch.as_tensor(ArenaView(ptr, nbytes), device=f"cuda:{local_rank}")
        chk = arena[:: max(1, nbytes // 65536)].to(torch.int32).sum().reshape(1).float()
        lo, hi = chk.clone(), chk.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        assert float(lo) == float(hi), "weight broadcast mismatch across replicas"
        tmax = torch.tensor([dt], device="cuda", dtype=torch.float64)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        bcast = {"bytes": nbytes, "seconds": float(tmax), "gbs": nbytes / float(tmax) / 1e9,
                 "how": "ncclBroadcast inside libhelixb200.so (hb_model_load_broadcast), CUDA events around the collective, max over ranks"}

    prompts = [session_prompt(rank * args.sessions + i, args.seq, desc.vocab) for i in range(args.sessions)]
    tokens_per_step = args.sessions * (args.seq + args.decode)
    e.start()
    for _ in range(args.warmup):
        got = serve_once(e, hb, prompts, args.decode)
        assert sum(map(len, got)) == args.sessions * args.decode

    sampler = ClockSampler(local_rank) if rank == 0 else None
    barrier()
    if sampler:
        sampler.start()
    s0 = e.stats()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        outs = serve_once(e, hb, prompts, args.decode)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    s1 = e.stats()
    barrier()
    clocks = sampler.stop() if sampler else None
    dev_ms = (s1["gpu_ms_prefill"] - s0["gpu_ms_prefill"]) + (s1["gpu_ms_decode"] - s0["gpu_ms_decode"])
    times = torch.tensor([dev_ms / 1e3, wall], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)  # max over ranks
    dev_s, wall_s = float(times[0]), float(times[1])
    launches = s1["kernel_launches"] - s0["kernel_launches"]
    prefill_steps = (s1["steps_prefill"] - s0["steps_prefill"]) / args.steps

    latency = serve_latency(e, hb, prompts, args.decode)
    latency_spread = latency_mixed = None
    if rank == 0:
        # arrivals spread over a second: with pure phases every later prompt's prefill step stalls the running streams;
        # with mixed steps (what the runtime passes: decode_with_prefill, 2048-token steps) they keep decoding
        latency_spread = serve_latency(e, hb, prompts, args.decode, spread_s=1.0)
        e.set_mixed(1, args.mixed_step_tokens)
        serve_once(e, hb, prompts[:4], 4)   # first use of the mixed path (paged prefill attention variants)
        latency_mixed = serve_latency(e, hb, prompts, args.decode, spread_s=1.0)
        latency_mixed["scheduler"] = f"decode_with_prefill=1, mixed_step_tokens={args.mixed_step_tokens}"
        e.set_mixed(0, 0)

    # ---- BASELINE configs[4] framing: a FIXED total of sessions, routed by the scheduler's rule from rank 0
    fixed = None
    if not args.no_fixed_total:
        total_sessions = args.fixed_total_sessions
        route = [route_least_active([0] * world, total_sessions) if rank == 0 else None]   # pickBestWarmSlot, scheduler.go:1958-2009
        if world > 1:
            dist.broadcast_object_list(route, src=0)
        mine = [i for i, r in enumerate(route[0]) if r == rank]
        ft_prompts = [session_prompt(10 ** 6 + i, args.seq, desc.vocab) for i in mine]
        serve_once(e, hb, ft_prompts[: max(1, len(ft_prompts) // 8)], 4)   # warm the batch sizes' graphs a little
        barrier()
        f0 = e.stats()
        tw = time.perf_counter()
        serve_once(e, hb, ft_prompts, args.decode)
        torch.cuda.synchronize()
        ft_wall = time.perf_counter() - tw
        f1 = e.stats()
        barrier()
        ft = torch.tensor([(f1["gpu_ms_prefill"] - f0["gpu_ms_prefill"]) / 1e3, (f1["gpu_ms_decode"] - f0["gpu_ms_decode"]) / 1e3, ft_wall],
                          device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ft, op=dist.ReduceOp.MAX)
        pre_s, dec_s, w_s = (float(x) for x in ft)
        fixed = {"sessions_total": total_sessions, "sessions_per_gpu": [route[0].count(r) for r in range(world)],
                 "routing": "replica.route_least_active on rank 0 (pickBestWarmSlot: fewest active requests, stable ties)",
                 "tokens_per_s": total_sessions * (args.seq + args.decode) / (pre_s + dec_s),
                 "decode_tokens_per_s": total_sessions * args.decode / dec_s, "prefill_tokens_per_s": total_sessions * args.seq / pre_s,
                 "e2e_tokens_per_s": total_sessions * (args.seq + args.decode) / w_s, "timing": "device time, max over ranks; one pass"}

    # ---- one profiled step: CUDA-event span around every launch on the engine stream
    e.set_profile(True)
    p0 = e.stats()
    serve_once(e, hb, prompts, args.decode)
    p1 = e.stats()
    e.set_profile(False)
    e.stop()
    fam = ["gemm_prefill", "attn_prefill", "attn_decode", "row_kernels", "gemm_decode"]
    prof = {}
    for i, name in enumerate(fam):
        ms = p1["prof_ms"][i] - p0["prof_ms"][i]
        work = p1["prof_work"][i] - p0["prof_work"][i]
        n = p1["prof_launches"][i] - p0["prof_launches"][i]
        prof[name] = {"ms": ms, "work": work, "launches": n}
    total_prof_ms = sum(v["ms"] for v in prof.values()) or 1.0
    peaks = measured_peaks()
    g = prof["gemm_prefill"]
    gemm_tf = g["work"] / (g["ms"] * 1e-3) / 1e12 if g["ms"] else 0.0
    gd = prof["gemm_decode"]
    gemm_dec_gbs = gd["work"] / (gd["ms"] * 1e-3) / 1e9 if gd["ms"] else 0.0
    ad = prof["attn_decode"]
    ap_ = prof["attn_prefill"]
    roofline = {"kernel": "gemm_tn_kernel (tcgen05, prefill steps)", "bound": "tensor", "achieved": gemm_tf,
                "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                "frac": gemm_tf / peaks["bf16_tflops_sustained"], "peak_source": peaks["source"] + " sustained cuBLAS bf16",
                "frac_of_nominal_2250": gemm_tf / 2250.0, "launches": g["launches"],
                "avg_launch_ms": g["ms"] / g["launches"] if g["launches"] else None,
                "share_of_step": g["ms"] / total_prof_ms, "traffic": ncu_traffic("gemm_prefill")}
    kernels = {
        "gemm_decode": {"bound": "hbm", "achieved": gemm_dec_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                        "frac": gemm_dec_gbs / peaks["hbm_gbs"], "share_of_step": gd["ms"] / total_prof_ms,
                        "launches": gd["launches"], "traffic": ncu_traffic("gemm_decode"),
                        "note": "event spans serialise the launches: the in-step overlap of consecutive kernels (PDL weight prefetch) "
                                "is not in these per-family numbers; phases.decode_hbm_frac is the whole-step figure"},
        "attn_decode": {"bound": "hbm", "achieved": ad["work"] / (ad["ms"] * 1e-3) / 1e9 if ad["ms"] else 0.0,
                        "peak": peaks["hbm_gbs"], "unit": "GB/s", "share_of_step": ad["ms"] / total_prof_ms,
                        "launches": ad["launches"]},
        "attn_prefill": {"bound": "tensor", "achieved": ap_["work"] / (ap_["ms"] * 1e-3) / 1e12 if ap_["ms"] else 0.0,
                         "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                         "share_of_step": ap_["ms"] / total_prof_ms, "launches": ap_["launches"]},
        "row_kernels": {"bound": "hbm", "share_of_step": prof["row_kernels"]["ms"] / total_prof_ms,
                        "launches": prof["row_kernels"]["launches"]},
    }
    for k in ("attn_decode", "attn_prefill"):
        kernels[k]["frac"] = kernels[k]["achieved"] / kernels[k]["peak"]
    # phase view (device time of the timed region)
    pre_ms = (s1["gpu_ms_prefill"] - s0["gpu_ms_prefill"]) / args.steps
    dec_ms = (s1["gpu_ms_decode"] - s0["gpu_ms_decode"]) / args.steps
    dec_steps = (s1["steps_decode"] - s0["steps_decode"]) / args.steps
    # algorithmic HBM bytes of one decode step (SURVEY.md §8d): GEMM weights 15.01 GB + KV read of every context
    ctx_mean = args.seq + args.decode / 2.0
    step_bytes = 15.01e9 + args.sessions * ctx_mean * 131072.0 if not args.layers else None
    phases = {"prefill_tokens_per_s": args.sessions * args.seq / (pre_ms * 1e-3) if pre_ms else None,
              "decode_tokens_per_s": args.sessions * args.decode / (dec_ms * 1e-3) if dec_ms else None,
              "prefill_ms": pre_ms, "decode_ms": dec_ms, "prefill_steps": prefill_steps,
              "decode_ms_per_step": dec_ms / dec_steps if dec_steps else None,
              "decode_hbm_gbs": step_bytes * dec_steps / (dec_ms * 1e-3) / 1e9 if step_bytes and dec_ms else None,
              "prefill_model_tflops": (args.sessions * args.seq * 14.50e9 + args.sessions * 1.05e9) / (pre_ms * 1e-3) / 1e12
              if pre_ms and not args.layers else None}
    if phases["decode_hbm_gbs"]:
        phases["decode_hbm_frac"] = phases["decode_hbm_gbs"] / peaks["hbm_gbs"]

    if rank == 0:
        # per-step host<->device traffic of the public path: prompt ids + per-step metadata in, sampled ids out
        h2d = args.sessions * args.seq * 4 * 3 + args.decode * args.sessions * 4 * 8
        d2h = args.sessions * (args.decode) * 4
        line = {"metric": METRIC, "value": world * tokens_per_step * args.steps / dev_s, "unit": UNIT, "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_s * 1e3 / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": workload_name(args),
                           "prefill_budget_tokens": args.max_batched_tokens, "cuda_graph_decode": not args.no_graphs,
                           "parallelism": f"replica x{world} (one ncclBroadcast of the weights, no data-path collective)",
                           "l2": "weights 16 GB + KV >> 126 MB L2: inputs larger than L2, no flush needed",
                           "value_timing": "CUDA events on the engine stream around every forward pass, summed; max over ranks",
                           "broadcast": bcast, "layers": desc.layers},
                "e2e": {"value": world * tokens_per_step * args.steps / wall_s, "unit": UNIT, "ms_per_step": wall_s * 1e3 / args.steps,
                        "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "api": "hb_submit/hb_wait/hb_poll (C ABI, host buffers, step-loop thread)"},
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "kernels": kernels, "phases": phases,
                "latency": latency, "latency_spread_arrivals": latency_spread, "latency_spread_arrivals_mixed_steps": latency_mixed,
                "fixed_total": fixed}
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_field(args.cpu_impl)
        print(json.dumps(line), flush=True)
    if args.dump_outputs:
        # what a client of hb_submit / hb_poll received in the last timed step: greedy token ids [session, decode step]
        dump_outputs(args.dump_outputs, {"tokens" + (f"_rank{rank}" if world > 1 else ""): np.array(outs, np.float64)},
                     DUMP_BYTES // world)
    e.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
