"""GPU: second opinion against the backend the reference actually delegates to (api/pkg/runner/vllm_runtime.go:163-252
spawns vLLM).  vLLM 0.22 served the seeded Llama-3-8B-shaped checkpoint (2 layers, the HF-pinned fixture's weights and
prompt; bf16, greedy, log-probabilities) once, and tests/golden/gen_vllm.py stored its answer in
tests/golden/vllm_llama3_8b_2layer.json.  This engine serves the same checkpoint; greedy token ids must agree until the
first near-tie and the chosen tokens' log-probabilities to 5e-2 (two independent bf16 implementations)."""
import json
import os

import numpy as np
import pytest

import helix_b200 as hb
from helix_b200 import configs
from oracle import weights

pytestmark = pytest.mark.gpu


def test_greedy_ids_and_logprobs_agree_with_vllm(golden_dir):
    with open(os.path.join(golden_dir, "vllm_llama3_8b_2layer.json")) as f:
        v = json.load(f)
    g = np.load(os.path.join(golden_dir, v["fixture"]))
    d = configs.llama3_8b()
    d.layers = int(g["layers"])
    sd = weights.llama_state_dict(d, int(g["seed"]), float(g["std"]))
    prompt = g["prompt"].tolist()
    with hb.Engine(hb.EngineConfig(max_seqs=2, max_ctx=1024, max_batched_tokens=1024, use_cuda_graphs=1)) as e:
        e.load_state_dict(d, sd)
        rids, outs = e.generate([prompt], hb.Sampling(max_tokens=8, logprobs=6))
        ids, lps = e.logprobs(rids[0])
    vllm_lp = [dict((int(t), lp) for t, lp in step) for step in v["logprobs"]]
    same = 0
    for i, (a, b) in enumerate(zip(outs[0], v["tokens"])):
        if a != b:
            break
        same += 1
        assert abs(float(lps[i, 0]) - vllm_lp[i][a]) <= 5e-2
    hf = g["greedy_tokens"].tolist()
    print(f"\n[vLLM second opinion] engine  {outs[0]}\n                      vLLM    {v['tokens']}\n                      HF fp32 {hf}; "
          f"identical for the first {same}/8 steps; engine logprobs {lps[:same, 0].round(4).tolist()}")
    assert same >= 3
    if same < 8:   # after a disagreement: it must be a near-tie in the engine's own distribution
        i = same
        alt = [float(lps[i, k]) for k in range(1, ids.shape[1]) if int(ids[i, k]) == v["tokens"][i]]
        assert alt and float(lps[i, 0]) - alt[0] <= 0.1, (i, outs[0], v["tokens"])
