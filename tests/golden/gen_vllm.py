"""Generates tests/golden/vllm_llama3_8b_2layer.json: vLLM's greedy continuation and log-probabilities on the seeded
Llama-3-8B-shaped checkpoint of llama3_8b_2layer.npz (2 layers, same weights and prompt).  vLLM is the backend Helix's
runner spawns (api/pkg/runner/vllm_runtime.go:163-252); it needs a GPU, so run this on one:

    python tests/golden/gen_vllm.py [OUT.json]

tests/test_vllm_second_opinion_gpu.py compares the engine with the stored result.
"""
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from helix_b200 import configs, weights_io  # noqa: E402
from oracle import weights  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
FIXTURE = "llama3_8b_2layer.npz"
MAX_TOKENS, LOGPROBS = 8, 5


def write_checkpoint(path, d, sd):
    weights_io.write_safetensors(os.path.join(path, "model.safetensors"), sd)
    cfg = {"architectures": ["LlamaForCausalLM"], "model_type": "llama", "hidden_size": d.hidden, "intermediate_size": d.ffn,
           "num_hidden_layers": d.layers, "num_attention_heads": d.heads, "num_key_value_heads": d.kv_heads, "head_dim": d.head_dim,
           "vocab_size": d.vocab, "max_position_embeddings": 8192, "rms_norm_eps": d.norm_eps, "rope_theta": d.rope_theta,
           "torch_dtype": "bfloat16", "tie_word_embeddings": False, "hidden_act": "silu", "bos_token_id": 128000, "eos_token_id": 128001}
    with open(os.path.join(path, "config.json"), "w") as f:
        json.dump(cfg, f)


def main(out):
    os.environ.setdefault("VLLM_LOGGING_LEVEL", "WARNING")
    os.environ.setdefault("HF_HUB_OFFLINE", "1")
    import vllm
    g = np.load(os.path.join(HERE, FIXTURE))
    d = configs.llama3_8b()
    d.layers = int(g["layers"])
    prompt = g["prompt"].tolist()
    with tempfile.TemporaryDirectory(prefix="hb_vllm_ckpt_") as ckpt:
        write_checkpoint(ckpt, d, weights.llama_state_dict(d, int(g["seed"]), float(g["std"])))
        llm = vllm.LLM(model=ckpt, skip_tokenizer_init=True, dtype="bfloat16", max_model_len=1024, max_num_seqs=4,
                       gpu_memory_utilization=0.3, enforce_eager=True, seed=0, enable_prefix_caching=False)
        sp = vllm.SamplingParams(temperature=0.0, max_tokens=MAX_TOKENS, ignore_eos=True, detokenize=False, logprobs=LOGPROBS)
        res = llm.generate([{"prompt_token_ids": prompt}], sp, use_tqdm=False)[0].outputs[0]
    result = {"fixture": FIXTURE, "vllm": vllm.__version__, "dtype": "bfloat16", "sampling": "greedy",
              "tokens": [int(t) for t in res.token_ids],
              # per generated token: [token id, log-probability] of the sampled token and the top LOGPROBS alternatives
              "logprobs": [sorted(([int(k), float(v.logprob)] for k, v in step.items()), key=lambda p: -p[1])
                           for step in res.logprobs]}
    with open(out, "w") as f:
        json.dump(result, f, indent=1)
        f.write("\n")
    print("vLLM", vllm.__version__, "greedy", result["tokens"])


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "vllm_llama3_8b_2layer.json"))
