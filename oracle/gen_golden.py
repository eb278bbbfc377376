"""Generate golden vectors by running the reference's OWN shard operator and wire codec.  TEST INFRA.

Run in the build container (needs /root/reference):  python -m oracle.gen_golden
Writes tests/golden/ref_layergroup_<cfg>.pt (a few hundred KB each).
``python -m oracle.gen_golden --portable`` writes tests/golden/ref_layergroup_eager_portable.json instead: SHA-256 of
every hop and of the last-4 logits of the eager runs, computed with the host-independent CPU arithmetic of
oracle/portable_cpu.py, so that tests/test_golden.py can check the oracle against them bit for bit on any x86-64 host.

What runs, unmodified, from the reference:
  * ``tensorlink.ml.injector.LayerGroupModule`` (injector.py:154-281) executing the HF decoder-layer loop
    body over each shard's layer subset;
  * ``tensorlink.ml.utils.tensor_to_bytes`` / ``bytes_to_tensor`` (utils.py:569-660) on every inter-shard hop.
The loop-body source handed to LayerGroupModule is the transformers 4.53 Qwen2 loop body (the version the
reference pins; its own AST finder does not match transformers 5.x loops, SURVEY.md F9).
Layers are the installed HF ``Qwen2DecoderLayer``/``Qwen3DecoderLayer`` with the seeded weights; host-side
embed / rotary / mask / final norm / lm_head are HF's (module.py:1023-1056 keeps them on the host).
"""
import hashlib
import json
import os
import sys

import torch

from oracle import portable_cpu
from oracle.ref_shim import import_reference
from tensorlink_b200.ml import configs as C
from tensorlink_b200.ml.weights import init_state_dict, synthetic_tokens
from tests.hf_util import hf_model

LOOP_BODY = """hidden_states = decoder_layer(
    hidden_states,
    attention_mask=causal_mask,
    position_ids=position_ids,
    position_embeddings=position_embeddings,
)"""
INPUT_VARS = ["hidden_states", "causal_mask", "position_ids", "position_embeddings"]
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def run(cfg, n_shards, B, S, attn, dtype=torch.bfloat16):
    injector, utils = import_reference()
    sd = init_state_dict(cfg, dtype=dtype)
    ids = synthetic_tokens(cfg, B, S)
    hf = hf_model(cfg, sd, attn, dtype)
    base, rem = divmod(cfg.n_layers, n_shards)
    bounds, a = [], 0
    for i in range(n_shards):
        b = a + base + (1 if i < rem else 0)
        bounds.append((a, b))
        a = b
    shards = [injector.LayerGroupModule(list(hf.model.layers[a:b]), INPUT_VARS, ["hidden_states"],
                                        LOOP_BODY, "decoder_layer", debug=False) for a, b in bounds]
    with torch.no_grad():
        x = hf.model.embed_tokens(ids)
        pos = torch.arange(S)[None].expand(B, -1)
        pe = hf.model.rotary_emb(x, pos)
        m = torch.full((S, S), torch.finfo(dtype).min, dtype=dtype).triu(1)[None, None].expand(B, 1, S, S)
        hops = []
        for sh in shards:
            kw = dict(hidden_states=x, causal_mask=m, position_ids=pos, position_embeddings=pe)
            wire = utils.tensor_to_bytes(kw)                      # user -> worker  (C1)
            kw = utils.bytes_to_tensor(wire)
            assert torch.equal(kw["hidden_states"], x) and kw["hidden_states"].dtype == dtype
            out = sh(**kw)
            back = utils.bytes_to_tensor(utils.tensor_to_bytes(out))   # worker -> user (C2)
            assert torch.equal(back["hidden_states"], out["hidden_states"])
            x = back["hidden_states"]
            hops.append(x.clone())
        logits = hf.lm_head(hf.model.norm(x))
        unsharded = hf(input_ids=ids).logits
    assert torch.equal(logits, unsharded), "reference sharded != unsharded HF"
    return {"cfg": cfg.name, "n_shards": n_shards, "attn": attn, "seed": 1234, "token_seed": 4321,
            "input_ids": ids, "hops": hops, "logits": logits, "bounds": bounds,
            "dtype": str(dtype)}


CASES = ((C.TINY_QWEN2, 2, 2, 24), (C.TINY_QWEN3, 3, 1, 17), (C.TINY_QWEN2_D128, 2, 1, 33))


def sha256_bf16(t):
    return hashlib.sha256(t.contiguous().view(torch.int16).numpy().tobytes()).hexdigest()


def portable():
    if not portable_cpu.active():          # read when torch loads: start again with the variables set
        os.execve(sys.executable, [sys.executable, "-m", "oracle.gen_golden", "--portable"], dict(os.environ, **portable_cpu.ENV))
    portable_cpu.apply()
    out = {}
    for cfg, n, B, S in CASES:
        g = run(cfg, n, B, S, "eager")
        out[cfg.name] = {"hops_sha256": [sha256_bf16(h) for h in g["hops"]], "logits_sha256": sha256_bf16(g["logits"][:, -4:, :])}
    path = os.path.join(OUT, "ref_layergroup_eager_portable.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
    print(path)


def main():
    os.makedirs(OUT, exist_ok=True)
    for cfg, n, B, S in CASES:
        for attn in ("eager", "sdpa"):
            g = run(cfg, n, B, S, attn)
            path = os.path.join(OUT, f"ref_layergroup_{cfg.name}_{attn}.pt")
            # keep fixtures small: logits for the last 4 positions only
            g["logits"] = g["logits"][:, -4:, :].clone()
            torch.save(g, path)
            print(path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    portable() if sys.argv[1:] == ["--portable"] else main()
