"""BASELINE config 1 (GPT-2 small, 2 CPU worker shards, one forward on (1,128) tokens): the reference's plumbing claim.

TEST INFRA.  Run in the build container (needs /root/reference):  python -m oracle.gen_golden_gpt2
What runs, unmodified, from the reference: ``LayerGroupModule`` (ml/injector.py:154-281) over blocks 0-5 and 6-11 of an
installed-HF ``GPT2LMHeadModel`` (124M, seeded random init, fp32, CPU) and the wire codec ``tensor_to_bytes`` /
``bytes_to_tensor`` (ml/utils.py:569-660) on every hop, exactly like oracle/gen_golden.py does for the Qwen shards.  The
reference's own loop finder cannot split GPT-2 (its ``for i, block in enumerate(self.h)`` is not matched,
ml/injector.py:75-90; SURVEY.md §8c), so the loop body is handed to LayerGroupModule by hand.  Result: the 2-shard
output equals the unsharded HF model BIT FOR BIT on CPU — the sharding + codec add no numeric change.  GPT-2 itself is
not on the B200 path (LayerNorm / GELU / learned positions have no kernels here: config 1 is the reference's CPU
plumbing case); tests/test_gpt2_plumbing_cpu.py re-runs the same 2-shard composition through THIS repo's wire codec
(oracle and product) on CPU and checks it against the fixture written here.  Both run with the host-independent CPU
arithmetic of oracle/portable_cpu.py, so that the SHA-256 comparison holds on any x86-64 host.
"""
import hashlib
import os
import sys

import torch

from oracle import portable_cpu
from oracle.ref_shim import import_reference

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "ref_gpt2_2shards.pt")
LOOP_BODY = """hidden_states = block(
    hidden_states,
    None,
    causal_mask,
    None,
    encoder_attention_mask=None,
    use_cache=False,
    position_ids=position_ids,
)"""
INPUT_VARS = ["hidden_states", "causal_mask", "position_ids"]


def gpt2_small(seed=1234):
    from transformers import GPT2Config, GPT2LMHeadModel
    torch.manual_seed(seed)
    cfg = GPT2Config(attn_implementation="eager")          # GPT-2 small defaults: 12 layers, 768, 12 heads, 50257
    m = GPT2LMHeadModel(cfg).eval()
    assert sum(p.numel() for p in m.parameters()) == 124_439_808
    return m


def tokens(seed=4321):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 50257, (1, 128), dtype=torch.int64, generator=g)


def host_side(m, ids):
    """What stays on the reference's user side (ml/module.py:1023-1056): embeddings, mask, final norm, lm_head."""
    S = ids.shape[1]
    pos = torch.arange(S)[None]
    x = m.transformer.wte(ids) + m.transformer.wpe(pos)
    mask = torch.full((S, S), torch.finfo(torch.float32).min).triu(1)[None, None]
    return x, mask, pos


def main():
    if not portable_cpu.active():          # read when torch loads: start again with the variables set
        os.execve(sys.executable, [sys.executable, "-m", "oracle.gen_golden_gpt2"], dict(os.environ, **portable_cpu.ENV))
    portable_cpu.apply()
    injector, utils = import_reference()
    m, ids = gpt2_small(), tokens()
    with torch.no_grad():
        x, mask, pos = host_side(m, ids)
        hops = []
        for a, b in ((0, 6), (6, 12)):
            shard = injector.LayerGroupModule(list(m.transformer.h[a:b]), INPUT_VARS, ["hidden_states"], LOOP_BODY, "block", debug=False)
            kw = utils.bytes_to_tensor(utils.tensor_to_bytes(dict(hidden_states=x, causal_mask=mask, position_ids=pos)))
            out = utils.bytes_to_tensor(utils.tensor_to_bytes(shard(**kw)))
            x = out["hidden_states"]
            hops.append(x.clone())
        logits = m.lm_head(m.transformer.ln_f(x))
        unsharded = m(input_ids=ids).logits
    assert torch.equal(logits, unsharded), "reference 2-shard GPT-2 != unsharded HF"
    fix = {"seed": 1234, "token_seed": 4321, "input_ids": ids, "bounds": [(0, 6), (6, 12)],
           "hop0_sha256": hashlib.sha256(hops[0].numpy().tobytes()).hexdigest(),
           "logits_sha256": hashlib.sha256(logits.numpy().tobytes()).hexdigest(),
           "hop0_tail": hops[0][:, -2:, :8].clone(), "logits_tail": logits[:, -1, :16].clone()}
    torch.save(fix, OUT)
    print("wrote", OUT, os.path.getsize(OUT), "bytes; sharded == unsharded bit for bit")


if __name__ == "__main__":
    main()
