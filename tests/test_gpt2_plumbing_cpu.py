"""BASELINE config 1: GPT-2 small (124M), 2 CPU shards (blocks 0-5 / 6-11), one forward on (1,128) synthetic tokens —
the reference's *plumbing* case (no GPU, no B200 kernels involved).

The fixture (tests/golden/ref_gpt2_2shards.pt, oracle/gen_golden_gpt2.py) was produced by the reference's own
``LayerGroupModule`` + wire codec and equals the unsharded HF model bit for bit.  Here the same two-shard composition
is run with THIS repo's wire codecs on the hop (the oracle restatement and the product codec ``p2p/wire.py``) and must
reproduce the reference's hop and logits exactly (fp32 on CPU: same ops, same order => bit-exact, compared by SHA-256),
i.e. a shard boundary + codec adds zero numeric change on this side as well.  Both the fixture and this run use the
host-independent CPU arithmetic of oracle/portable_cpu.py (fp32 GEMMs and the random init are otherwise ISA-specific in
the last bit), which must be in place when torch loads, so the composition runs in a subprocess (this file as a script)."""
import hashlib
import os
import subprocess
import sys

import torch

from oracle import portable_cpu
from oracle import wire_oracle as W
from tensorlink_b200.p2p import wire

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIX = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_gpt2_2shards.pt")


def _sha(t):
    return hashlib.sha256(t.contiguous().numpy().tobytes()).hexdigest()


def _two_shard_runs(fix):
    """For each of this repo's codecs (oracle, product): hop 0 and the logits of the two-shard composition, as SHA-256
    plus a few values; and whether the logits equal the unsharded HF model's bit for bit."""
    from transformers import GPT2Config, GPT2LMHeadModel
    torch.manual_seed(fix["seed"])
    m = GPT2LMHeadModel(GPT2Config(attn_implementation="eager")).eval()
    assert sum(p.numel() for p in m.parameters()) == 124_439_808           # SURVEY.md §8 model table
    ids = fix["input_ids"]
    S = ids.shape[1]
    runs = []
    with torch.no_grad():
        pos = torch.arange(S)[None]
        x = m.transformer.wte(ids) + m.transformer.wpe(pos)
        mask = torch.full((S, S), torch.finfo(torch.float32).min).triu(1)[None, None]
        for codec_enc, codec_dec in ((W.encode, W.decode), (wire.encode, wire.decode)):
            h = x
            hops = []
            for a, b in fix["bounds"]:
                live_ins = codec_dec(codec_enc({"hidden_states": h, "causal_mask": mask, "position_ids": pos}))   # user -> worker
                y = live_ins["hidden_states"]
                for blk in m.transformer.h[a:b]:                                   # the shard = the loop body over its blocks
                    y = blk(y, None, live_ins["causal_mask"], None, encoder_attention_mask=None, use_cache=False,
                            position_ids=live_ins["position_ids"])
                h = codec_dec(codec_enc({**live_ins, "hidden_states": y}))["hidden_states"]                         # worker -> user
                hops.append(h)
            logits = m.lm_head(m.transformer.ln_f(h))
            runs.append({"hop0_sha256": _sha(hops[0]), "logits_sha256": _sha(logits), "hop0_tail": hops[0][:, -2:, :8].clone(),
                         "logits_tail": logits[:, -1, :16].clone()})
        unsharded_equal = bool(torch.equal(logits, m(input_ids=ids).logits))
    return runs, unsharded_equal


def test_gpt2_two_cpu_shards_equal_the_reference_and_unsharded_hf(tmp_path):
    out = tmp_path / "runs.pt"
    r = subprocess.run([sys.executable, os.path.abspath(__file__), str(out)], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, PYTHONPATH=ROOT, **portable_cpu.ENV))
    assert r.returncode == 0, r.stderr[-3000:]
    fix = torch.load(FIX)
    runs, unsharded_equal = torch.load(out)
    assert len(runs) == 2
    for got in runs:
        assert got["hop0_sha256"] == fix["hop0_sha256"] and got["logits_sha256"] == fix["logits_sha256"]
        assert torch.equal(got["hop0_tail"], fix["hop0_tail"]) and torch.equal(got["logits_tail"], fix["logits_tail"])
    assert unsharded_equal                                                      # == unsharded HF, bit for bit


if __name__ == "__main__":
    portable_cpu.apply()
    torch.save(_two_shard_runs(torch.load(FIX)), sys.argv[1])
