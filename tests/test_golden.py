"""Oracle vs golden vectors produced by the reference's own LayerGroupModule + wire codec
(oracle/gen_golden.py; fixtures committed under tests/golden/).

The eager comparison is bit for bit, and with torch's default ISA-specific CPU kernels a bf16 run differs in the last bit
from one CPU to another.  So the oracle's eager runs use the host-independent arithmetic of oracle/portable_cpu.py, which
must be in place when torch loads (a subprocess: this file run as a script), and are checked against the SHA-256 of the
reference's eager runs under the same arithmetic (ref_layergroup_eager_portable.json)."""
import glob
import json
import os
import subprocess
import sys

import pytest
import torch

from oracle import portable_cpu
from oracle import shard_oracle as O
from oracle.gen_golden import sha256_bf16
from tensorlink_b200.ml import configs as C
from tensorlink_b200.ml.weights import init_state_dict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "ref_layergroup_*.pt")))
PORTABLE = os.path.join(os.path.dirname(__file__), "golden", "ref_layergroup_eager_portable.json")


def test_fixtures_present():
    assert len(GOLDEN) == 6


def _oracle_hops(g, attn_mode):
    cfg = C.get_config(g["cfg"])
    sd = init_state_dict(cfg, seed=g["seed"])
    m = O.OracleModel(cfg, sd, attn_mode)
    ids = g["input_ids"]
    B, S = ids.shape
    with torch.no_grad():
        x = torch.nn.functional.embedding(ids, m.embed)
        cos, sin = O.rope_tables(cfg, torch.arange(S)[None].expand(B, -1), x.dtype)
        hops = []
        for a, b in g["bounds"]:
            x = O.wire_hop(O.shard_forward(cfg, m.layers[a:b], list(range(a, b)), x, cos, sin, attn_mode))
            hops.append(x)
        logits = torch.nn.functional.linear(O.rmsnorm(x, m.norm, cfg.rms_eps), m.head)[:, -4:, :]
    return hops, logits


def _eager_digests(paths):
    """{config name: SHA-256 of the oracle's eager hops and last-4 logits} on the inputs of each eager fixture."""
    out = {}
    for p in paths:
        g = torch.load(p)
        hops, logits = _oracle_hops(g, "eager")
        out[g["cfg"]] = {"hops_sha256": [sha256_bf16(h) for h in hops], "logits_sha256": sha256_bf16(logits)}
    return out


@pytest.fixture(scope="module")
def portable_eager_digests():
    r = subprocess.run([sys.executable, os.path.abspath(__file__)], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, PYTHONPATH=ROOT, **portable_cpu.ENV))
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout.splitlines()[-1])


@pytest.mark.parametrize("path", [p for p in GOLDEN if p.endswith("_eager.pt")], ids=os.path.basename)
def test_oracle_bit_exact_vs_reference_layergroup_eager(path, portable_eager_digests):
    cfg = torch.load(path)["cfg"]
    with open(PORTABLE) as f:
        want = json.load(f)[cfg]
    assert portable_eager_digests[cfg] == want


@pytest.mark.parametrize("path", [p for p in GOLDEN if p.endswith("_sdpa.pt")], ids=os.path.basename)
def test_oracle_sdpa_math_vs_reference_layergroup_sdpa(path):
    """Tolerance: the spread between the reference's own eager and sdpa runs (its bf16 noise floor)."""
    g = torch.load(path)
    ge = torch.load(path.replace("_sdpa.pt", "_eager.pt"))
    hops, logits = _oracle_hops(g, "sdpa_math")
    for got, ref, ref_e in zip(hops, g["hops"], ge["hops"]):
        floor = O.rel_l2(ref_e, ref)
        assert O.rel_l2(got, ref) <= 1.25 * floor + 1e-6
    assert O.rel_l2(logits, g["logits"]) <= 1.25 * O.rel_l2(ge["logits"], g["logits"])


if __name__ == "__main__":
    portable_cpu.apply()
    print(json.dumps(_eager_digests([p for p in GOLDEN if p.endswith("_eager.pt")])))
