#!/usr/bin/env python
"""Embedding backward alone (native.embed_bwd, id sort included) at one training step's tokens: 4096 tokens x
H = 3584 into the Qwen2.5-7B vocabulary, for uniform ids and for one id taking the whole batch.  CUDA events; one JSON
line per id set, with the card's name and power limit and the time as a fraction of a training step (--step-ms)."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tensorlink_b200 import native as nat  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--tokens", type=int, default=4096)
    ap.add_argument("--hidden", type=int, default=3584)
    ap.add_argument("--vocab", type=int, default=152064)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--step-ms", type=float, default=195.0, help="training step time the kernel is compared with")
    a = ap.parse_args()
    nat.require_device()
    g = torch.Generator(device="cuda").manual_seed(0)
    dout = torch.randn(a.tokens, a.hidden, generator=g, device="cuda").bfloat16()
    table = torch.zeros(a.vocab, a.hidden, dtype=torch.bfloat16, device="cuda")
    id_sets = {"uniform": torch.randint(0, a.vocab, (a.tokens,), generator=g, device="cuda"),
               "one_id": torch.full((a.tokens,), 151643, dtype=torch.int64, device="cuda")}
    for name, ids in id_sets.items():
        for _ in range(10):
            nat.embed_bwd(ids, dout, table)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(a.iters):
            nat.embed_bwd(ids, dout, table)
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) / a.iters * 1e3
        print(json.dumps({"ids": name, "tokens": a.tokens, "hidden": a.hidden, "us": round(us, 2),
                          "fraction_of_step": round(us / (a.step_ms * 1e3), 6), "card": card()}), flush=True)
