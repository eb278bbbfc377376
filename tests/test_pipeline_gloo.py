"""CPU (gloo) tests of the pipeline host logic with world_size 2 and 3 (first / middle / last stage): plan -> stages, forward
hops, generate with ids hopping back, micro-batch rotation, streaming, EOS early stop, left-padded batches, loss
broadcast, backward routing, tied embeddings on two ranks (SURVEY.md §8e)."""
import os
import socket
import subprocess
import sys

import pytest
import torch

from oracle import portable_cpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.parametrize("world", [2, 3])
def test_pipeline_host_logic(tmp_path, world):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "pipeline_worker.py"), str(tmp_path)]
    env = dict(os.environ, PYTHONPATH=ROOT, **portable_cpu.ENV)
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    errs = "".join(open(p).read() for p in sorted(map(str, tmp_path.glob("err*.txt"))))
    assert r.returncode == 0, errs or r.stderr[-3000:]
    res = [torch.load(tmp_path / f"rank{i}.pt") for i in range(world)]
    r0 = res[0]
    assert r0["logits_equal"] and r0["stream_ok"] and r0["stream_stop_ok"]
    for r_ in res:                                                  # every rank holds every result
        assert r_["gen_equal"] and r_["gen2_equal"] and r_["eos_ok"] and r_["eos_stop_ok"] and r_["left_pad_ok"] and r_["odd_batch_ok"]
        assert r_["loss_close"] and r_["gather_ok"]
        # bf16 autograd in pieces (a gradient crossing a rank boundary is rounded to bf16 once more) vs one graph
        assert r_["grad_worst_rel_l2"] < 2e-2 and r_["tied_rel_l2"] < 2e-2
        assert r_["n_params_with_grad"] >= 9 and r_["bytes_sent"] > 0
