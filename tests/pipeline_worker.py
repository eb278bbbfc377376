"""Run under torchrun (gloo, CPU): exercises DistributedModel's multi-rank host logic with the oracle stage.

Started with the host-independent CPU arithmetic of oracle/portable_cpu.py: the pipelined results are compared bit for bit
with one unsharded oracle run, and with the default ISA-specific kernels the two ways of blocking the same math round
differently on some CPUs."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import portable_cpu  # noqa: E402
from oracle import shard_oracle as O  # noqa: E402
from tensorlink_b200.ml import DistributedModel  # noqa: E402
from tensorlink_b200.ml import configs as C  # noqa: E402
from tensorlink_b200.ml.weights import init_state_dict, synthetic_tokens  # noqa: E402
from tensorlink_b200.p2p.link import init_process_group_from_env  # noqa: E402
from tests.oracle_stage import OracleStage  # noqa: E402


def main(out_dir):
    portable_cpu.apply()
    init_process_group_from_env("gloo")
    rank, world = dist.get_rank(), dist.get_world_size()
    cfg = C.TINY_QWEN2_D128
    sd = init_state_dict(cfg)
    res = {}

    # 1) inference forward with logits gathered to rank 0, and the plan handed in explicitly (reference schema)
    from tensorlink_b200.ml import graphing
    plan = graphing.make_plan(cfg, world)
    dm = DistributedModel(cfg, training=False, config=plan, max_batch=4, max_seq=64, _stage_factory=OracleStage, device="cpu")
    ids = synthetic_tokens(cfg, 2, 12)
    out = dm(ids if rank == 0 else None, gather_logits=True)
    if rank == 0:
        with torch.no_grad():
            ref = O.OracleModel(cfg, sd, "sdpa_math").logits(ids)
        res["logits_equal"] = bool(torch.equal(out.logits, ref))
    # the whole model's state dict gathered on the first rank (reference: parameters(distributed=True, load=True))
    whole = dm.state_dict(gather=True)
    if rank == 0:
        res["gather_ok"] = bool(set(whole) == set(sd) and all(torch.equal(whole[k], sd[k]) for k in sd))
    else:
        res["gather_ok"] = bool(0 < len(whole) < len(sd))
    # 2) greedy generate, single micro-batch and 2 micro-batches in flight; streaming callback on rank 0
    class Streamer:
        def __init__(self):
            self.cols, self.ended = [], False

        def put(self, t):
            self.cols.append(t.clone())

        def end(self):
            self.ended = True
    st = Streamer()
    gen = dm.generate(ids if rank == 0 else None, max_new_tokens=6, streamer=st)
    dm2 = DistributedModel(cfg, training=False, n_pipelines=2, max_batch=4, max_seq=64, _stage_factory=OracleStage, device="cpu")
    ids4 = synthetic_tokens(cfg, 4, 9)
    gen2 = dm2.generate(ids4 if rank == 0 else None, max_new_tokens=5)
    ref_gen = O.OracleModel(cfg, sd, "sdpa_math").generate(ids, 6)
    ref_gen2 = O.OracleModel(cfg, sd, "sdpa_math").generate(ids4, 5)
    # HF stopping semantics through the pipeline: every rank returns the same trimmed / padded result
    from tensorlink_b200.ml.module import apply_eos
    eos = int(ref_gen2[1, 9 + 2])
    gen_eos = dm2.generate(ids4 if rank == 0 else None, max_new_tokens=5, eos_token_id=eos, pad_token_id=0)
    res["eos_ok"] = bool(torch.equal(gen_eos, apply_eos(ref_gen2, 9, eos, 0)) and gen_eos.shape[1] <= ref_gen2.shape[1])
    # ... and the loop really stops: 40 tokens requested, both rows (copies of one prompt) emit EOS within the first 3 steps, the ranks agree
    # at the step-16 check (ids in flight are drained first) and return the prompt plus the tokens up to that EOS
    twin = ids4[[1, 1]].contiguous()
    ref_twin = O.OracleModel(cfg, sd, "sdpa_math").generate(twin, 5)
    eos2 = int(ref_twin[0, 9 + 2])
    stop = dm2.generate(twin if rank == 0 else None, max_new_tokens=40, eos_token_id=eos2, pad_token_id=0)
    res["eos_stop_ok"] = bool(torch.equal(stop, apply_eos(ref_twin, 9, eos2, 0)) and stop.shape[1] < 9 + 40)
    res["eos_stop_steps"] = int(getattr(dm2.stage, "n_decode_calls", -1))
    # left-padded batch with its attention_mask: every row equals its own unpadded generation, pads stay in front
    lens, Sp, PAD = [9, 6, 9, 4], 9, 3
    rows = [synthetic_tokens(cfg, 1, L, seed=300 + i)[0] for i, L in enumerate(lens)]
    pids = torch.full((4, Sp), PAD, dtype=torch.int64)
    pmask = torch.zeros(4, Sp, dtype=torch.int64)
    for r, (t, L) in enumerate(zip(rows, lens)):
        pids[r, Sp - L:], pmask[r, Sp - L:] = t, 1
    padded = dm2.generate(pids if rank == 0 else None, attention_mask=pmask if rank == 0 else None, max_new_tokens=4,
                          pad_token_id=PAD)
    ok = tuple(padded.shape) == (4, Sp + 4) and bool(torch.equal(padded[:, :Sp], pids))
    for r, (t, L) in enumerate(zip(rows, lens)):
        want, margins = O.OracleModel(cfg, sd, "sdpa_math").generate(t[None], 4, return_margins=True)
        for k in range(4):                                  # exact until the first step the oracle itself cannot resolve
            if margins[0, k] < 0.05:
                break
            ok = ok and int(padded[r, Sp + k]) == int(want[0, L + k])
    res["left_pad_ok"] = ok
    # a batch the requested micro-batch count does not divide (3 rows, n_pipelines = 2 -> one micro-batch of 3 rows)
    ids3 = synthetic_tokens(cfg, 3, 7, seed=77)
    dm3 = DistributedModel(cfg, training=False, n_pipelines=2, max_batch=6, max_seq=64, _stage_factory=OracleStage, device="cpu")
    gen3 = dm3.generate(ids3 if rank == 0 else None, max_new_tokens=4)
    res["odd_batch_ok"] = bool(torch.equal(gen3, O.OracleModel(cfg, sd, "sdpa_math").generate(ids3, 4)))
    # streamer + early stop: the callback sees exactly the columns the (stopped) loop produced, then end()
    st2 = Streamer()
    stop2 = dm2.generate(twin if rank == 0 else None, max_new_tokens=40, eos_token_id=eos2, pad_token_id=0, streamer=st2)
    if rank == 0:
        cols = torch.stack(st2.cols, 1)
        k = stop2.shape[1] - 9                 # new tokens that survive the EOS trim; the streamer saw at least those
        res["stream_stop_ok"] = bool(st2.ended and 1 <= k <= cols.shape[1] < 40 and torch.equal(cols[:, :k], stop2[:, 9:]))
    res["gen_equal"] = bool(torch.equal(gen, ref_gen))          # every rank holds the result
    res["gen2_equal"] = bool(torch.equal(gen2, ref_gen2))
    if rank == 0:
        res["stream_ok"] = st.ended and torch.equal(torch.stack(st.cols, 1), ref_gen[:, 12:])
    # 3) training step: loss on every rank, backward through the ranks, grads match single-process autograd
    dmt = DistributedModel(cfg, training=True, n_pipelines=2, max_batch=4, max_seq=64, _stage_factory=OracleStage, device="cpu",
                           optimizer=torch.optim.Adam)
    tids = synthetic_tokens(cfg, 4, 16)
    o = dmt(tids if rank == 0 else None, labels=tids if rank == 0 else None)
    o.loss.backward()
    ref_sd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    ref_loss, _ = O.OracleModel(cfg, ref_sd, "sdpa_math").loss(tids, tids)
    ref_loss.backward()
    res["loss_close"] = abs(float(o.loss) - float(ref_loss)) < 2e-3
    worst = 0.0
    for k, v in dmt.stage.sd.items():
        if v.grad is not None and ref_sd[k].grad is not None:
            worst = max(worst, O.rel_l2(v.grad, ref_sd[k].grad))
    res["grad_worst_rel_l2"] = worst
    res["n_params_with_grad"] = sum(v.grad is not None for v in dmt.stage.sd.values())
    res["bytes_sent"] = dmt.link.bytes_sent
    # tied embeddings split over the two ranks (embedding on rank 0, lm_head on rank 1): after backward both copies hold
    # embedding gradient + lm_head gradient = the single-process gradient of the shared tensor
    tcfg = C.TINY_QWEN2
    tsd = init_state_dict(tcfg)
    dtie = DistributedModel(tcfg, training=True, n_pipelines=2, max_batch=4, max_seq=64, _stage_factory=OracleStage, device="cpu",
                            optimizer=torch.optim.Adam)
    tt = synthetic_tokens(tcfg, 4, 12)
    dtie(tt if rank == 0 else None, labels=tt if rank == 0 else None).loss.backward()
    rsd = {k: v.clone().requires_grad_(True) for k, v in tsd.items()}
    rsd["lm_head.weight"] = rsd["model.embed_tokens.weight"]
    O.OracleModel(tcfg, rsd, "sdpa_math").loss(tt, tt)[0].backward()
    if dtie.link.first or dtie.link.last:
        mine = dtie.stage.sd["model.embed_tokens.weight" if dtie.link.first else "lm_head.weight"].grad
        res["tied_rel_l2"] = O.rel_l2(mine, rsd["model.embed_tokens.weight"].grad)
    else:
        res["tied_rel_l2"] = 0.0                # a middle stage holds neither copy
    torch.save(res, os.path.join(out_dir, f"rank{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    try:
        main(sys.argv[1])
    except Exception:
        import traceback
        with open(os.path.join(sys.argv[1], f"err{os.environ.get('RANK', '0')}.txt"), "w") as f:
            traceback.print_exc(file=f)
        raise
