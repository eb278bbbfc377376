"""Backward / optimizer kernels and the whole training step against the oracle's autograd (CPU).

Gradient tolerances follow tests/test_model_gpu.py: per-op kernels are compared with autograd of the oracle's
restatement of the same op in fp32 on the same bf16 inputs (rel-L2 <= 4e-3: one bf16 rounding of the output is
~2e-3); the full step is compared against fp32 autograd of the oracle model with the chain criteria
(accuracy <= 1.25x / agreement <= 2x the bf16 oracle's own distance from fp32)."""
import pytest
import torch
import torch.nn.functional as F

from oracle import shard_oracle as O
from tensorlink_b200.ml import configs as C
from tensorlink_b200.ml.weights import init_state_dict, synthetic_tokens

pytestmark = pytest.mark.gpu
TOL = 4e-3


@pytest.fixture(scope="module")
def nat():
    from tensorlink_b200 import native
    native.require_device()
    return native


def rnd(*shape, seed=0, std=1.0, dtype=torch.bfloat16):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(*shape, generator=g) * std).to(dtype)


@pytest.mark.parametrize("M,I,gate_std", [pytest.param(M, I, s, id=f"{M}-{I}" + ("" if s == 1.0 else f"-gate{s:g}"))
                                          for M, I, s in [(7, 64, 1.0), (300, 4864, 1.0), (3, 4, 1.0), (5, 12, 1.0),
                                                          (4096, 18944, 1.0), (64, 896, 20.0), (64, 896, 100.0)]])
def test_swiglu_fwd_bwd(nat, M, I, gate_std):
    """(4096, 18944): the 7B bench shape, many grid-stride sweeps; gate std 20 / 100: saturated sigmoid, no NaN or Inf."""
    g, u, dh = rnd(M, I, seed=1, std=gate_std), rnd(M, I, seed=2), rnd(M, I, seed=3)
    gu = torch.stack([g, u], dim=2).reshape(M, 2 * I).contiguous()
    h = torch.empty(M, I, dtype=torch.bfloat16, device="cuda")
    nat.swiglu_fwd(gu.cuda(), h)
    assert torch.equal(h.cpu(), F.silu(g) * u)
    gf, uf = g.float().requires_grad_(), u.float().requires_grad_()
    (F.silu(gf) * uf).backward(dh.float())
    dgu = torch.empty(M, 2 * I, dtype=torch.bfloat16, device="cuda")
    nat.swiglu_bwd(gu.cuda(), dh.cuda(), dgu)
    got = dgu.cpu().view(M, I, 2)
    assert torch.isfinite(got).all()
    assert O.rel_l2(got[..., 0], gf.grad) <= TOL and O.rel_l2(got[..., 1], uf.grad) <= TOL


@pytest.mark.parametrize("rows,H", [(5, 128), (300, 896), (64, 3584), (33, 4096), (1, 1024), (1, 1032), (1, 2048),
                                    (1, 8192), (16384, 896), (16384, 3584)])
def test_rmsnorm_bwd(nat, rows, H):
    """Warp kernel (H <= 1024) and block kernel with 1 / 2 / 4 / 8 vectors per thread; 16384 rows: many rows per block.
    dw accumulates into a non-zero fp32 accumulator, a second call adds to it, and dw_accum=None leaves it alone."""
    x, dy, add = rnd(rows, H, seed=4, std=2.0), rnd(rows, H, seed=5), rnd(rows, H, seed=6)
    w = (1 + 0.1 * torch.randn(H)).bfloat16()
    xf, wf = x.float().requires_grad_(), w.float().requires_grad_()
    O.rmsnorm(xf, wf, 1e-6).backward(dy.float())
    rstd = torch.rsqrt(x.float().pow(2).mean(-1) + 1e-6).cuda()
    dx = torch.empty(rows, H, dtype=torch.bfloat16, device="cuda")
    dw0 = rnd(H, seed=7, dtype=torch.float32) * float(wf.grad.norm()) / H ** 0.5
    dw = dw0.cuda()
    nat.rmsnorm_bwd(x.cuda(), w.cuda(), dy.cuda(), rstd, dx, dw)
    assert O.rel_l2(dx.cpu(), xf.grad) <= TOL
    assert O.rel_l2(dw.cpu() - dw0, wf.grad) <= TOL
    nat.rmsnorm_bwd(x.cuda(), w.cuda(), dy.cuda(), rstd, dx, dw, dx_add=add.cuda())
    assert O.rel_l2(dx.cpu(), xf.grad + add.float()) <= TOL
    assert O.rel_l2(dw.cpu() - dw0, 2 * wf.grad) <= TOL
    before = dw.clone()
    nat.rmsnorm_bwd(x.cuda(), w.cuda(), dy.cuda(), rstd, dx, None)
    assert O.rel_l2(dx.cpu(), xf.grad) <= TOL
    assert torch.equal(dw, before)


@pytest.mark.parametrize("cfg,B,S,T_tab", [
    pytest.param(C.TINY_QWEN2, 2, 19, 64, id="tiny-qwen2"), pytest.param(C.TINY_QWEN2_D128, 2, 19, 64, id="tiny-qwen2-d128"),
    pytest.param(C.QWEN3_8B, 2, 2048, 4096, id="qwen3-8b"), pytest.param(C.QWEN25_7B, 2, 1024, 4096, id="qwen2.5-7b"),
    pytest.param(C.QWEN25_05B, 4, 512, 4096, id="qwen2.5-0.5b")])
def test_rope_kv_bwd(nat, cfg, B, S, T_tab):
    """Model configs: GQA groups of 4 and 7, d = 64 and 128, positions up to 2047 in a table as long as a trainer's."""
    d, n_h, n_kv = cfg.head_dim, cfg.n_heads, cfg.n_kv_heads
    q = rnd(B, n_h, S, d, seed=7).float().requires_grad_()
    k = rnd(B, n_kv, S, d, seed=8).float().requires_grad_()
    n_rep = n_h // n_kv
    dq = rnd(B, S, n_h, d, seed=9)
    dk_p, dv_p = rnd(B, n_h, S, d, seed=10), rnd(B, n_h, S, d, seed=11)          # one partial per query head
    dk = dk_p.float().view(B, n_kv, n_rep, S, d).sum(2)
    dv = dv_p.float().view(B, n_kv, n_rep, S, d).sum(2)
    cos, sin = O.rope_tables(cfg, torch.arange(S)[None].expand(B, -1), torch.bfloat16)
    qr, kr = O.apply_rope(q, k, cos.float(), sin.float())
    (qr * dq.transpose(1, 2).float()).sum().backward(retain_graph=True)
    (kr * dk.float()).sum().backward()
    ct, st = nat.rope_table(O.rope_inv_freq(cfg).cuda(), T_tab)
    dqkv = torch.empty(B * S, cfg.qkv_dim, dtype=torch.bfloat16, device="cuda")
    nat.rope_kv_bwd(dq.cuda().reshape(B * S, -1), dk_p.cuda(), dv_p.cuda(), dqkv, ct, st, S, n_h, n_kv, d)
    got = dqkv.cpu().view(B, S, n_h + 2 * n_kv, d)
    assert O.rel_l2(got[:, :, :n_h].transpose(1, 2), q.grad) <= TOL
    assert O.rel_l2(got[:, :, n_h:n_h + n_kv].transpose(1, 2), k.grad) <= TOL
    assert O.rel_l2(got[:, :, n_h + n_kv:].transpose(1, 2), dv) <= TOL
    dv_seq = dv_p.float().view(B, n_kv, n_rep, S, d)[:, :, 0].clone()
    for r in range(1, n_rep):                     # the kernel's order: fp32 partial sums, one rounding
        dv_seq += dv_p.float().view(B, n_kv, n_rep, S, d)[:, :, r]
    assert torch.equal(got[:, :, n_h + n_kv:].transpose(1, 2), dv_seq.bfloat16())


@pytest.mark.parametrize("B,S,n_h,n_kv,d,impl", [
    (2, 64, 4, 2, 64, "mma"), (1, 100, 14, 2, 64, "mma"), (2, 130, 4, 2, 128, "mma"), (1, 257, 8, 8, 128, "mma"),
    (2, 128, 4, 2, 128, "tc"), (2, 130, 4, 2, 128, "tc"), (1, 257, 8, 8, 128, "tc"), (2, 192, 14, 2, 64, "tc"),
    (1, 321, 4, 4, 64, "tc"), (2, 512, 28, 4, 128, "tc"), (1, 1024, 32, 8, 128, "tc"),
    (8, 512, 28, 4, 128, "default"), (2, 1024, 32, 8, 128, "default"), (4, 512, 14, 2, 64, "default"),
    (2, 127, 4, 2, 128, "default"), (2, 128, 4, 2, 128, "default")])
def test_attn_bwd(nat, B, S, n_h, n_kv, d, impl, monkeypatch):
    """dQ, dK, dV vs fp32 autograd: the mma.sync kernels (short sequences, TL_ATTN_BWD=mma) and the tcgen05 kernels (from one
    128-row tile upwards; sequence lengths off the 64 / 128 tile grid, GQA groups 1..7, both head sizes); "default": no
    override, the bench / Qwen3-8B / 0.5B shapes and both sides of the 128-row dispatch boundary."""
    if impl == "default":
        monkeypatch.delenv("TL_ATTN_BWD", raising=False)
    else:
        monkeypatch.setenv("TL_ATTN_BWD", impl)
    _check_attn_bwd(nat, B, S, n_h, n_kv, d, std=0.7)


def test_attn_bwd_peaked_softmax(nat, monkeypatch):
    """q, k with std 3: near one-hot attention rows (large logits, P close to 0 / 1).  Here dS = P * (dP - D) cancels,
    and D = rowsum(dO * O) is taken from the bf16 forward output, so bf16 attention itself is off fp32 by more than 4e-3:
    the attention rule of tests/test_kernels_gpu.py applies (no less accurate than the same math in bf16 autograd)."""
    monkeypatch.delenv("TL_ATTN_BWD", raising=False)
    _check_attn_bwd(nat, 2, 256, 8, 2, 128, std=3.0, vs_bf16_autograd=True)


def _check_attn_bwd(nat, B, S, n_h, n_kv, d, std, vs_bf16_autograd=False):
    q, k, v = rnd(B, S, n_h, d, seed=12, std=std), rnd(B, n_kv, S, d, seed=13, std=std), rnd(B, n_kv, S, d, seed=14)
    do = rnd(B, S, n_h * d, seed=15)
    qf, kf, vf = q.float().requires_grad_(), k.float().requires_grad_(), v.float().requires_grad_()
    n_rep = n_h // n_kv
    s = (qf.transpose(1, 2) @ O.repeat_kv(kf, n_rep).transpose(2, 3)) * d ** -0.5 + O.causal_mask(S, S, torch.float32)
    of = (F.softmax(s, -1) @ O.repeat_kv(vf, n_rep)).transpose(1, 2).reshape(B, S, -1)
    of.backward(do.float())
    tol = {"q": TOL, "k": TOL, "v": TOL}
    if vs_bf16_autograd:
        qb, kb, vb = q.clone().requires_grad_(), k.clone().requires_grad_(), v.clone().requires_grad_()
        sb = (qb.transpose(1, 2) @ O.repeat_kv(kb, n_rep).transpose(2, 3)) * d ** -0.5 + O.causal_mask(S, S, torch.bfloat16)
        (F.softmax(sb, -1) @ O.repeat_kv(vb, n_rep)).transpose(1, 2).reshape(B, S, -1).backward(do)
        for n, gb, gf in (("q", qb.grad, qf.grad), ("k", kb.grad, kf.grad), ("v", vb.grad, vf.grad)):
            tol[n] = max(TOL, 1.25 * O.rel_l2(gb, gf))
        print("bf16 autograd vs fp32 (x1.25):", tol)
    T_max = S + 3
    kc = torch.zeros(B, n_kv, T_max, d, dtype=torch.bfloat16)
    vc = torch.zeros_like(kc)
    kc[:, :, :S], vc[:, :, :S] = k, v
    kc, vc = kc.cuda(), vc.cuda()
    out = torch.empty(B, S, n_h * d, dtype=torch.bfloat16, device="cuda")
    lse = torch.empty(B, n_h, S, dtype=torch.float32, device="cuda")
    nat.attn_prefill_fwd(q.cuda(), kc, vc, out, lse, B, S, 0, n_h, n_kv, d, d ** -0.5)
    # the trainer allocates dq / dk / dv with torch.empty: every element below S must be written
    dq = torch.full((B, S, n_h, d), float("nan"), dtype=torch.bfloat16, device="cuda")
    dk = torch.full((B, n_h, T_max, d), float("nan"), dtype=torch.bfloat16, device="cuda")   # one partial per query head
    dv = torch.full_like(dk, float("nan"))
    ws = torch.empty(nat.attn_bwd_ws(B, S, n_h), dtype=torch.uint8, device="cuda")
    nat.attn_bwd(q.cuda(), kc, vc, out, do.cuda(), lse, dq, dk, dv, ws, B, S, n_h, n_kv, d, d ** -0.5)
    assert torch.isfinite(dq).all() and torch.isfinite(dk[:, :, :S]).all() and torch.isfinite(dv[:, :, :S]).all()
    dks = dk.cpu().float().view(B, n_kv, n_rep, T_max, d).sum(2)
    dvs = dv.cpu().float().view(B, n_kv, n_rep, T_max, d).sum(2)
    errs = {"q": O.rel_l2(dq.cpu(), qf.grad), "k": O.rel_l2(dks[:, :, :S], kf.grad), "v": O.rel_l2(dvs[:, :, :S], vf.grad)}
    print("kernel vs fp32:", errs)
    assert all(errs[n] <= tol[n] for n in errs), (errs, tol)
    for t in (dk, dv):                           # rows past S: left alone or zero, never anything else
        tail = t[:, :, S:]
        assert (torch.isnan(tail) | (tail == 0)).all()


@pytest.mark.parametrize("M,V", [(5, 1024), (64, 151936)])
def test_cross_entropy(nat, M, V):
    logits = rnd(M, V, seed=16, std=2.0)
    labels = torch.randint(0, V, (M,))
    labels[1] = -100
    lf = logits.float().requires_grad_()
    n_valid = int((labels != -100).sum())
    loss = F.cross_entropy(lf, labels, ignore_index=-100)
    loss.backward()
    ls = torch.zeros(1, dtype=torch.float32, device="cuda")
    nv = torch.zeros(1, dtype=torch.int32, device="cuda")
    d = torch.empty(M, V, dtype=torch.bfloat16, device="cuda")
    nat.ce_fwd_bwd(logits.cuda(), labels.cuda(), ls, nv, d, 1.0 / n_valid)
    assert int(nv) == n_valid
    assert abs(float(ls) / n_valid - float(loss)) <= 1e-4 * abs(float(loss))
    assert O.rel_l2(d.cpu(), lf.grad) <= TOL
    assert d.cpu()[1].abs().sum() == 0


def test_embed_bwd_colsum_add(nat):
    ids = torch.tensor([[3, 7, 3, 9]])
    dout = rnd(4, 64, seed=17)
    dt = torch.zeros(16, 64, dtype=torch.bfloat16, device="cuda")
    nat.embed_bwd(ids.cuda(), dout.cuda(), dt)
    ref = torch.zeros(16, 64).index_add_(0, ids.view(-1), dout.float())
    assert O.rel_l2(dt.cpu(), ref) <= TOL
    dy = rnd(300, 1152, seed=18)
    db = torch.ones(1152, dtype=torch.float32, device="cuda")
    nat.colsum(dy.cuda(), db)
    assert O.rel_l2(db.cpu(), 1 + dy.float().sum(0)) <= 1e-5
    a, b = rnd(4096, seed=19), rnd(4096, seed=20)
    ad = a.cuda()
    nat.add_inplace(ad, b.cuda())
    assert torch.equal(ad.cpu(), a + b)


def test_adamw_matches_torch(nat):
    p0, g = rnd(5000, seed=21), rnd(5000, seed=22, std=0.1)
    for decoupled, wd in ((False, 0.0), (False, 0.01), (True, 0.01)):
        ref = p0.float().clone().requires_grad_()
        opt = (torch.optim.AdamW if decoupled else torch.optim.Adam)([ref], lr=1e-2, weight_decay=wd)
        p = p0.cuda().clone()
        m = torch.zeros(5000, dtype=torch.float32, device="cuda")
        v = torch.zeros_like(m)
        for t in range(1, 4):
            ref.grad = g.float()
            opt.step()
            nat.adamw_step(p, g.cuda(), m, v, 1e-2, 0.9, 0.999, 1e-8, wd, t, decoupled)
            ref.data = ref.data.bfloat16().float()        # the parameter lives in bf16
        assert O.rel_l2(p.cpu(), ref.data) <= 1e-3


def _oracle_grads(cfg, ids, dtype, attn="sdpa_math"):
    sd = {k: v.to(dtype).clone().requires_grad_(True) for k, v in init_state_dict(cfg).items()}
    if cfg.tied:
        sd["lm_head.weight"] = sd["model.embed_tokens.weight"]
    loss, _ = O.OracleModel(cfg, sd, attn).loss(ids, ids)
    loss.backward()
    return float(loss), {k: v.grad for k, v in sd.items() if v.grad is not None}


@pytest.mark.parametrize("cfg", [C.TINY_QWEN2, C.TINY_QWEN2_D128, C.TINY_QWEN3], ids=lambda c: c.name)
@pytest.mark.parametrize("n_mb", [1, 2])
def test_training_step_vs_oracle_autograd(cfg, n_mb):
    from tensorlink_b200.ml import DistributedModel
    ids = synthetic_tokens(cfg, 4, 48)
    loss32, g32 = _oracle_grads(cfg, ids, torch.float32)
    loss16, g16 = _oracle_grads(cfg, ids, torch.bfloat16)
    dm = DistributedModel(cfg, training=True, n_pipelines=n_mb, max_batch=4, max_seq=64, optimizer=torch.optim.Adam)
    opt = dm.create_optimizer(lr=1e-3)
    dm.train()
    opt.zero_grad()
    out = dm(ids, labels=ids)
    out.loss.backward()
    torch.cuda.synchronize()
    print(f"{cfg.name} n_mb={n_mb}: loss gpu {float(out.loss):.6f} oracle_bf16 {loss16:.6f} oracle_fp32 {loss32:.6f}")
    assert abs(float(out.loss) - loss32) <= max(2 * abs(loss16 - loss32), 2e-3)
    got = dm.stage.params.hf_state_dict(grads=True)
    worst = 0.0
    names = ["model.layers.0.self_attn.q_norm.weight", "model.layers.2.self_attn.k_norm.weight",
             "model.layers.0.self_attn.k_proj.weight"] if cfg.qk_norm else ["model.layers.0.self_attn.k_proj.bias"]
    for name in names + ["model.layers.0.self_attn.q_proj.weight",
                 "model.layers.1.self_attn.o_proj.weight", "model.layers.2.mlp.gate_proj.weight",
                 "model.layers.2.mlp.up_proj.weight", "model.layers.3.mlp.down_proj.weight",
                 "model.layers.0.input_layernorm.weight", "model.layers.3.post_attention_layernorm.weight",
                 "model.norm.weight", "model.embed_tokens.weight"] + ([] if cfg.tied else ["lm_head.weight"]):
        e_ref = O.rel_l2(g16[name], g32[name])
        e_gpu = O.rel_l2(got[name].cpu(), g32[name])
        print(f"  {name}: gpu-vs-fp32 {e_gpu:.3e} oracle_bf16-vs-fp32 {e_ref:.3e}")
        worst = max(worst, e_gpu / e_ref)
        assert e_gpu <= 1.5 * e_ref + 2e-3, name
    # optimizer step moves the parameters the way torch.optim.Adam does on the same gradients
    before = dm.stage.params.flat.clone()
    opt.step()
    delta = (dm.stage.params.flat.float() - before.float())
    nz = dm.stage.params.grad != 0
    assert float(delta[nz].abs().mean()) > 1e-4            # first Adam step: |delta| ~ lr for every touched weight
    assert float(delta[~nz].abs().max()) == 0.0


def test_training_loss_decreases():
    from tensorlink_b200.ml import DistributedModel
    cfg = C.TINY_QWEN2_D128
    ids = synthetic_tokens(cfg, 4, 32)
    dm = DistributedModel(cfg, training=True, max_batch=4, max_seq=64, optimizer=torch.optim.AdamW)
    opt = dm.create_optimizer(lr=2e-3, weight_decay=0.01)
    losses = []
    for _ in range(8):
        opt.zero_grad()
        out = dm(input_ids=ids, labels=ids)
        out.loss.backward()
        opt.step()
        losses.append(float(out.loss))
    print("losses", [round(l, 4) for l in losses])
    assert losses[-1] < losses[0] - 0.5


@pytest.mark.parametrize("n_mb", [1, 2], ids=["one_mb", "two_mb_split_head"])
def test_upstream_gradient_scales_every_parameter(n_mb):
    """``(loss * c).backward()`` (gradient accumulation, loss scaling): EVERY gradient is multiplied by c — including
    the lm_head and final-norm gradients, which are produced during the forward pass — and a training-mode forward
    that is never followed by backward leaves the gradient arena untouched (autograd semantics of the reference,
    ml/worker.py:271)."""
    from tensorlink_b200.ml import DistributedModel
    for cfg in (C.TINY_QWEN2_D128, C.TINY_QWEN2):                 # untied and tied lm_head
        ids = synthetic_tokens(cfg, 2, 24)
        dm = DistributedModel(cfg, training=True, n_pipelines=n_mb, max_batch=2, max_seq=32, optimizer=torch.optim.Adam)
        opt = dm.create_optimizer(lr=1e-3)
        opt.zero_grad()
        dm(ids, labels=ids).loss.backward()
        assert dm.stage.trainer.head_split == (n_mb > 1)
        full = {k: v.clone() for k, v in dm.stage.params.hf_state_dict(grads=True).items()}
        opt.zero_grad()
        dm(ids, labels=ids)                                        # forward only: nothing may reach the arena
        untouched = dm.stage.params.hf_state_dict(grads=True)
        assert all(float(v.float().abs().sum()) == 0.0 for v in untouched.values())
        (dm(ids, labels=ids).loss * 0.5).backward()
        half = dm.stage.params.hf_state_dict(grads=True)
        for k, v in full.items():
            if "norm" in k or k.endswith(".bias"):
                # gains / biases are summed over row blocks with fp32 atomics: the order varies from run to run
                assert O.rel_l2(half[k].float() * 2, v.float()) <= 2e-3, k
            else:
                assert torch.equal(half[k].float() * 2, v.float()), k   # a power of two: exact in bf16
        # accumulation: a second backward without zero_grad adds the same gradient again
        (dm(ids, labels=ids).loss * 0.5).backward()
        acc = dm.stage.params.hf_state_dict(grads=True)
        for k in ("lm_head.weight", "model.norm.weight", "model.layers.0.mlp.down_proj.weight", "model.embed_tokens.weight"):
            assert O.rel_l2(acc[k], full[k]) <= 4e-3, k


def test_deferred_weight_gradients_equal_per_micro_batch_accumulation():
    """n micro-batches: one weight-gradient GEMM per weight over all tokens of the step (fp32 accumulation over the
    whole contraction) vs the single-micro-batch step on the same rows — same loss, gradients within one bf16 rounding."""
    from tensorlink_b200.ml import DistributedModel
    cfg = C.TINY_QWEN3
    ids = synthetic_tokens(cfg, 4, 32)
    out = {}
    for n_mb in (1, 4):
        dm = DistributedModel(cfg, training=True, n_pipelines=n_mb, max_batch=4, max_seq=32, optimizer=torch.optim.Adam)
        opt = dm.create_optimizer(lr=1e-3)
        opt.zero_grad()
        o = dm(ids, labels=ids)
        o.loss.backward()
        out[n_mb] = (float(o.loss), dm.stage.params.hf_state_dict(grads=True))
        assert dm.stage.trainer.defer_w == (n_mb > 1)
        opt.step()
        torch.cuda.synchronize()
    assert abs(out[1][0] - out[4][0]) < 2e-3
    for k, v in out[1][1].items():
        assert O.rel_l2(out[4][1][k], v) <= 6e-3, k


def test_layerwise_adam_on_side_stream_equals_one_launch(monkeypatch):
    """``TL_ADAM_OVERLAP=1`` (opt-in: measured slower on the 7B step, DESIGN.md §4.4): the update of layer j starts as
    soon as its gradients are final; parameters after two steps equal the default single-launch update bit for bit."""
    from tensorlink_b200.ml import DistributedModel
    cfg = C.TINY_QWEN3
    ids = synthetic_tokens(cfg, 4, 32)
    res = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("TL_ADAM_OVERLAP", mode)
        dm = DistributedModel(cfg, training=True, n_pipelines=2, max_batch=4, max_seq=32, optimizer=torch.optim.AdamW, seed=5)
        opt = dm.create_optimizer(lr=1e-3, weight_decay=0.01)
        for _ in range(2):
            opt.zero_grad()
            dm(ids, labels=ids).loss.backward()
            opt.step()
        if hasattr(opt, "wait"):
            opt.wait()
        torch.cuda.synchronize()
        res[mode] = dm.stage.params.flat.clone()
    # norm-gain gradients are summed with fp32 atomics: allow their last-bit noise, everything else is identical
    diff = (res["0"].float() - res["1"].float()).abs()
    assert float((diff > 0).float().mean()) < 1e-3 and float(diff.max()) <= 2e-3 * float(res["0"].float().abs().max())


def test_other_optimizer_classes_step_like_torch():
    """``optimizer=torch.optim.SGD`` (any Optimizer subclass, like the reference's worker accepts, ml/worker.py:1309-1327):
    the class's own step runs on the device over the flat arena; the update equals lr * (momentum-filtered) gradient."""
    from tensorlink_b200.ml import DistributedModel
    cfg = C.TINY_QWEN2_D128
    ids = synthetic_tokens(cfg, 2, 24)
    dm = DistributedModel(cfg, training=True, max_batch=2, max_seq=32, optimizer=torch.optim.SGD)
    opt = dm.create_optimizer(lr=0.5, momentum=0.0)
    opt.zero_grad()
    out = dm(ids, labels=ids)
    out.loss.backward()
    p = dm.stage.params
    p.grad_settle()
    before, g = p.flat.float().clone(), p.grad.float().clone()
    opt.step()
    want = (before - 0.5 * g).bfloat16().float()
    assert O.rel_l2(p.flat.float(), want) <= 1e-3 and float((p.flat.float() - before).abs().sum()) > 0
    losses = [float(out.loss)]
    for _ in range(5):
        opt.zero_grad()
        o = dm(ids, labels=ids)
        o.loss.backward()
        opt.step()
        losses.append(float(o.loss))
    assert losses[-1] < losses[0]
    with pytest.raises(TypeError):
        DistributedModel(cfg, training=True, max_batch=2, max_seq=32, optimizer="sgd").create_optimizer(lr=0.1)
