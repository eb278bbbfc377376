"""Training kernels at the shapes and in the modes the trainer (ml/train.py) calls them with.

References: fp64 sums (embedding backward, GEMMs, column sums), fp32 autograd (q/k-norm backward, cross-entropy) and
torch.optim (AdamW).  Tolerances are the suite's: one bf16 rounding per output, rel-L2 <= 1e-3 against the rounded
reference; backward ops rel-L2 <= 4e-3 against fp32 autograd on the same bf16 inputs; fp32 outputs 1e-5 (1e-4 for
long contractions); exact wherever the kernel's arithmetic is fixed."""
import pytest
import torch
import torch.nn.functional as F

from oracle import shard_oracle as O

pytestmark = pytest.mark.gpu
TOL, TOL_BWD = 1e-3, 4e-3


@pytest.fixture(scope="module")
def nat():
    from tensorlink_b200 import native
    native.require_device()
    return native


def rnd(*shape, seed=0, std=1.0, dtype=torch.bfloat16, device="cpu"):
    g = torch.Generator(device=device).manual_seed(seed)
    return (torch.randn(*shape, generator=g, device=device) * std).to(dtype)


# ---------------------------------------------------------------------------------------------- embedding backward
def _embed_ref(ids, dout, V):
    """fp64 sum of each id's rows (same bf16 rows as the kernel), and the touched ids."""
    ref = torch.zeros(V, dout.shape[1], dtype=torch.float64, device=dout.device)
    ok = (ids >= 0) & (ids < V)
    ref.index_add_(0, ids[ok], dout[ok].double())
    return ref, torch.unique(ids[ok])


def _rel(a, b):
    """rel-L2 in fp64 on the device (the large optimizer arenas)."""
    a, b = a.double().flatten(), b.double().flatten()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def _rows_rel_l2(got, want):
    """rel-L2 of every row on its own (fp64)."""
    got, want = got.double(), want.double()
    return (got - want).norm(dim=1) / want.norm(dim=1).clamp_min(1e-30)


@pytest.mark.parametrize("H", [896, 3584])
@pytest.mark.parametrize("k", [1, 2, 17, 300, 4096])
def test_embed_bwd_repeated_id(nat, k, H):
    """One id that occurs k times (a frequent token, a padding id): its row is the fp32 sum rounded once, not k bf16
    roundings.  torch's own CUDA embedding backward on the same rows is printed beside it for comparison."""
    V = 1000
    ids = torch.full((k,), 17, dtype=torch.int64, device="cuda")
    dout = rnd(k, H, seed=k, device="cuda")
    dt = torch.zeros(V, H, dtype=torch.bfloat16, device="cuda")
    nat.embed_bwd(ids, dout, dt)
    ref, _ = _embed_ref(ids, dout, V)
    err = O.rel_l2(dt[17], ref[17])
    w = torch.zeros(V, H, dtype=torch.bfloat16, device="cuda", requires_grad=True)
    F.embedding(ids, w).backward(dout)
    print(f"k={k} H={H}: tl_embed_bwd rel-L2 {err:.2e}, torch CUDA embedding backward {O.rel_l2(w.grad[17], ref[17]):.2e}")
    assert err <= TOL_BWD
    assert int(torch.count_nonzero(dt[:17])) == 0 and int(torch.count_nonzero(dt[18:])) == 0


def _zipf_ids(n, V, seed, pad_id, n_pad):
    """Token ids of a heavy-tailed batch: a seeded Zipf-like draw over V (rank r with weight 1/(r+1)^1.1, ranks
    shuffled over the vocabulary) plus a block of one padding id."""
    g = torch.Generator().manual_seed(seed)
    w = 1.0 / torch.arange(1, V + 1, dtype=torch.float64) ** 1.1
    ranks = torch.multinomial(w, n - n_pad, replacement=True, generator=g)
    ids = torch.randperm(V, generator=g)[ranks]
    return torch.cat([ids, torch.full((n_pad,), pad_id, dtype=torch.int64)])


def test_embed_bwd_zipf_batch(nat):
    """A 4096-token step over the Qwen2.5-7B vocabulary with a heavy-tailed id distribution and 512 padding tokens:
    every touched row within 4e-3 of the fp64 sum, every other row left at zero."""
    V, H, n = 152064, 3584, 4096
    ids = _zipf_ids(n, V, seed=3, pad_id=151643, n_pad=512).cuda()
    counts = torch.bincount(ids, minlength=V)
    print(f"zipf batch: {int((counts > 0).sum())} distinct ids, most frequent x{int(counts.max())}, "
          f"second x{int(counts.topk(2).values[1])}")
    dout = rnd(n, H, seed=4, device="cuda")
    dt = torch.zeros(V, H, dtype=torch.bfloat16, device="cuda")
    nat.embed_bwd(ids, dout, dt)
    ref, touched = _embed_ref(ids, dout, V)
    untouched = torch.ones(V, dtype=torch.bool, device="cuda")
    untouched[touched] = False
    assert int(torch.count_nonzero(dt[untouched])) == 0
    errs = _rows_rel_l2(dt[touched], ref[touched])
    worst = int(errs.argmax())
    print(f"zipf batch: worst touched row rel-L2 {float(errs[worst]):.2e} (id seen x{int(counts[touched[worst]])})")
    assert float(errs.max()) <= TOL_BWD


def test_embed_bwd_accumulates_into_nonzero_table(nat):
    """Successive micro-batches (and the tied-embedding delta) add into a non-zero bf16 gradient: each call gives
    bf16(table + fp32 sum of its rows), one rounding per call."""
    V, H = 4096, 896
    g = torch.Generator().manual_seed(6)
    table = rnd(V, H, seed=7, device="cuda")
    want = table.clone()
    dt = table.clone()
    hit = torch.zeros(V, dtype=torch.bool, device="cuda")
    for call in range(2):
        ids = torch.cat([torch.full((300,), 5), torch.randint(0, V // 2, (724,), generator=g)])
        ids = ids[torch.randperm(ids.numel(), generator=g)].cuda()
        dout = rnd(ids.numel(), H, seed=10 + call, device="cuda")
        nat.embed_bwd(ids, dout, dt)
        ref, touched = _embed_ref(ids, dout, V)
        want = (want.double() + ref).bfloat16()
        hit[touched] = True
    assert O.rel_l2(dt, want) <= TOL
    assert O.rel_l2(dt[5], want[5]) <= TOL
    assert torch.equal(dt[~hit], table[~hit])


def test_embed_bwd_skips_out_of_range_ids(nat):
    V, H = 512, 64
    ids = torch.tensor([-100, 3, -1, V, 3, V + 7, 0, V - 1, -100], device="cuda")
    dout = rnd(ids.numel(), H, seed=8, device="cuda")
    dt = torch.zeros(V, H, dtype=torch.bfloat16, device="cuda")
    nat.embed_bwd(ids, dout, dt)
    ref, touched = _embed_ref(ids, dout, V)
    assert sorted(touched.tolist()) == [0, 3, V - 1]
    assert O.rel_l2(dt, ref.bfloat16()) <= TOL
    assert torch.equal(dt[0], dout[6]) and torch.equal(dt[V - 1], dout[7])


def test_embed_bwd_is_deterministic(nat):
    V, H = 152064, 3584
    ids = _zipf_ids(4096, V, seed=9, pad_id=151643, n_pad=256).cuda()
    dout = rnd(ids.numel(), H, seed=10, device="cuda")
    a = torch.zeros(V, H, dtype=torch.bfloat16, device="cuda")
    b = torch.zeros_like(a)
    nat.embed_bwd(ids, dout, a)
    nat.embed_bwd(ids, dout, b)
    assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------- training GEMMs
def _sample_rows(M, tile, n_rand, seed):
    """All rows when few; else the first and the last (partial) row tile and a seeded sample in between."""
    if M <= 3 * tile + n_rand:
        return torch.arange(M)
    last = (M - 1) // tile * tile
    g = torch.Generator().manual_seed(seed)
    mid = torch.randint(tile, last, (n_rand,), generator=g)
    return torch.unique(torch.cat([torch.arange(tile), torch.arange(last, M), mid]))


# (M, N, K) = (out features, in features, tokens): qkv of 0.5B; qkv, wo, gate/up, down and lm_head of 7B
WGRAD_SHAPES = [(1152, 896, 4096), (896, 896, 4096), (4608, 3584, 4096), (3584, 3584, 4096), (37888, 3584, 4096),
                (3584, 18944, 4096), (152064, 3584, 2048),
                (1152, 896, 1), (1152, 896, 7), (1152, 896, 63), (1152, 896, 65), (1152, 896, 1003),
                (4608, 3584, 1), (4608, 3584, 7), (4608, 3584, 63), (4608, 3584, 65), (4608, 3584, 1003)]


@pytest.mark.parametrize("M,N,K", WGRAD_SHAPES)
def test_gemm_weight_grad_trainer_flags(nat, M, N, K):
    """dW += dY^T X as every weight-gradient GEMM of the trainer runs it: A = dY [tokens, out] and B = X [tokens, in]
    both MN-major, EPI_ACCUM into a non-zero bf16 C, K = token count (any K, odd ones included).  (896, 896) and
    (1152, 896) fill too few 256x256 tiles for the CTA-pair kernel; the 7B shapes run on it.  The bf16 epilogue rounds
    like autograd's ``grad += dW``: the product is rounded to bf16, then the sum (gemm_common.cuh); a fresh gradient
    (no EPI_ACCUM) is the product rounded once."""
    tiles2 = ((M + 255) // 256) * ((N + 255) // 256)
    print(f"M={M} N={N} K={K}: {'2-CTA' if tiles2 * 3 >= torch.cuda.get_device_properties(0).multi_processor_count else '1-CTA'}")
    dy = rnd(K, M, seed=1, device="cuda")
    x = rnd(K, N, seed=2, std=0.5, device="cuda")
    c0 = rnd(M, N, seed=3, device="cuda") * 0.5 * K ** 0.5
    c = c0.clone()
    nat.gemm(dy, x, out=c, flags=nat.A_MN_MAJOR | nat.B_MN_MAJOR | nat.EPI_ACCUM, M=M, K=K, N=N)
    rows = _sample_rows(M, 256, 512, seed=M + K).cuda()
    prod = (dy[:, rows].double().t() @ x.double()).bfloat16()
    assert O.rel_l2(c[rows], (c0[rows].double() + prod.double()).bfloat16()) <= TOL
    fresh = nat.gemm(dy, x, flags=nat.A_MN_MAJOR | nat.B_MN_MAJOR, M=M, K=K, N=N)
    assert O.rel_l2(fresh[rows], prod) <= TOL


# dgrads: [tokens, K] · W given as [K, N] (B MN-major), bf16 out.  d_act, dh2, d_attn, dh1 of 7B; dhn of one lm_head chunk
DGRAD_SHAPES = [(4096, 18944, 3584), (4096, 3584, 37888), (4096, 3584, 3584), (4096, 3584, 4608), (2048, 3584, 152064),
                (1, 3584, 4608), (127, 3584, 4608), (129, 3584, 4608), (1, 896, 1152), (127, 896, 1152), (129, 896, 1152)]


@pytest.mark.parametrize("M,N,K", DGRAD_SHAPES)
def test_gemm_data_grad_trainer_flags(nat, M, N, K):
    a = rnd(M, K, seed=4, device="cuda")
    w = rnd(K, N, seed=5, std=K ** -0.5, device="cuda")
    got = nat.gemm(a, w, flags=nat.B_MN_MAJOR, N=N)
    assert got.dtype == torch.bfloat16 and tuple(got.shape) == (M, N)
    rows = _sample_rows(M, 128, 512, seed=M + K).cuda()
    want = (a[rows].double() @ w.double()).bfloat16()
    assert O.rel_l2(got[rows], want) <= TOL


# ---------------------------------------------------------------------------------------------- q/k-norm backward
@pytest.mark.parametrize("n,n_h,n_kv,d", [(192, 4, 2, 128), (192, 4, 2, 64), (4096, 32, 8, 128), (4096, 14, 2, 64)])
def test_qk_norm_bwd(nat, n, n_h, n_kv, d):
    """Qwen3's q/k RMSNorm over the head dim: dqkv's q and k slices are replaced by the gradient w.r.t. the pre-norm
    vectors, the gain gradients add into non-zero fp32 accumulators, the v slice comes back bit for bit."""
    heads, eps = n_h + 2 * n_kv, 1e-6
    qkv = rnd(n, heads * d, seed=1, std=2.0)
    dqkv0 = rnd(n, heads * d, seed=2)
    qn, kn = (1 + 0.1 * rnd(d, seed=3, dtype=torch.float32)).bfloat16(), (1 + 0.1 * rnd(d, seed=4, dtype=torch.float32)).bfloat16()
    x = qkv.view(n, heads, d)[:, :n_h + n_kv].float().requires_grad_()
    wq, wk = qn.float().requires_grad_(), kn.float().requires_grad_()
    y = torch.cat([O.rmsnorm(x[:, :n_h], wq, eps), O.rmsnorm(x[:, n_h:], wk, eps)], dim=1)
    y.backward(dqkv0.view(n, heads, d)[:, :n_h + n_kv].float())
    acc_q0, acc_k0 = rnd(d, seed=5, dtype=torch.float32), rnd(d, seed=6, dtype=torch.float32)
    acc_q, acc_k = acc_q0.cuda(), acc_k0.cuda()
    dqkv = dqkv0.cuda()
    nat.qk_norm_bwd(qkv.cuda(), dqkv, qn.cuda(), kn.cuda(), acc_q, acc_k, eps, n_h, n_kv, d)
    got = dqkv.cpu().view(n, heads, d)
    assert O.rel_l2(got[:, :n_h + n_kv], x.grad) <= TOL_BWD
    assert torch.equal(got[:, n_h + n_kv:], dqkv0.view(n, heads, d)[:, n_h + n_kv:])
    assert O.rel_l2(acc_q.cpu() - acc_q0, wq.grad) <= TOL_BWD
    assert O.rel_l2(acc_k.cpu() - acc_k0, wk.grad) <= TOL_BWD


# ---------------------------------------------------------------------------------------------- cross-entropy
@pytest.mark.parametrize("M,V,std", [(2048, 152064, 2.0), (2048, 151936, 2.0), (256, 151936, 20.0)])
def test_cross_entropy_in_place_chunks(nat, M, V, std):
    """As the trainer's lm_head chunk loop runs it: dlogits written over the logits, two chunks adding into one
    loss_sum / n_valid, labels at 0 and V - 1 and ignored rows, a grad_scale that is not 1/n."""
    logits = rnd(M, V, seed=11, std=std, device="cuda")
    g = torch.Generator().manual_seed(12)
    labels = torch.randint(0, V, (M,), generator=g)
    labels[0], labels[1], labels[2], labels[M // 2 + 1], labels[-1] = 0, V - 1, -100, V - 1, 0
    labels = labels.cuda()
    scale = 0.37
    lf = logits.double().requires_grad_()
    loss = F.cross_entropy(lf, labels, ignore_index=-100, reduction="sum")
    (loss * scale).backward()
    n_valid = int((labels != -100).sum())
    ls = torch.zeros(1, dtype=torch.float32, device="cuda")
    nv = torch.zeros(1, dtype=torch.int32, device="cuda")
    buf = logits.clone()
    for a, e in ((0, M // 2), (M // 2, M)):
        nat.ce_fwd_bwd(buf[a:e], labels[a:e], ls, nv, buf[a:e], scale)
    assert int(nv) == n_valid
    assert abs(float(ls) - float(loss)) <= 1e-4 * abs(float(loss))
    assert O.rel_l2(buf, lf.grad) <= TOL_BWD
    assert int(torch.count_nonzero(buf[2])) == 0
    for r in (0, 1, M // 2 + 1, M - 1):         # the one-hot sits in the row's first or last 8-wide vector
        lab = int(labels[r])
        assert abs(float(buf[r, lab]) - float(lf.grad[r, lab])) <= 1e-2 * abs(float(lf.grad[r, lab]))


def test_cross_entropy_all_ignored_chunk(nat):
    M, V = 64, 151936
    logits = rnd(M, V, seed=13, device="cuda")
    labels = torch.full((M,), -100, dtype=torch.int64, device="cuda")
    ls = torch.full((1,), 3.5, dtype=torch.float32, device="cuda")
    nv = torch.full((1,), 7, dtype=torch.int32, device="cuda")
    nat.ce_fwd_bwd(logits, labels, ls, nv, logits, 0.37)
    assert float(ls) == 3.5 and int(nv) == 7
    assert int(torch.count_nonzero(logits)) == 0


# ---------------------------------------------------------------------------------------------- bias column sums
@pytest.mark.parametrize("M", [1, 255, 257, 4096])
@pytest.mark.parametrize("N", [4608, 1152, 66])
def test_colsum(nat, M, N):
    """db (fp32, non-zero) += column sums of dqkv, contiguous and as a strided view (row pitch > N)."""
    for ld in (N, N + 136):
        full = rnd(M, ld, seed=M + ld, device="cuda")
        dy = full[:, :N]
        db0 = rnd(N, seed=N, dtype=torch.float32, device="cuda")
        db = db0.clone()
        nat.colsum(dy, db)
        assert O.rel_l2(db - db0, dy.double().sum(0)) <= 1e-5, ld


# ---------------------------------------------------------------------------------------------- small helpers
@pytest.mark.parametrize("n", [5003, 1 << 20, 10_000_003])
def test_f32_to_bf16_accum(nat, n):
    src = rnd(n, seed=1, dtype=torch.float32, device="cuda")
    dst0 = rnd(n, seed=2, device="cuda")
    for accumulate in (False, True):
        dst = dst0.clone()
        nat.f32_to_bf16_accum(src, dst, accumulate)
        want = (src + dst0.float()).bfloat16() if accumulate else src.bfloat16()
        assert torch.equal(dst, want), accumulate


@pytest.mark.parametrize("dtype,n", [(torch.bfloat16, 4096), (torch.bfloat16, 10_000_008), (torch.float32, 5003),
                                     (torch.float32, 10_000_003)])
def test_scale_add(nat, dtype, n):
    """a = (accumulate ? a : 0) + scale * b with one rounding, and the aliased call commit_head makes
    (``a is b``, accumulate=False: a *= scale)."""
    scale = 0.37
    s64 = float(torch.tensor(scale, dtype=torch.float32))
    a0, b = rnd(n, seed=3, dtype=dtype, device="cuda"), rnd(n, seed=4, dtype=dtype, device="cuda")
    for accumulate in (False, True):
        a = a0.clone()
        nat.scale_add(a, b, scale, accumulate=accumulate)
        want = (a0.double() if accumulate else 0) + s64 * b.double()
        assert torch.equal(a, want.float().to(dtype)), accumulate
    a = a0.clone()
    nat.scale_add(a, a, scale, accumulate=False)
    assert torch.equal(a, (s64 * a0.double()).float().to(dtype))


# ---------------------------------------------------------------------------------------------- AdamW
@pytest.mark.parametrize("n", [5003, (1 << 24) + 5])
@pytest.mark.parametrize("decoupled", [False, True], ids=["adam_l2", "adamw"])
def test_adamw_trajectory_matches_torch(nat, n, decoupled):
    """50 steps with changing gradients, betas / eps off their defaults, weight decay.  Each step torch.optim starts
    from the kernel's own bf16 parameter, so the trajectories cannot drift apart: the moments agree in fp32 and the
    new parameter is bf16(p_old + torch's update) except at rounding boundaries (<= 1 % of elements, by one ulp).
    The default (streaming) load/store mode only: TL_ADAM_STREAM is read once per process."""
    lr, betas, eps, wd = 2e-3, (0.8, 0.95), 1e-6, 0.1
    p = rnd(n, seed=21, device="cuda")
    m = torch.zeros(n, dtype=torch.float32, device="cuda")
    v = torch.zeros_like(m)
    ref = p.float().clone().requires_grad_()
    opt = (torch.optim.AdamW if decoupled else torch.optim.Adam)([ref], lr=lr, betas=betas, eps=eps, weight_decay=wd,
                                                                 foreach=False)
    for t in range(1, 51):
        g = rnd(n, seed=100 + t, std=0.1 * (1 + t % 7), device="cuda")
        p_old = p.clone()
        with torch.no_grad():
            ref.copy_(p_old.float())
        ref.grad = g.float()
        opt.step()
        nat.adamw_step(p, g, m, v, lr, betas[0], betas[1], eps, wd, t, decoupled)
        st = opt.state[ref]
        assert _rel(m, st["exp_avg"]) <= 1e-6, t
        assert _rel(v, st["exp_avg_sq"]) <= 1e-6, t
        want = ref.detach().bfloat16()
        diff = p != want
        assert float(diff.float().mean()) <= 0.01, t
        # one bf16 ulp at the operands' scale: where p_old and the update nearly cancel, fp32 op-order differences
        # are relative to |p_old|, not to the tiny result
        scale = torch.maximum(p_old.float().abs(), want.float().abs())
        ulp = torch.ldexp(torch.ones_like(scale), torch.frexp(scale).exponent - 8)
        assert bool(((p.float() - want.float()).abs() <= ulp).all()), t
        assert float((p.float() - p_old.float()).abs().mean()) > 0, t
