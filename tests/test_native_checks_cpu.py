"""Shape checks of the training wrappers in native.py that guard raw-pointer kernels: a mismatch raises before any
launch (no device needed), instead of the kernel reading or writing past a buffer."""
import pytest
import torch

from tensorlink_b200 import native

bf = torch.bfloat16


def _attn_args(B=2, S=16, n_h=4, n_kv=2, d=64, T_max=16, dk_T=None, v_T=None):
    z = lambda *s: torch.zeros(*s, dtype=bf)
    kc, vc = z(B, n_kv, T_max, d), z(B, n_kv, T_max if v_T is None else v_T, d)
    dk = z(B, n_h, T_max if dk_T is None else dk_T, d)
    return (z(B, S, n_h, d), kc, vc, z(B, S, n_h * d), z(B, S, n_h * d), torch.zeros(B, n_h, S), z(B, S, n_h, d), dk,
            z(*dk.shape), torch.zeros(16, dtype=torch.uint8), B, S, n_h, n_kv, d, d ** -0.5)


@pytest.mark.parametrize("kw", [dict(dk_T=12), dict(dk_T=20), dict(v_T=12), dict(T_max=8)])
def test_attn_bwd_rejects_mismatched_shapes(kw):
    with pytest.raises(AssertionError) as e:
        native.attn_bwd(*_attn_args(**kw))
    assert "device tensor" not in str(e.value)


def _rope_args(B=2, S=16, n_h=4, n_kv=2, d=64, dk_T=16, dv_T=None, n_tok=None, tab=32):
    z = lambda *s: torch.zeros(*s, dtype=bf)
    n = B * S if n_tok is None else n_tok
    return (z(n, n_h * d), z(B, n_h, dk_T, d), z(B, n_h, dk_T if dv_T is None else dv_T, d), z(n, (n_h + 2 * n_kv) * d),
            z(tab, d // 2), z(tab, d // 2), S, n_h, n_kv, d)


@pytest.mark.parametrize("kw", [dict(dk_T=12), dict(dv_T=20), dict(n_tok=24), dict(tab=8)])
def test_rope_kv_bwd_rejects_mismatched_shapes(kw):
    with pytest.raises(AssertionError) as e:
        native.rope_kv_bwd(*_rope_args(**kw))
    assert "device tensor" not in str(e.value)


@pytest.mark.parametrize("ids_n,dout_shape", [(5, (4, 64)), (4, (4, 32)), (4, (3, 64)), (4, (4, 128))])
def test_embed_bwd_rejects_mismatched_shapes(ids_n, dout_shape):
    with pytest.raises(AssertionError) as e:
        native.embed_bwd(torch.zeros(ids_n, dtype=torch.int64), torch.zeros(*dout_shape, dtype=bf), torch.zeros(16, 64, dtype=bf))
    assert "device tensor" not in str(e.value)
