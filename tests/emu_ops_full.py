"""torch (CPU) emulations of the full-attention operators of `geoformer_b200.ops` (`full_attention`,
`full_attention_window`), with the kernels' argument contracts, on top of tests/emu_ops.py.

TEST INFRASTRUCTURE ONLY.  `install(monkeypatch)` installs every emulation of tests/emu_ops.py and these two; calls are
counted in emu_ops.CALLS like the others."""
from __future__ import annotations

import math

import torch

from tests import emu_ops
from tests.emu_ops import CALLS, _count  # noqa: F401  (re-exported: tests read the counters from here)


def full_attention(q, ldq, k, ldk, v, ldv, n, l, s, heads, dim):
    """gf_full_attention / gf_dense_kv_h16 + gf_full_attention_tc: softmax(Q K^T / sqrt(dim)) V of each query row
    against all s key rows of its sample (plain projections, no feature map); fp32 message."""
    _count("full_attention")
    return _full(q, ldq, k, ldk, v, ldv, n, l, s, heads, dim)


def full_attention_window(q, ldq, k, ldk, v, ldv, n_windows, tokens, heads, dim):
    """gf_full_attention_window(_f16): window m's query rows against window m's key / value rows; fp32 message."""
    _count("full_attention_window")
    return _full(q, ldq, k, ldk, v, ldv, n_windows, tokens, tokens, heads, dim)


def _full(q, ldq, k, ldk, v, ldv, n, l, s, heads, dim):
    assert q.stride(0) == ldq and k.stride(0) == ldk and v.stride(0) == ldv and q.dtype == k.dtype == v.dtype
    c = heads * dim
    Q = q[:, :c].float().reshape(n, l, heads, dim)
    K = k[:, :c].float().reshape(n, s, heads, dim)
    V = v[:, :c].float().reshape(n, s, heads, dim)
    p = torch.softmax(torch.einsum("nlhd,nshd->nlsh", Q, K) / math.sqrt(dim), dim=2)
    return torch.einsum("nlsh,nshd->nlhd", p, V).reshape(n * l, c).contiguous()


def install(monkeypatch):
    from geoformer_b200 import ops
    emu_ops.install(monkeypatch)
    for name in ("full_attention", "full_attention_window"):
        assert hasattr(ops, name), name
        monkeypatch.setattr(ops, name, globals()[name])
