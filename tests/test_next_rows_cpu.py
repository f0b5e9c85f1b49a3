"""CPU tests (-m "not gpu") of the §8f next rows either side of the hot paths: rotary embedding of the attention
prologue and the vision token framing. The oracles are checked against fixtures produced by EXECUTING the reference's
own functions (tools/make_golden_next_rows_from_reference.py), and the numerical design of the CUDA kernel (angles
rebuilt from 64 inverse frequencies, cos/sin rounded once from double) is checked against the reference's table."""
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TAGS = ("t1e4", "t5e7")


@pytest.mark.parametrize("tag", TAGS)
def test_rope_oracle_is_bit_exact_vs_reference_fixture(tag):
    from oracle import rope as R
    g = np.load(os.path.join(GOLD, "rope_reference.npz"))
    oq, ok = R.rope_reference(g[tag + "_xq"], g[tag + "_xk"], g[tag + "_pos"], float(g[tag + "_theta"]),
                              int(g[tag + "_max_pos"]))
    assert np.array_equal(oq, g[tag + "_oq"]) and np.array_equal(ok, g[tag + "_ok"])


@pytest.mark.parametrize("tag", TAGS)
def test_rope_kernel_angle_scheme_matches_reference_table(tag):
    """float32(float64(pos)*float64(inv_freq)) then correctly rounded cos/sin: <= 1 ulp from the reference table,
    including positions near 2^20 with theta 5e7 (angles up to ~1e6 rad)."""
    from lwm_b200.rope import precompute_inv_freq
    g = np.load(os.path.join(GOLD, "rope_reference.npz"))
    inv = precompute_inv_freq(128, float(g[tag + "_theta"]))
    ang = (g[tag + "_pos"].astype(np.float64)[..., None] * inv.astype(np.float64)).astype(np.float32)
    c = np.cos(ang.astype(np.float64)).astype(np.float32)
    s = np.sin(ang.astype(np.float64)).astype(np.float32)

    def ulps(a, b):
        return np.max(np.abs(a.view(np.int32).astype(np.int64) - b.view(np.int32).astype(np.int64)))
    big = np.abs(g[tag + "_cos"]) > 1e-3          # ulp distance is only meaningful away from the zero crossings
    assert ulps(c[big], g[tag + "_cos"][big]) <= 1
    big = np.abs(g[tag + "_sin"]) > 1e-3
    assert ulps(s[big], g[tag + "_sin"][big]) <= 1
    assert np.abs(c - g[tag + "_cos"]).max() <= 6e-8 and np.abs(s - g[tag + "_sin"]).max() <= 6e-8


def test_rope_is_a_rotation():
    """size-independent property: norms of every (even, odd) pair are preserved; conj undoes the rotation"""
    from oracle import rope as R
    rng = np.random.default_rng(0)
    x = rng.standard_normal((1, 64, 2, 128)).astype(np.float32)
    pos = rng.integers(0, 1 << 20, (1, 64))
    table = R.precompute_freqs_cis(128, 1 << 20, 5e7)
    y, _ = R.apply_rotary_emb(x, x, np.take(table, pos, axis=0))
    n0 = np.hypot(x[..., 0::2], x[..., 1::2])
    n1 = np.hypot(y[..., 0::2], y[..., 1::2])
    assert np.allclose(n0, n1, rtol=1e-5, atol=1e-6)
    back, _ = R.apply_rotary_emb(y, y, np.conj(np.take(table, pos, axis=0)))
    assert np.allclose(back, x, atol=2e-6)


@pytest.mark.parametrize("tag", ("f1", "f5", "f9sel4"))
def test_vision_token_oracle_matches_reference_processor(tag):
    from oracle import vision_tokens as V
    g = np.load(os.path.join(GOLD, "vision_tokens_reference.npz"))
    tokens, mask = V.vision_field(g[tag + "_codes"].tolist(), [32000], [32001, 32002],
                                  max_n_frames=int(g[tag + "_max_n_frames"]))
    # the fixture wraps the field in bos ... eos (data.py:167-170, 236-239)
    assert [1] + tokens + [2] == g[tag + "_tokens"].tolist()
    assert [False] + mask + [False] == g[tag + "_vision_mask"].tolist()


def test_vision_token_roundtrip_and_host_selection():
    from oracle import vision_tokens as V
    from lwm_b200.vision_tokens import select_frames, vision_mask
    rng = np.random.default_rng(2)
    codes = rng.integers(0, 8192, 7 * 256)
    toks = V.frame_tokens(codes)
    assert len(toks) == 7 * 257 and toks[256] == 8192 and toks[-1] == 8193
    assert np.array_equal(V.unframe_tokens(toks).reshape(-1), codes)
    assert select_frames(7, -1) is None and select_frames(7, 7) is None
    assert select_frames(9, 4).tolist() == np.linspace(0, 8, 4).astype(int).tolist()
    assert vision_mask(3, 1, 2) == V.vision_field(codes[:768], [0], [0, 0])[1]
    # shape handling of the un-framing host code (pure views, no kernel)
    import torch
    from lwm_b200 import _lib
    from lwm_b200.vision_tokens import _as_frames
    assert _as_frames(torch.zeros(257), 256).shape == (1, 257)            # a single framed image, flat
    assert _as_frames(torch.zeros(5 * 257), 256).shape == (5, 257)
    assert _as_frames(torch.zeros(2, 257), 256).shape == (2, 257)         # vision_generation.py:159-160
    assert _as_frames(torch.zeros(2, 3 * 257), 256).shape == (2, 3, 257)  # vision_generation.py:219-221
    with pytest.raises(_lib.LwmError):
        _as_frames(torch.zeros(300), 256)


def test_call_site_mask_helpers():
    """host mirrors of lwm/llama.py:526-537 (mask -> additive finfo.min bias) and :574-591 (decode mask)"""
    import torch
    from lwm_b200.ringattention import attention_bias_from_mask, decode_attention_mask
    m = torch.tensor([[0, 0, 1, 1, 1], [1, 1, 1, 1, 0]])
    for dt in (torch.bfloat16, torch.float32):
        b = attention_bias_from_mask(m, dt)
        assert b.shape == (2, 1, 1, 5) and b.dtype == dt
        assert b[0, 0, 0].tolist() == [torch.finfo(dt).min] * 2 + [0.0] * 3
        assert b[1, 0, 0, -1].item() == torch.finfo(dt).min
    # numpy restatement of llama.py:574-577, 586-587
    Q, shift, K = 3, 4, 9
    pad = np.ones((2, K), dtype=np.int64)
    pad[0, :2] = 0
    causal = np.arange(K)[None] <= (np.arange(Q) + shift)[:, None]
    want = np.logical_and(np.broadcast_to(pad[:, None, None, :] > 0, (2, 1, Q, K)), causal[None, None])
    got = decode_attention_mask(torch.from_numpy(pad), Q, shift)
    assert got.dtype == torch.bool and np.array_equal(got.numpy(), want)


def test_import_surface_of_the_ringattention_package_and_blockwise_ffn():
    """lwm/llama.py:30 imports four names from `ringattention`; blockwise_feedforward == the un-chunked cell"""
    import torch
    from ringattention import blockwise_feedforward, ringattention, ringattention_inference, ringattention_jax
    assert ringattention_jax is ringattention and callable(ringattention_inference)
    torch.manual_seed(0)
    w1, w2, w3 = [torch.randn(16, 64, requires_grad=True), torch.randn(64, 16, requires_grad=True),
                  torch.randn(16, 64, requires_grad=True)]

    def cell(x):                                     # the LLaMA MLP shape (llama.py:623-661): w2(silu(w1 x) * w3 x)
        return (torch.nn.functional.silu(x @ w1) * (x @ w3)) @ w2
    x = torch.randn(2, 32, 16, requires_grad=True)
    ref = cell(x)
    g = torch.randn_like(ref)
    ref_grads = torch.autograd.grad(ref, (x, w1, w2, w3), g)
    for pre_remat in (True, False):
        out = blockwise_feedforward(cell, x, 8, pre_remat=pre_remat)
        assert torch.allclose(out, ref, atol=1e-6)
        grads = torch.autograd.grad(out, (x, w1, w2, w3), g)
        for a, b in zip(grads, ref_grads):
            assert torch.allclose(a, b, atol=1e-4, rtol=1e-5)
    with pytest.raises(ValueError):
        blockwise_feedforward(cell, x, 5)
