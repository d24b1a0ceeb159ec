"""CPU pins of the float64 stage reference (tests/stage_ref.py) that the GPU stage tests compare
the kernels with: with every rounding point switched off it must be the plain Llama forward of
`oracle.llama_oracle` and reproduce the reference project's numbers (tests/golden/layer_arith.json)
to fp32 precision."""
import pytest
import torch

from oracle import llama_oracle as orc
from tests import golden_util as gu
from tests import stage_ref as sr

LLAMA3 = {"rope_type": "llama3", "factor": 32.0, "low_freq_factor": 1.0, "high_freq_factor": 4.0,
          "original_max_position_embeddings": 8192}
LINEAR = {"rope_type": "linear", "factor": 4.0}


def _cfg(dims):
    return dict(head_dim=dims.head_dim, heads=dims.heads, kv_heads=dims.kv_heads,
                rope_theta=dims.rope_theta, rope_scaling=dims.rope_scaling, rms_eps=dims.rms_eps)


def _forward(w64, ids, rnd):
    """All layers on `ids` from an empty cache -> (logits, k and v of layer 0)."""
    d = w64.dims
    x = w64.embed[torch.tensor(ids)]
    pos = torch.arange(len(ids))
    empty = torch.zeros(0, d.kv_heads, d.head_dim, dtype=torch.float64)
    k0 = v0 = None
    for L in w64.layers:
        x, k, v, _ = sr.decoder_layer(x, L, pos, empty, empty, _cfg(d), rnd)
        if k0 is None:
            k0, v0 = k, v
    return sr.lm_head(x, w64.final_norm, w64.lm_head, d.rms_eps, rnd), k0, v0


@pytest.mark.parametrize("case", gu.load("layer_arith.json")["cases"], ids=lambda c: c["model"])
def test_unrounded_reference_is_the_oracle_and_the_reference_numbers(case):
    dims, sd = gu.state_dict_for(case, alpha_key=False)
    w32 = orc.weights_from_state_dict(dims, sd)
    w64 = orc.weights_from_state_dict(dims, sd, dtype=torch.float64)
    prompt = case["prompt"]
    logits, k0, v0 = _forward(w64, prompt, rnd=False)
    kv = orc.KVStore(dims.layers)
    want = orc.step_all_layers(w32, prompt, kv).double()
    fp32 = dict(rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(logits, want, **fp32)
    torch.testing.assert_close(k0.transpose(0, 1), kv.k[0].double(), **fp32)
    torch.testing.assert_close(v0.transpose(0, 1), kv.v[0].double(), **fp32)
    # the reference project's own forward (same tolerance as tests/test_oracle_golden.py)
    gold = dict(rtol=2e-4, atol=2e-5)
    torch.testing.assert_close(logits[-1], torch.tensor(case["full_logits_last"], dtype=torch.float64), **gold)
    torch.testing.assert_close(logits[3], torch.tensor(case["full_logits_row3"], dtype=torch.float64), **gold)
    torch.testing.assert_close(k0[-1, 0], torch.tensor(case["k_cache_l0_h0_last"], dtype=torch.float64), **gold)
    torch.testing.assert_close(v0[-1, 0], torch.tensor(case["v_cache_l0_h0_last"], dtype=torch.float64), **gold)
    # with the kernels' rounding points the logits move by bf16-sized amounts, not more
    rounded, _, _ = _forward(w64, prompt, rnd=True)
    assert float((rounded - logits).abs().max()) < 0.02 * float(logits.abs().max())


@pytest.mark.parametrize("scaling", [None, LINEAR, LLAMA3], ids=["default", "linear", "llama3"])
@pytest.mark.parametrize("head_dim,theta", [(128, 10000.0), (64, 500000.0), (32, 10000.0)])
def test_rope_table_is_the_oracle_table(scaling, head_dim, theta):
    dims = orc.LlamaDims(vocab=8, hidden=head_dim, inter=8, layers=1, heads=1, kv_heads=1,
                         head_dim=head_dim, rope_theta=theta, rope_scaling=scaling)
    pos = torch.cat([torch.arange(0, 130), torch.tensor([4095, 4096, 8191, 8192, 16383])])
    cos, sin = sr.rope_cos_sin(pos, head_dim, theta, scaling)
    want_cos, want_sin = orc.rope_tables(dims, pos, torch.float32)
    half = head_dim // 2
    torch.testing.assert_close(cos, want_cos[:, :half].double(), rtol=0, atol=2e-6)
    torch.testing.assert_close(sin, want_sin[:, :half].double(), rtol=0, atol=2e-6)
    if scaling is LLAMA3:       # the three llama3 bands all occur at these widths
        inv = sr.rope_inv_freq(head_dim, theta)
        assert not torch.equal(sr.rope_inv_freq(head_dim, theta, scaling), inv)


def test_rotation_matches_the_oracle_rotate_half():
    g = torch.Generator().manual_seed(0)
    x = torch.randn(5, 3, 64, generator=g, dtype=torch.float64)      # [s, heads, hd]
    pos = torch.arange(100, 105)
    cos, sin = sr.rope_cos_sin(pos, 64, 10000.0)
    dims = orc.LlamaDims(vocab=8, hidden=64, inter=8, layers=1, heads=3, kv_heads=3, head_dim=64)
    c, s = orc.rope_tables(dims, pos, torch.float64)
    want = orc.apply_rope(x.transpose(0, 1), c, s).transpose(0, 1)
    torch.testing.assert_close(sr.rotate(x, cos, sin), want, rtol=1e-6, atol=1e-6)


def test_argmax_lowest_index_wins_ties():
    logits = torch.tensor([[1.0, 3.0, 3.0, 2.0], [-5.0, -5.0, -7.0, -5.0], [0.0, 0.0, 0.0, 0.0]],
                          dtype=torch.float64)
    assert sr.argmax_lowest(logits).tolist() == [1, 0, 0]


def test_ulp_error_counts_bf16_steps():
    ref = torch.tensor([1.0, 1.0, -3.0, 1e-6], dtype=torch.float64)
    one_up = torch.tensor([1.0 + 2 ** -7, 1.0, -3.0 - 2 ** -6, 0.0], dtype=torch.float64)
    err = sr.ulp_error(one_up, ref, floor=2.0 ** -20)
    assert err.tolist()[:3] == [1.0, 0.0, 1.0]
    assert float(err[3]) == pytest.approx(1e-6 / 2 ** -20)
    rows = torch.tensor([[3.0, 4.0], [0.0, 1e-3]], dtype=torch.float64)
    assert sr.row_floor(rows).flatten().tolist() == [2.0 ** -6, 2.0 ** -18]
