"""GPU: the tcgen05 / TMEM LM head (csrc/lmhead_tc.cuh, LSK_LMHEAD_TC=1).  Executed for the first
time in round 2: correct, but slower than the mma.sync head at decode widths (3.6 vs 5.7 TB/s at
7 rows — profiles/r2_unrun_experimental_1gpu.log), so it stays opt-in; these tests keep it honest."""
import pytest
import torch

from tests import golden_util as gu

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("n,k,m", [(256, 256, 1), (1000, 512, 7), (32000, 4096, 7), (32000, 4096, 16),
                                   (16032, 5120, 1)])
def test_tcgen05_lm_head_matches_a_torch_reference(n, k, m):
    """lmhead_tc.cuh stand-alone: fp32 logits of rmsnorm(x) . W^T within bf16-operand tolerance of
    a torch fp32 reference that rounds the normalised activations to bf16 like the kernel does
    (fp32 accumulate: |err| <= ~1e-3 * sqrt(k) * |w| |x| worst case; we allow 2e-2 absolute on
    unit-variance inputs), and the fused arg-max must be the arg-max of the kernel's own logits."""
    import ctypes as C
    from layerskip_b200 import _lib
    lib = _lib.load()
    g = torch.Generator(device="cuda").manual_seed(n + k + m)
    w = (torch.randn(n, k, generator=g, device="cuda") * 0.05).to(torch.bfloat16)
    x = torch.randn(m, k, generator=g, device="cuda")
    nw = (1.0 + 0.1 * torch.randn(k, generator=g, device="cuda")).to(torch.bfloat16)
    logits = torch.full((m, n), float("nan"), device="cuda")
    bv = torch.zeros(16, device="cuda")
    bi = torch.zeros(16, dtype=torch.int32, device="cuda")
    ms = C.c_float(0)
    torch.cuda.synchronize()
    _lib.check(lib.lsk_test_lmhead_tc(w.data_ptr(), n, k, x.data_ptr(), nw.data_ptr(), 1e-5, m,
                                      logits.data_ptr(), bv.data_ptr(), bi.data_ptr(), 20, C.byref(ms)))
    torch.cuda.synchronize()
    rstd = torch.rsqrt((x * x).mean(-1, keepdim=True) + 1e-5)
    xn = (nw.float() * (x * rstd)).to(torch.bfloat16).float()
    ref = xn @ w.float().T
    assert torch.isfinite(logits).all()
    assert float((logits - ref).abs().max()) < 2e-2
    assert torch.equal(bi[:m].long(), logits.argmax(-1))        # ties: lowest index, like torch
    assert torch.equal(bv[:m], logits.max(-1).values)
    print(f"tcgen05 lm head n={n} k={k} m={m}: {ms.value * 1e3:.1f} us, "
          f"{n * k * 2 / (ms.value * 1e-3) / 1e9:.0f} GB/s")


@pytest.mark.parametrize("name", ["gqa128_a0.1", "mha128_a0.1"])
def test_engine_with_tcgen05_lm_head_stays_exact_and_within_the_margin_gate(name, monkeypatch):
    """LSK_LMHEAD_TC=1: every LM head (draft, verify, autoregressive) goes through the tcgen05
    kernel, so speculative == autoregressive must still hold exactly; against the oracle the usual
    margin gate applies (accumulation order differs from the mma.sync head)."""
    from layerskip_b200 import GenerationConfig
    from layerskip_b200.strategy import (B200AutoRegressiveGenerationStrategy,
                                         B200SelfSpeculativeGenerationStrategy)
    from oracle import llama_oracle as orc
    from tests import parity_util as pu
    from tests.test_gpu_engine import _Model
    monkeypatch.setenv("LSK_LMHEAD_TC", "1")
    case = next(c for c in gu.spec_cases() if c["name"] == name)
    dims, sd = gu.state_dict_for(case)
    model, w = _Model(dims, sd), orc.weights_from_state_dict(dims, sd)
    spec = B200SelfSpeculativeGenerationStrategy(max_ctx=512)
    ar = B200AutoRegressiveGenerationStrategy(engine_cache=spec.engines)
    try:
        def generate(prompt, n):
            cfg = GenerationConfig(**{**case["cfg"], "max_steps": n})
            return spec.generate_token_ids(model, prompt, case["eos"], cfg).predicted_tokens
        flips, gaps = pu.check_stream(w, case["prompt"], case["reference"]["spec_tokens"], generate)
        s = spec.generate_token_ids(model, case["prompt"], case["eos"], GenerationConfig(**case["cfg"]))
        a = ar.generate_token_ids(model, case["prompt"], case["eos"],
                                  GenerationConfig(**{**case["cfg"], "exit_layer": -1, "num_speculations": -1}))
    finally:
        spec.engines.close()
    assert s.predicted_tokens == a.predicted_tokens
    assert flips <= 4, gaps


@pytest.mark.parametrize("value", [0.5, -0.001], ids=["positive", "all_negative"])
@pytest.mark.parametrize("n,i,j", [(1005, 5, 1002), (1005, 130, 1001), (32001, 37 * 16 + 11, 31999)])
def test_tcgen05_lm_head_tie_goes_to_the_lowest_index_and_padding_rows_never_win(n, i, j, value):
    """Rows i < j (different 128-row tiles and rows inside them) each hold `value` in one column and
    zeros elsewhere; the normed activations are exactly 1, so both logits equal `value` bit for bit.
    Every other row is negative everywhere.  With n % 16 != 0 the last tile has padding rows, which
    would win with logit 0 when `value` < 0 if they leaked into the arg-max."""
    import ctypes as C
    from layerskip_b200 import _lib
    lib = _lib.load()
    k, m = 256, 7
    g = torch.Generator(device="cuda").manual_seed(n + i)
    w = -(torch.rand(n, k, generator=g, device="cuda") * 0.01 + 0.001)
    w[i] = 0
    w[j] = 0
    w[i, 3] = value
    w[j, k - 5] = value
    w = w.to(torch.bfloat16)
    x = torch.ones(m, k, device="cuda")
    nw = torch.ones(k, dtype=torch.bfloat16, device="cuda")
    logits = torch.full((m, n), float("nan"), device="cuda")
    bv = torch.zeros(16, device="cuda")
    bi = torch.zeros(16, dtype=torch.int32, device="cuda")
    ms = C.c_float(0)
    torch.cuda.synchronize()
    _lib.check(lib.lsk_test_lmhead_tc(w.data_ptr(), n, k, x.data_ptr(), nw.data_ptr(), 1e-5, m,
                                      logits.data_ptr(), bv.data_ptr(), bi.data_ptr(), 1, C.byref(ms)))
    torch.cuda.synchronize()
    assert torch.equal(logits[:, i], logits[:, j]) and torch.equal(logits[:, i], logits.max(-1).values)
    assert bi[:m].tolist() == [i] * m
    assert torch.equal(bv[:m], logits[:, i])
