"""TEST INFRASTRUCTURE ONLY — writes tests/golden/*.json from the UNMODIFIED reference.

Run in the build container (needs /root/reference):   python oracle/gen_golden.py

For every case a tiny random-init Llama (weights = oracle.random_state_dict(seed), so any
machine can rebuild them bit-for-bit from the seed; a checksum is stored to prove it) is
loaded into HuggingFace `LlamaForCausalLM`, and the reference's own
`SelfSpeculativeGenerationStrategy` / `AutoRegressiveGenerationStrategy`
(/root/reference/self_speculation/*.py, imported through oracle/ref_shim.py) produce:
  * the generated token list and acceptance rate,
  * a per-round trace (drafted, matched, tokens emitted) captured by wrapping — not editing —
    `single_step_speculation` (self_speculation_generator.py:102-229),
  * for the arithmetic fixture: exit-layer hidden rows and logits from `forward_early` /
    `forward` (llama_model_utils.py:155-276) on a fixed prompt.
"""
from __future__ import annotations

import json
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import llama_oracle as orc  # noqa: E402
from oracle import ref_shim  # noqa: E402

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")

MODELS = {
    # name: (vocab, hidden, inter, layers, heads, kv_heads, head_dim)
    "survey_mha32": (512, 256, 688, 4, 8, 8, 32),      # SURVEY.md Appendix C tiny config
    "tiny_mha128": (512, 256, 704, 4, 2, 2, 128),      # engine-compatible (head_dim 128)
    "tiny_gqa128": (640, 512, 1408, 6, 4, 2, 128),     # engine-compatible, grouped KV
}


def dims_of(name: str) -> orc.LlamaDims:
    v, h, i, l, nh, nkv, hd = MODELS[name]
    return orc.LlamaDims(vocab=v, hidden=h, inter=i, layers=l, heads=nh, kv_heads=nkv,
                         head_dim=hd, rms_eps=1e-5, rope_theta=10000.0)


def checksum(sd) -> str:
    acc = 0.0
    for k in sorted(sd):
        t = sd[k].to(torch.float64)
        acc += float((t.abs().sum() + (t * torch.arange(1, t.numel() + 1, dtype=torch.float64)
                                       .view(t.shape) % 7).sum()))
    return f"{acc:.6f}"


def build_hf(dims: orc.LlamaDims, sd):
    from transformers import LlamaConfig, LlamaForCausalLM
    cfg = LlamaConfig(vocab_size=dims.vocab, hidden_size=dims.hidden,
                      intermediate_size=dims.inter, num_hidden_layers=dims.layers,
                      num_attention_heads=dims.heads, num_key_value_heads=dims.kv_heads,
                      head_dim=dims.head_dim, max_position_embeddings=2048,
                      rms_norm_eps=dims.rms_eps, tie_word_embeddings=False)
    model = LlamaForCausalLM(cfg)
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not [m for m in missing if "rotary" not in m], missing
    assert not unexpected, unexpected
    return model.eval()


CASES = [
    # name, model, seed, damp_from, alpha, prompt, eos, cfg
    dict(name="survey_a0.1", model="survey_mha32", seed=0, damp_from=2, alpha=0.1,
         prompt=list(range(3, 19)), eos=[511],
         cfg=dict(max_steps=20, exit_layer=2, num_speculations=4, sample=False)),
    dict(name="mha128_a1.0", model="tiny_mha128", seed=1, damp_from=2, alpha=1.0,
         prompt=[5, 9, 200, 31, 7, 77, 123, 45, 300, 2, 19], eos=[511],
         cfg=dict(max_steps=24, exit_layer=2, num_speculations=4, sample=False)),
    dict(name="mha128_a0.3", model="tiny_mha128", seed=1, damp_from=2, alpha=0.3,
         prompt=[5, 9, 200, 31, 7, 77, 123, 45, 300, 2, 19], eos=[511],
         cfg=dict(max_steps=24, exit_layer=2, num_speculations=4, sample=False)),
    dict(name="mha128_a0.1", model="tiny_mha128", seed=1, damp_from=2, alpha=0.1,
         prompt=[5, 9, 200, 31, 7, 77, 123, 45, 300, 2, 19], eos=[511],
         cfg=dict(max_steps=40, exit_layer=2, num_speculations=6, sample=False)),
    dict(name="mha128_a0.03_e1", model="tiny_mha128", seed=2, damp_from=1, alpha=0.03,
         prompt=[17, 4, 4, 250], eos=[511],
         cfg=dict(max_steps=33, exit_layer=1, num_speculations=3, sample=False)),
    dict(name="mha128_a0_full", model="tiny_mha128", seed=3, damp_from=3, alpha=0.0,
         prompt=[400, 401, 402, 403, 404, 405, 406, 407], eos=[511],
         cfg=dict(max_steps=30, exit_layer=3, num_speculations=8, sample=False)),
    dict(name="gqa128_a0.1", model="tiny_gqa128", seed=4, damp_from=3, alpha=0.1,
         prompt=[11, 500, 23, 8, 639, 100, 100, 7, 345, 222, 3, 90, 91, 92, 93, 94, 95],
         eos=[639],
         cfg=dict(max_steps=48, exit_layer=3, num_speculations=6, sample=False)),
    dict(name="gqa128_a0.05_long", model="tiny_gqa128", seed=5, damp_from=2, alpha=0.05,
         prompt=list(range(20, 20 + 70)), eos=[639],
         cfg=dict(max_steps=64, exit_layer=2, num_speculations=5, sample=False)),
    dict(name="mha128_prompt1", model="tiny_mha128", seed=6, damp_from=2, alpha=0.1,
         prompt=[42], eos=[511],
         cfg=dict(max_steps=12, exit_layer=2, num_speculations=4, sample=False)),
    dict(name="mha128_steps2", model="tiny_mha128", seed=6, damp_from=2, alpha=0.1,
         prompt=[42, 43, 44], eos=[511],
         cfg=dict(max_steps=2, exit_layer=2, num_speculations=4, sample=False)),
    dict(name="mha128_steps3", model="tiny_mha128", seed=6, damp_from=2, alpha=0.1,
         prompt=[42, 43, 44], eos=[511],
         cfg=dict(max_steps=3, exit_layer=2, num_speculations=4, sample=False)),
    # EOS cases are completed below (the eos id is taken from the no-EOS run's own output)
    dict(name="mha128_eos_mid", model="tiny_mha128", seed=1, damp_from=2, alpha=0.1,
         prompt=[5, 9, 200, 31, 7, 77, 123, 45, 300, 2, 19], eos="from_output:9",
         cfg=dict(max_steps=40, exit_layer=2, num_speculations=6, sample=False)),
    dict(name="gqa128_eos_two", model="tiny_gqa128", seed=4, damp_from=3, alpha=0.1,
         prompt=[11, 500, 23, 8, 639, 100, 100, 7, 345, 222, 3, 90, 91, 92, 93, 94, 95],
         eos="from_output:20,5",
         cfg=dict(max_steps=48, exit_layer=3, num_speculations=6, sample=False)),
    # sampling: replayable only on the CPU RNG — pins the oracle's sampling path draw for draw
    dict(name="mha128_sample_s1", model="tiny_mha128", seed=1, damp_from=2, alpha=0.1,
         prompt=[5, 9, 200, 31, 7, 77, 123, 45, 300, 2, 19], eos=[511], torch_seed=1,
         cfg=dict(max_steps=32, exit_layer=2, num_speculations=4, sample=True,
                  temperature=0.6, top_k=0, top_p=0.9)),
    dict(name="mha128_sample_s2_topk", model="tiny_mha128", seed=1, damp_from=2, alpha=0.3,
         prompt=[5, 9, 200, 31, 7, 77, 123, 45, 300, 2, 19], eos=[511], torch_seed=2,
         cfg=dict(max_steps=32, exit_layer=2, num_speculations=5, sample=True,
                  temperature=0.9, top_k=12, top_p=0.95)),
    dict(name="gqa128_sample_s3", model="tiny_gqa128", seed=4, damp_from=3, alpha=0.1,
         prompt=[11, 500, 23, 8], eos=[639], torch_seed=3,
         cfg=dict(max_steps=40, exit_layer=3, num_speculations=6, sample=True,
                  temperature=0.6, top_k=0, top_p=0.9)),
]


def run_reference(ref, model, prompt, eos, cfg, torch_seed=None):
    GC = ref.generator_base.GenerationConfig
    Spec = ref.self_speculation_generator.SelfSpeculativeGenerationStrategy
    AR = ref.autoregressive_generator.AutoRegressiveGenerationStrategy
    rounds = []

    class Traced(Spec):
        def single_step_speculation(self, **kw):
            before = len(kw["output_ids"])
            res = super().single_step_speculation(**kw)
            _inp, out_ids, past, n_match, n_spec = res
            rounds.append(dict(d_req=int(kw["num_speculations"]), d_actual=int(n_spec),
                               n_matches=int(n_match), emitted=[int(t) for t in out_ids[before:]],
                               kv_len_after=int(past[0][0].shape[2])))
            return res

    gc = GC(generation_strategy="self_speculative", **cfg)
    with torch.inference_mode():
        if torch_seed is not None:
            torch.manual_seed(torch_seed)
        spec = Traced().generate_token_ids(model, list(prompt), list(eos), gc)
        ar_cfg = dict(cfg)
        ar_cfg["exit_layer"] = -1
        ar_cfg["num_speculations"] = -1
        if torch_seed is not None:
            torch.manual_seed(torch_seed)
        ar = AR().generate_token_ids(model, list(prompt), list(eos), GC(**ar_cfg))
        ee_cfg = dict(cfg)
        ee_cfg["num_speculations"] = -1
        if torch_seed is not None:
            torch.manual_seed(torch_seed)
        early = AR().generate_token_ids(model, list(prompt), list(eos), GC(**ee_cfg))
    return dict(spec_tokens=[int(t) for t in spec.predicted_tokens],
                acceptance_rate=float(spec.acceptance_rate),
                ar_tokens=[int(t) for t in ar.predicted_tokens],
                early_exit_tokens=[int(t) for t in early.predicted_tokens],
                rounds=rounds)


def main() -> None:
    ref = ref_shim.load_reference()
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    out_cases = []
    for case in CASES:
        dims = dims_of(case["model"])
        sd = orc.random_state_dict(dims, case["seed"], case["damp_from"], case["alpha"])
        model = build_hf(dims, sd)
        eos = case["eos"]
        if isinstance(eos, str):
            idxs = [int(x) for x in eos.split(":")[1].split(",")]
            probe = run_reference(ref, model, case["prompt"], [dims.vocab - 1], case["cfg"])
            eos = [probe["spec_tokens"][i] for i in idxs]
        res = run_reference(ref, model, case["prompt"], eos, case["cfg"],
                            case.get("torch_seed"))
        rec = dict(name=case["name"], model=case["model"], dims=list(MODELS[case["model"]]),
                   weight_seed=case["seed"], damp_from=case["damp_from"], alpha=case["alpha"],
                   weights_checksum=checksum(sd), prompt=case["prompt"], eos=eos,
                   torch_seed=case.get("torch_seed"), cfg=case["cfg"], reference=res)
        out_cases.append(rec)
        print(f"{case['name']:24s} n_out={len(res['spec_tokens']):3d} "
              f"acc={res['acceptance_rate']:.3f} rounds={len(res['rounds'])} "
              f"spec==ar:{res['spec_tokens'] == res['ar_tokens']}")
    with open(os.path.join(GOLDEN_DIR, "spec_traces.json"), "w") as f:
        json.dump(dict(generator="oracle/gen_golden.py", reference="facebookresearch/LayerSkip "
                       "self_speculation/* run unmodified under oracle/ref_shim.py",
                       torch=torch.__version__, cases=out_cases), f, indent=1)

    # ---- arithmetic fixture: the reference's forward / forward_early on a fixed prompt
    arith = []
    lmu = ref.llama_model_utils
    for mname, seed, exit_layer in (("tiny_mha128", 1, 2), ("tiny_gqa128", 4, 3),
                                    ("survey_mha32", 0, 2)):
        dims = dims_of(mname)
        sd = orc.random_state_dict(dims, seed, None, 1.0)
        model = build_hf(dims, sd)
        g = torch.Generator().manual_seed(99)
        prompt = torch.randint(3, dims.vocab - 1, (1, 13), generator=g)
        with torch.inference_mode():
            full = lmu.forward(model, prompt, None)
            early = lmu.forward_early(model, prompt, None, exit_layer, None)
            # one decode step on top of the early cache (seq=1 path)
            nxt = torch.tensor([[int(early.logits[0, -1].argmax())]])
            early2 = lmu.forward_early(model, nxt, early.past_key_values, exit_layer,
                                       early.exit_query_cache)
        arith.append(dict(
            model=mname, dims=list(MODELS[mname]), weight_seed=seed,
            weights_checksum=checksum(sd), exit_layer=exit_layer,
            prompt=[int(t) for t in prompt[0]],
            full_logits_last=[float(x) for x in full.logits[0, -1]],
            full_logits_row3=[float(x) for x in full.logits[0, 3]],
            early_logits_last=[float(x) for x in early.logits[0, -1]],
            exit_hidden_last=[float(x) for x in early.exit_query_cache[0, -1]],
            k_cache_l0_h0_last=[float(x) for x in early.past_key_values[0][0][0, 0, -1]],
            v_cache_l0_h0_last=[float(x) for x in early.past_key_values[0][1][0, 0, -1]],
            step2_token=int(nxt), step2_logits=[float(x) for x in early2.logits[0, -1]]))
    with open(os.path.join(GOLDEN_DIR, "layer_arith.json"), "w") as f:
        json.dump(dict(generator="oracle/gen_golden.py", cases=arith), f)
    print("wrote", GOLDEN_DIR)


RERUN_CASE = "mha128_a0.1"


def rerun() -> None:
    """Run the reference once more on one committed case (seeded weights, prompt, eos and settings
    read back from spec_traces.json) and store its whole result as reference_rerun.json, so the
    suite can check the fixture against an independent run without the reference tree."""
    import transformers
    ref = ref_shim.load_reference()
    with open(os.path.join(GOLDEN_DIR, "spec_traces.json")) as f:
        case = next(c for c in json.load(f)["cases"] if c["name"] == RERUN_CASE)
    dims = orc.LlamaDims(*case["dims"])
    sd = orc.random_state_dict(dims, case["weight_seed"], case["damp_from"], case["alpha"])
    res = run_reference(ref, build_hf(dims, sd), case["prompt"], case["eos"], case["cfg"],
                        case.get("torch_seed"))
    with open(os.path.join(GOLDEN_DIR, "reference_rerun.json"), "w") as f:
        json.dump(dict(generator="oracle/gen_golden.py --rerun", case=RERUN_CASE,
                       torch=torch.__version__, transformers=transformers.__version__,
                       reference=res), f, indent=1)
    print("wrote", os.path.join(GOLDEN_DIR, "reference_rerun.json"))


if __name__ == "__main__":
    rerun() if "--rerun" in sys.argv else main()
