"""Host-side logic of bench.py and of the synthetic fixtures that needs no GPU: the roofline numerator (algorithmic weight bytes of
one draft -> verify -> accept cycle, SURVEY.md 8d), the weight-spec generator shared by both arms, and the closed-vocabulary
permutation-bigram target behind `--fixture correlated` / tests/test_fullshape_gpu.py."""
import argparse

import torch

import bench
from eagle_b200 import synthetic as syn


def _args(model, layers=0):
    return argparse.Namespace(model=model, dtype=bench.MODELS[model]["dtype"], tree="dynamic", fixture="random", layers=layers, temperature=0.0)


def test_cycle_bytes_match_the_survey_figure_for_the_headline_config():
    tcfg, hcfg, eagle3 = bench.model_configs(_args("llama3-8b"))
    cyc, verify = bench.weight_bytes_per_cycle(tcfg, hcfg, eagle3, 6)
    # DESIGN.md 4 / SURVEY 8d: 15.009 GB verify (32 x 436.2 MB + 1.051 GB lm_head) + 5.34 GB draft (7 x 0.749 GB + 0.101 GB fc)
    assert abs(verify / 1e9 - 15.009) < 0.01
    assert abs(cyc / 1e9 - 20.35) < 0.01


def test_weight_specs_cover_the_reference_state_dict_keys():
    for model in ("llama3-8b", "llama2-13b"):
        tcfg, hcfg, eagle3 = bench.model_configs(_args(model, layers=2))
        names = {(w, n) for w, n, _, _ in bench.weight_specs(tcfg, hcfg, eagle3)}
        assert ("t", "model.layers.1.mlp.down_proj.weight") in names and ("t", "lm_head.weight") in names
        if eagle3:
            assert ("h", "midlayer.self_attn.q_proj.weight") in names and ("h", "fc.weight") in names and ("h", "lm_head.weight") in names
        else:
            assert ("h", "layers.0.self_attn.q_proj.weight") in names and ("h", "fc.bias") in names
        for w, n, shape, kind in bench.weight_specs(tcfg, hcfg, eagle3):
            if n.endswith("q_proj.weight") and w == "h":
                assert shape[1] == (2 if eagle3 else 1) * hcfg["hidden_size"]  # EAGLE-3 attends over cat(norm(emb), norm(hidden))


def test_workload_names_identify_the_baseline_config():
    a = _args("llama2-13b")
    a.temperature = 1.0
    assert "sampling(T=1)" in bench.workload_name(a) and "configs[3]" in bench.baseline_config(a)
    assert "configs[2]" in bench.baseline_config(_args("llama3-8b"))
    assert "configs[4]" in bench.baseline_config(_args("llama3-70b"))


def test_dump_outputs_writes_the_call_result_as_float64(tmp_path):
    import numpy as np
    bench.dump_outputs(str(tmp_path / "out"), torch.tensor([[5, 128255, 7]]), 2, 1)
    got = {n: np.load(tmp_path / "out" / f"{n}.npy") for n in ("ids", "new_token", "idx")}
    assert all(a.dtype == np.float64 for a in got.values())
    assert got["ids"].tolist() == [[5.0, 128255.0, 7.0]] and float(got["new_token"]) == 2.0 and float(got["idx"]) == 1.0


def test_closed_set_bigram_target_keeps_the_continuation_inside_the_draft_vocabulary():
    cfg = syn.target_config("tiny")
    W = syn.make_target_weights(cfg, 3, torch.bfloat16)
    used = syn.draft_vocab_ids(cfg["vocab_size"], 256)
    E_before = W["model.embed_tokens.weight"].clone()
    syn.make_bigram_target_(W, cfg, residual_eps=0.5, closed_set=used)
    # lm_head row perm[t] = head_scale * (scaled) emb[t]: recover perm and check it maps the set onto itself
    lm, E = W["lm_head.weight"].float(), W["model.embed_tokens.weight"].float()
    perm = (E @ lm.t()).argmax(-1)  # the row most aligned with emb[t]
    inside = torch.zeros(cfg["vocab_size"], dtype=torch.bool)
    inside[used] = True
    assert bool(inside[perm[used]].all()), "a draft-vocabulary token must be followed by a draft-vocabulary token"
    assert not bool(inside[perm[~inside]].any())
    assert torch.equal(torch.sort(perm).values, torch.arange(cfg["vocab_size"]))  # still a permutation
    assert not torch.equal(E_before, W["model.embed_tokens.weight"])  # embeddings were rescaled in place
