"""Generate tests/golden/*.pt by running the UNMODIFIED reference on CPU.

Runs only in the build container (needs /root/reference; the GPU box has no reference).
The reference is imported with three environment shims that live here, not in the
reference (SURVEY.md 8c): (1) stub eagle.model.modeling_qwen3_kv (does not import on
transformers 5.x), (2) reset rope_scaling=None + rope_theta on configs, (3) bypass hub /
tokenizer construction by assembling EaModel by hand.

    python -m oracle.make_golden            # writes tests/golden/*.pt

Weights are NOT stored: they come from eagle_b200.synthetic factories (seeded), which the
tests re-run.  Stored: prompts, per-cycle tree tensors, verify arg-max per node, accept
results, the generated ids, and a few floating-point tensors for tolerance checks.
"""
from __future__ import annotations

import os
import random
import sys
import types

import torch
import torch.nn as nn

REF = "/root/reference"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, "tests", "golden")


def import_reference():
    sys.dont_write_bytecode = True
    sys.path.insert(0, REF)
    stub = types.ModuleType("eagle.model.modeling_qwen3_kv")
    stub.Qwen3ForCausalLM = object
    sys.modules["eagle.model.modeling_qwen3_kv"] = stub  # shim 1
    if not torch.cuda.is_available():
        torch.cuda.synchronize = lambda *a, **k: None
    import eagle.model.ea_model as em
    from eagle.model.modeling_llama_kv import LlamaForCausalLM as KVLlama
    from eagle.model.cnets import Model as Head3
    from eagle.model.cnets1 import Model as Head1
    from eagle.model.configs import EConfig
    from transformers import LlamaConfig
    return em, KVLlama, Head3, Head1, EConfig, LlamaConfig


class StandInTokenizer:
    eos_token_id = -12345

    def convert_tokens_to_ids(self, _):
        return -12346


def build_reference_model(tcfg: dict, tW, hcfg: dict, hW, eagle3: bool, dtype, total_token, depth, top_k):
    em, KVLlama, Head3, Head1, EConfig, LlamaConfig = import_reference()
    keys = ("vocab_size", "hidden_size", "intermediate_size", "num_hidden_layers", "num_attention_heads",
            "num_key_value_heads", "rms_norm_eps", "max_position_embeddings")
    cfg = LlamaConfig(**{k: tcfg[k] for k in keys}, pad_token_id=0, tie_word_embeddings=False)
    cfg.rope_scaling = None  # shim 2
    cfg.rope_theta = tcfg["rope_theta"]
    base = KVLlama(cfg)
    miss = base.load_state_dict(tW, strict=False)
    assert not miss.unexpected_keys and all("rotary_emb" in k for k in miss.missing_keys), miss
    base = base.to(dtype).eval()
    extra = {}
    if eagle3:
        extra["draft_vocab_size"] = hcfg["draft_vocab_size"]
    ecfg = EConfig(**{k: hcfg[k] for k in keys}, pad_token_id=0, **extra)
    ecfg.rope_scaling = None
    ecfg.rope_theta = hcfg["rope_theta"]
    Head = Head3 if eagle3 else Head1
    head = Head(ecfg, bias=hcfg.get("bias", True), total_tokens=total_token, depth=depth, top_k=top_k,
                threshold=1.0, load_emb=False)
    if eagle3 and hcfg["draft_vocab_size"] == hcfg["vocab_size"]:
        del head.d2t, head.t2d  # ea_model.py:74-75
    missing = head.load_state_dict(hW, strict=False)
    assert not [m for m in missing.missing_keys if "rotary" not in m], missing
    m = em.EaModel.__new__(em.EaModel)  # shim 3
    nn.Module.__init__(m)
    m.base_model, m.config, m.use_eagle3 = base, base.config, eagle3
    m.hidden_size, m.vocab_size = tcfg["hidden_size"], tcfg["vocab_size"]
    m.tokenizer = StandInTokenizer()
    m.ea_layer = head
    m.ea_layer.diff_device = False
    m.ea_layer.to(dtype)
    m.ea_layer.init_tree()
    m.eval()
    return m, em


def run_and_capture(m, em, prompt, sampling_seed=None, **gen_kw):
    """Run reference eagenerate, recording per-cycle tensors by wrapping its own step functions."""
    import eagle.model.ea_model as emod
    rec = {"cycles": [], "trees": []}
    orig_topk_gen = m.ea_layer.topK_genrate
    orig_tree_dec = emod.tree_decoding
    orig_eval = emod.evaluate_posterior
    orig_topk = torch.topk
    state = {}

    def topk_gen(hidden_states, input_ids, head, logits_processor):
        seen = []

        def spy_topk(x, k, *a, **kw):
            seen.append((x, k))
            return orig_topk(x, k, *a, **kw)

        torch.topk = spy_topk
        try:
            out = orig_topk_gen(hidden_states, input_ids, head, logits_processor)
        finally:
            torch.topk = orig_topk
        scores_flat = seen[-1][0]
        rec["trees"].append(dict(in_hidden=hidden_states.clone(), in_ids=input_ids.clone(),
                                 scores_flat=scores_flat.clone(),
                                 draft_tokens=out[0].clone(), retrieve=out[1].clone(),
                                 tree_mask=out[2].clone(), tree_pos=out[3].clone()))
        return out

    def tree_dec(model, tree_candidates, past_key_values, tree_position_ids, input_ids, retrieve_indices):
        logits, hidden_state, outputs = orig_tree_dec(model, tree_candidates, past_key_values, tree_position_ids,
                                                      input_ids, retrieve_indices)
        state["hidden_new"] = hidden_state
        state["prev_len"] = input_ids.shape[1]
        return logits, hidden_state, outputs

    def eval_post(logits, candidates, logits_processor):
        best, acc, sample_p = orig_eval(logits, candidates, logits_processor)
        rec["cycles"].append(dict(candidates=candidates.clone(), leaf_argmax=torch.argmax(logits, dim=-1).clone(),
                                  best=int(best), accept_length=int(acc), prev_len=state["prev_len"],
                                  hidden_new=state["hidden_new"].clone() if len(rec["cycles"]) < 2 else None))
        return best, acc, sample_p

    m.ea_layer.topK_genrate = topk_gen
    emod.tree_decoding = tree_dec
    emod.evaluate_posterior = eval_post
    try:
        if sampling_seed is not None:
            torch.manual_seed(sampling_seed)
            random.seed(sampling_seed)
        ids, new_token, idx = m.eagenerate(prompt, log=True, **gen_kw)
    finally:
        m.ea_layer.topK_genrate = orig_topk_gen
        emod.tree_decoding = orig_tree_dec
        emod.evaluate_posterior = orig_eval
    rec.update(prompt=prompt.clone(), ids=ids.clone(), new_token=int(new_token), idx=int(idx))
    return rec


from eagle_b200.synthetic import FIXTURES, base_fixture, fixture_models, make_prompt  # noqa: E402,F401  (the fixture registry lives with the weight factories)

# Fixtures stored without the per-phase hidden states (head input `in_hidden`, verify features `hidden_new`): no test reads them
# for these fixtures, and at the TP-8-shardable width they would take the file past 1 MB.
NO_HIDDEN_STATES = {"e3_tp8_bf16"}


# Stop conditions of the driver loop (ea_model.py:290-299).  The tokenizer's EOS / <|eot_id|> id is set to the token the greedy
# golden run emits at the given index of its continuation, so the run must stop after the cycle that commits it.
STOP_FIXTURES = {
    # name: (base fixture, which id, index into the base run's new tokens, extra gen kwargs)
    "e3_corr_bf16_EOS": ("e3_corr_bf16", "eos", 20, {}),
    "e3_corr_bf16_EOT": ("e3_corr_bf16", "eot", 9, {"is_llama3": True}),
    "e3_corr_bf16_MAXLEN": ("e3_corr_bf16", None, 0, {"max_length": 120, "max_new_tokens": 400}),   # length limit :250, :298
}


def make_stop_goldens(only=()):
    for fx, (base, which, index, extra) in STOP_FIXTURES.items():
        if only and fx not in only:
            continue
        plen, pseed, gen_kw, _ = FIXTURES[base]
        tcfg, tW, hcfg, hW, eagle3, dtype, tree = fixture_models(base)
        m, em = build_reference_model(tcfg, tW, hcfg, hW, eagle3, dtype, **tree)
        prompt = make_prompt(tcfg["vocab_size"], plen, pseed)
        base_ids = torch.load(os.path.join(GOLD, base + ".pt"), weights_only=False)["ids"]
        stop_id = int(base_ids[0, plen + index]) if which else None
        tok = StandInTokenizer()
        if which == "eos":
            tok.eos_token_id = stop_id
        elif which == "eot":
            tok.convert_tokens_to_ids = lambda _t, _i=stop_id: _i
        m.tokenizer = tok
        kw = dict(gen_kw)
        kw.update(extra)
        ids, new_token, idx = m.eagenerate(prompt, log=True, **kw)
        rec = dict(prompt=prompt.clone(), ids=ids.clone(), new_token=int(new_token), idx=int(idx), gen_kw=kw, tree=tree,
                   which=which, stop_id=stop_id, torch_version=torch.__version__)
        out = os.path.join(GOLD, fx + ".pt")
        torch.save(rec, out)
        print(f"{fx}: stop id {stop_id} ({which}) -> new_token={rec['new_token']} cycles={rec['idx'] + 1} len={ids.shape[1]}")



STATIC_TREES = {
    # name: choices (None -> the reference's own eagle/model/choices.py:mc_sim_7b_63)
    "mc_sim_7b_63": None,
    "mc_sim_7b_63_shuffled": "shuffle",
    "chain4": [[0], [0, 0], [0, 0, 0], [0, 0, 0, 0]],
    "flat3": [[0], [1], [2]],
    "wide": [[0], [1], [2], [3], [4], [0, 0], [0, 1], [0, 3], [1, 0], [1, 2], [2, 0], [0, 0, 0], [0, 0, 1], [0, 1, 0],
             [1, 0, 0], [1, 0, 4], [0, 0, 0, 0]],
    "gap": [[0], [1], [0, 0], [1, 0], [1, 0, 0]],  # parent-with-grandchildren is NOT a prefix of its level
}


def make_static_goldens():
    """tests/golden/static_tree.pt: the reference's fixed-tree integer buffers, generate_candidates, and the token
    table of EAGLEModel.topK_genrate (modeling_eagle.py:863-957, greedy) on the e1_rand_bf16 head weights."""
    import_reference()
    import eagle.model.utils as ru
    import eagle.modeling_eagle as me
    from eagle.model.choices import mc_sim_7b_63
    rec = {"trees": {}, "torch_version": torch.__version__}
    g = torch.Generator().manual_seed(77)
    for name, ch in STATIC_TREES.items():
        if ch is None:
            ch = [list(c) for c in mc_sim_7b_63]
        elif ch == "shuffle":
            ch = [list(c) for c in mc_sim_7b_63]
            perm = torch.randperm(len(ch), generator=g).tolist()
            ch = [ch[i] for i in perm]
        v10 = ru.generate_tree_buffers(ch, "cpu")          # TOPK = 10 (utils.py:13)
        v5 = me.generate_tree_buffers(ch, "cpu")           # TOPK = 5
        try:
            d5 = me.generate_tree_buffers_for_eagle(ch, "cpu")  # TOPK = 5
        except IndexError:  # a depth-1 tree has no node with children: the reference cannot build draft buffers for it
            d5 = None
        n_rows = 1 + (sum(int(t.numel()) for t in d5["tree_indices"]) if d5 else 0)
        cands = {}
        for topk, vb in ((10, v10), (5, v5)):
            table = torch.randint(0, 1000, (1, n_rows, topk), generator=g)
            sample_token = torch.randint(0, 1000, (1, 1), generator=g)
            if int(vb["tree_indices"].max()) <= n_rows * topk:
                cart, tree_c = ru.generate_candidates(table, vb["tree_indices"], vb["retrieve_indices"], sample_token, None)
                cands[topk] = dict(table=table, sample_token=sample_token, cart=cart, tree_candidates=tree_c)
        rec["trees"][name] = dict(choices=ch, verify10=v10, verify5=v5, draft5=d5, candidates=cands)
        print(f"static {name}: nodes={len(ch) + 1} leaves={v10['retrieve_indices'].shape[0]} "
              f"levels={[int(t.numel()) for t in d5['tree_indices']] if d5 else None} "
              f"repeat={d5['repeat_nums'] if d5 else None}")

    # --- static level-by-level growth on a tiny EAGLE-1 head
    tcfg, tW, hcfg, hW, eagle3, dtype, _ = fixture_models("e1_rand_bf16")
    assert not eagle3 and hcfg["rope_theta"] == 10000.0  # EAGLERotaryEmbedding has a fixed base (modeling_eagle.py:95)
    cfg = me.EAGLE_Config(vocab_size=hcfg["vocab_size"], hidden_size=hcfg["hidden_size"],
                          intermediate_size=hcfg["intermediate_size"], num_hidden_layers=1,
                          num_attention_heads=hcfg["num_attention_heads"],
                          num_key_value_heads=hcfg["num_key_value_heads"], rms_norm_eps=hcfg["rms_norm_eps"],
                          max_position_embeddings=hcfg["max_position_embeddings"], pad_token_id=0)
    cfg.rope_scaling = None
    grow = {}
    for name in ("mc_sim_7b_63", "wide", "gap", "chain4"):
        ch = rec["trees"][name]["choices"]
        model = me.EAGLEModel(cfg, bias=True)
        miss = model.load_state_dict(hW, strict=False)
        assert not miss.unexpected_keys and not [k for k in miss.missing_keys if "rotary" not in k], miss
        model = model.to(dtype).eval()
        model.device = torch.device("cpu")
        model.diff_device = False
        model.tree = ch
        model.init_tree()
        head = nn.Linear(hcfg["hidden_size"], hcfg["vocab_size"], bias=False)
        head.weight.data = tW["lm_head.weight"].clone()
        head = head.to(dtype)
        P, a = 19, 2
        hidden = (torch.randn(1, P, hcfg["hidden_size"], generator=g) * 0.5).to(dtype)
        ids = torch.randint(0, hcfg["vocab_size"] - 200, (1, P + 1), generator=g)
        model.reset_kv()
        t1, _, _ = model.topK_genrate(hidden, ids, head, None, attention_mask=torch.ones(1, P, dtype=torch.long))
        # second call: a+1 new feature rows on top of the stable KV (modeling_eagle.py:1536-1549)
        hidden2 = (torch.randn(1, a + 1, hcfg["hidden_size"], generator=g) * 0.5).to(dtype)
        new_ids = torch.randint(0, hcfg["vocab_size"] - 200, (1, a + 1), generator=g)
        draft_ids = torch.cat((ids[:, -1:], new_ids), dim=1)
        t2, _, _ = model.topK_genrate(hidden2, draft_ids, head, None,
                                      attention_mask=torch.ones(1, P + a + 1, dtype=torch.long), len_posi=P + a + 1)
        grow[name] = dict(hidden=hidden, ids=ids, table=t1[0].clone(), hidden2=hidden2,
                          full_ids2=torch.cat((ids, new_ids), dim=1), table2=t2[0].clone())
        print(f"static growth {name}: table {tuple(t1.shape)} / {tuple(t2.shape)}")
    rec["growth"] = grow
    out = os.path.join(GOLD, "static_tree.pt")
    torch.save(rec, out)
    print("wrote", out, os.path.getsize(out), "bytes")


def main():
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    if len(sys.argv) > 1 and sys.argv[1] == "static":
        make_static_goldens()
        return
    only = [a for a in sys.argv[1:] if a in FIXTURES or a in STOP_FIXTURES]
    if not only or any(a in STOP_FIXTURES for a in only):
        if not only:
            pass  # the base goldens are (re)generated first, below, then the stop runs
        else:
            make_stop_goldens([a for a in only if a in STOP_FIXTURES])
            only = [a for a in only if a in FIXTURES]
            if not only:
                return
    for fx, (plen, pseed, gen_kw, sseed) in FIXTURES.items():
        if only and fx not in only:
            continue
        model_name = base_fixture(fx)
        tcfg, tW, hcfg, hW, eagle3, dtype, tree = fixture_models(model_name)
        m, em = build_reference_model(tcfg, tW, hcfg, hW, eagle3, dtype, **tree)
        prompt = make_prompt(tcfg["vocab_size"], plen, pseed)
        rec = run_and_capture(m, em, prompt, sampling_seed=sseed, **gen_kw)
        if fx in NO_HIDDEN_STATES:
            for t in rec["trees"]:
                del t["in_hidden"]
            for c in rec["cycles"]:
                c["hidden_new"] = None
        naive = m.naivegenerate(prompt, temperature=0.0, max_new_tokens=gen_kw["max_new_tokens"],
                                max_length=gen_kw["max_length"]) if sseed is None else None
        rec["naive_ids"] = naive
        rec["gen_kw"] = gen_kw
        rec["tree"] = tree
        rec["torch_version"] = torch.__version__
        out = os.path.join(GOLD, fx + ".pt")
        torch.save(rec, out)
        tau = rec["new_token"] / (rec["idx"] + 1)
        accs = [c["accept_length"] for c in rec["cycles"]]
        print(f"{fx}: new_token={rec['new_token']} cycles={rec['idx'] + 1} tau={tau:.2f} accept={accs} "
              f"bytes={os.path.getsize(out)}")
        if naive is not None:
            n = min(naive.shape[1], rec["ids"].shape[1])
            print("   greedy == naive prefix:", bool((naive[0, :n] == rec["ids"][0, :n]).all()))
    if not only:
        make_stop_goldens()
        make_static_goldens()


if __name__ == "__main__":
    main()
