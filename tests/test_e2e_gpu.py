"""End-to-end parity on the B200: the CUDA engine behind `EaModel` against the reference-generated
golden vectors (tests/golden, produced by the unmodified reference) and the CPU oracle.

Bar (north star): identical accepted-token sequences under greedy decoding.  Greedy speculative decoding
emits the target's own greedy continuation, so sequence parity reduces to arg-max stability of the
tree-attention forward.  On the correlated fixtures (peaked distributions, large margins) the sequences,
accept lengths and trees must match the reference exactly; on random-weight fixtures (near-uniform logits,
bf16 top-2 margins below summation-order noise) we require the first cycles to match and report the rest.
"""
import pytest
import torch

from oracle.make_golden import FIXTURES, fixture_models
from tests.fixtures import build_oracle, load_golden

pytestmark = pytest.mark.gpu

ULP = {torch.bfloat16: 2.0 ** -7, torch.float16: 2.0 ** -10}


def tree_paths(draft_tokens, tree_mask):
    """Canonical, sibling-order-free form of a draft tree: the multiset of root->node token paths.  torch.topk leaves
    the order of equal model-dtype scores unspecified, so two correct builders may order tied siblings differently."""
    T = draft_tokens.shape[-1]
    toks = draft_tokens.reshape(-1).tolist()
    m = tree_mask.reshape(T, T)
    paths = []
    for i in range(T):
        anc = [j for j in range(T) if m[i, j] > 0]
        paths.append(tuple(toks[j] for j in anc))
    return sorted(paths)


def node_map(dt_a, tm_a, dt_b, tm_b):
    """node index in tree a -> node index in tree b with the same token path (None if absent)."""
    T = dt_a.shape[-1]

    def keyed(dt, tm):
        toks = dt.reshape(-1).tolist()
        m = tm.reshape(T, T)
        return {tuple(toks[j] for j in range(T) if m[i, j] > 0): i for i in range(T)}

    ka, kb = keyed(dt_a, tm_a), keyed(dt_b, tm_b)
    return {ia: kb.get(path) for path, ia in ka.items()}


def build_engine(fx, flags=0, max_length=512):
    from eagle_b200 import EaModel
    tcfg, tW, hcfg, hW, eagle3, dtype, tree = fixture_models(fx)
    m = EaModel.from_state_dicts(tcfg, tW, hcfg, hW, use_eagle3=eagle3, torch_dtype=dtype, max_length=max_length, flags=flags, **tree)
    return m, dtype


@pytest.mark.parametrize("flags", [1, 0], ids=["simt-gemm", "tcgen05"])
@pytest.mark.parametrize("fx", ["e3_corr_bf16", "e1_corr_fp16", "e3_gqa_bf16"])
def test_correlated_fixture_identical_to_reference(fx, flags):
    g = load_golden(fx)
    m, _ = build_engine(fx, flags)
    ids, new_token, idx = m.eagenerate(g["prompt"].cuda(), log=True, **g["gen_kw"])
    assert ids.cpu().tolist() == g["ids"].tolist()
    assert (new_token, idx) == (g["new_token"], g["idx"])
    assert m.stats()["kernel_launches"] > 0


@pytest.mark.parametrize("fx", ["e3_corr_bf16", "e1_corr_fp16", "e3_rand_bf16", "e1_rand_bf16"])
def test_first_tree_and_stepwise_state(fx):
    """prefill -> tree 0 in the reference's own formats, then cycle-by-cycle accept results."""
    g = load_golden(fx)
    m, dtype = build_engine(fx)
    first = m.prefill(g["prompt"].cuda())
    t0 = g["trees"][0]
    assert first == int(t0["draft_tokens"][0, 0]), "first token (arg-max of the prefill's last row)"
    dt, ri, tm, tp = m.get_tree()
    corr = "corr" in fx
    # The tree is compared through sibling-order-free root->node token paths.  The high-confidence part of the tree (the
    # draft's top-1 chain, which is what gets accepted) must be there; the low-probability filler nodes carry
    # model-dtype log-probs that tie in bf16/fp16 and torch.topk orders ties arbitrarily, so they are only reported.
    ours, ref = tree_paths(dt, tm), tree_paths(t0["draft_tokens"], t0["tree_mask"])
    assert dt.shape == t0["draft_tokens"].shape and int(dt[0, 0]) == int(t0["draft_tokens"][0, 0])
    assert bool((tm[0, 0].diagonal() == 1).all()) and bool((tm[0, 0, :, 0] == 1).all())
    shared = len(set(ours) & set(ref))
    print(f"{fx}: first tree shares {shared}/{len(ref)} root->node paths with the reference tree")
    if corr:
        gc0 = g["cycles"][0]
        accepted = tuple(gc0["candidates"][gc0["best"], : gc0["accept_length"] + 1].tolist())
        for d in range(1, len(accepted) + 1):
            assert accepted[:d] in set(ours), f"accepted prefix {accepted[:d]} missing from the engine's tree"
        if ours == ref and torch.equal(dt, t0["draft_tokens"]):  # no tie reordering: everything must be bit-identical
            assert torch.equal(tm, t0["tree_mask"]) and torch.equal(tp, t0["tree_pos"]) and torch.equal(ri, t0["retrieve"])
    n_cycles = len(g["cycles"]) if corr else 1
    for c in range(n_cycles):
        toks, nxt = m.step()
        am, best, acc, n = m.get_verify()
        gc = g["cycles"][c]
        want = gc["candidates"][gc["best"], : gc["accept_length"] + 1].tolist()
        assert toks == want, f"cycle {c}: committed tokens {toks} != reference {want}"
        assert acc == gc["accept_length"]


def test_verify_features_close_to_reference():
    """EAGLE-3 feature taps of the first verify pass vs the reference's hidden_state_new (bf16 tolerance)."""
    fx = "e3_corr_bf16"
    g = load_golden(fx)
    m, dtype = build_engine(fx)
    m.prefill(g["prompt"].cuda())
    dt, ri, tm, tp = m.get_tree()
    m.step()
    feats = m.debug_read("verify_features")
    t0 = g["trees"][0]
    nm = node_map(dt, tm, t0["draft_tokens"], t0["tree_mask"])  # tied filler nodes may differ between the two trees
    mine = [i for i in range(dt.shape[-1]) if nm[i] is not None]
    assert len(mine) >= 8, "too few common tree nodes to compare"
    feats = feats[torch.tensor(mine)]
    want = g["cycles"][0]["hidden_new"][0].float()[torch.tensor([nm[i] for i in mine])]
    err = (feats - want).abs()
    tol = 0.02 + 4 * ULP[dtype] * want.abs()
    frac_bad = float((err > tol).float().mean())
    assert frac_bad < 1e-3, f"{frac_bad:.4%} of feature elements off; max err {float(err.max()):.4f}"


@pytest.mark.parametrize("fx", ["e3_rand_bf16", "e1_rand_bf16"])
def test_random_weights_lossless_and_reported(fx):
    """Random weights (tau = 1): the engine's greedy spec-decode output must equal ITS OWN vanilla greedy output
    (losslessness, the reference's own invariant, speed.py relies on it) and we report agreement with the reference."""
    g = load_golden(fx)
    m, _ = build_engine(fx)
    ids = m.eagenerate(g["prompt"].cuda(), **g["gen_kw"]).cpu()
    naive = m.naivegenerate(g["prompt"].cuda(), max_new_tokens=g["gen_kw"]["max_new_tokens"], max_length=g["gen_kw"]["max_length"]).cpu()
    n = min(ids.shape[1], naive.shape[1])
    assert ids[0, :n].tolist() == naive[0, :n].tolist(), "speculative output differs from vanilla greedy"
    ref = g["ids"]
    k = min(ids.shape[1], ref.shape[1])
    agree = int((ids[0, :k] == ref[0, :k]).long().cumprod(0).sum())
    P = g["prompt"].shape[1]
    print(f"[{fx}] tokens identical to the reference: {agree - P}/{k - P} generated")
    # Margin-aware bar: greedy decoding is a chain of arg-max decisions; the engine must reproduce the reference's token at EVERY
    # position up to the first decision the reference itself takes with a top-2 logit margin below 2 ulps of the model dtype
    # (below that, fp32 summation order decides and no two correct implementations agree -- DESIGN.md 2).
    ref_model, (_, _, _, _, _, dtype, _) = build_oracle(fx)
    hidden, _ = ref_model.target.forward(ref[:, : k - 1], ref_model._kv(512))
    logits = ref_model.target.lm_head(hidden)[0, P - 1:].float()  # row j decides generated token j
    top2 = logits.topk(2, dim=-1).values
    spacing = torch.exp2(torch.floor(torch.log2(top2[:, 0].abs().clamp_min(1e-30)))) * ULP[dtype]
    margin_ulps = (top2[:, 0] - top2[:, 1]) / spacing
    fragile = (margin_ulps < 2.0).nonzero().flatten()
    must_match = int(fragile[0]) if fragile.numel() else k - P
    print(f"{fx}: identical generated-token prefix vs reference {agree - P}/{k - P}; first sub-2-ulp decision of the reference at "
          f"generated token {must_match} (min margin {float(margin_ulps.min()):.2f} ulp)")
    assert agree - P >= must_match, f"diverged at generated token {agree - P}, before the first fragile decision ({must_match})"


@pytest.mark.parametrize("fx", ["e3_corr_bf16", "e1_corr_fp16"])
def test_naive_generate_identical_to_reference(fx):
    g = load_golden(fx)
    m, _ = build_engine(fx)
    out = m.naivegenerate(g["prompt"].cuda(), max_new_tokens=g["gen_kw"]["max_new_tokens"], max_length=g["gen_kw"]["max_length"])
    assert out.cpu().tolist() == g["naive_ids"].tolist()


def test_ea_generate_yields_every_cycle():
    fx = "e3_corr_bf16"
    g = load_golden(fx)
    m, _ = build_engine(fx)
    outs = list(m.ea_generate(g["prompt"].cuda(), **g["gen_kw"]))
    assert len(outs) == g["idx"] + 1
    assert outs[-1].cpu().tolist() == g["ids"].tolist()


def test_engine_reuse_across_calls():
    """State persists between calls like the reference's cached KV (ea_model.py:227-241): a second call on the
    same model must give the same answer."""
    fx = "e3_corr_bf16"
    g = load_golden(fx)
    m, _ = build_engine(fx)
    a = m.eagenerate(g["prompt"].cuda(), **g["gen_kw"]).cpu()
    b = m.eagenerate(g["prompt"].cuda(), **g["gen_kw"]).cpu()
    assert a.tolist() == b.tolist() == g["ids"].tolist()


def test_sampling_posterior_is_lossless_monte_carlo():
    """temperature = 1 (config 4's mode): the SECOND generated token -- the first one decided by the speculative-sampling
    posterior (accepted draft token, or the residual-distribution bonus) -- must be distributed exactly like the target's
    own next-token distribution.  Same idea as the reference's only test (eagle/testbug/testbbug.py: histogram of
    eagenerate(temperature=1.0) outputs vs the target categorical), on the tiny random-weight EAGLE-3 fixture."""
    fx = "e3_rand_bf16"
    g = load_golden(fx)
    m, dtype = build_engine(fx)
    prompt = g["prompt"]
    P = prompt.shape[1]
    m.set_uniforms([0.5])
    torch.manual_seed(0)
    t1 = int(m.eagenerate(prompt.cuda(), temperature=1.0, max_new_tokens=0, max_length=512)[0, P])
    ref, _ = build_oracle(fx)
    kv = ref._kv(512)
    hidden, _ = ref.target.forward(torch.cat((prompt, torch.tensor([[t1]])), dim=1), kv)
    p2 = torch.softmax(ref.target.lm_head(hidden)[0, -1].float(), dim=-1)
    order = torch.argsort(p2, descending=True)
    n_buckets, n_trials = 16, 2400
    cum = torch.cumsum(p2[order], 0)
    bucket_of = torch.empty_like(order)
    bucket_of[order] = torch.clamp((cum * n_buckets).long(), max=n_buckets - 1)
    expected = torch.zeros(n_buckets).index_add_(0, bucket_of, p2) * n_trials
    counts = torch.zeros(n_buckets)
    accepted_second = 0
    for i in range(n_trials):
        m.set_uniforms([0.5])          # pins the first token; everything after comes from the seeded counter RNG
        torch.manual_seed(1000 + i)
        ids, new_token, idx = m.eagenerate(prompt.cuda(), temperature=1.0, max_new_tokens=1, max_length=512, log=True)
        assert int(ids[0, P]) == t1
        counts[bucket_of[int(ids[0, P + 1])]] += 1
        accepted_second += int(new_token > idx + 1)
    chi2 = float(((counts - expected) ** 2 / expected).sum())
    print(f"sampling losslessness: chi2={chi2:.1f} over {n_buckets} equal-mass buckets, {n_trials} trials")
    assert chi2 < 45.0, f"second-token histogram deviates from the target distribution: chi2={chi2:.1f} (df=15)"


def test_sampling_generation_runs_and_is_reproducible():
    fx = "e3_corr_bf16"
    g = load_golden(fx)
    m, _ = build_engine(fx)
    torch.manual_seed(7)
    a = m.eagenerate(g["prompt"].cuda(), temperature=1.0, max_new_tokens=32, max_length=512).cpu()
    torch.manual_seed(7)
    b = m.eagenerate(g["prompt"].cuda(), temperature=1.0, max_new_tokens=32, max_length=512).cpu()
    assert a.tolist() == b.tolist() and a.shape[1] > g["prompt"].shape[1] + 32
    # large-margin target (p(top-1) ~ 1): sampling at T=1 reproduces the greedy continuation
    assert a[0, : g["ids"].shape[1]].tolist()[: a.shape[1]] == g["ids"][0, : a.shape[1]].tolist()[: g["ids"].shape[1]]


def test_consecutive_sampling_calls_draw_fresh_seeds():
    """ADVICE r1: every temperature > 0 call used to replay one random stream.  Two calls after ONE torch.manual_seed must
    differ (the reference advances the global RNG), re-seeding must reproduce the pair."""
    fx = "e3_rand_bf16"  # near-uniform target: samples differ whenever the uniforms do
    g = load_golden(fx)
    m, _ = build_engine(fx)
    prompt = g["prompt"].cuda()
    torch.manual_seed(11)
    a = m.eagenerate(prompt, temperature=1.0, max_new_tokens=16, max_length=512).cpu().tolist()
    b = m.eagenerate(prompt, temperature=1.0, max_new_tokens=16, max_length=512).cpu().tolist()
    c = m.naivegenerate(prompt, temperature=1.0, max_new_tokens=16, max_length=512).cpu().tolist()
    assert a != b, "two consecutive sampling calls returned the same sample"
    torch.manual_seed(11)
    a2 = m.eagenerate(prompt, temperature=1.0, max_new_tokens=16, max_length=512).cpu().tolist()
    b2 = m.eagenerate(prompt, temperature=1.0, max_new_tokens=16, max_length=512).cpu().tolist()
    c2 = m.naivegenerate(prompt, temperature=1.0, max_new_tokens=16, max_length=512).cpu().tolist()
    assert (a, b, c) == (a2, b2, c2)
    # greedy calls do not consume the generator
    torch.manual_seed(11)
    m.eagenerate(prompt, max_new_tokens=4, max_length=512)
    a3 = m.eagenerate(prompt, temperature=1.0, max_new_tokens=16, max_length=512).cpu().tolist()
    assert a3 == a


def test_naive_generate_streams_token_by_token():
    """ea_model.py:485-558 yields after every decoded token (the round-1 version ran the whole generation first)."""
    fx = "e3_corr_bf16"
    g = load_golden(fx)
    m, _ = build_engine(fx)
    P = g["prompt"].shape[1]
    kw = dict(max_new_tokens=g["gen_kw"]["max_new_tokens"], max_length=g["gen_kw"]["max_length"])
    gen = m.naive_generate(g["prompt"].cuda(), **kw)
    first = next(gen)
    assert first.shape[1] == P + 1 and first[0, :P].cpu().tolist() == g["prompt"][0].tolist()
    cyc_before = m.stats()["kernel_launches"]
    second = next(gen)
    assert second.shape[1] == P + 2 and m.stats()["kernel_launches"] > cyc_before  # the work happens between yields
    outs = [first, second] + list(gen)
    assert outs[-1].cpu().tolist() == g["naive_ids"].tolist()
    assert [o.shape[1] for o in outs] == list(range(P + 1, P + 1 + len(outs)))


def test_total_token_minus_one_self_tunes():
    """total_token=-1 (ea_model.py:148-168): the engine times the target forward at {40,48,50,56,60} rows and keeps one."""
    from eagle_b200 import EaModel
    fx = "e3_corr_bf16"
    g = load_golden(fx)
    tcfg, tW, hcfg, hW, eagle3, dtype, tree = fixture_models(fx)
    tree = dict(tree, total_token=-1)
    m = EaModel.from_state_dicts(tcfg, tW, hcfg, hW, use_eagle3=eagle3, torch_dtype=dtype, max_length=512, **tree)
    assert m.ea_layer.total_tokens + 1 in (40, 48, 50, 56, 60) and len(m.tuned_times_ms) == 5
    ids = m.eagenerate(g["prompt"].cuda(), **g["gen_kw"]).cpu()
    n = min(ids.shape[1], g["ids"].shape[1])  # greedy spec decoding is lossless whatever the tree size: same token stream
    assert ids[0, :n].tolist() == g["ids"][0, :n].tolist()
    dt, _, _, _ = m.get_tree()
    assert dt.shape[-1] == m.ea_layer.total_tokens + 1
