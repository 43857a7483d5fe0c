"""Static draft tree on the B200 (SURVEY.md 8 row a11): the engine's fixed-tree mode against the CPU oracle
(oracle/static_tree.py, pinned bit-for-bit on the reference's own buffers / generate_candidates / EAGLEModel.topK_genrate
by tests/test_static_tree_cpu.py) and against reference-generated goldens where the kernel has one."""
import ctypes as C

import pytest
import torch

from oracle import eagle_oracle as orc
from oracle import static_tree as stt
from oracle.make_golden import fixture_models, make_prompt
from tests.fixtures import load_golden, to_cfg

pytestmark = pytest.mark.gpu

DT = {torch.bfloat16: 0, torch.float16: 1}


def _lib():
    from eagle_b200 import _lib
    return _lib.load(), _lib


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("rows,V,k", [(1, 1024, 5), (4, 32000, 10), (11, 128256, 10), (64, 4096, 16)])
def test_topk_raw_kernel(dtype, rows, V, k):
    lib, L = _lib()
    g = torch.Generator().manual_seed(rows * 7 + k)
    x = (torch.randn(rows, V, generator=g) * 3).to(dtype)
    xd = x.cuda()
    tv = torch.empty(rows, k, dtype=torch.float32, device="cuda")
    ti = torch.empty(rows, k, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    L.check(lib.eb200_k_topk_raw(DT[dtype], xd.data_ptr(), rows, V, k, tv.data_ptr(), ti.data_ptr(), None))
    want = torch.topk(x.float(), k, dim=-1)
    assert torch.equal(tv.cpu(), want.values)                                   # same values in the same order
    assert torch.equal(torch.gather(x.float(), 1, ti.cpu().long()), want.values)  # indices point at those values
    for r in range(rows):
        idx = ti[r].cpu().tolist()
        assert len(set(idx)) == k
        vals = want.values[r].tolist()
        for a in range(k - 1):  # ties: lowest index first
            if vals[a] == vals[a + 1]:
                assert idx[a] < idx[a + 1]


@pytest.mark.parametrize("name", ["mc_sim_7b_63", "wide", "gap", "chain4"])
def test_generate_candidates_kernel_matches_reference(name):
    lib, L = _lib()
    t = load_golden("static_tree")["trees"][name]
    for topk, c in t["candidates"].items():
        vb = stt.verify_buffers(t["choices"], topk)
        table = c["table"].reshape(-1, topk).to(torch.int32).contiguous()
        ti = vb["tree_indices"].to(torch.int32).contiguous()
        T = ti.numel()
        out = torch.empty(T, dtype=torch.int64)
        L.check(lib.eb200_k_generate_candidates(table.data_ptr(), table.shape[0], topk, None, 0, ti.data_ptr(), T,
                                                int(c["sample_token"]), out.data_ptr()))
        assert torch.equal(out[None], c["tree_candidates"])
        # with a draft->target offset table (cnets.py:712-713): tokens are remapped before the gather
        d2t = torch.randint(0, 5000, (1000,), generator=torch.Generator().manual_seed(3), dtype=torch.int64)
        L.check(lib.eb200_k_generate_candidates(table.data_ptr(), table.shape[0], topk, d2t.data_ptr(), 1000, ti.data_ptr(), T,
                                                int(c["sample_token"]), out.data_ptr()))
        mapped = c["table"] + d2t[c["table"]]
        _, want = stt.generate_candidates(mapped, vb["tree_indices"], vb["retrieve_indices"], c["sample_token"])
        assert torch.equal(out[None], want)


def _engine(fx, choices, topk, max_length=512, flags=0):
    from eagle_b200 import EaModel
    tcfg, tW, hcfg, hW, eagle3, dtype, _ = fixture_models(fx)
    m = EaModel.from_state_dicts(tcfg, tW, hcfg, hW, use_eagle3=eagle3, torch_dtype=dtype, max_length=max_length, flags=flags,
                                 top_k=topk, tree_choices=choices)
    o = orc.OracleEaModel(to_cfg(tcfg), tW, to_cfg(hcfg), hW, eagle3, top_k=topk, tree_choices=choices)
    return m, o, tcfg


@pytest.mark.parametrize("topk", [5, 10])
@pytest.mark.parametrize("fx", ["e3_corr_bf16", "e1_corr_fp16", "e3_gqa_bf16"])
def test_static_generation_identical_to_oracle(fx, topk):
    """mc_sim_7b_63 tree, greedy: same ids / new_token / idx as the oracle's static eagenerate, cycle by cycle the same
    committed tokens and accept lengths, and the fixed mask / positions / retrieve paths bit-identical."""
    m, o, tcfg = _engine(fx, stt.MC_SIM_7B_63, topk)
    prompt = make_prompt(tcfg["vocab_size"], 29, 11)
    o.cycle_log = []
    want_ids, want_new, want_idx = o.eagenerate(prompt, max_new_tokens=40, max_length=512, log=True)
    ids, new_token, idx = m.eagenerate(prompt.cuda(), max_new_tokens=40, max_length=512, log=True)
    assert ids.cpu().tolist() == want_ids.tolist()
    assert (new_token, idx) == (want_new, want_idx)
    assert new_token / (idx + 1) > 2.0, "fixture should accept several tokens per cycle on the static tree"
    # step-wise
    first = m.prefill(prompt.cuda())
    c0 = o.cycle_log[0]
    assert first == int(c0["draft_tokens"][0, 0])
    vb = stt.verify_buffers(stt.MC_SIM_7B_63, topk)
    same = total = 0
    for c, oc in enumerate(o.cycle_log):
        dt, ri, tm, tp = m.get_tree()
        assert torch.equal(tm, vb["tree_attn_mask"]) and torch.equal(tp, vb["tree_position_ids"])
        assert torch.equal(ri, vb["retrieve_indices"])
        assert int(dt[0, 0]) == int(oc["draft_tokens"][0, 0])
        # cascade-aware comparison: a node counts as a divergence only if every ancestor carries the oracle's token and its own
        # token differs (children of a differing node differ trivially)
        eq = (dt == oc["draft_tokens"])[0]
        anc_ok = torch.tensor([bool(eq[[j for j in range(dt.shape[-1]) if tm[0, 0, i, j] > 0 and j != i]].all()) for i in range(dt.shape[-1])])
        same += int((eq & anc_ok).sum())
        total += int(anc_ok.sum())
        toks, nxt = m.step()
        am, best, acc, n = m.get_verify()
        want = torch.cat((oc["draft_tokens"], torch.full((1, 1), -1, dtype=torch.long)), dim=1)[0, oc["retrieve"]][
            oc["best"], : oc["accept_length"] + 1].tolist()
        assert toks == want, f"cycle {c}: committed {toks} != oracle {want}"
        assert acc == oc["accept_length"] and nxt == oc["bonus"]
    print(f"static {fx} top_k={topk}: {same}/{total} tree tokens (nodes with identical ancestors) identical to the oracle over {len(o.cycle_log)} cycles")
    # first-divergence nodes are bf16/fp16 exact ties among low-probability filler children (torch.topk orders ties arbitrarily, the
    # kernel by index); they never sit on a committed path (checked token by token above)
    assert same / total >= 0.95, f"{total - same}/{total} tree nodes diverge from the oracle under identical ancestors"


@pytest.mark.parametrize("name", ["wide", "gap", "chain4"])
def test_static_other_trees(name):
    choices = load_golden("static_tree")["trees"][name]["choices"]
    m, o, tcfg = _engine("e3_corr_bf16", choices, 5)
    prompt = make_prompt(tcfg["vocab_size"], 41, 5)
    want = o.eagenerate(prompt, max_new_tokens=24, max_length=512, log=True)
    got = m.eagenerate(prompt.cuda(), max_new_tokens=24, max_length=512, log=True)
    assert got[0].cpu().tolist() == want[0].tolist() and got[1:] == want[1:]


def test_static_random_head_with_d2t_is_lossless():
    """Random EAGLE-3 head with a reduced draft vocabulary (d2t remap in the candidate gather): whatever the head proposes,
    greedy speculative decoding over the fixed tree must reproduce the engine's own vanilla greedy continuation."""
    m, o, tcfg = _engine("e3_rand_bf16", stt.MC_SIM_7B_63, 10)
    prompt = make_prompt(tcfg["vocab_size"], 37, 10).cuda()
    ids = m.eagenerate(prompt, max_new_tokens=24, max_length=512).cpu()
    naive = m.naivegenerate(prompt, max_new_tokens=24, max_length=512).cpu()
    n = min(ids.shape[1], naive.shape[1])
    assert ids[0, :n].tolist() == naive[0, :n].tolist()
    dt, ri, tm, tp = m.get_tree()
    assert int(dt.max()) < tcfg["vocab_size"] and int(dt.min()) >= 0


def test_static_sampling_runs_and_stops():
    """temperature > 0 over the fixed tree uses the same q == 1 posterior (utils.py:375-415); smoke + determinism."""
    m, o, tcfg = _engine("e3_corr_bf16", stt.MC_SIM_7B_63, 10)
    prompt = make_prompt(tcfg["vocab_size"], 29, 11).cuda()
    torch.manual_seed(7)
    a = m.eagenerate(prompt, temperature=1.0, max_new_tokens=24, max_length=512).cpu()
    torch.manual_seed(7)
    b = m.eagenerate(prompt, temperature=1.0, max_new_tokens=24, max_length=512).cpu()
    assert a.tolist() == b.tolist() and a.shape[1] > prompt.shape[1] + 24


def test_switch_back_to_dynamic_tree():
    from eagle_b200 import EaModel
    lib, L = _lib()
    fx = "e3_corr_bf16"
    g = load_golden(fx)
    tcfg, tW, hcfg, hW, eagle3, dtype, tree = fixture_models(fx)
    m = EaModel.from_state_dicts(tcfg, tW, hcfg, hW, use_eagle3=eagle3, torch_dtype=dtype, max_length=512, **tree)
    # a tree that does not fit the engine's total_token / depth is refused
    flat = (C.c_int32 * 3)(0, 0, 0)
    lens = (C.c_int32 * 2)(1, 2)
    with pytest.raises(L.EngineError, match="total_token"):
        L.check(lib.eb200_set_static_tree(m._h, flat, lens, 2))
    L.check(lib.eb200_set_static_tree(m._h, None, None, 0))
    ids, new_token, idx = m.eagenerate(g["prompt"].cuda(), log=True, **g["gen_kw"])
    assert ids.cpu().tolist() == g["ids"].tolist() and (new_token, idx) == (g["new_token"], g["idx"])
