"""The stage checks of tests/test_tower_parity.py (tests/tower_stages.py) on an fp64 CPU tower with injected faults.

The tower: two vision-style blocks (d = 128, 2 heads, 3 sequences of 50 tokens = 150 rows, so the last 128-row tile is
partial), deep prompts spliced into both layers, no pruning.  It stores what the native tower stores and rounds where the
native stand-alone formulation rounds (LayerNorm outputs, weights, qkv, o, h and QuickGELU(h) to bf16; the residual
stream in fp32), so the correct tower must pass every stage at the GPU's bounds.  Each fault below is one that a
whole-model metric dilutes over the rest of the tower; the stage checks must reject it and name the (layer, stage,
block) where it was made."""
import pytest
import torch
import torch.nn.functional as F

from tests import tower_stages as ts

D, H, S, L, N_CTX, LAYERS = 128, 2, 3, 50, 2, 2
ROW0 = L - N_CTX
E = 64


def _bf(t):
    return t.bfloat16().double()


@pytest.fixture(scope="module")
def tower():
    g = torch.Generator().manual_seed(0)

    def u(shape, bound):
        return (torch.rand(shape, generator=g, dtype=torch.float64) * 2 - 1) * bound

    def n(shape, std):
        return torch.randn(shape, generator=g, dtype=torch.float64) * std

    # the synthetic vision tower's distributions (mudpt_b200/synthetic.py: torch defaults)
    blocks = []
    for _ in range(LAYERS):
        blocks.append({"ln_1.weight": 1 + n(D, 0.1), "ln_1.bias": n(D, 0.1), "attn.in_proj_weight": u((3 * D, D), (6 / (4 * D)) ** 0.5),
                       "attn.in_proj_bias": n(3 * D, 0.02), "attn.out_proj.weight": u((D, D), D ** -0.5),
                       "attn.out_proj.bias": n(D, 0.02), "ln_2.weight": 1 + n(D, 0.1), "ln_2.bias": n(D, 0.1),
                       "mlp.c_fc.weight": u((4 * D, D), D ** -0.5), "mlp.c_fc.bias": u(4 * D, D ** -0.5),
                       "mlp.c_proj.weight": u((D, 4 * D), (4 * D) ** -0.5), "mlp.c_proj.bias": u(D, (4 * D) ** -0.5)})
    return {"blocks": [{k: v.float() for k, v in b.items()} for b in blocks], "x0": n((S * L, D), 1.0).float(),
            "x0_ragged": n((sum(RAGGED.lengths), D), 1.0).float(),
            "prompts": n((LAYERS, N_CTX, D), 1.0).float(), "ln_g": (1 + n(D, 0.1)).float(), "ln_b": n(D, 0.1).float(),
            "proj": n((D, E), D ** -0.5).float()}


GEO = ts.Geometry(lengths=[L] * S, H=H, causal=False, row0=ROW0, n_ctx=N_CTX, spliced=[0, 1], sel=[s * L for s in range(S)])
# a ragged causal (text-like) tower: packed rows (162, a partial last tile), EOT rows inside their sequences
RAGGED = ts.Geometry(lengths=[40, 55, 37, 30], H=H, causal=True, row0=1, n_ctx=N_CTX, spliced=[0, 1], sel=[30, 40 + 50, 95 + 20, 132 + 29])


def _attention(qkv, geo, causal):
    """(o, lse) of the packed rows: fp64 attention, lse in the kernels' layout (sequence s: [H, len_s] at off[s] * H)"""
    off = geo.off
    o = ts._attention(qkv.double(), ts.Geometry(**{**geo.__dict__, "causal": causal}), False)
    lse = torch.cat([ts._attn_lse2_ref(qkv[off[s]:off[s + 1]].double(), 1, n, H, causal).flatten() for s, n in enumerate(geo.lengths)])
    return o, lse


def run(tw, fault=None, geo=GEO):
    """(saved operands {(name, layer): tensor}, features) of the tower, with one fault: "bias_tail" (c_proj bias missing
    on the last, partial 128-row tile of layer 0), "splice_late" (layer 0's deep prompt spliced into layer 1 instead),
    "ln2_gamma" (layer 1's LN2 with layer 0's gamma), "ln1_gamma"
    (layer 0's LN1 with layer 1's gamma), "last_mask" (the pruned last block's EOT queries see every key of
    their sequence), "lse_seq2" (one lse entry of sequence 2 of layer 0 off by 1e-3)."""
    ops = {}
    S = geo.S
    pr = geo.prompt_rows("cpu").flatten()
    x = (tw["x0"] if geo is GEO else tw["x0_ragged"]).clone()
    rows = x.shape[0]
    for i in range(LAYERS):
        w = tw["blocks"][i]
        if fault == "splice_late":
            if i == 1:
                x[pr] = tw["prompts"][0].repeat(S, 1)
        else:
            x[pr] = tw["prompts"][i].repeat(S, 1)
        ops["x_in", i] = x
        g1 = tw["blocks"][1]["ln_1.weight"] if (fault == "ln1_gamma" and i == 0) else w["ln_1.weight"]
        a = _bf(F.layer_norm(x.double(), (D,), g1.double(), w["ln_1.bias"].double(), ts.LN_EPS))
        qkv = (a @ _bf(w["attn.in_proj_weight"]).t() + w["attn.in_proj_bias"].double()).bfloat16()
        ops["qkv", i] = qkv
        o, lse = _attention(qkv, geo, geo.causal)
        if fault == "lse_seq2" and i == 0:
            lse[geo.off[2] * H + 7] += 1e-3
        ops["o", i], ops["lse", i] = o.bfloat16(), lse.float()
        if fault == "last_mask" and i == LAYERS - 1:  # (the saved o is right: the rows the pruned block gathers are not)
            o = _attention(qkv, geo, False)[0]
        xm = (x.double() + o.bfloat16().double() @ _bf(w["attn.out_proj.weight"]).t() + w["attn.out_proj.bias"].double()).float()
        ops["x_mid", i] = xm
        g2 = tw["blocks"][0]["ln_2.weight"] if (fault == "ln2_gamma" and i == 1) else w["ln_2.weight"]
        a = _bf(F.layer_norm(xm.double(), (D,), g2.double(), w["ln_2.bias"].double(), ts.LN_EPS))
        h = a @ _bf(w["mlp.c_fc.weight"]).t() + w["mlp.c_fc.bias"].double()
        ops["h", i] = h.bfloat16()
        bias = w["mlp.c_proj.bias"].double().expand(rows, D).clone()
        if fault == "bias_tail" and i == 0:
            bias[128:] = 0
        x = (xm.double() + _bf(ts.quick_gelu(h)) @ _bf(w["mlp.c_proj.weight"]).t() + bias).float()
    ops["x_in", LAYERS] = x
    feats = F.layer_norm(x[geo.sel].double(), (D,), tw["ln_g"].double(), tw["ln_b"].double(), ts.LN_EPS) @ tw["proj"].double()
    return ops, feats.float()


def check(tw, ops, feats, geo=GEO, fused=False, pruned=False):
    return ts.check_tower(lambda name, i: ops[name, i], lambda i: tw["blocks"][i], LAYERS, geo, tw["prompts"], fused, pruned,
                          feats, tw["ln_g"], tw["ln_b"], tw["proj"])


def _cos(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float(a @ b / (a.norm() * b.norm()))


def test_correct_tower_passes_every_stage(tower):
    rep = check(tower, *run(tower))
    assert rep.failures() == [], rep.table("correct tower")
    assert set(rep.worst()) == {"splice", "ln1_qkv", "attn", "lse", "out_proj", "ln2_fc", "c_proj", "head"}
    # the bf16 roundings are visible to the checks (not an fp64 identity), well inside the bounds
    assert 0.05 < rep.worst()["ln1_qkv"][0] < 0.9, rep.table("correct tower")


def test_c_proj_bias_lost_on_the_partial_tile(tower):
    """Rejected at layer 0, c_proj, on the tile of rows 128..149; the whole-model feature cosine accepts it."""
    ops, feats = run(tower, "bias_tail")
    first = check(tower, ops, feats).failures()[0]
    assert first[:2] == (0, "c_proj") and first[3][0] == 128 and first[2] > 5, first
    _, good = run(tower)
    assert _cos(feats, good) >= 0.999


def test_deep_prompt_spliced_one_layer_late(tower):
    first = check(tower, *run(tower, "splice_late")).failures()[0]
    assert first[:2] == (0, "splice") and first[3] == (0,), first


def test_ln2_with_another_layers_gamma(tower):
    fails = check(tower, *run(tower, "ln2_gamma")).failures()
    assert fails and fails[0][:2] == (1, "ln2_fc"), fails
    assert {(f[0], f[1]) for f in fails} == {(1, "ln2_fc")}, fails  # teacher forcing: nothing downstream is blamed


def test_report_names_unwritten_blocks():
    """A NaN (unwritten) element fails its block with an infinite ratio."""
    ref = torch.randn(300, 256, dtype=torch.float64)
    out = ref.bfloat16()
    out[260, 200] = float("nan")
    r, blk = ts.gemm_tiles(out, ref)
    assert r == float("inf") and blk == (256, 128)


@pytest.mark.parametrize("fused", [False, True])
def test_ragged_pruned_tower(tower, fused):
    """The paths only the native towers reach otherwise: packed causal rows with per-class lse, the pruned last block on
    the EOT rows, the fused-LayerNorm bound.  The correct tower passes; a last block whose EOT queries see the keys after
    them fails last_block on a sequence whose EOT is not its last row; one wrong lse entry of sequence 2 fails lse there;
    an LN1 with another layer's gamma fails ln1_qkv under either bound; an LN2 with another layer's gamma in the pruned
    last block fails last_block."""
    rep = check(tower, *run(tower, geo=RAGGED), RAGGED, fused, True)
    assert rep.failures() == [], rep.table("ragged, pruned")
    assert set(rep.worst()) == {"splice", "ln1_qkv", "attn", "lse", "out_proj", "ln2_fc", "c_proj", "last_block"}
    first = check(tower, *run(tower, "last_mask", RAGGED), RAGGED, fused, True).failures()[0]
    assert first[:2] == (LAYERS - 1, "last_block") and first[3][0] in (0, 1, 2), first
    first = check(tower, *run(tower, "lse_seq2", RAGGED), RAGGED, fused, True).failures()[0]
    assert first[:3] == (0, "lse", first[2]) and first[3][0] == 2 and first[2] > 5, first
    first = check(tower, *run(tower, "ln1_gamma", RAGGED), RAGGED, fused, True).failures()[0]
    assert first[:2] == (0, "ln1_qkv"), first
    first = check(tower, *run(tower, "ln2_gamma", RAGGED), RAGGED, fused, True).failures()[0]
    assert first[:2] == (1, "last_block"), first
