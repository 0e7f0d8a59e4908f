"""Pin the CPU oracle to the reference through golden vectors made by tests/golden/make_golden.py."""
import pytest
import torch

from oracle import separator_oracle as O
from sepreformer_b200.configs import MODEL_SHAPES

from _util import check_generator_stable, load_golden, model_state, rel_l2, seeded_input

SEP_CASES = ["sep_base_small", "sep_base_exact16", "sep_base_medium", "sep_large_whamr_small", "sep_large_wham_small",
             "sep_large_medium"]


def _run_oracle(gold, dtype):
    name = str(gold["model"])
    shape = MODEL_SHAPES[name]
    sd = model_state(name, int(gold["wseed"]))
    x = seeded_input(int(gold["xseed"]), int(gold["batch"]), shape.feat, int(gold["t_enc"]))
    check_generator_stable(gold, sd, x)
    p = {k: v.to(dtype) for k, v in sd.items() if v.is_floating_point()}
    with torch.no_grad():
        return O.separator_forward(x.to(dtype), p, heads=shape.heads, num_stages=shape.num_stages,
                                   num_spks=shape.num_spks, maxlen=shape.maxlen,
                                   per_stage_split=shape.per_stage_split)


@pytest.mark.parametrize("tag", SEP_CASES)
def test_separator_oracle_matches_reference_golden_fp64(tag):
    if tag in ("sep_base_medium", "sep_large_medium"):
        pytest.skip("covered in fp32 below (fp64 at T=2000 takes a while)")
    gold = load_golden(tag)
    last, stages = _run_oracle(gold, torch.float64)
    st = int(gold["stride"])
    # golden was stored as float32 of the reference's fp64 output -> agreement limited by that rounding
    assert rel_l2(last[..., ::st], gold["last"]) < 1e-7
    for i, s in enumerate(stages):
        assert rel_l2(s[..., ::st], gold[f"stage{i}"]) < 1e-7
    assert abs(float(last.norm()) - float(gold["last_norm"])) < 1e-9 * float(gold["last_norm"])


@pytest.mark.parametrize("tag", SEP_CASES)
def test_separator_oracle_fp32_close_to_golden(tag):
    gold = load_golden(tag)
    last, stages = _run_oracle(gold, torch.float32)
    st = int(gold["stride"])
    assert last.shape[-1] % 16 == 0
    assert rel_l2(last[..., ::st], gold["last"]) < 2e-5
    for i, s in enumerate(stages):
        assert rel_l2(s[..., ::st], gold[f"stage{i}"]) < 2e-5


@pytest.mark.parametrize("tag,model", [("blocks_base", "SepReformer_Base_WSJ0"), ("blocks_large", "SepReformer_Large_DM_WSJ0")])
def test_block_oracles_match_reference_golden(tag, model):
    gold = load_golden(tag)
    shape = MODEL_SHAPES[model]
    p = {k: v.double() for k, v in model_state(model, int(gold["wseed"])).items() if v.is_floating_point()}
    b, td, t, f = int(gold["batch"]), int(gold["td"]), int(gold["t"]), shape.feat
    x = seeded_input(int(gold["xseed"]), b * 2, t, f).double()
    pe = p["pos_emb.pe_k.weight"]
    h, ml = shape.heads, shape.maxlen
    got = {
        "gcfn": O.gcfn(x, p, "dec_stages.1.g_block_2.block.gcfn."),
        "cla": O.cla(x, p, "dec_stages.1.l_block_1.block.cla."),
        "ega": O.ega(x, p, "dec_stages.1.g_block_3.block.ega.", h, td, pe, ml),
        "global": O.global_block(x, p, "enc_stages.2.g_block_1.", h, td, pe, ml),
        "local": O.local_block(x, p, "enc_stages.2.l_block_2."),
        "spkattn": O.spk_attention(x, p, "dec_stages.1.spk_attn_1.", h, 2),
        "downconv": O.down_conv(x, p, "enc_stages.2.downconv."),
        "spksplit": O.spk_split(x[:b], p, "spk_split_block.", 2),
        "fusion": O.fuse(seeded_input(int(gold["xseed"]) + 1, b * 2, t // 2, f).double(), x, p, "simple_fusion.2."),
    }
    for k, v in got.items():
        assert v.shape == gold[k].shape, k
        assert rel_l2(v, gold[k]) < 1e-7, k


def test_fast_conv_equals_definition():
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 50, 8, generator=g, dtype=torch.float64)
    for k, pad, stride in ((3, 1, 1), (65, 32, 1), (5, 2, 2)):
        w = torch.randn(8, 1, k, generator=g, dtype=torch.float64)
        b = torch.randn(8, generator=g, dtype=torch.float64)
        a = O.dwconv_time(x, w, b, pad, stride, fast=False)
        c = O.dwconv_time(x, w, b, pad, stride, fast=True)
        assert a.shape == c.shape and rel_l2(a, c) < 1e-12


def test_pad_quirk_no_pad_when_multiple():
    x = torch.zeros(1, 96, 4)
    assert O.pad_frames(x, 16).shape[1] == 96
    assert O.pad_frames(torch.zeros(1, 97, 4), 16).shape[1] == 112


def test_pit_sisnri_permutation_invariant():
    g = torch.Generator().manual_seed(0)
    s1, s2 = torch.randn(3, 4000, generator=g), torch.randn(3, 4000, generator=g)
    mix = s1 + s2
    e1 = s1 + 0.1 * torch.randn(3, 4000, generator=g)
    e2 = s2 + 0.1 * torch.randn(3, 4000, generator=g)
    a = O.pit_si_snri([e1, e2], [s1, s2], mix)
    b = O.pit_si_snri([e2, e1], [s1, s2], mix)
    assert torch.allclose(a, b) and float(a.min()) > 15.0


def test_oracle_matches_live_reference():
    """The reference Separator's fp64 output, stored in fp64: agreement to 1e-12, not just float32 rounding."""
    gold = load_golden("sep_base_fp64")
    st = int(gold["stride"])
    sd = model_state("SepReformer_Base_WSJ0", 7)
    x = seeded_input(5, 1, 128, 203).double()
    with torch.no_grad():
        yo, so = O.separator_forward(x, {k: v.double() for k, v in sd.items() if v.is_floating_point()})
    assert len(so) == sum(k.startswith("stage") and not k.endswith("_norm") for k in gold)
    for key, t in [("last", yo)] + [(f"stage{i}", s) for i, s in enumerate(so)]:
        assert t[..., ::st].shape == gold[key].shape, key
        assert rel_l2(t[..., ::st], gold[key]) < 1e-12, key
        assert abs(float(t.norm()) - float(gold[key + "_norm"])) < 1e-12 * float(gold[key + "_norm"]), key
