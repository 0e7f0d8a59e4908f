"""Generate the golden vectors under tests/golden/ by running the *reference itself*.

Needs a checkout of the original SepReformer project (github.com/dmlguq456/SepReformer), found as
oracle/install_reference.py finds it (``SEPREFORMER_REFERENCE``, else ``/root/reference``); the tests only read what
this writes:

    python tests/golden/make_golden.py [case ...]

For every case the reference ``Separator`` (or one of its block classes) is instantiated from the
reference's own configs.yaml, loaded (strict) with ``sepreformer_b200.params.seeded_state(seed)`` -
weights that any machine can regenerate from the seed - and run in fp64 on a seeded input; the fp64
output is stored as float32.  A few weight/input checksums are stored too so that a silent change of
the random generator would be detected rather than misread as a parity failure.
"""
import importlib
import os
import sys

import numpy as np
import torch
import yaml

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle.install_reference import SRC as REF  # noqa: E402
sys.path.insert(0, REF)

from loguru import logger  # noqa: E402

logger.remove()

from sepreformer_b200.configs import MODEL_SHAPES  # noqa: E402
from sepreformer_b200.params import ParamTree, separator_spec, seeded_state, state_shapes  # noqa: E402


def seeded_input(seed, *shape):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


def checksums(sd):
    keys = sorted(k for k in sd if not k.endswith("num_batches_tracked"))
    picks = [keys[0], keys[len(keys) // 3], keys[2 * len(keys) // 3], keys[-1]]
    return np.array([float(sd[k].double().abs().sum()) for k in picks]), np.array(picks)


def ref_separator(model_name):
    mod = importlib.import_module(f"models.{model_name}.modules.module")
    cfg = yaml.full_load(open(os.path.join(REF, "models", model_name, "configs.yaml")))["config"]["model"]["module_separator"]
    return mod.Separator(**cfg).eval(), mod


def separator_case(tag, model_name, batch, t_enc, wseed, xseed, stride=1):
    shape = MODEL_SHAPES[model_name]
    ref, _ = ref_separator(model_name)
    sd = seeded_state(state_shapes(ParamTree(separator_spec(shape))), seed=wseed)
    ref.load_state_dict(sd, strict=True)
    ref = ref.double()
    x = seeded_input(xseed, batch, shape.feat, t_enc)
    with torch.no_grad():
        last, stages = ref(x.double())
    wsum, wkeys = checksums(sd)
    out = dict(model=np.array(model_name), batch=batch, t_enc=t_enc, wseed=wseed, xseed=xseed, stride=stride,
               wsum=wsum, wkeys=wkeys, xsum=float(x.double().abs().sum()),
               last=last[..., ::stride].float().numpy(),
               last_norm=float(last.norm()))
    for i, s in enumerate(stages):
        out[f"stage{i}"] = s[..., ::stride].float().numpy()
        out[f"stage{i}_norm"] = float(s.norm())
    np.savez_compressed(os.path.join(HERE, tag + ".npz"), **out)
    print(tag, last.shape, float(last.norm()))


def block_cases(tag, model_name, wseed, xseed, batch=2, td=3):
    """One call of each reference block class on channels-last input; prefixes name the weights used."""
    shape = MODEL_SHAPES[model_name]
    ref, mod = ref_separator(model_name)
    sd = seeded_state(state_shapes(ParamTree(separator_spec(shape))), seed=wseed)
    ref.load_state_dict(sd, strict=True)
    ref = ref.double()
    f, r = shape.feat, 4
    t = td * r
    x = seeded_input(xseed, batch * 2, t, f).double()          # [B*S, T, F] channels-last
    pos = torch.arange(td)
    pos_k, _ = ref.pos_emb((pos[:, None] - pos[None, :]).long())
    out = dict(model=np.array(model_name), wseed=wseed, xseed=xseed, batch=batch, td=td, t=t)
    with torch.no_grad():
        dec = ref.dec_stages[1]
        enc = ref.enc_stages[2]
        out["gcfn"] = dec.g_block_2.block["gcfn"](x).float().numpy()                      # dec_stages.1.g_block_2.block.gcfn.
        out["cla"] = dec.l_block_1.block["cla"](x).float().numpy()                        # dec_stages.1.l_block_1.block.cla.
        out["ega"] = dec.g_block_3.block["ega"](x.transpose(1, 2), pos_k).float().numpy()  # dec_stages.1.g_block_3.block.ega.
        out["global"] = enc.g_block_1(x.transpose(1, 2), pos_k).transpose(1, 2).float().numpy()   # enc_stages.2.g_block_1.
        out["local"] = enc.l_block_2(x).float().numpy()                                    # enc_stages.2.l_block_2.
        out["spkattn"] = dec.spk_attn_1(x.transpose(1, 2), 2).transpose(1, 2).float().numpy()     # dec_stages.1.spk_attn_1.
        out["downconv"] = enc.downconv(x).float().numpy()                                  # enc_stages.2.downconv.
        split = ref.spk_split_blocks[1] if shape.per_stage_split else ref.spk_split_block
        out["spksplit"] = split(x[:batch].transpose(1, 2)).transpose(1, 2).float().numpy()
        low = seeded_input(xseed + 1, batch * 2, t // 2, f).double()
        up = torch.nn.functional.interpolate(low.transpose(1, 2), size=t)
        out["fusion"] = ref.simple_fusion[2](torch.cat([up, x.transpose(1, 2)], 1)).transpose(1, 2).float().numpy()
    np.savez_compressed(os.path.join(HERE, tag + ".npz"), **out)
    print(tag, {k: v.shape for k, v in out.items() if hasattr(v, "shape") and v.ndim > 1})


def _ref_model(model_name):
    cfg = yaml.full_load(open(os.path.join(REF, "models", model_name, "configs.yaml")))["config"]["model"]
    return importlib.import_module(f"models.{model_name}.model").Model, cfg


def _strided(out, key, t, stride, dtype):
    out[key] = t[..., ::stride].to(dtype).numpy()
    out[key + "_norm"] = float(t.double().norm())


def model_shell_case(tag, stride=4):
    """tests/test_model_shell.py: the reference Model in fp64 with the oracle's seeded shell weights."""
    from _util import model_state, seeded_input
    from test_model_shell import shell_state
    Model, cfg = _ref_model("SepReformer_Base_WSJ0")
    ref = Model(**cfg).eval()
    ref.separator.load_state_dict(model_state("SepReformer_Base_WSJ0", 7), strict=True)
    missing, unexpected = ref.load_state_dict(shell_state(), strict=False)
    assert not unexpected and all(not k.startswith(("audio_encoder", "feature_projector", "out_layer.", "audio_decoder")) for k in missing)
    ref = ref.double()
    mix = 0.1 * seeded_input(9, 2, 4000).double()
    with torch.no_grad():
        audio, _ = ref(mix)
    out = dict(stride=stride)
    for s, a in enumerate(audio):
        _strided(out, f"audio{s}", a, stride, torch.float64)
    np.savez_compressed(os.path.join(HERE, tag + ".npz"), **out)
    print(tag, [a.shape for a in audio])


def pit_criterion_case(tag):
    """tests/test_model_shell.py: the reference's PIT_SISNRi (utils/implements/criterions.py) on three seeded trials;
    the two packages it imports but this path never touches are stubbed."""
    import types
    for missing in ("mir_eval", "mir_eval.separation", "torchaudio", "torchaudio.transforms"):
        if missing not in sys.modules:
            try:
                __import__(missing)
            except Exception:
                mod = types.ModuleType(missing)
                mod.bss_eval_sources = None
                mod.MelScale = object
                sys.modules[missing] = mod
    from utils.implements.criterions import PIT_SISNRi
    from test_model_shell import pit_trials
    crit = PIT_SISNRi(device=torch.device("cpu"), num_spks=2, scale_inv=True)
    vals = []
    for e, (s1, s2), mix in pit_trials():
        v, _ = crit(estims=e, mixture=mix, input_sizes=torch.tensor([mix.shape[-1]]), target_attr=[s1, s2], eps=1.0e-15)
        vals.append(float(v))
    np.savez_compressed(os.path.join(HERE, tag + ".npz"), pit_sisnri=np.array(vals))
    print(tag, vals)


def separator_fp64_case(tag, stride=8):
    """tests/test_oracle_golden.py: the reference Separator in fp64, stored in fp64 (compared at 1e-12)."""
    from _util import model_state
    ref, _ = ref_separator("SepReformer_Base_WSJ0")
    ref.load_state_dict(model_state("SepReformer_Base_WSJ0", 7), strict=True)
    ref = ref.double()
    x = seeded_input(5, 1, 128, 203).double()
    with torch.no_grad():
        last, stages = ref(x)
    out = dict(stride=stride)
    _strided(out, "last", last, stride, torch.float64)
    for i, s in enumerate(stages):
        _strided(out, f"stage{i}", s, stride, torch.float64)
    np.savez_compressed(os.path.join(HERE, tag + ".npz"), **out)
    print(tag, last.shape, [s.shape for s in stages])


def model_level_case(tag, model_name="SepReformer_Base_WSJ0", stride=16):
    """tests/test_model_gpu.py: the stock reference Model in fp32 with every entry of its state_dict seeded
    (``seeded_state`` in state_dict order), on the seeded mixtures of that test; audio and the four auxiliary heads."""
    import json
    from test_model_gpu import mixtures
    Model, cfg = _ref_model(model_name)
    ref = Model(**cfg).eval()
    ref.load_state_dict(seeded_state(state_shapes(ref), seed=1), strict=True)
    mix, _, _ = mixtures(2, 8000)
    with torch.inference_mode():
        audio, aux = ref(mix)
    out = dict(model=np.array(model_name), cfg=np.array(json.dumps(cfg)), keys=np.array(list(ref.state_dict())), stride=stride)
    for s, a in enumerate(audio):
        _strided(out, f"audio{s}", a, stride, torch.float32)
    for i, heads in enumerate(aux):
        for s, a in enumerate(heads):
            _strided(out, f"aux{i}_{s}", a, stride, torch.float32)
    np.savez_compressed(os.path.join(HERE, tag + ".npz"), **out)
    print(tag, audio[0].shape, len(aux))


if __name__ == "__main__":
    sys.path.insert(0, os.path.dirname(HERE))      # the tests' helpers, for the cases that mirror a test
    only = set(sys.argv[1:])        # optional: regenerate just the named cases

    def separator_case(tag, *a, _f=separator_case, **k):      # noqa: F811
        if not only or tag in only:
            _f(tag, *a, **k)

    def block_cases(tag, *a, _f=block_cases, **k):            # noqa: F811
        if not only or tag in only:
            _f(tag, *a, **k)

    separator_case("sep_base_small", "SepReformer_Base_WSJ0", batch=2, t_enc=157, wseed=1, xseed=11)
    separator_case("sep_base_exact16", "SepReformer_Base_WSJ0", batch=1, t_enc=96, wseed=2, xseed=12)
    separator_case("sep_base_medium", "SepReformer_Base_WSJ0", batch=1, t_enc=1997, wseed=1, xseed=13, stride=8)
    separator_case("sep_large_whamr_small", "SepReformer_Large_DM_WHAMR", batch=1, t_enc=150, wseed=3, xseed=14)
    separator_case("sep_large_wham_small", "SepReformer_Large_DM_WHAM", batch=2, t_enc=79, wseed=4, xseed=15)
    # F = 256 at a length where every persistent kernel walks several tiles per CTA at the full-rate stages
    separator_case("sep_large_medium", "SepReformer_Large_DM_WSJ0", batch=1, t_enc=2003, wseed=5, xseed=16, stride=8)
    block_cases("blocks_base", "SepReformer_Base_WSJ0", wseed=1, xseed=21)
    block_cases("blocks_large", "SepReformer_Large_DM_WSJ0", wseed=5, xseed=22)
    for tag, case in (("model_shell_base", model_shell_case), ("pit_criterion", pit_criterion_case),
                      ("sep_base_fp64", separator_fp64_case), ("model_base", model_level_case)):
        if not only or tag in only:
            case(tag)
