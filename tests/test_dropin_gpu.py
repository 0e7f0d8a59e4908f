"""The north-star drop-in claim exercised end to end on the GPU (VERDICT r1 row J1): the reference's own ``Model``
(model.py:27,41) built after ``sepreformer_b200.install()`` runs on the B200 and agrees with the stock reference
``Model`` on the CPU - directly and under ``torch.nn.parallel.data_parallel`` as engine.py:165-167 calls it.

Needs the runnable copy of the reference's model files (``oracle/_ref``, made by ``build()`` from a checkout of the
original project; git-ignored): ``install()`` patches the reference's own ``Model`` code."""
import pytest
import torch

import sepreformer_b200
from sepreformer_b200.params import seeded_state, state_shapes

from _util import REF_DIR, reference_model_config, reference_model_module, rel_l2

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(REF_DIR is None, reason="no oracle/_ref: build() found no checkout of the original project")]

NAME = "SepReformer_Base_WSJ0"


def _models():
    mm = reference_model_module(NAME)
    cfg = reference_model_config(NAME)
    stock_sep = mm.Separator
    torch.manual_seed(0)
    ref = mm.Model(**cfg).eval()
    # non-trivial separator weights (default LayerScale 1e-5 would hide every block), stock init for the shell
    ref.separator.load_state_dict(seeded_state(state_shapes(ref.separator), seed=1), strict=True)
    try:
        sepreformer_b200.install(mm)
        ours = mm.Model(**cfg).eval()
    finally:
        mm.Separator = stock_sep
    assert isinstance(ours.separator, sepreformer_b200.Separator)
    missing, unexpected = ours.load_state_dict(ref.state_dict(), strict=True)
    assert not missing and not unexpected
    assert list(ours.state_dict().keys()) == list(ref.state_dict().keys())
    return ref, ours


def _mix(b, n=8000, seed=5):
    g = torch.Generator().manual_seed(seed)
    return 0.05 * torch.randn(b, n, generator=g) + 0.05 * torch.randn(b, n, generator=g)


def test_reference_model_with_installed_separator_matches_stock_reference():
    ref, ours = _models()
    mix = _mix(2)
    ours = ours.cuda()
    with torch.inference_mode():
        want, want_aux = ref(mix)
        got, got_aux = ours(mix.cuda())
    for s in range(2):
        err = rel_l2(got[s].cpu(), want[s])
        print(f"speaker {s}: model output rel-L2 {err:.2e}")
        assert err < 1e-3
    for a, b in zip(got_aux, want_aux):          # the four auxiliary heads consume the per-stage outputs
        assert rel_l2(a[0].cpu(), b[0]) < 1e-3
    # the drop-in separator refuses the training path instead of silently skipping gradients (engine.py:64)
    ours.train()
    with torch.no_grad(), pytest.raises(RuntimeError, match="inference-only"):
        ours(mix.cuda())


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_data_parallel_two_devices_packs_once_per_device():
    ref, ours = _models()
    ours = ours.cuda(0)
    mix = _mix(4)
    sh = ours.separator._sh()
    with torch.inference_mode():
        want, _ = ref(mix)
        packs = []
        for _ in range(3):
            got, _ = torch.nn.parallel.data_parallel(ours, mix.cuda(0), device_ids=[0, 1])
            packs.append(sh.packs)
    assert sorted(sh.handles) == [0, 1]
    assert packs[0] == 2 and packs[1] == 2 and packs[2] == 2, packs       # one pack per device, none afterwards
    for s in range(2):
        assert rel_l2(got[s].cpu(), want[s]) < 1e-3
