"""The model-shell restatement used for the SI-SNRi metric is pinned to the reference Model (golden vectors made by
tests/golden/make_golden.py from the original project)."""
import torch

from oracle import separator_oracle as O

from _util import load_golden, model_state, rel_l2, seeded_input


def shell_state(feat=128, seed=3):
    g = torch.Generator().manual_seed(seed)
    u = lambda *s: (torch.rand(*s, generator=g) * 2 - 1)
    return {
        "audio_encoder.conv1d.weight": u(256, 1, 16) / 4.0,
        "feature_projector.norm.weight": 1 + 0.1 * u(256), "feature_projector.norm.bias": 0.1 * u(256),
        "feature_projector.conv1d.weight": u(feat, 256, 1) / 16.0,
        "out_layer.end_conv1x1.0.weight": u(4 * feat, feat) / feat ** 0.5, "out_layer.end_conv1x1.0.bias": 0.1 * u(4 * feat),
        "out_layer.end_conv1x1.2.weight": u(256, 2 * feat) / (2 * feat) ** 0.5, "out_layer.end_conv1x1.2.bias": 0.1 * u(256),
        "audio_decoder.weight": u(256, 1, 16) / 16.0,
    }


def test_shell_matches_reference_model():
    gold = load_golden("model_shell_base")
    st = int(gold["stride"])
    shell = shell_state()
    ref_keys = [str(k) for k in load_golden("model_base")["keys"]]        # the reference Model's state_dict keys
    missing = set(ref_keys) - set(shell)
    assert set(shell) <= set(ref_keys)
    assert all(not k.startswith(("audio_encoder", "feature_projector", "out_layer.", "audio_decoder")) for k in missing)
    sd = model_state("SepReformer_Base_WSJ0", 7)
    mix = 0.1 * seeded_input(9, 2, 4000).double()
    with torch.no_grad():
        p64 = {k: v.double() for k, v in sd.items() if v.is_floating_point()}
        shell64 = {k: v.double() for k, v in shell.items()}
        audio = O.model_forward(mix, shell64, lambda f: O.separator_forward(f, p64)[0])
    for s, a in enumerate(audio):
        b = gold[f"audio{s}"]
        assert a[..., ::st].shape == b.shape
        assert rel_l2(a[..., ::st], b) < 1e-10
        assert abs(float(a.norm()) - float(gold[f"audio{s}_norm"])) < 1e-10 * float(gold[f"audio{s}_norm"])


def test_si_snri_of_perfect_estimate_is_large():
    g = torch.Generator().manual_seed(1)
    s1, s2 = torch.randn(2, 8000, generator=g), torch.randn(2, 8000, generator=g)
    v = O.pit_si_snri([s2 + 1e-3 * s1, s1 + 1e-3 * s2], [s1, s2], s1 + s2)      # swapped order: PIT must find it
    assert float(v.min()) > 40.0


def pit_trials():
    """Three seeded (estimates, targets, mixture) trials; the last lists the estimates in the other speaker order."""
    g = torch.Generator().manual_seed(4)
    for trial in range(3):
        n = 4000 + 37 * trial
        s1, s2 = torch.randn(1, n, generator=g), torch.randn(1, n, generator=g)
        e = [s2 + 0.3 * torch.randn(1, n, generator=g), s1 + 0.1 * torch.randn(1, n, generator=g)]
        yield (e[::-1] if trial == 2 else e), (s1, s2), s1 + s2


def test_oracle_pit_si_snri_matches_reference_criterion():
    """oracle.pit_si_snri (the checker of the device-side metric kernel) against the reference's own PIT_SISNRi
    (utils/implements/criterions.py:221-260) on the same trials."""
    want = load_golden("pit_criterion")["pit_sisnri"]
    trials = list(pit_trials())
    assert len(trials) == len(want)
    for (e, tgt, mix), ref_val in zip(trials, want):
        got = O.pit_si_snri(e, list(tgt), mix)            # already divided by num_spks (engine.py:132)
        assert abs(float(ref_val) / 2 - float(got)) < 1e-4
