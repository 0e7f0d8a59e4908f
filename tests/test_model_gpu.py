"""The model-level path (SURVEY.md 8f rows n1-n4): waveform -> AudioEncoder/FeatureProjector -> separator -> OutputLayer ->
AudioDecoder -> waveforms in ONE C-ABI call (sepref_model_forward), against the CPU oracle's model shell (pinned to the
reference Model in test_model_shell.py), the reference Model itself through golden vectors, and the device-side
batched PIT SI-SNRi against the oracle's restatement of criterions.py:221-260."""
import pytest
import torch

import sepreformer_b200
from oracle import separator_oracle as O
from sepreformer_b200 import MODEL_SHAPES, separator_kwargs
from sepreformer_b200.params import seeded_state, state_shapes

from _util import load_golden, rel_l2

pytestmark = pytest.mark.gpu

_cache = {}


def model_kwargs(name):
    shape = MODEL_SHAPES[name]
    f = shape.feat
    return dict(num_stages=shape.num_stages, num_spks=shape.num_spks,
                module_audio_enc=dict(in_channels=1, out_channels=256, kernel_size=16, stride=4, groups=1, bias=False),
                module_feature_projector=dict(num_channels=256, in_channels=256, out_channels=f, kernel_size=1, bias=False),
                module_separator=separator_kwargs(shape),
                module_output_layer=dict(in_channels=256, out_channels=f, num_spks=shape.num_spks),
                module_audio_dec=dict(in_channels=256, out_channels=1, kernel_size=16, stride=4, bias=False))


def gpu_model(name):
    if name not in _cache:
        _cache.clear()
        shape = MODEL_SHAPES[name]
        torch.manual_seed(3)
        m = sepreformer_b200.Model(**model_kwargs(name), per_stage_split=shape.per_stage_split)      # stock torch init for the shell
        m.separator.load_state_dict(seeded_state(state_shapes(m.separator), seed=1), strict=True)
        with torch.no_grad():                                                                         # non-trivial GroupNorm affine
            m.feature_projector.norm.weight.add_(0.1 * torch.randn(256))
            m.feature_projector.norm.bias.add_(0.1 * torch.randn(256))
        _cache[name] = m.cuda().eval()
    return _cache[name]


def mixtures(b, n, seed=5):
    g = torch.Generator().manual_seed(seed)
    s1, s2 = 0.05 * torch.randn(b, n, generator=g), 0.05 * torch.randn(b, n, generator=g)
    return s1 + s2, s1, s2


def oracle_audio(m, mix):
    sd = {k: v.detach().cpu() for k, v in m.state_dict().items() if v.is_floating_point()}
    sep = {k[len("separator."):]: v for k, v in sd.items() if k.startswith("separator.")}
    s = m.separator.shape_
    kw = dict(heads=s.heads, num_stages=s.num_stages, num_spks=s.num_spks, maxlen=s.maxlen, per_stage_split=s.per_stage_split, fast=True)
    with torch.no_grad():
        return O.model_forward(mix, sd, lambda f: O.separator_forward(f, sep, **kw)[0])


@pytest.mark.parametrize("path", [1, 2])
@pytest.mark.parametrize("name,b,n", [("SepReformer_Base_WSJ0", 2, 8000), ("SepReformer_Base_WSJ0", 3, 5002),
                                      ("SepReformer_Large_DM_WSJ0", 1, 4000)])
def test_model_forward_matches_oracle(name, b, n, path):
    m = gpu_model(name)
    m.separator.gemm_path = path
    m.compute_aux = False
    mix, _, _ = mixtures(b, n)
    want = oracle_audio(m, mix)
    with torch.inference_mode():
        got, aux = m(mix.cuda())
    assert aux == [] and len(got) == 2
    for s in range(2):
        assert got[s].shape == want[s].shape == (b, ((n - 16) // 4) * 4 + 16)
        err = rel_l2(got[s].cpu(), want[s])
        print(f"{name} B={b} n={n} path={path} speaker {s}: audio rel-L2 {err:.2e}")
        assert err < 1e-3


def test_model_host_requests_equal_device_call():
    m = gpu_model("SepReformer_Base_WSJ0")
    m.separator.gemm_path = 2
    m.compute_aux = False
    mixes = [mixtures(2 + (i & 1), 6000 + 400 * i, seed=20 + i)[0] for i in range(4)]
    with torch.inference_mode():
        want = [torch.stack(m(x.cuda())[0]).cpu() for x in mixes]
        got = [None] * len(mixes)
        for i, x in enumerate(mixes):
            if i >= 2:
                got[i - 2] = m.wait_host(i & 1).clone()
            m.submit_host(x.pin_memory(), i & 1)
        for i in range(len(mixes) - 2, len(mixes)):
            got[i] = m.wait_host(i & 1).clone()
    for a, b in zip(want, got):
        assert torch.equal(a, b)


def test_device_pit_si_snri_matches_oracle():
    m = gpu_model("SepReformer_Base_WSJ0")
    g = torch.Generator().manual_seed(9)
    b, n = 5, 8000
    s1, s2 = torch.randn(b, n, generator=g), torch.randn(b, n, generator=g)
    mix = s1 + s2
    e1 = s1 + 0.1 * torch.randn(b, n, generator=g) + 0.3          # offsets: the metric removes means
    e2 = s2 + 0.2 * torch.randn(b, n, generator=g)
    est = torch.stack([e2, e1])                                   # swapped: PIT must pick the other permutation
    est[:, 3] = torch.stack([e1[3], e2[3]])                       # ... except for utterance 3
    pad = torch.zeros(2, b, 12)
    want = O.pit_si_snri([est[0], est[1]], [s1, s2], mix)
    got = m.pit_si_snri(torch.cat([est, pad], -1).cuda(), torch.stack([s1, s2]).cuda(), mix.cuda()).cpu()
    assert got.shape == (b, 3)
    assert torch.allclose(got[:, 0] / 2, want, atol=2e-4), (got[:, 0] / 2, want)
    assert torch.allclose(got[:, 1] + got[:, 2], got[:, 0], atol=1e-4)


def test_si_snri_delta_through_the_model_path():
    """North-star metric on the whole GPU path: |SI-SNRi(ours) - SI-SNRi(oracle)| <= 0.05 dB."""
    m = gpu_model("SepReformer_Base_WSJ0")
    m.separator.gemm_path = 2
    m.compute_aux = False
    mix, s1, s2 = mixtures(3, 8000, seed=77)
    want = oracle_audio(m, mix)
    n = mix.shape[-1]
    a = O.pit_si_snri([e[..., :n] for e in want], [s1, s2], mix)
    with torch.inference_mode():
        got, _ = m(mix.cuda())
        dev = m.pit_si_snri(torch.stack(got), torch.stack([s1, s2]).cuda(), mix.cuda()).cpu()[:, 0] / 2
    delta = float((a - dev).abs().max())
    print(f"SI-SNRi oracle {a.tolist()} device path {dev.tolist()} delta {delta:.5f} dB")
    assert delta <= 0.05


def test_model_level_install_matches_reference_model_including_aux_heads():
    """install(level="model") against the stock reference Model (tests/golden/make_golden.py): same state_dict keys in
    the same order, and the same audio and auxiliary-head outputs on the same seeded weights and mixtures."""
    import json
    import types
    gold = load_golden("model_base")
    st = int(gold["stride"])
    cfg = json.loads(str(gold["cfg"]))
    mm = sepreformer_b200.install(types.ModuleType("model"), level="model")
    ours = mm.Model(**cfg)
    assert isinstance(ours, sepreformer_b200.Model)
    assert list(ours.state_dict()) == [str(k) for k in gold["keys"]]
    sd = seeded_state(state_shapes(ours), seed=1)
    ours = ours.cuda().eval()
    ours.load_state_dict(sd, strict=True)          # AFTER .cuda(): the load hook must re-pack the weights
    mix, _, _ = mixtures(2, 8000)
    with torch.inference_mode():
        got, got_aux = ours(mix.cuda())
    for s in range(2):
        err = rel_l2(got[s].cpu()[..., ::st], gold[f"audio{s}"])
        print(f"model-level install, speaker {s}: rel-L2 {err:.2e}")
        assert got[s].shape[-1] == mix.shape[-1] and err < 1e-3
    assert len(got_aux) == 4
    for i, heads in enumerate(got_aux):
        for s in range(2):
            want = gold[f"aux{i}_{s}"]
            assert heads[s][..., ::st].shape == want.shape and rel_l2(heads[s].cpu()[..., ::st], want) < 1e-3


def test_cuda_graph_replay_is_bit_identical_and_cheap_to_enqueue():
    """SEPREF_OPT_CUDA_GRAPH (VERDICT r1 weak #8): the second call of a shape captures, later calls replay one graph
    launch; results equal the eager launches bit for bit; the host side of a B = 1, 4 s forward drops below 0.3 ms."""
    import time
    from sepreformer_b200 import _lib
    m = gpu_model("SepReformer_Base_WSJ0")
    sep = m.separator
    sep.gemm_path = 2
    sep.write_stage_outputs = False
    x = torch.randn(1, 128, 7997, generator=torch.Generator().manual_seed(3)).cuda()
    with torch.inference_mode():
        sep.use_cuda_graph = False
        want = sep(x)[0].clone()
        for _ in range(3):
            sep(x)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(20):
            sep(x)
        eager_ms = (time.perf_counter() - t0) * 1e3 / 20
        torch.cuda.synchronize()
        sep.use_cuda_graph = True
        h = sep.handle()
        r0 = _lib.lib().sepref_graph_replay_count(h)
        for _ in range(4):                                   # eager, capture, replay, replay
            got = sep(x)[0]
        torch.cuda.synchronize()
        assert _lib.lib().sepref_graph_replay_count(h) - r0 >= 3
        assert torch.equal(got, want)
        t0 = time.perf_counter()
        for _ in range(20):
            sep(x)
        graph_ms = (time.perf_counter() - t0) * 1e3 / 20
        torch.cuda.synchronize()
        assert torch.equal(sep(x)[0], want)
        # the model-level call through a graph, too
        m.compute_aux = False
        mix, _, _ = mixtures(1, 32000, seed=8)
        sep.use_cuda_graph = False
        wa = torch.stack(m(mix.cuda())[0]).clone()
        sep.use_cuda_graph = True
        for _ in range(3):
            ga = torch.stack(m(mix.cuda())[0])
        assert torch.equal(ga, wa)
    sep.use_cuda_graph = False
    sep.write_stage_outputs = True
    print(f"host time per B=1 4 s forward: eager {eager_ms:.3f} ms, graph replay {graph_ms:.3f} ms")
    assert graph_ms < 0.3
