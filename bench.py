#!/usr/bin/env python
"""bench.py - separator frames/sec on B200 (BASELINE.json metric), one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload c2|c4|c5|c1] [--model NAME] [--seconds S] [--batch B] [--dump-outputs DIR]

Workloads (BASELINE.json configs, SURVEY.md 8d; weights are seeded random values of the real architecture - the
reference checkpoint is a Git-LFS pointer, SURVEY.md F3 - hence `"data": "synthetic"`):
  c2 (default; configs[1], and configs[2] per GPU)  SepReformer_Base_WSJ0, 32 utterances x 4 s @ 8 kHz per GPU (7997 frames each)
  c4 (configs[3])                                    SepReformer_Large_DM_WHAMR, 16 x 4 s per GPU
  c5 (configs[4] per GPU)                            SepReformer_Large_DM_WSJ0, 8 x 10 s per GPU (19997 frames, 1250 pooled keys)
  c1 (configs[0] shape)                              SepReformer_Base_WSJ0, 1 utterance of sample_WSJ.wav's length (18396 frames)
A "step" is one separator forward over the per-GPU batch.

  value        frames/s, inputs resident in HBM, CUDA events around exactly K steps, max over ranks
  e2e          frames/s through the host-buffer C-ABI entry (pinned host buffers in and out; H2D + D2H inside the timed
               region) - the number to hold against the reference arm
  roofline     the dominant kernel (fused GCFN): algorithmic FLOPs / its time measured live with CUDA events recorded by
               the library on the launching stream; plus whole-step tensor and HBM fractions
  parity       checked on the TIMED configuration: two utterances of the timed batch against the fp32 CUDA-core path,
               finiteness of the whole output, and the SI-SNRi delta against the CPU oracle on a short mixture
  reference_gpu  the reference's own Separator (oracle/_ref, eager PyTorch) on the same B200, fp32 and allow_tf32
  cpu_baseline / --impl reference: the reference's Separator (oracle/_ref; else its restatement in oracle/) on the
               host cores

--dump-outputs DIR writes what the last timed step returned (the separator's last-stage output and its per-stage outputs)
as DIR/<name>.npy, float32; arrays too large for a 60 MB budget are sampled at fixed seeded positions, and
DIR/manifest.json records each array's shape and whether it was sampled.  The inputs depend on the arguments alone, so
two builds can be compared output for output.  (--impl reference times the CPU reference and has no outputs to dump.)

N > 1: launched by torch.distributed.run, one rank per GPU; utterances shard (weak scaling); the only collective is an
all-gather of the per-utterance metric vector, inside the timed region as the last thing each step does.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

ENC_K, ENC_S, ENC_C = 16, 4, 256
WORKLOADS = {
    "c2": dict(model="SepReformer_Base_WSJ0", samples=32000, batch=32, tag="configs[1]"),
    "c4": dict(model="SepReformer_Large_DM_WHAMR", samples=32000, batch=16, tag="configs[3]"),
    "c5": dict(model="SepReformer_Large_DM_WSJ0", samples=80000, batch=8, tag="configs[4] per GPU"),
    "c1": dict(model="SepReformer_Base_WSJ0", samples=73596, batch=1, tag="configs[0] shape (sample_WSJ.wav length)"),
}
REF_COPY = os.path.join(ROOT, "oracle", "_ref")
DUMP_BYTES = 60 << 20


def frames_of(samples):
    return (samples - ENC_K) // ENC_S + 1


def synth_features(batch, feat, seed, device, samples):
    """Separator input as the model shell would produce it (reference module.py:12-35, model.py:39-40):
    mixture -> Conv1d(1,256,k16,s4)+GELU -> GroupNorm(1) -> 1x1 conv to F.  Random-init shell, seeded."""
    g = torch.Generator().manual_seed(seed)
    s1 = 0.05 * torch.randn(batch, samples, generator=g)
    s2 = 0.05 * torch.randn(batch, samples, generator=g)
    enc_w = (torch.rand(ENC_C, 1, ENC_K, generator=g) * 2 - 1) / ENC_K ** 0.5
    proj_w = (torch.rand(feat, ENC_C, 1, generator=g) * 2 - 1) / ENC_C ** 0.5
    mix = (s1 + s2).to(device)
    with torch.no_grad():
        e = torch.nn.functional.gelu(torch.nn.functional.conv1d(mix[:, None], enc_w.to(device), stride=ENC_S))
        e = torch.nn.functional.group_norm(e, 1, eps=1e-8)
        x = torch.nn.functional.conv1d(e, proj_w.to(device))
    return x.contiguous()


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_burst=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def algorithmic_flops(F, B, Tp):
    """SURVEY.md 8d: separator MACs per padded frame = 571.375 F^2 + 1779.8 F + 0.3984375 T F; GCFN alone is
    41.5 token-calls per padded frame of 9F^2 + 18F MACs."""
    total = 2.0 * (571.375 * F * F + 1779.8 * F + 0.3984375 * Tp * F) * B * Tp
    gcfn = 2.0 * (9 * F * F + 18 * F) * 41.5 * B * Tp
    return total, gcfn


def algorithmic_hbm_bytes(F, B, Tp, weight_bytes):
    """SURVEY.md 8d: one read and one write of [tok, F] fp32 per fused block, 83 block-passes per padded frame."""
    return 83.0 * 2 * 4 * F * B * Tp + weight_bytes


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(int(float(r[1])) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit())
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        mx = max((int(float(r[2])) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()), default=None)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ reference legs
def seeded_separator_state(model):
    from sepreformer_b200 import MODEL_SHAPES
    from sepreformer_b200.params import ParamTree, separator_spec, seeded_state, state_shapes
    shape = MODEL_SHAPES[model]
    return shape, seeded_state(state_shapes(ParamTree(separator_spec(shape))), seed=1)


def reference_separator(model):
    """The reference's own Separator (unmodified files under oracle/_ref, oracle/install_reference.py) with the seeded
    weights loaded; None when the copy is not there."""
    if not os.path.isdir(os.path.join(REF_COPY, "models", model)):
        return None
    import importlib
    import yaml
    if REF_COPY not in sys.path:
        sys.path.insert(0, REF_COPY)
    from loguru import logger
    logger.remove()
    mod = importlib.import_module(f"models.{model}.modules.module")
    cfg = yaml.full_load(open(os.path.join(REF_COPY, "models", model, "configs.yaml")))["config"]["model"]["module_separator"]
    sep = mod.Separator(**cfg).eval()
    _, sd = seeded_separator_state(model)
    sep.load_state_dict(sd, strict=True)
    return sep


def cpu_forward_fn(model, x):
    """(callable, kind): the reference Separator on the CPU when oracle/_ref is present, else the oracle port."""
    ref = reference_separator(model)
    if ref is not None:
        return (lambda: ref(x)), "reference"
    from oracle import separator_oracle as O
    shape, sd = seeded_separator_state(model)
    p = {k: v for k, v in sd.items() if v.is_floating_point()}
    return (lambda: O.separator_forward(x, p, heads=shape.heads, num_stages=shape.num_stages, num_spks=shape.num_spks,
                                        maxlen=shape.maxlen, per_stage_split=shape.per_stage_split, fast=True)), "port"


def time_cpu(model, samples, batch, steps, warmup, thread_candidates=None):
    """Times the reference's CPU path on this host.  PyTorch's CPU throughput on these many-core hosts peaks well below
    the logical core count (oversubscribed threads are several times slower), so a short proxy picks the thread count;
    every count tried is reported."""
    from sepreformer_b200 import MODEL_SHAPES
    feat = MODEL_SHAPES[model].feat
    ncpu = os.cpu_count() or 1
    # (the full logical-core count is not tried: 128 threads took 105 s per 1-s proxy forward on the GPU host, 64 took 0.5 s, 8-16 0.1 s)
    cands = thread_candidates or sorted({c for c in (8, 16, 32, 64) if c <= ncpu})
    xs = synth_features(1, feat, 7, "cpu", 4000 + ENC_K)
    fn_s, kind = cpu_forward_fn(model, xs)
    tried = {}
    with torch.inference_mode():
        for c in cands:
            torch.set_num_threads(c)
            fn_s()
            t = time.perf_counter()
            fn_s()
            tried[c] = time.perf_counter() - t
        best = min(tried, key=tried.get)
        torch.set_num_threads(best)
        x = synth_features(batch, feat, 1234, "cpu", samples)
        fn, kind = cpu_forward_fn(model, x)
        for _ in range(warmup):
            fn()
        ts = []
        for _ in range(steps):
            t = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t)
    total = sum(ts)
    return dict(fps=batch * x.shape[-1] * steps / total, ms=total / steps * 1e3, best_ms=min(ts) * 1e3, threads=best, kind=kind,
                proxy_s={str(k): round(v, 3) for k, v in tried.items()}, logical_cores=ncpu)


def cpu_model_name():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown CPU"


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    model, samples = wl["model"], wl["samples"]
    batch = 1
    steps = args.steps
    r = time_cpu(model, samples, batch, steps, args.warmup)
    what = ("the reference's own Separator (unmodified files, oracle/_ref)" if r["kind"] == "reference"
            else "oracle/ restatement of the reference Separator (oracle/_ref not present)")
    line = {
        "impl": "reference", "metric": "separator frames/sec", "value": r["fps"], "unit": "frames/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": args.warmup, "ms_per_step": r["ms"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{model} separator forward, {samples} samples @ 8 kHz 2-spk ({frames_of(samples)} frames/utt), "
                               f"CPU sample of {batch} utterance per step", "global_batch": batch, "frames_per_utt": frames_of(samples)},
        "cpu_baseline": {"value": r["fps"], "unit": "frames/s", "cores": r["threads"], "kind": r["kind"],
                         "sample": f"{steps} steps x {batch} utterance of the same synthetic workload: {what}, eager fp32 torch CPU, "
                                   f"inference_mode, on {cpu_model_name()} ({r['logical_cores']} logical cores); thread count chosen by a "
                                   f"1-s-utterance proxy, seconds per proxy forward by thread count: {r['proxy_s']}"},
        "e2e": {"value": r["fps"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def time_reference_on_gpu(model, x_dev, steps=3):
    """SURVEY.md 8d / BASELINE.md 3: the reference Separator itself, eager PyTorch on this B200 (the honest GPU
    baseline): fp32, and again with TF32 matmuls allowed.  Returns None when oracle/_ref is absent."""
    ref = reference_separator(model)
    if ref is None:
        return None
    out = {}
    ref = ref.to(x_dev.device)
    try:
        for name, tf32 in (("fp32", False), ("allow_tf32", True)):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.backends.cudnn.allow_tf32 = tf32
            with torch.inference_mode():
                for _ in range(2):
                    ref(x_dev)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(steps):
                    ref(x_dev)
                e1.record()
                torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[name] = {"ms_per_step": ms, "value": x_dev.shape[0] * x_dev.shape[-1] / (ms * 1e-3), "unit": "frames/s"}
    finally:
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = True
    del ref
    torch.cuda.empty_cache()
    out["what"] = ("reference Separator (oracle/_ref, unmodified), eager PyTorch on this GPU, inference_mode, same batch and "
                   f"weights, {steps} timed forwards after 2 warm-ups, CUDA events")
    return out


def dump_outputs(outdir, arrays):
    """Each array as <outdir>/<name>.npy in float32; one larger than its share of DUMP_BYTES is replaced by the elements at
    a seeded, sorted set of flat (row-major) positions, the same positions for the same shape on every run.
    <outdir>/manifest.json gives, per name, the array's shape and, when sampled, the seed and sample size."""
    import numpy as np
    os.makedirs(outdir, exist_ok=True)
    cap = DUMP_BYTES // 4 // len(arrays)
    manifest = {}
    for name, t in arrays.items():
        a = t.detach().float()
        manifest[name] = {"shape": list(a.shape), "dtype": "float32", "sampled": a.numel() > cap}
        if a.numel() > cap:
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:cap].sort().values
            a = a.reshape(-1)[idx.to(a.device)]
            manifest[name].update(sample="torch.randperm(numel, Generator().manual_seed(0))[:n].sort()", seed=0, n=cap)
        np.save(os.path.join(outdir, name + ".npy"), a.cpu().numpy())
    with open(os.path.join(outdir, "manifest.json"), "w") as f:
        json.dump(manifest, f, indent=1)


# ------------------------------------------------------------------------------------------------ parity on the timed config
def shell_state(feat, seed=3):
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


def parity_block(sep, x_dev, last_timed, model, skip_oracle):
    """Evidence that the timed configuration computes the right thing (VERDICT r1 weak #3)."""
    S = sep.shape_.num_spks
    nchk = min(2, x_dev.shape[0])
    path, graph = sep.gemm_path, sep.use_cuda_graph
    finite = bool(torch.isfinite(last_timed).all())
    a = last_timed[: nchk * S].double().clone()     # (graph mode hands out the same output buffers on every call)
    sep.gemm_path, sep.use_cuda_graph = 0, False
    ref0, _ = sep(x_dev[:nchk].contiguous())
    sep.gemm_path, sep.use_cuda_graph = path, graph
    b = ref0.double()
    out = {"finite": finite,
           "rel_l2_vs_fp32_path": float((a - b).norm() / b.norm()),
           "utterances_checked": nchk, "tolerance": 1e-3}
    if not skip_oracle:
        from oracle import separator_oracle as O
        shape, sd = seeded_separator_state(model)
        p = {k: v for k, v in sd.items() if v.is_floating_point()}
        shell = shell_state(shape.feat)
        g = torch.Generator().manual_seed(77)
        n = 8000                                   # 1 s mixtures: the oracle side costs about a second
        s1, s2 = 0.05 * torch.randn(2, n, generator=g), 0.05 * torch.randn(2, n, generator=g)
        mix = s1 + s2
        kw = dict(heads=shape.heads, num_stages=shape.num_stages, num_spks=shape.num_spks, maxlen=shape.maxlen,
                  per_stage_split=shape.per_stage_split, fast=True)
        est_ref = O.model_forward(mix, shell, lambda f: O.separator_forward(f, p, **kw)[0])
        est_gpu = O.model_forward(mix, shell, lambda f: sep(f.to(x_dev.device))[0].cpu())
        sa = O.pit_si_snri([e[..., :n] for e in est_ref], [s1, s2], mix)
        sb = O.pit_si_snri([e[..., :n] for e in est_gpu], [s1, s2], mix)
        out["si_snri_delta_db"] = float((sa - sb).abs().max())
        out["si_snri_bound_db"] = 0.05
        out["si_snri_note"] = "2 x 1 s synthetic mixtures through the same model shell (oracle/), separator = CPU oracle vs this library"
    out["ok"] = bool(out["finite"] and out["rel_l2_vs_fp32_path"] < 1e-3 and out.get("si_snri_delta_db", 0.0) <= 0.05)
    return out


def model_kwargs(shape):
    from sepreformer_b200 import separator_kwargs
    f = shape.feat
    return dict(num_stages=shape.num_stages, num_spks=shape.num_spks,
                module_audio_enc=dict(in_channels=1, out_channels=256, kernel_size=16, stride=4, groups=1, bias=False),
                module_feature_projector=dict(num_channels=256, in_channels=256, out_channels=f, kernel_size=1, bias=False),
                module_separator=separator_kwargs(shape),
                module_output_layer=dict(in_channels=256, out_channels=f, num_spks=shape.num_spks),
                module_audio_dec=dict(in_channels=256, out_channels=1, kernel_size=16, stride=4, bias=False))


def run_ours(args, wl):
    import torch.distributed as dist
    from sepreformer_b200 import MODEL_SHAPES, Model
    from sepreformer_b200.params import seeded_state, state_shapes

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)

    model_name, samples = wl["model"], wl["samples"]
    shape = MODEL_SHAPES[model_name]
    B, T = wl["batch"], frames_of(samples)
    # the whole model with the reference's module surface (stock torch init for the shell, seeded separator weights);
    # `sep` is its separator - the hot path the metric is quoted on
    torch.manual_seed(3)
    model = Model(**model_kwargs(shape), per_stage_split=shape.per_stage_split)
    model.separator.load_state_dict(seeded_state(state_shapes(model.separator), seed=1))
    model = model.to(dev).eval()
    model.compute_aux = False            # inference: the training-time auxiliary heads are not evaluated (engine.py:165 drops them)
    sep = model.separator
    sep.use_cuda_graph = not args.no_cuda_graph     # replay one captured graph per forward instead of ~260 launch calls
    sep.write_stage_outputs = True       # the four per-stage outputs of Separator.forward are produced, as in the reference
    g = torch.Generator().manual_seed(1234 + rank)
    s1 = 0.05 * torch.randn(B, samples, generator=g)
    s2 = 0.05 * torch.randn(B, samples, generator=g)
    mix_host = (s1 + s2).pin_memory()
    mix_dev = mix_host.to(dev)
    tgt_dev = torch.stack([s1, s2]).to(dev)
    # separator input exactly as this model's shell produces it (module.py:12-35); deterministic convolutions, so the
    # same arguments give the same input on every run
    with torch.no_grad(), torch.backends.cudnn.flags(enabled=True, deterministic=True):
        e = torch.nn.functional.gelu(model.audio_encoder.conv1d(mix_dev[:, None]))
        x_dev = model.feature_projector.conv1d(model.feature_projector.norm(e)).contiguous()
        del e
    x_host = x_dev.cpu().pin_memory()
    Tp = sep.padded_frames(T)
    frames_step = B * T
    F = shape.feat
    with torch.inference_mode():         # separated waveforms of this batch, resident: what the metric kernel reads every step
        audio_dev = torch.stack(model(mix_dev)[0]).contiguous()

    from sepreformer_b200.sharding import gather_utterance_values

    def step_device():
        out = sep(x_dev)
        if world > 1:     # the path's only exchange (SURVEY 8e): per-utterance PIT SI-SNRi rows [B_local, 3], computed on the
            # device (k_pit_sisnri), all-gathered into global utterance order on every rank
            gather_utterance_values(model.pit_si_snri(audio_dev, tgt_dev, mix_dev), B * world)
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput
    with torch.inference_mode():
        for _ in range(args.warmup):
            step_device()
        barrier()
        clocks = ClockSampler(local)
        if rank == 0:
            clocks.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            last_timed, stages_timed = step_device()
        e1.record()
        barrier()
        ms_total = e0.elapsed_time(e1)
        launches = sep.last_launch_count * args.steps
        clk = clocks.stop() if rank == 0 else None
        if args.dump_outputs and rank == 0:      # before any other call reuses the graph's output buffers
            dump_outputs(args.dump_outputs, {"last": last_timed, **{f"stage{i}": t for i, t in enumerate(stages_timed)}})
        del stages_timed

        # ---- the timed configuration is checked (rank 0; after the timed region)
        parity = parity_block(sep, x_dev, last_timed, model_name, args.no_cpu_baseline) if rank == 0 else None
        del last_timed

        # ---- dominant kernel timed live with CUDA events on the launching stream (separate pass, same inputs)
        prof = sep.profile_kernels(x_dev, steps=max(1, min(args.steps, 5)))

        # ---- the same step with kind::tf32 operands (reported beside the headline for comparison)
        nt = max(3, min(args.steps, 5))
        sep.gemm_path = 1
        for _ in range(2):
            step_device()
        barrier()
        t0e, t1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0e.record()
        for _ in range(nt):
            step_device()
        t1e.record()
        barrier()
        ms_tf32 = t0e.elapsed_time(t1e) / nt
        sep.gemm_path = 2

        # ---- end to end through the host-buffer C-ABI calls: every step copies its inputs from pinned host memory
        # and its result back to host memory inside the timed region.  Serving-loop form (submit / wait, two
        # requests in flight: the copies of steps i-1 / i+1 overlap the kernels of step i); the wall clock below
        # therefore includes one exposed H2D at the start and one exposed D2H at the end of the K steps.
        n_out = model.output_samples(samples)
        wav_outs = [torch.empty(shape.num_spks, B, n_out, dtype=torch.float32, pin_memory=True) for _ in range(2)]
        feat_outs = [torch.empty(B * shape.num_spks, shape.feat, Tp, dtype=torch.float32, pin_memory=True) for _ in range(2)]

        def consume(out_h):      # read the step's result on the host; N > 1: the sharded path's exchange step
            v = out_h.reshape(-1)[:: max(1, out_h.numel() // (2 * B))][: 2 * B].reshape(B, 2)
            if world > 1:
                gather_utterance_values(v.to(dev), B * world)
            return float(v.sum())

        def pipelined(steps, submit, wait):
            for i in range(steps):
                slot = i & 1
                if i >= 2:
                    consume(wait(slot))
                submit(slot)
            for i in range(max(0, steps - 2), steps):
                consume(wait(i & 1))

        def timed(submit, wait):
            pipelined(max(2, min(args.warmup, 4)), submit, wait)
            torch.cuda.synchronize()
            barrier()
            t0 = time.perf_counter()
            pipelined(args.steps, submit, wait)
            torch.cuda.synchronize()
            ms = (time.perf_counter() - t0) * 1e3
            barrier()
            return ms

        # headline e2e: the user-level call - a mixture goes in, separated waveforms come back (sepref_model_submit_host)
        ms_e2e = timed(lambda slot: model.submit_host(mix_host, slot, dev, out=wav_outs[slot]), lambda slot: model.wait_host(slot, dev))
        # the round-1 boundary for comparison: F-channel features in and out (sepref_separator_submit_host)
        ms_sync = timed(lambda slot: sep.submit_host(x_host, slot, dev, out=feat_outs[slot]), lambda slot: sep.wait_host(slot, dev)[0]) / args.steps
        del feat_outs

        # ---- host time of one call at a latency-bound size (B = 1): what the caller's thread spends per forward
        x1 = x_dev[:1].contiguous()
        for _ in range(3):
            sep(x1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(10):
            sep(x1)
        host_ms_b1 = (time.perf_counter() - t0) * 1e3 / 10      # enqueue time only: no synchronize inside the loop
        torch.cuda.synchronize()

        ref_gpu = None
        if rank == 0 and world == 1 and not args.no_reference_gpu:
            try:
                ref_gpu = time_reference_on_gpu(model_name, x_dev)
            except Exception as e:      # e.g. out of memory at the reference's intermediate sizes: report, do not fail the bench
                ref_gpu = {"error": f"{type(e).__name__}: {str(e)[:200]}"}

    t = torch.tensor([ms_total, ms_e2e, ms_sync], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e, ms_sync = float(t[0]), float(t[1]), float(t[2])

    if rank == 0:
        peaks = measured_peaks()
        ms_step = ms_total / args.steps
        flops_step, gcfn_flops = algorithmic_flops(F, B, Tp)
        weight_bytes = sum(v.numel() * 4 for v in sep.state_dict().values() if v.is_floating_point())
        hbm_bytes = algorithmic_hbm_bytes(F, B, Tp, weight_bytes)
        f16_peak = peaks["bf16_sustained"]
        roof = None
        if prof and prof.get("gcfn_ms", 0) > 0:
            ach = gcfn_flops / (prof["gcfn_ms"] * 1e-3) / 1e12
            traffic = None
            for name in ("r2_gcfn_traffic.json", "r1_gcfn_traffic.json"):
                tpath = os.path.join(ROOT, "profiles", name)
                if os.path.exists(tpath) and wl is WORKLOADS["c2"]:
                    traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
                    break
            roof = {"kernel": f"sepref::tc::k_gcfn<{F},F16> (fused GCFN block: tcgen05 kind::f16, TMEM accumulators, TMA weight slabs)",
                    "bound": "tensor", "achieved": ach, "peak": f16_peak, "unit": "TFLOP/s", "frac": ach / f16_peak,
                    "traffic": traffic, "launches_per_step": prof["gcfn_launches"],
                    "avg_launch_ms": prof["gcfn_ms"] / max(1, prof["gcfn_launches"]),
                    "share_of_step": prof["gcfn_ms"] / ms_step,
                    "algorithmic_flops_per_step": gcfn_flops,
                    "hbm_frac": hbm_bytes / (ms_step * 1e-3) / 1e9 / peaks["hbm_gbs"],
                    "whole_step": {"algorithmic_flops": flops_step, "tensor_frac": flops_step / (ms_step * 1e-3) / 1e12 / f16_peak,
                                   "algorithmic_hbm_bytes": hbm_bytes, "achieved_gbs": hbm_bytes / (ms_step * 1e-3) / 1e9,
                                   "hbm_peak_gbs": peaks["hbm_gbs"]},
                    "peak_source": f"{peaks['source']}: sustained dense bf16 {peaks['bf16_sustained']:.0f} TFLOP/s (fp16 and bf16 "
                                   f"issue at the same rate), HBM copy {peaks['hbm_gbs']:.0f} GB/s; frac is recomputable from kernel_ms.gcfn_ms"}
        cpu = None if args.no_cpu_baseline else time_cpu(model_name, samples, 1, 2, 1, thread_candidates=[16, 32])
        line = {
            "metric": "separator frames/sec", "value": frames_step * world * args.steps / (ms_total * 1e-3), "unit": "frames/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16 operands (11-bit significand = TF32's; row-scaled weights; range-checked at pack time, TF32 where unbounded), f32 accumulate, f32 activations and I/O",
            "data": "synthetic",
            "config": {"workload": f"{model_name} separator forward ({wl['tag']}): batch {B}/GPU x {samples} samples @ 8 kHz 2-spk, {T} frames/utt",
                       "global_batch": B * world, "frames_per_utt": T, "parallelism": f"dp{world} (utterance sharding)",
                       "l2": f"inputs ({x_host.numel() * 4 / 1e6:.0f} MB) and activations (GBs) exceed the 126 MB L2; no explicit flush",
                       "launch": "CUDA graph replay (SEPREF_OPT_CUDA_GRAPH)" if sep.use_cuda_graph else "individual kernel launches",
                       "exchange": "N > 1: all-gather of per-utterance PIT SI-SNRi rows [B_local, 3] computed by k_pit_sisnri on the device"},
            "e2e": {"value": frames_step * world * args.steps / (ms_e2e * 1e-3), "unit": "frames/s",
                    "h2d_bytes_per_step": mix_host.numel() * 4, "d2h_bytes_per_step": shape.num_spks * B * n_out * 4,
                    "ms_per_step": ms_e2e / args.steps,
                    "mode": "sepreformer_b200.Model.submit_host / wait_host (sepref_model_submit_host): mixtures [B, samples] from pinned "
                            "host memory -> encoder, projector, separator, output layer, decoder on the GPU -> waveforms [2, B, n_out] back "
                            "to pinned host memory; 2 requests in flight, host wall clock over the K steps (H2D + kernels + D2H inside)",
                    "feature_boundary": {"value": frames_step * world / (ms_sync * 1e-3), "ms_per_step": ms_sync,
                                         "h2d_bytes_per_step": x_host.numel() * 4, "d2h_bytes_per_step": B * shape.num_spks * F * Tp * 4,
                                         "note": "round-1 boundary: sepref_separator_submit_host, F-channel features in and out"}},
            "gpu_launches": launches, "clocks": clk, "roofline": roof, "parity": parity,
            "cpu_baseline": None if cpu is None else {
                "value": cpu["fps"], "unit": "frames/s", "cores": cpu["threads"], "kind": cpu["kind"],
                "sample": f"2 timed forwards of 1 utterance of the same synthetic workload on the host cores ({cpu_model_name()}, "
                          f"{cpu['logical_cores']} logical), {cpu['threads']} threads (proxy seconds by thread count {cpu['proxy_s']}); "
                          + ("reference Separator from oracle/_ref" if cpu["kind"] == "reference" else "oracle/ restatement")},
            "reference_gpu": ref_gpu,
            "host_enqueue_ms_b1": host_ms_b1,
            "kernel_ms": prof,
            "tf32": {"value": frames_step * world / (ms_tf32 * 1e-3), "ms_per_step": ms_tf32,
                     "note": "same step with gemm_path=1 (tcgen05 kind::tf32 operands)"},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--model", default=None, help="override the workload's model directory name")
    ap.add_argument("--seconds", type=float, default=None, help="override the utterance length (seconds @ 8 kHz)")
    ap.add_argument("--batch", type=int, default=None, help="utterances per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU legs (oracle SI-SNRi check and cpu_baseline)")
    ap.add_argument("--no-reference-gpu", action="store_true", help="skip timing the reference Separator on the GPU")
    ap.add_argument("--no-cuda-graph", action="store_true", help="launch every kernel individually (SEPREF_OPT_CUDA_GRAPH off)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs to DIR/<name>.npy (float32, seeded sample above 60 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs applies to --impl ours: the reference arm times the CPU reference and returns nothing")
    wl = WORKLOADS[args.workload]
    if args.model or args.seconds or args.batch:
        wl = dict(wl)
        if args.model:
            wl["model"] = args.model
        if args.seconds:
            wl["samples"] = int(round(args.seconds * 8000))
        if args.batch:
            wl["batch"] = args.batch
        wl["tag"] = wl["tag"] + " (overridden)"
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
