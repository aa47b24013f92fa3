#!/usr/bin/env python
"""bench.py -- FAcodec encode -> quantize -> decode throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path (encoder -> quantizer(n_c=2, codes) -> decoder) over one
batch of synthetic 4 s 24 kHz utterances (PseudoDataset law, meldataset.py:67-68); the workload
is BASELINE configs[1]: 32 utterances per GPU (weak scaling: every rank gets its own 32).
Prints ONE JSON line on rank 0 (contract in the task statement):
  value      = audio-seconds per second, whole job, inputs resident in HBM (CUDA events, max over ranks)
  e2e        = same metric through Codec.forward_host: pinned HOST buffers, H2D + D2H inside the timed region
  roofline   = dominant kernel family (the two tcgen05 conv kernels conv_tc_kernel + conv_tcp_kernel, ~80 % of a step):
               algorithmic FLOPs / device time, from CUDA events recorded around every launch in a separate
               instrumented pass (fac_profile_*); traffic = DRAM bytes per launch of that family from the committed
               ncu launch list (profiles/roofline_r02.json)
  cpu_baseline = the oracle port (oracle/facodec_oracle.py = the reference's own ATen call sequence)
               timed on this box's host cores on a bounded sample
--impl reference times that CPU path alone (the reference is 100% Python/PyTorch, so the validated restatement
stands in: kind "port").
--dump-outputs DIR writes what the last timed step returned (waveforms, the three code tensors, timbre vectors of rank 0)
as DIR/<name>.npy, so that two builds can be compared output for output on the same seeded inputs.
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

SR = 24000
UTT_SECONDS = 4
UTT_SAMPLES = SR * UTT_SECONDS
BATCH_PER_GPU = 32
METRIC = "audio_seconds_per_second"
UNIT = "24kHz audio-s/s (encode+VQ+decode)"
DTYPE = ("f32 I/O and accumulation; every product is a 3-MMA split of fp32 operands: fp16 hi + 2^11-scaled fp16 lo "
         "(22 mantissa bits, register-promoted accumulation) upstream of the VQ, bf16 hi + bf16 lo (16 bits) downstream")
GFLOP_PER_AUDIO_S = 118.44     # SURVEY.md 8(d): 473.75 GFLOP per 4 s utterance
MB_PER_AUDIO_S = 320.3         # SURVEY.md 8(d): fused-block fp32 bytes per audio-second


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], tflops=d.get("bf16_tflops_sustained", d["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, tflops=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dump_outputs(out_dir, arrays, limit_bytes=64 << 20):
    """Writes each tensor as out_dir/<name>.npy: float32, or float64 for integer tensors (code indices stay exact)."""
    import numpy as np
    host = {}
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        host[name] = a.astype(np.float64 if a.dtype.kind in "iub" else np.float32)
    total = sum(a.nbytes for a in host.values())
    if total > limit_bytes:
        raise ValueError(f"outputs take {total} bytes, more than the {limit_bytes} a dump may hold")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def usable_cores():
    """Host threads this process may actually use: min(cpu_count, affinity mask, cgroup CPU quota)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = min(n, max(1, int(int(q) / int(per))))
    except Exception:
        pass
    return n


def cpu_reference_run(steps, warmup, sample_utts=4):
    """The reference's CPU path (oracle port) on this box's host cores: B=sample_utts x 4 s per step."""
    import torch
    from facodec_b200 import synth
    from oracle import facodec_oracle as O
    cores = usable_cores()
    torch.set_num_threads(cores)
    sds = synth.synth_state_dicts(0)
    x = synth.synth_waves(sample_utts, UTT_SAMPLES)
    for _ in range(warmup):
        O.codec_forward(sds, x, n_c=2)
    t0 = time.perf_counter()
    for _ in range(steps):
        O.codec_forward(sds, x, n_c=2)
    dt = time.perf_counter() - t0
    value = sample_utts * UTT_SECONDS * steps / dt
    return value, dt / steps * 1e3, cores, f"{sample_utts} x 4 s utterances per step, {steps} steps, fp32, torch {torch.__version__} CPU, {torch.get_num_threads()} threads"


def library_baseline(x, dev, steps=2):
    """SURVEY.md 8(d) "library" baseline: the reference's ATen call sequence (the oracle restatement = what the reference's
    nn.Modules execute: cuDNN convs / LSTM, cuBLAS, cuFFT) run by PyTorch eager on the same B200, fp32 with TF32 disabled,
    on one configs[1] batch.  Returns None when it cannot run (e.g. out of memory)."""
    import torch
    from facodec_b200 import synth
    from oracle import facodec_oracle as O
    try:
        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False
        sds = synth.synth_state_dicts(0)
        sds_gpu = {k: {n: t.to(dev) for n, t in sd.items()} for k, sd in sds.items()}
        with torch.no_grad():
            O.codec_forward(sds_gpu, x, n_c=2)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(steps):
                O.codec_forward(sds_gpu, x, n_c=2)
            b.record()
            torch.cuda.synchronize()
        ms = a.elapsed_time(b) / steps
        del sds_gpu
        torch.cuda.empty_cache()
        return {"value": x.shape[0] * UTT_SECONDS / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps,
                "kind": "reference ATen op sequence (oracle restatement) under PyTorch eager on this GPU: cuDNN/cuBLAS/cuFFT, "
                        "fp32, TF32 off, torch " + torch.__version__}
    except RuntimeError as e:
        return {"unavailable": str(e).splitlines()[0][:200]}


def vq_bench(args, rank, local_rank, world):
    """BASELINE configs[3]: quantize/rvq.py ResidualVQ (4 quantizers x 1024 entries, 1024 -> 8) over 2^20 frames per GPU.
    Metric: frames per second through facodec_b200.ResidualVQ (channels-last [B, T, 1024] in and out, indices [4, B, T]);
    roofline: HBM, algorithmic bytes = 4 KB read + 4 KB written + 32 B of indices per frame; parity: every index of a
    sample of frames against the CPU oracle."""
    import torch
    import torch.distributed as dist
    import facodec_b200 as fb
    from facodec_b200 import distributed as D
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    B, T = 1024, 1024
    frames = B * T
    rvq = fb.ResidualVQ(num_quantizers=4, codebook_size=10, dim=1024, codebook_dim=8, commitment=0.25).eval()
    g = torch.Generator(device=dev).manual_seed(7 + rank)
    x = torch.randn(B, T, 1024, device=dev, generator=g)
    for _ in range(max(1, args.warmup)):
        q, idx, _, _ = rvq(x, channels_last=True, return_all=False)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(args.steps):
        q, idx, _, _ = rvq(x, channels_last=True, return_all=False)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b)
    if world > 1:
        dist.barrier()
        ms = D.max_over_ranks(ms, dev)
    value = world * frames * args.steps / (ms * 1e-3)
    peaks = load_peaks()
    bytes_per_frame = 2 * 4096 + 4 * 8
    gbs = frames * bytes_per_frame / (ms / args.steps * 1e-3) / 1e9
    parity = None
    if rank == 0:
        from oracle import facodec_oracle as O
        torch.set_num_threads(usable_cores())
        ns = 16
        layers = [dict(in_w=rvq._folded(i, "in_proj"), in_b=rvq._p[f"layers/{i}/in_proj/bias"].detach().cpu(),
                       out_w=rvq._folded(i, "out_proj"), out_b=rvq._p[f"layers/{i}/out_proj/bias"].detach().cpu(),
                       codebook=rvq._p[f"layers/{i}/_codebook/weight"].detach().cpu()) for i in range(4)]
        with torch.no_grad():
            qo, io, _, _ = O.fvq_residual_vq(layers, x[:ns].transpose(1, 2).cpu())
        nbad = int((idx[:, :ns].cpu() != io).sum())
        parity = {"frames_checked": ns * T, "indices_checked": int(io.numel()), "indices_differing": nbad,
                  "max_abs_err_quantized": float((q[:ns].transpose(1, 2).cpu() - qo).abs().max())}
        print(json.dumps({"metric": "rvq_frames_per_second", "value": value, "unit": "frames/s (4 codebooks x 1024 entries, 1024 -> 8)",
                          "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 / int64", "data": "synthetic",
                          "config": {"workload": "BASELINE configs[3]: FVQ+RVQ codebook-distance microbench, 1024-dim latents x 4 codebooks "
                                                 "x 1024 entries, 2^20 frames per GPU (B=1024, T=1024), channels-last",
                                     "l2": "8.6 GB of input + output per step >> 126 MB L2"},
                          "roofline": {"kernel": "rvq_kernel (warp per frame)", "bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"],
                                       "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"], "traffic": None,
                                       "algorithmic_bytes_per_frame": bytes_per_frame, "peak_source": peaks["source"]},
                          "parity": parity, "gpu_launches": args.steps}))
    if world > 1:
        dist.destroy_process_group()
    return 0


def trainfwd_bench(args, rank, local_rank, world):
    """BASELINE configs[4], the part of it this repo builds: the training step's FORWARD (encoder -> quantizer n_c=2 ->
    decoder, train.py:265-272, eval-mode arithmetic) plus the forward of the reference's own reconstruction loss
    (losses.py:65-89) between input and reconstruction, fp32-faithful, 8 utterances x 4 s per GPU (batch 64 on 8 GPUs).
    No backward, no discriminators, no audiotools losses (DESIGN.md section 0, row f3).  Parity: the loss value of the first
    timed batch against the CPU oracle fed with the GPU's reconstruction."""
    import torch
    import torch.distributed as dist
    import facodec_b200 as fb
    from facodec_b200 import distributed as D
    from facodec_b200 import losses, synth
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    B = 8
    sds = synth.synth_state_dicts(0) if rank == 0 else None
    if world > 1:
        sds = D.broadcast_state_dicts(sds, 0, dev)
    model = fb.build_model(with_predictors=True)
    for k in ("encoder", "quantizer", "decoder"):
        model[k].load_state_dict(sds[k]); model[k].eval()
    model.fa_predictors.eval()                      # synthetic default weights (PyTorch-init statistics), identical on every rank
    codec = fb.Codec(model)
    xs = [synth.synth_waves(B, UTT_SAMPLES, seed=1000 + 17 * rank + i).to(dev) for i in range(4)]

    def step(x):
        # train.py:265-272: encoder -> quantizer -> fa_predictors(quantized, timbre) -> decoder, then the loss forward
        z = model.encoder(x)
        outs, quantized, commit, cb, timbre = model.quantizer(z, x, n_c=2)
        model.fa_predictors(quantized, timbre)
        y = model.decoder(outs)
        return y, losses.reconstruction_loss(x, y)

    for i in range(max(3, args.warmup)):
        step(xs[i % 4])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(args.steps):
        y, L = step(xs[i % 4])
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b)
    if world > 1:
        dist.barrier()
        ms = D.max_over_ranks(ms, dev)
    # loss-only timing (device events) and parity on rank 0
    a.record()
    for i in range(args.steps):
        losses.reconstruction_loss(xs[i % 4], y)
    b.record()
    torch.cuda.synchronize()
    ms_loss = a.elapsed_time(b) / args.steps
    if rank == 0:
        from oracle import facodec_oracle as O
        torch.set_num_threads(usable_cores())
        x0 = xs[(args.steps - 1) % 4]
        with torch.no_grad():
            Lo = float(O.reconstruction_loss(x0.cpu(), y.cpu()))
        value = world * B * UTT_SECONDS * args.steps / (ms * 1e-3)
        print(json.dumps({"metric": "train-step forward + reconstruction loss, 24 kHz audio-seconds per second", "value": value, "unit": UNIT,
                          "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps,
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "f32 I/O; 3-MMA split products (see the codec line); loss sums in fp64", "data": "synthetic",
                          "config": {"workload": "BASELINE configs[4], forward half only: encoder -> quantizer -> fa_predictors -> decoder "
                                                 "(train.py:265-272, eval arithmetic) + losses.reconstruction_loss forward (losses.py:65-89), "
                                                 "8 x 4 s utterances per GPU; no backward, no discriminator, no audiotools losses",
                                     "l2": "inputs rotate over 4 distinct batches; the loss alone streams ~1.5 GB of scratch per step"},
                          "loss_ms_per_step": ms_loss,
                          "parity": {"loss_gpu": float(L), "loss_oracle_cpu": Lo, "rel_err": abs(float(L) - Lo) / abs(Lo)},
                          "gpu_launches": 400 * args.steps}))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=12)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-library-baseline", action="store_true")
    ap.add_argument("--workload", default="codec", choices=["codec", "vq", "trainfwd"],
                    help="codec = BASELINE configs[1] (the headline); vq = configs[3] FVQ/RVQ codebook-distance microbench; "
                         "trainfwd = the forward half of configs[4] (codec forward + losses.reconstruction_loss)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the outputs of the last one as DIR/<name>.npy (codec workload, --impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.workload != "codec" or args.impl != "ours"):
        ap.error("--dump-outputs writes the outputs of the codec workload's timed path (--workload codec --impl ours)")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    config = {"workload": f"BASELINE configs[1]: batch={BATCH_PER_GPU} x 4 s 24 kHz mono utterances per GPU, full codec "
                          "forward (encoder -> quantizer n_c=2 with codes -> decoder), reference config.yml geometry",
              "utterances_per_gpu": BATCH_PER_GPU, "utterance_samples": UTT_SAMPLES,
              "parallelism": f"dp{world} (utterance sharding, replicas, no hot-path collective)",
              "l2": "per-step working set (~10 GB of activations) >> 126 MB L2; inputs rotate over 4 distinct batches"}

    if args.workload == "vq":
        return vq_bench(args, rank, local_rank, world)
    if args.workload == "trainfwd":
        return trainfwd_bench(args, rank, local_rank, world)

    if args.impl == "reference":
        if rank != 0:
            return 0
        # exactly K timed steps after W warm-up steps; each step is a bounded sample of the workload (2 of the 32
        # utterances, ~5 s of CPU work) so that the whole run ends within a few minutes
        steps = max(1, args.steps)
        value, ms, cores, sample = cpu_reference_run(steps, max(0, args.warmup), sample_utts=2)
        config = dict(config)
        config["workload"] = ("bounded sample of BASELINE configs[1]: batch=2 x 4 s 24 kHz mono utterances per step (2 of the 32 "
                              "utterances of a configs[1] batch; same model, same n_c=2 forward), CPU only -- throughput-normalised "
                              "metric, see cpu_baseline.sample")
        config["utterances_per_step"] = 2
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
                          "steps": steps, "warmup": max(0, args.warmup), "ms_per_step": ms, "higher_is_better": True,
                          "scaling": "weak", "vs_baseline": None, "dtype": "f32 (ATen CPU kernels)", "data": "synthetic",
                          "config": config,
                          "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
                          "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return 0

    import torch
    import torch.distributed as dist
    import facodec_b200 as fb
    from facodec_b200 import distributed as D
    from facodec_b200 import synth

    assert torch.cuda.is_available(), "bench.py --impl ours needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    # ---- weights: rank 0 builds the checkpoint, ONE broadcast moves it (NCCL over NVLink) ----
    sds = synth.synth_state_dicts(0) if rank == 0 else None
    if world > 1:
        sds = D.broadcast_state_dicts(sds, src=0, device=dev)
    model = fb.build_model()
    for k in ("encoder", "quantizer", "decoder"):
        model[k].load_state_dict(sds[k])
        model[k].eval()
    codec = fb.Codec(model)
    eng = codec.engine

    # ---- inputs: 4 distinct batches of 32 utterances per rank, resident in HBM ----
    nrot = 4
    waves = synth.synth_waves(BATCH_PER_GPU * nrot, UTT_SAMPLES, seed=114514 + rank)
    xs = [waves[i * BATCH_PER_GPU:(i + 1) * BATCH_PER_GPU].contiguous().to(dev) for i in range(nrot)]
    xs_host = [waves[i * BATCH_PER_GPU:(i + 1) * BATCH_PER_GPU].contiguous().pin_memory() for i in range(nrot)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(steps):
            fn(i)
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b)
        barrier()
        return D.max_over_ranks(ms, dev) if world > 1 else ms

    # ---- device-resident throughput ----
    for i in range(args.warmup):
        codec.forward(xs[i % nrot], n_c=2)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    last = []

    def step(i):
        out = codec.forward(xs[i % nrot], n_c=2)
        if i == args.steps - 1:
            last.append(out)

    ms_total = timed(step, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        y_last, codes_last, timbre_last = last[0]
        dump_outputs(args.dump_outputs, {"y": y_last, "codes_p": codes_last[0], "codes_c": codes_last[1],
                                         "codes_r": codes_last[2], "timbre": timbre_last})
    del last
    launches = codec.launch_count() * args.steps
    audio_s = world * BATCH_PER_GPU * UTT_SECONDS * args.steps
    value = audio_s / (ms_total * 1e-3)

    # ---- end to end: pinned host in, host out ----
    out_bufs = None
    y0, c0 = codec.forward_host(xs_host[0], n_c=2)
    out_bufs = (y0, c0[0], c0[1], c0[2])
    for i in range(max(1, args.warmup - 1)):
        codec.forward_host(xs_host[i % nrot], n_c=2, out=out_bufs)
    ms_e2e = timed(lambda i: codec.forward_host(xs_host[i % nrot], n_c=2, out=out_bufs), args.steps)
    e2e_value = audio_s / (ms_e2e * 1e-3)
    h2d = xs_host[0].numel() * 4
    d2h = y0.numel() * 4 + sum(c.numel() * 8 for c in c0)

    # ---- roofline of the dominant kernel family, instrumented pass (events around every launch) ----
    import ctypes
    peaks = load_peaks()
    L, h = eng.L, eng.handle
    L.fac_profile_reset(h)
    L.fac_profile_enable(h, 1)
    nprof = 2
    for i in range(nprof):
        codec.forward(xs[i % nrot], n_c=2)
    torch.cuda.synchronize()
    L.fac_profile_enable(h, 0)
    fam = {}
    for name in ("conv_tc", "conv_tcp", "conv_tt", "conv", "lstm_rec", "fa_quantize"):
        ms, fl, by, n = ctypes.c_double(), ctypes.c_double(), ctypes.c_double(), ctypes.c_longlong()
        L.fac_profile_get(h, name.encode(), ctypes.byref(ms), ctypes.byref(fl), ctypes.byref(by), ctypes.byref(n))
        fam[name] = dict(ms=ms.value / nprof, flops=fl.value / nprof, bytes=by.value / nprof, launches=n.value // nprof)
    L.fac_profile_reset(h)
    # dominant kernels: the two tcgen05 conv kernels (same mainloop; conv_tcp adds register promotion)
    conv = {k: fam["conv_tc"][k] + fam["conv_tcp"][k] + fam["conv_tt"][k] for k in ("ms", "flops", "bytes", "launches")}
    conv_tflops = conv["flops"] / (conv["ms"] * 1e-3) / 1e12 if conv["ms"] > 0 else 0.0
    traffic, traffic_src = None, None
    try:
        rj = json.load(open(os.path.join(ROOT, "profiles", "roofline_r02.json")))
        traffic = rj["conv_family"]["dram_bytes_per_launch"]
        traffic_src = rj["conv_family"]["source"]
    except Exception:
        pass
    pipe_ops = 3.0 * fam["conv_tc"]["flops"] + 6.0 * fam["conv_tcp"]["flops"] + 3.0 * fam["conv_tt"]["flops"]   # bf16-equivalent tensor work issued
    roofline = {"kernel": "tcgen05 conv family: conv_tc_kernel (kind::f16, bf16 hi/lo split, layers downstream of the VQ) + "
                          "conv_tt_kernel (transposed formulation, time = MMA N = 256, fp16 hi + scaled-lo split with "
                          "register-promoted accumulation, layers upstream of the VQ; conv_tcp_kernel is its TF32 fallback): all "
                          "eligible Conv1d/ConvTranspose1d/Linear layers",
                "family_ms_per_step": {k: fam[k]["ms"] for k in ("conv_tc", "conv_tcp", "conv_tt")},
                "bound": "tensor", "achieved": conv_tflops, "peak": peaks["tflops"], "unit": "TFLOP/s",
                "frac": conv_tflops / peaks["tflops"], "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": f"{peaks['source']} bf16 dense sustained (MEASURED_PEAKS.json)",
                "note": "achieved counts ALGORITHMIC fp32 FLOPs (2*MACs) per launch / mean launch time; an fp32-faithful "
                        "product costs 3 MMAs (bf16 / fp16 splits; 3 half-rate MMAs for the TF32 fallback), so the tensor pipe does >= 3x "
                        "this work; traffic is DRAM read+write bytes per launch (ncu), to compare with "
                        "per_launch.algorithmic_gb_per_step / launches_per_step",
                "tensor_pipe_frac_est": pipe_ops / (conv["ms"] * 1e-3) / 1e12 / peaks["tflops"] if conv["ms"] > 0 else 0.0,
                "per_launch": {"launches_per_step": conv["launches"], "avg_ms": conv["ms"] / max(1, conv["launches"]),
                               "algorithmic_gflop_per_step": conv["flops"] / 1e9,
                               "algorithmic_gb_per_step": conv["bytes"] / 1e9,
                               "achieved_gbs": conv["bytes"] / (conv["ms"] * 1e-3) / 1e9 if conv["ms"] > 0 else 0.0},
                "share_of_step": conv["ms"] / (ms_total / args.steps),
                "other_families_ms_per_step": {k: v["ms"] for k, v in fam.items() if k not in ("conv_tc", "conv_tcp", "conv_tt")},
                "whole_path": {"hbm_roofline_audio_s_per_s": peaks["hbm_gbs"] * 1e3 / MB_PER_AUDIO_S,
                               "tensor_roofline_audio_s_per_s": peaks["tflops"] * 1e3 / GFLOP_PER_AUDIO_S,
                               "frac_of_hbm_roofline": value / world / (peaks["hbm_gbs"] * 1e3 / MB_PER_AUDIO_S),
                               "frac_of_tensor_roofline": value / world / (peaks["tflops"] * 1e3 / GFLOP_PER_AUDIO_S)}}

    # ---- configs[0]: single 4 s utterance latency (B = 1), device-resident and end to end ----
    x1 = xs[0][:1].contiguous()
    x1h = xs_host[0][:1].contiguous().pin_memory()
    for _ in range(3):
        codec.forward(x1, n_c=2)
    nlat = 20
    ms_b1 = timed(lambda i: codec.forward(x1, n_c=2), nlat) / nlat
    o1 = codec.forward_host(x1h, n_c=2)
    ob1 = (o1[0], o1[1][0], o1[1][1], o1[1][2])
    ms_b1_e2e = timed(lambda i: codec.forward_host(x1h, n_c=2, out=ob1), nlat) / nlat
    latency = {"workload": "BASELINE configs[0]: single 4 s 24 kHz utterance, full codec forward, 1 GPU",
               "ms_device_resident": ms_b1, "ms_e2e_host_buffers": ms_b1_e2e,
               "audio_s_per_s": UTT_SECONDS / (ms_b1 * 1e-3), "launches": codec.launch_count()}
    try:    # the same forward replayed from one CUDA graph (Codec.forward_graphed)
        for _ in range(2):
            codec.forward_graphed(x1, n_c=2)
        latency["ms_cuda_graph_replay"] = timed(lambda i: codec.forward_graphed(x1, n_c=2), nlat) / nlat
    except Exception as exc:   # report, do not hide: the eager numbers above stand on their own
        latency["cuda_graph_error"] = str(exc).splitlines()[0][:200]

    # ---- library baseline (rank 0, N=1 only): the reference's own ATen call sequence under PyTorch eager on THIS GPU ----
    library = None
    if rank == 0 and world == 1 and not args.no_library_baseline:
        library = library_baseline(xs[0], dev)

    # ---- CPU baseline (rank 0, N=1 only): bounded sample of the same workload ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, _, cores, sample = cpu_reference_run(steps=2, warmup=1)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}

    if rank == 0:
        print(json.dumps({"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                          "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
                          "scaling": "weak", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
                          "config": config, "clocks": clocks,
                          "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                                  "ms_per_step": ms_e2e / args.steps},
                          "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
                          "library_baseline": library, "latency_b1": latency}))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
