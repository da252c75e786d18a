#!/usr/bin/env python
"""bench.py - headline benchmark of parakeet_b200: one JSON result line on stdout.

Workload (BASELINE.json configs[1]): Parallel WaveGAN generator inference, batch 32, 80-mel x 400 frames -> 3.84 M
samples of 24 kHz audio per step, CSMSC generator (30 residual layers, 64/128 channels, upsample [4,5,3,5]), random
weights of that architecture, synthetic N(0,1) mel + noise.  One step = one pass of the generator over one batch.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

--dump-outputs DIR writes the waveform the last timed step computed on rank 0 (B, 1, T float32, 15 MB) to DIR/wav.npy; the
weights and inputs are seeded, so two builds run with the same arguments can be compared output for output.

N > 1 is launched by torchrun (one rank per GPU); utterances are independent, so every rank runs its own batch of 32
with no data-path collective (weak scaling) and `value` is the whole-job aggregate.  The same line also carries, at every N,
`cfg3_strong` (BASELINE cfg 3: FastSpeech2 -> PWG synthesis of the SAME 32 utterances sharded over the ranks, results gathered
on rank 0 and copied to the host: strong scaling) and `cfg5_train` (BASELINE cfg 5: FastSpeech2 training step on a global
batch of 64 with the NCCL all-reduce of the flat gradient; all-reduce time and bus bandwidth reported separately).
`--impl reference` times the reference algorithm's CPU path (the torch-CPU oracle restatement; PaddlePaddle itself is not
installable here, see DESIGN.md) with all host threads on a bounded sample of the same workload; the `cpu_baseline` of the
N=1 line uses the same procedure and sample (cpu_leg).
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

BATCH, FRAMES, HOP = 32, 400, 300
FLOP_PER_SAMPLE_LAYER = 2 * (128 * (3 * 64 + 80) + 128 * 64)       # 86 016: conv k3 + aux 1x1 + skip/out 1x1 (SURVEY 8d)
FLOP_PER_SAMPLE = 30 * FLOP_PER_SAMPLE_LAYER + 2 * 64 * 64 + 2 * 64 + 2 * 64  # 2 588 928


def peaks():
    p = dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            m = json.load(f)
        p.update(hbm_gbs=m["hbm_gbs"], bf16_tflops=m["bf16_tflops"],
                 bf16_tflops_sustained=m.get("bf16_tflops_sustained", m["bf16_tflops"]), source="measured (MEASURED_PEAKS.json)")
    except Exception:
        pass
    return p


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "samples": len(sm),
                "reasons": sorted(reasons)}


def cpu_reference_step(params, x, c):
    import torch
    from oracle import pwg as opwg
    with torch.no_grad():
        return opwg.generator_forward(params, x, c)


def pick_cpu_threads(params, x, c):
    """The CPU path is timed at its best thread count (oversubscribing small convs on a 100+ core host is slower)."""
    import torch
    cores = os.cpu_count() or 1
    best, best_t = cores, None
    xs, cs = x[:1, :, :HOP * 40].contiguous(), c[:1, :, :44].contiguous()
    for n in sorted({cores, max(cores // 2, 1), max(cores // 4, 1), 32, 16, 8} & set(range(1, cores + 1)), reverse=True):
        torch.set_num_threads(n)
        cpu_reference_step(params, xs, cs)
        t0 = time.perf_counter()
        cpu_reference_step(params, xs, cs)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best


CPU_SAMPLE_UTTS = 1          # bounded sample of the CPU legs: 1 of the 32 utterances (400 mel frames = 120 000 samples) per step


def cpu_leg(steps, warmup, seed=2):
    """ONE procedure for both CPU numbers (`cpu_baseline` of the N=1 line and the `--impl reference` arm): the torch-CPU oracle
    restatement of PWGGenerator.forward with the CSMSC architecture, the same bounded sample per step, thread count picked
    once, `warmup` untimed passes, then `steps` timed passes.  -> (samples/s, cores, sample description, seconds per step)."""
    import torch
    from oracle import pwg as opwg
    params = opwg.fold_weight_norm(opwg.synth_params(seed, weight_norm=True))
    x, c = opwg.synth_inputs(seed, batch=CPU_SAMPLE_UTTS, mel_frames=FRAMES)
    cores = pick_cpu_threads(params, x, c)
    for _ in range(max(warmup, 1)):
        cpu_reference_step(params, x, c)
    t0 = time.perf_counter()
    for _ in range(steps):
        cpu_reference_step(params, x, c)
    dt = (time.perf_counter() - t0) / steps
    sample = (f"{CPU_SAMPLE_UTTS} of {BATCH} utterances (400 mel frames = {FRAMES * HOP} samples) per step, torch-CPU fp32 oracle port, "
              f"{max(warmup, 1)} warm-up + {steps} timed passes, best of several thread counts = {cores} of {os.cpu_count()} host threads")
    return CPU_SAMPLE_UTTS * FRAMES * HOP / dt, cores, sample, dt


def workload_config(world):
    return {"workload": "pwg_generator_b32_mel400_24k", "global_batch": BATCH * world, "per_gpu_batch": BATCH,
            "mel_frames": FRAMES, "hop": HOP, "parallelism": f"batch-sharded x{world}, no collective",
            "l2": "inputs and working set (3 GB) larger than L2; no flush needed"}


def run_reference(args, rank):
    """The reference algorithm's CPU implementation (oracle restatement) on the host cores, bounded sample per step."""
    if rank != 0:
        return
    v, cores, sample, dt = cpu_leg(args.steps, args.warmup)
    print(json.dumps({
        "impl": "reference", "metric": "audio-samples/sec", "value": v, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus),
        "cpu_baseline": {"value": v, "unit": "samples/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def ljspeech_fastspeech2(dev, seed=1, **kw):
    """LJSpeech yaml (examples/fastspeech2/ljspeech/conf/default.yaml:33-75), vocab 80, random-init weights."""
    from parakeet_b200.models import FastSpeech2
    return FastSpeech2(80, 80, adim=384, aheads=2, elayers=4, eunits=1536, dlayers=4, dunits=1536,
                       positionwise_layer_type="conv1d", positionwise_conv_kernel_size=3, duration_predictor_layers=2,
                       duration_predictor_chans=256, duration_predictor_kernel_size=3, postnet_layers=5, postnet_filts=5,
                       postnet_chans=256, pitch_predictor_layers=5, pitch_predictor_chans=256, pitch_predictor_kernel_size=5,
                       pitch_embed_kernel_size=1, energy_predictor_layers=2, energy_predictor_chans=256,
                       energy_predictor_kernel_size=3, energy_embed_kernel_size=1, device=dev, seed=seed, **kw)


def cfg3_strong_scaling(gen, dev, rank, world, steps, barrier, max_over_ranks):
    """BASELINE cfg 3: FastSpeech2 + Parallel WaveGAN end-to-end synthesis of the SAME 32 utterances at every N (strong
    scaling): parallel.shard_indices deals them out by length, every rank synthesises its slice as one ragged batch
    (phoneme ids from pinned host memory), the padded results are gathered on rank 0 over NCCL and copied to pinned host
    memory - all inside the timed region."""
    import math
    import torch
    import torch.distributed as dist
    from parakeet_b200.parallel import shard_indices
    fs = ljspeech_fastspeech2(dev)
    sd = dict(fs.state_dict())
    sd["duration_predictor.linear.bias"] = torch.tensor([math.log(8.0)])   # predicted durations ~7 frames / phoneme
    fs.set_state_dict(sd)
    g = torch.Generator().manual_seed(3)                                    # same utterances on every rank
    lengths = torch.randint(60, 141, (BATCH,), generator=g).tolist()
    ids_all = torch.zeros(BATCH, max(lengths), dtype=torch.int64)
    for i, n in enumerate(lengths):
        ids_all[i, :n] = torch.randint(1, 79, (n,), generator=g)
    noise_seed = 1234
    mine = shard_indices(lengths, world, rank)
    n_mine = len(mine)
    assert n_mine * world == BATCH, "32 utterances divide evenly over 1/2/4/8 ranks"
    my_len = [lengths[i] for i in mine]
    ids_h = torch.zeros(n_mine, max(my_len), dtype=torch.int64)
    for r, i in enumerate(mine):
        ids_h[r, :lengths[i]] = ids_all[i, :lengths[i]]
    ids_h, il_h = ids_h.pin_memory(), torch.tensor(my_len, dtype=torch.int64).pin_memory()
    host_out = {}

    def step():
        ids, il = ids_h.to(dev, non_blocking=True), il_h.to(dev, non_blocking=True)
        mel, olens, _ = fs.batch_inference(ids, il)
        L = mel.shape[1]
        cc = mel.transpose(1, 2)
        cc = torch.cat([cc[:, :, :1].expand(-1, -1, 2), cc, cc[:, :, -1:].expand(-1, -1, 2)], dim=-1).contiguous()
        gn = torch.Generator(device=dev).manual_seed(noise_seed)
        noise = torch.randn(n_mine, 1, L * HOP, device=dev, generator=gn)
        wav = gen(noise, cc, lens=(olens * HOP).to(torch.int32))[:, 0]          # (n_mine, L * HOP), zeros past each utterance
        if world > 1:
            lmax = torch.tensor([wav.shape[1]], device=dev, dtype=torch.int64)
            dist.all_reduce(lmax, op=dist.ReduceOp.MAX)                         # common padded length for the gather
            pad = torch.zeros(n_mine, int(lmax.item()), device=dev)
            pad[:, :wav.shape[1]] = wav
            parts = [torch.empty_like(pad) for _ in range(world)] if rank == 0 else None
            dist.gather(pad, parts, dst=0)
            lens_parts = [torch.empty(n_mine, dtype=torch.int64, device=dev) for _ in range(world)] if rank == 0 else None
            dist.gather(olens.to(torch.int64), lens_parts, dst=0)
            if rank == 0:
                full, ol = torch.stack(parts), torch.stack(lens_parts)          # (world, n_mine, Lpad)
        else:
            full, ol = wav.unsqueeze(0), olens.to(torch.int64).unsqueeze(0)
        if rank == 0:
            key = tuple(full.shape)
            if key not in host_out:
                host_out.clear()
                host_out[key] = (torch.empty(full.shape, dtype=torch.float32).pin_memory(), torch.empty(ol.shape, dtype=torch.int64).pin_memory())
            host_out[key][0].copy_(full, non_blocking=True)
            host_out[key][1].copy_(ol, non_blocking=True)
            return host_out[key]
        return None

    import torch
    for _ in range(3):
        res = step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        res = step()
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1)) / steps
    if rank != 0:
        return None
    frames = int(res[1].sum())
    return {"workload": "fastspeech2+pwg synthesis of the same 32 utterances (60..140 phonemes), sharded by length over the ranks",
            "scaling": "strong", "n_gpus": world, "utterances_per_gpu": n_mine, "ms_per_step": ms, "mel_frames": frames,
            "samples_per_s": frames * HOP / (ms * 1e-3), "mel_frames_per_s": frames / (ms * 1e-3),
            "h2d_bytes_per_step": int(ids_h.numel() * 8 + il_h.numel() * 8) * world,
            "d2h_bytes_per_step": int(res[0].numel() * 4 + res[1].numel() * 8),
            "collectives": "1 all_reduce(MAX) of the padded length + 2 gathers of the results to rank 0 (NCCL)" if world > 1 else "none"}


def cfg5_train_step(dev, rank, world, steps, barrier, max_over_ranks):
    """BASELINE cfg 5: FastSpeech2 training step (forward + backward + ONE NCCL all-reduce of the flat gradient + Adam) on a
    global batch of 64 synthetic utterances split evenly over the ranks (strong scaling: 64 / N per GPU, 8 per GPU at N = 8)."""
    import torch
    import torch.distributed as dist
    from parakeet_b200.data import synthetic_fastspeech2_batch as synth_train_batch
    from parakeet_b200.training import FastSpeech2TrainStep
    GLOBAL = 64
    per = GLOBAL // world
    yaml_rates = dict(transformer_enc_dropout_rate=0.2, transformer_enc_positional_dropout_rate=0.2, transformer_enc_attn_dropout_rate=0.2,
                      transformer_dec_dropout_rate=0.2, transformer_dec_positional_dropout_rate=0.2, transformer_dec_attn_dropout_rate=0.2,
                      pitch_predictor_dropout=0.5, energy_predictor_dropout=0.5, pitch_embed_dropout=0.0, energy_embed_dropout=0.0)
    m = ljspeech_fastspeech2(dev, stop_gradient_from_pitch_predictor=True, **yaml_rates)   # same seed -> same weights on every rank
    ts = FastSpeech2TrainStep(m, learning_rate=1e-3, dropout=True, seed=1000 + rank)       # conf/default.yaml:56-74 dropout rates
    g = torch.Generator().manual_seed(5)
    lengths = torch.randint(60, 141, (GLOBAL,), generator=g).tolist()
    batch = synth_train_batch(55, lengths[rank * per:(rank + 1) * per])
    batch = {k: v.to(dev) for k, v in batch.items()}
    frames_local = torch.tensor([float(batch["speech_lengths"].sum())], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(frames_local)
    for _ in range(2):
        losses = ts.step(batch)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        losses = ts.step(batch)
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1)) / steps
    ar_ms, bus = None, None
    nbytes = ts.gflat.numel() * 4
    if world > 1:                                            # the exchange step alone (same buffer, same call)
        for _ in range(2):
            ts.buffers.all_reduce_grads(ts.group)
        barrier()
        e0.record()
        for _ in range(5):
            ts.buffers.all_reduce_grads(ts.group)
        e1.record()
        barrier()
        ar_ms = max_over_ranks(e0.elapsed_time(e1)) / 5
        bus = 2 * (world - 1) / world * nbytes / (ar_ms * 1e-3) / 1e9
    if rank != 0:
        return None
    return {"workload": "fastspeech2 training step with the yaml's dropout rates, global batch 64 (T ~ U{60..140} phonemes, durations U{2..12})", "scaling": "strong",
            "n_gpus": world, "per_gpu_batch": per, "ms_per_step": ms, "steps_per_s": 1e3 / ms,
            "mel_frames_per_s": float(frames_local.item()) / (ms * 1e-3), "loss": [float(v) for v in losses],
            "grad_allreduce_bytes": nbytes, "allreduce_ms": ar_ms, "allreduce_bus_gbs": bus,
            "collectives": "1 all_reduce(SUM) of the flat fp32 gradient per step (NCCL)" if world > 1 else "none"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-extra", action="store_true", help="skip the FastSpeech2 / end-to-end extras and the CPU baseline")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's output (rank 0) to DIR/wav.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return run_reference(args, rank)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    from parakeet_b200 import _lib
    from parakeet_b200.models import PWGGenerator

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=240))   # a failed rank must not hang the job
    lib = _lib.lib()

    # CSMSC generator_params (examples/GANVocoder/parallelwave_gan/baker/conf/default.yaml:23-45), random-init weights
    gen = PWGGenerator(layers=30, stacks=3, residual_channels=64, gate_channels=128, skip_channels=64, aux_channels=80,
                       aux_context_window=2, upsample_scales=[4, 5, 3, 5], use_weight_norm=True, device=dev, seed=2)
    gen.remove_weight_norm()                     # as synthesize.py does before inference
    g_in = torch.Generator().manual_seed(1002 + rank)
    c_h = torch.randn(BATCH, 80, FRAMES, generator=g_in)
    c_h = torch.cat([c_h[:, :, :1].expand(-1, -1, 2), c_h, c_h[:, :, -1:].expand(-1, -1, 2)], dim=-1).contiguous()  # replicate pad
    x_h = torch.randn(BATCH, 1, FRAMES * HOP, generator=g_in)
    x_h, c_h = x_h.pin_memory(), c_h.pin_memory()
    x, c = x_h.to(dev), c_h.to(dev)
    samples_per_step = BATCH * FRAMES * HOP

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    # ---------------- device-resident timed region ----------------
    for _ in range(args.warmup):
        y = gen(x, c)
    gen._layer_events = []                     # (start, end) CUDA events around the 30 residual-layer launches of each step
    sampler = ClockSampler(local_rank)
    sampler.start()
    t_wait = time.time()
    while not sampler.lines and time.time() - t_wait < 3.0:     # nvidia-smi needs a moment to emit its first sample
        y = gen(x, c)
        torch.cuda.synchronize()
    barrier()
    first_line = len(sampler.lines)
    launches0 = lib.pk_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        y = gen(x, c)
    e1.record()
    barrier()
    launches = lib.pk_launch_count() - launches0
    sampler.lines = sampler.lines[max(first_line - 1, 0):]      # samples taken during the timed region (+ the one straddling its start)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:        # before the sections below call gen again
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "wav.npy"), y.float().cpu().numpy())
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    layer_ms = [a.elapsed_time(b) for a, b in gen._layer_events]
    gen._layer_events = None
    ms_per_step = ms_total / args.steps
    value = world * samples_per_step * args.steps / (ms_total * 1e-3)

    # ---------------- end to end through the public API with host buffers ----------------
    wav_h = torch.empty(BATCH, 1, FRAMES * HOP, dtype=torch.float32).pin_memory()
    for _ in range(2):
        wav_h.copy_(gen(x_h.to(dev, non_blocking=True), c_h.to(dev, non_blocking=True)), non_blocking=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        xd = x_h.to(dev, non_blocking=True)
        cd = c_h.to(dev, non_blocking=True)
        wav_h.copy_(gen(xd, cd), non_blocking=True)
    e1.record()
    barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))
    e2e_value = world * samples_per_step * args.steps / (ms_e2e * 1e-3)

    # ---------------- the other two multi-GPU configurations of BASELINE.json (every rank takes part) ----------------
    cfg3 = cfg5 = None
    if not args.no_extra:
        try:
            cfg3 = cfg3_strong_scaling(gen, dev, rank, world, max(args.steps // 2, 3), barrier, max_over_ranks)
        except Exception as ex:
            cfg3 = {"error": repr(ex)}
        try:
            cfg5 = cfg5_train_step(dev, rank, world, 5, barrier, max_over_ranks)
        except Exception as ex:
            cfg5 = {"error": repr(ex)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk = peaks()
    layer_launch_ms = sum(layer_ms) / max(len(layer_ms), 1) / 30.0            # average residual-layer kernel duration
    flops_per_launch = FLOP_PER_SAMPLE_LAYER * samples_per_step               # algorithmic (one pass), 330 GFLOP
    achieved_tf = flops_per_launch / (layer_launch_ms * 1e-3) / 1e12
    fcond = PWGGenerator._frame_cond()
    kernel = "pk::fc::pwg_layer_fc_kernel" if fcond else "pk::pwg_layer_pair_kernel"
    # dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of that kernel at this exact configuration, from the committed
    # `ncu --set full` capture (profiles/roofline_traffic.json, written by scripts/ncu_traffic.py from the .ncu-rep); null when
    # no capture of the current kernel is on file
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            ent = json.load(f).get(kernel)
        if ent:
            traffic, traffic_src = ent["dram_bytes_per_launch"], ent.get("source")
    except Exception:
        pass
    bytes_per_sample = (256 + 256 + 512) if fcond else (256 + 256 + 512 + 320)   # x rd, x wr, skip rmw (+ conditioning planes)
    roofline = {"bound": "tensor", "kernel": kernel, "achieved": achieved_tf, "peak": pk["bf16_tflops_sustained"],
                "unit": "TFLOP/s", "frac": achieved_tf / pk["bf16_tflops_sustained"],
                "traffic": traffic, "traffic_unit": "bytes/launch", "traffic_source": traffic_src,
                "peak_source": pk["source"] + ", sustained bf16 (kernel timed inside a long step)",
                "launch_ms": layer_launch_ms, "launches_per_step": 30,
                "note": "algorithmic FLOPs of the reference's block (86 016 per sample per layer); split-bf16 operands execute 3 "
                        "tensor-core passes per product (+ the residual pass)",
                "hbm_algorithmic_bytes_per_launch": samples_per_step * bytes_per_sample,
                "hbm_algorithmic_gbs": (samples_per_step * bytes_per_sample) / (layer_launch_ms * 1e-3) / 1e9,
                "hbm_peak_gbs": pk["hbm_gbs"]}

    out = {"metric": "audio-samples/sec", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "bf16x3 (split-bf16 operands, fp32 accumulate; fp32-grade, 1e-3 parity)", "data": "synthetic",
           "config": workload_config(world),
           "clocks": clocks, "gpu_launches": int(launches),
           "e2e": {"value": e2e_value, "unit": "samples/s", "ms_per_step": ms_e2e / args.steps,
                   "h2d_bytes_per_step": int(x_h.numel() * 4 + c_h.numel() * 4), "d2h_bytes_per_step": int(wav_h.numel() * 4),
                   "api": "PWGGenerator.forward(x, c) with pinned host tensors"},
           "roofline": roofline}
    if cfg3 is not None:
        out["cfg3_strong"] = cfg3
    if cfg5 is not None:
        out["cfg5_train"] = cfg5

    if not args.no_extra and world == 1:      # single-GPU side metrics; the scaling runs report the headline + cfg3 / cfg5 only
        try:
            import math
            fs = ljspeech_fastspeech2(dev)
            sd = dict(fs.state_dict())
            sd["duration_predictor.linear.bias"] = torch.tensor([math.log(8.0)])   # predicted durations ~7 frames / phoneme
            fs.set_state_dict(sd)
            g = torch.Generator().manual_seed(3)
            lengths = torch.randint(60, 141, (BATCH,), generator=g).tolist()
            ids = torch.zeros(BATCH, max(lengths), dtype=torch.int64)
            for i, n in enumerate(lengths):
                ids[i, :n] = torch.randint(1, 79, (n,), generator=g)
            il = torch.tensor(lengths, dtype=torch.int64)
            ids, il = ids.to(dev), il.to(dev)
            for _ in range(3):
                mel, olens, _ = fs.batch_inference(ids, il)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(args.steps):
                mel, olens, _ = fs.batch_inference(ids, il)
            e1.record()
            torch.cuda.synchronize()
            fs_ms = e0.elapsed_time(e1) / args.steps
            frames = int(olens.sum())
            out["extra"] = {"fastspeech2_b32": {"mel_frames_per_s": frames / (fs_ms * 1e-3), "ms_per_step": fs_ms, "frames": frames}}
            # WaveFlow (cfg4): 64 channels, 8 flows x 8 layers, n_group 16, batch 16, 400 mel frames -> 102 128 samples each
            from parakeet_b200.models import ConditionalWaveFlow
            wf = ConditionalWaveFlow([16, 16], 8, 8, 16, 64, 80, (3, 3), device=dev, seed=4)
            sdw = dict(wf.state_dict())
            gw = torch.Generator().manual_seed(4)
            for k_ in sdw:
                if "output_proj" in k_:      # the reference zero-initialises these (identity flow); use small random values
                    sdw[k_] = (torch.rand(sdw[k_].shape, generator=gw) * 2 - 1) * 0.05
            wf.set_state_dict(sdw)
            melw = (torch.randn(16, 80, FRAMES, generator=gw) * 0.5 - 3).to(dev)
            zw = torch.randn(16, 256 * FRAMES - 272, generator=gw).to(dev)
            for _ in range(3):               # eager call, graph capture, first replay
                wf.infer(melw, z=zw)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(3):
                aw = wf.infer(melw, z=zw)
            e1.record()
            torch.cuda.synchronize()
            wf_ms = e0.elapsed_time(e1) / 3
            out["extra"]["waveflow_b16_c64"] = {"samples_per_s": aw.numel() / (wf_ms * 1e-3), "ms_per_step": wf_ms,
                                                "note": "cfg4; one persistent dataflow launch per flow (pk_waveflow_flow), one CUDA graph per call"}
            # the same batch on the reference's shipped WaveFlow config (examples/waveflow/config.py: 128 residual channels)
            del wf
            wf2 = ConditionalWaveFlow([16, 16], 8, 8, 16, 128, 80, (3, 3), device=dev, seed=5)
            for _ in range(3):
                wf2.infer(melw, z=zw)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(3):
                aw = wf2.infer(melw, z=zw)
            e1.record()
            torch.cuda.synchronize()
            wf_ms = e0.elapsed_time(e1) / 3
            out["extra"]["waveflow_b16_c128"] = {"samples_per_s": aw.numel() / (wf_ms * 1e-3), "ms_per_step": wf_ms,
                                                 "note": "shipped config (128 channels), same batch as cfg4"}
            del wf2
            # Parallel WaveGAN training step (the workload of the reference's own benchmark harness, tests/benchmark/PWGAN/
            # run_benchmark.sh: batch 6, batch_max_steps 25 500, metric sequences/s), past discriminator_train_start_steps: generator
            # step with the adversarial term + discriminator step
            from parakeet_b200.models import PWGDiscriminator
            from parakeet_b200.training import PWGTrainStep
            gen_t = PWGGenerator(layers=30, stacks=3, residual_channels=64, gate_channels=128, skip_channels=64, aux_channels=80,
                                 aux_context_window=2, upsample_scales=[4, 5, 3, 5], use_weight_norm=True, device=dev, seed=5)
            dis_t = PWGDiscriminator(device=dev, seed=6)
            pts = PWGTrainStep(gen_t, dis_t, discriminator_train_start_steps=0)
            pts.iteration = 1
            gt = torch.Generator().manual_seed(9)
            bt, ft = 6, 85
            wav_t = (torch.randn(bt, 1, ft * HOP, generator=gt) * 0.3).to(dev)
            mel_t = torch.randn(bt, 80, ft + 4, generator=gt).to(dev)
            for _ in range(2):
                lt = pts.update_core((wav_t, mel_t))
            torch.cuda.synchronize()
            e0.record()
            for _ in range(5):
                lt = pts.update_core((wav_t, mel_t))
            e1.record()
            torch.cuda.synchronize()
            pt_ms = e0.elapsed_time(e1) / 5
            out["extra"]["pwg_train_step_b6"] = {"sequences_per_s": bt / (pt_ms * 1e-3), "samples_per_s": bt * ft * HOP / (pt_ms * 1e-3),
                                                 "ms_per_step": pt_ms, "generator_loss": float(lt["generator_loss"]),
                                                 "discriminator_loss": float(lt["discriminator_loss"]),
                                                 "note": "PWGUpdater.update_core: G step (MR-STFT + adversarial) + D step, batch 6 x 25 500 samples, "
                                                         "unfused training formulation (separate tcgen05 GEMMs + element-wise kernels)"}
        except Exception as ex:  # extras must never break the headline line
            out.setdefault("extra", {})["error"] = repr(ex)
    if not args.no_extra and world == 1:
        # CPU baseline (rank 0, N=1 only): the same procedure and sample as the `--impl reference` arm (cpu_leg), fewer passes
        v, cores, sample, _ = cpu_leg(steps=2, warmup=1)
        out["cpu_baseline"] = {"value": v, "unit": "samples/s", "cores": cores, "kind": "port", "sample": sample}
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
