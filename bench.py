#!/usr/bin/env python
"""bench.py -- throughput of the two WaveNet hot paths on B200, with roofline and the CPU baseline beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload all|generate|train]
                    [--dump-outputs DIR]

Under torchrun (N>1) every rank runs; rank 0 prints ONE JSON line.  Every timed loop runs --steps iterations.

Primary metric (BASELINE.json configs[1]): generate_fast samples/sec -- layers=10, blocks=5, 256 channels,
16000 samples (1 s of 16 kHz audio), single stream; a "step" is one full generate_fast run.  At N>1 each rank runs
an independent replica (the path does not shard; SURVEY.md section 8e).
Secondary metric, same JSON line under "train": training-forward mu-law frames/sec (configs[2] shape: B=8 per GPU,
L=16000, output_length=10885), batch-sharded over the ranks (weak scaling; the forward has no collective).

`value` is device-timed with inputs resident in HBM; `e2e` goes through the reference-facing Python API with host
buffers.  `cpu_baseline` / `--impl reference` time the CPU port of the reference (oracle/) on the host cores.

`--dump-outputs DIR` (e.g. bench_outputs/, which git ignores) writes what the last timed step returned, as float32
.npy files, so that two builds can be compared output for output (the inputs are seeded): DIR/generate_indices.npy,
the (1, 16000) sampled class indices, and with the training forward DIR/train_logits.npy, a fixed seeded sample of
TRAIN_DUMP_ROWS of its (87080, 256) logits, whose row numbers are in DIR/train_logits_rows.npy.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "pytorch-wavenet_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np
import torch

GEN_KW = dict(layers=10, blocks=5, dilation_channels=256, residual_channels=256, skip_channels=256,
              end_channels=256, classes=256, output_length=16000 - 5116 + 1, kernel_size=2, bias=False)
GEN_SAMPLES = 16000
TRAIN_B, TRAIN_L = 8, 16000
TEMPERATURE = 1.0
TRAIN_DUMP_ROWS = 8192
GEN_WORKLOAD = ("cfg2 generate_fast: layers=10 blocks=5 ch=256 classes=256, 16000 samples, single stream, temperature=1.0, "
                "seeded random-init weights")


# ------------------------------------------------------------------------------------------------ helpers
def measured_peaks(what="hbm"):
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        if what == "tensor":
            return float(d["bf16_tflops_sustained"]), "measured sustained cuBLAS bf16 (MEASURED_PEAKS.json)"
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return (1400.0 if what == "tensor" else 6650.0), "fallback (B200_PROFILING.md)"


def captured_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed `ncu --set full` capture
    (profiles/traffic.json, written by tools/ncu_summary.py traffic ...); None when there is no capture of it."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(path):
        return None, None
    with open(path) as f:
        d = json.load(f)
    e = d.get(kernel)
    return (e["dram_bytes_per_launch"], e["source"]) if e else (None, None)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); power.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        os.unlink(self.path)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def dist_setup(n_gpus):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    else:
        torch.cuda.set_device(0)
    return world, rank, local


def barrier_sync(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(x, world):
    if world == 1:
        return x
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def build_model(kw, seed=0):
    import wavenet_model as wmod
    torch.manual_seed(seed)
    return wmod.WaveNetModel(**kw)


class L2Flush:
    def __init__(self):
        self.buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def __call__(self):
        self.buf.fill_(1)


def write_outputs(path, arrays):
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------ generation
def bench_generate(args, world, rank, dump=None):
    model = build_model(GEN_KW).cuda()
    rt = model._runtime()
    NS, n = 1, GEN_SAMPLES
    s = rt.sampler(NS)
    dev = rt.device()
    first = torch.full((NS, 1), 128, dtype=torch.int32, device=dev)
    np.random.seed(rank)
    uni = torch.from_numpy(np.random.random_sample((NS, n))).to(dev)
    out = torch.zeros(NS, n, dtype=torch.int32, device=dev)
    flush = L2Flush()

    def step():
        rt.generate_resident(s, first, 1, n, TEMPERATURE, 0.0, out, d_uni=uni)

    for _ in range(args.warmup):
        step()
    barrier_sync(world)
    clocks = ClockSampler(torch.cuda.current_device())
    clocks.start()
    evs = []
    t_wall0 = time.perf_counter()
    for _ in range(args.steps):
        flush()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step()
        e1.record()
        evs.append((e0, e1))
    barrier_sync(world)
    t_wall = time.perf_counter() - t_wall0
    if dump is not None:                  # before the argmax run below reuses `out`
        dump["generate_indices"] = out.cpu().numpy().astype(np.float32)
    clk = clocks.stop()
    ms = sum(a.elapsed_time(b) for a, b in evs)
    ms = max_over_ranks(ms, world)
    value = world * NS * n * args.steps / (ms / 1e3)

    # end to end through the reference-facing API: host first_samples / numpy RNG in, float64 waveform out
    model.generate_fast(256, temperature=TEMPERATURE)                     # warm
    barrier_sync(world)
    t0 = time.perf_counter()
    e2e_steps = args.steps
    for _ in range(e2e_steps):
        audio = model.generate_fast(n, temperature=TEMPERATURE)
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0, world)
    assert audio.shape == (n,) and np.isfinite(audio).all()
    e2e = {"value": world * n * e2e_steps / e2e_s, "unit": "samples/s",
           "h2d_bytes_per_step": int(rt.h2d_bytes_last), "d2h_bytes_per_step": int(rt.d2h_bytes_last),
           "api": "WaveNetModel.generate_fast(16000, temperature=1.0) -> float64 ndarray"}

    import ctypes, native
    # argmax path, for reference
    t_arg = []
    for _ in range(args.steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rt.generate_resident(s, first, 1, n, 0.0, 0.0, out)
        e1.record()
        torch.cuda.synchronize()
        t_arg.append(e0.elapsed_time(e1))

    # cfg4: 64 independent streams batched on one GPU (aggregate samples/s); shorter run, same per-sample cost
    batched = None

    def run_streams(NB, nb):
        sb = rt.sampler(NB)
        first_b = torch.full((NB, 1), 128, dtype=torch.int32, device=dev)
        uni_b = torch.from_numpy(np.random.random_sample((NB, nb))).to(dev)
        out_b = torch.zeros(NB, nb, dtype=torch.int32, device=dev)
        rt.generate_resident(sb, first_b, 1, 64, TEMPERATURE, 0.0, out_b[:, :64].contiguous(), d_uni=uni_b[:, :64].contiguous())
        tb = []
        for _ in range(args.steps):
            flush()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rt.generate_resident(sb, first_b, 1, nb, TEMPERATURE, 0.0, out_b, d_uni=uni_b)
            e1.record()
            torch.cuda.synchronize()
            tb.append(e0.elapsed_time(e1))
        g_, b_, x_ = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        native.lib().wn_gen_launch_info(sb["handle"], ctypes.byref(g_), ctypes.byref(b_), ctypes.byref(x_))
        return max_over_ranks(min(tb), world), g_.value, b_.value

    if not args.no_batched:
        NB, nb = 64, 1000
        sb = rt.sampler(NB)
        first_b = torch.full((NB, 1), 128, dtype=torch.int32, device=dev)
        uni_b = torch.from_numpy(np.random.random_sample((NB, nb))).to(dev)
        out_b = torch.zeros(NB, nb, dtype=torch.int32, device=dev)
        rt.generate_resident(sb, first_b, 1, 64, TEMPERATURE, 0.0, out_b[:, :64].contiguous(), d_uni=uni_b[:, :64].contiguous())
        tb = []
        for _ in range(args.steps):
            flush()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rt.generate_resident(sb, first_b, 1, nb, TEMPERATURE, 0.0, out_b, d_uni=uni_b)
            e1.record()
            torch.cuda.synchronize()
            tb.append(e0.elapsed_time(e1))
        tbm = max_over_ranks(min(tb), world)
        gb_, bb_, _bars = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        native.lib().wn_gen_launch_info(sb["handle"], ctypes.byref(gb_), ctypes.byref(bb_), ctypes.byref(_bars))
        # the same kernel where its 16-CTA clusters are all co-resident (7 x 8 streams) and at the 8-CTA variant's capacity
        t56, g56, _ = run_streams(56, nb)
        t120, g120, _ = run_streams(120, nb)
        other = {"56_streams": {"value": world * 56 * nb / (t56 / 1e3), "us_per_step": t56 * 1e3 / nb, "grid": g56},
                 "120_streams": {"value": world * 120 * nb / (t120 / 1e3), "us_per_step": t120 * 1e3 / nb, "grid": g120}}
        batched = {"workload": "cfg4: 64 independent streams, same net, 1000 samples per stream, temperature=1.0",
                   "kernel": "gen_kernel_cl8 (8 streams per cluster, mma.sync bf16 hi/lo pairs, st.async block exchange)",
                   "us_per_step": tbm * 1e3 / nb, "other_stream_counts": other,
                   "value": world * NB * nb / (tbm / 1e3), "unit": "samples/s (aggregate over streams)",
                   "per_stream_samples_per_s": nb / (tbm / 1e3), "ms_per_launch": tbm, "grid": gb_.value, "block": bb_.value,
                   "distinct_streams": int(len({tuple(r) for r in out_b[:, :32].cpu().numpy().tolist()}))}

    g, b, bars = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    native.lib().wn_gen_launch_info(s["handle"], ctypes.byref(g), ctypes.byref(b), ctypes.byref(bars))
    weight_bytes = 4 * sum(p.numel() for p in model.parameters())
    per_launch_ms = ms / args.steps
    peak, peak_src = measured_peaks()
    # algorithmic bytes per launch: every sample touches all weights once (79.4 MB fp32: they do not fit on chip) plus
    # k ring columns read and one written per layer
    alg_bytes = n * (weight_bytes + 50 * 3 * 256 * 4)
    kid = native.lib().wn_gen_kernel_id(s["handle"])
    kname = {6: "gen_kernel_cl8", 3: "gen_kernel_fast", 4: "gen_kernel_cluster", 2: "gen_kernel_ll", 1: "gen_kernel", 5: "gen_kernel_x2"}[kid]
    traffic, tsrc = captured_traffic(kname)
    sm_mhz = clk.get("sm_mhz") or 1965.0
    macs = sum(p.numel() for p in model.parameters()) - 256 * 256      # start conv is a gather
    issue_peak = 148 * 128 * sm_mhz * 1e6                               # FMA lanes per second at the clock seen
    roof = {"kernel": kname, "bound": "hbm", "achieved": alg_bytes / (per_launch_ms / 1e3) / 1e9, "peak": peak,
            "unit": "GB/s", "frac": alg_bytes / (per_launch_ms / 1e3) / 1e9 / peak,
            "traffic": None if traffic is None else traffic, "traffic_source": tsrc, "peak_source": peak_src,
            "us_per_sample": per_launch_ms * 1e3 / n, "exchange_stages_per_sample": bars.value,
            "us_per_exchange_stage": per_launch_ms * 1e3 / n / bars.value, "grid": g.value, "block": b.value,
            "issue": {"fma_per_sample": macs, "achieved_gfma_s": macs * n / (per_launch_ms / 1e3) / 1e9,
                      "peak_gfma_s": issue_peak / 1e9, "frac": macs * n / (per_launch_ms / 1e3) / issue_peak}}
    gen_dtype = ("bf16 hi/lo operand pairs, 3 MMAs per product, f32 accumulate (f32-class: logits within 2e-5 of the f32 "
                 "kernels, 1e-4 of the reference)") if kid == 6 else "f32"
    return dict(value=value, dtype=gen_dtype, ms_per_step=ms / args.steps, clocks=clk, e2e=e2e, roofline=roof,
                argmax_samples_per_s=n / (min(t_arg) / 1e3), wall_s=t_wall, launches=args.steps, batched=batched)


# ------------------------------------------------------------------------------------------------ training forward
def train_alg_bytes(model, B, L, dense_input):
    """SURVEY.md section 8d: per layer e*B*(R*T_in + R*T_out + 2*S*T_final); start and head added."""
    import wavenet_model as wmod
    dil = [d for d, _ in model.dilations]
    plan = wmod.StackPlan(dil, model.kernel_size, L)
    R, S, C = model.residual_channels, model.skip_channels, model.classes
    e = 4
    per_layer = []
    for i in range(len(dil)):
        t_in, t_out = L - plan.in_start[i], L - plan.out_start[i]
        per_layer.append(e * B * (R * t_in + R * t_out + (1 if i == 0 else 2) * S * plan.t_final))
    start = B * L * (C * e if dense_input else 1) + e * B * R * L
    head = e * B * (S * plan.t_final + C * model.output_length)
    flops = sum(2 * B * (L - plan.out_start[i]) * (2 * model.kernel_size * R * model.dilation_channels +
                                                     model.dilation_channels * R) +
                2 * B * plan.t_final * model.dilation_channels * S for i in range(len(dil)))
    return per_layer, start, head, flops


def bench_train(args, world, rank, dump=None):
    kw = dict(GEN_KW)
    model = build_model(kw).cuda()
    rt = model._runtime()
    B, L = TRAIN_B, TRAIN_L
    idx = torch.randint(0, 256, (B, L), generator=torch.Generator().manual_seed(1234 + rank))
    d_idx = idx.to(torch.uint8).cuda()
    flush = L2Flush()
    with torch.no_grad():
        for _ in range(args.warmup):
            y = model.forward_indices(d_idx)
        barrier_sync(world)
        clocks = ClockSampler(torch.cuda.current_device())
        clocks.start()
        evs, bevs = [], []
        for _ in range(args.steps):
            flush()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            rt.block_events = (b0, b1)
            e0.record()
            y = model.forward_indices(d_idx)
            e1.record()
            evs.append((e0, e1)); bevs.append((b0, b1))
        rt.block_events = None
        barrier_sync(world)
        clk = clocks.stop()
        if dump is not None:
            rows = torch.randperm(y.shape[0], generator=torch.Generator().manual_seed(0))[:TRAIN_DUMP_ROWS].sort().values
            dump["train_logits_rows"] = rows.numpy().astype(np.float32)
            dump["train_logits"] = y[rows.to(y.device)].float().cpu().numpy()
        fwd_mode = getattr(rt, "last_block_mode", "ffma")
        ms = max_over_ranks(sum(a.elapsed_time(b) for a, b in evs), world)
        block_ms = sum(a.elapsed_time(b) for a, b in bevs) / args.steps
        value = world * B * L * args.steps / (ms / 1e3)

        # end to end through forward(): pinned host one-hot in, logits read back
        x_host = torch.zeros(B, 256, L).scatter_(1, idx.view(B, 1, L), 1.0).pin_memory()
        y_host = torch.empty(B * model.output_length, 256).pin_memory()
        model(x_host.cuda(non_blocking=True))
        barrier_sync(world)
        t0 = time.perf_counter()
        e2e_steps = args.steps
        for _ in range(e2e_steps):
            y = model(x_host.cuda(non_blocking=True))
            y_host.copy_(y, non_blocking=True)
            torch.cuda.synchronize()
        e2e_s = max_over_ranks(time.perf_counter() - t0, world)
        e2e = {"value": world * B * L * e2e_steps / e2e_s, "unit": "frames/s",
               "h2d_bytes_per_step": int(x_host.numel() * 4), "d2h_bytes_per_step": int(y_host.numel() * 4),
               "api": "WaveNetModel.forward((8,256,16000) one-hot fp32 from pinned host) -> logits copied to host"}
        # index API (uint8 indices in, argmax of logits out): the traffic-minimal use of the same kernels
        idx_host = idx.to(torch.uint8).pin_memory()
        am_host = torch.empty(B * model.output_length, dtype=torch.int64).pin_memory()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            am = model.forward_indices(idx_host.cuda(non_blocking=True)).argmax(1)
            am_host.copy_(am, non_blocking=True)
            torch.cuda.synchronize()
        e2e_idx_s = max_over_ranks(time.perf_counter() - t0, world)
    # opt-in single-pass TF32 blocks (outside the 1e-4 parity bar; reported for the HBM-bound regime only)
    fast = None
    if getattr(rt, "last_block_mode", "") == "tc" and args.variants:
        with torch.no_grad():
            y_exact = model.forward_indices(d_idx)
            rt.fast_tf32 = True
            for _ in range(2):
                y_fast = model.forward_indices(d_idx)
            fe = []
            for _ in range(args.steps):
                flush()
                b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                rt.block_events = (b0, b1)
                y_fast = model.forward_indices(d_idx)
                torch.cuda.synchronize()
                fe.append(b0.elapsed_time(b1))
            rt.block_events = None
            rt.fast_tf32 = False
            err = float((y_fast - y_exact).abs().max() / y_exact.abs().max())
        fms = sum(fe) / len(fe)
        per_layer_f, _, _, _ = train_alg_bytes(model, B, L, dense_input=False)
        hbm_peak, _ = measured_peaks()
        # pass A writes z and pass B reads it back: 2 more activation passes than the fused algorithmic minimum
        fast = {"mode": "single-pass TF32 blocks (opt-in, NOT the parity path)", "blocks_ms_per_step": fms,
                "logits_max_rel_err_vs_exact": err,
                "hbm_algorithmic_gbs": sum(per_layer_f) / (fms / 1e3) / 1e9,
                "hbm_frac_of_measured_peak": sum(per_layer_f) / (fms / 1e3) / 1e9 / hbm_peak}
        # the other fp32-class operand split, for comparison (3xTF32 when bf16 pairs are the default and vice versa)
        other = "tf32x3" if getattr(rt, "tc_precision", "tf32x3") == "bf16x2" else "bf16x2"
        keep = rt.tc_precision
        with torch.no_grad():
            rt.tc_precision = other
            for _ in range(2):
                y_other = model.forward_indices(d_idx)
            oe = []
            for _ in range(args.steps):
                flush()
                b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                rt.block_events = (b0, b1)
                y_other = model.forward_indices(d_idx)
                torch.cuda.synchronize()
                oe.append(b0.elapsed_time(b1))
            rt.block_events = None
            rt.tc_precision = keep
        fast["other_operand_split"] = {"operand_split": other, "blocks_ms_per_step": sum(oe) / len(oe),
                                       "logits_max_rel_diff_vs_default_split": float((y_other - y_exact).abs().max() / y_exact.abs().max())}
        del y_exact, y_fast, y_other
    # full training step on the same shapes: forward (saving activations) + backward + per-block gradient all-reduce
    import torch.nn.functional as F
    import data_parallel as dp
    import wavenet_training as wt
    red = dp.make_data_parallel(model)
    target = torch.randint(0, 256, (B * model.output_length,), generator=torch.Generator().manual_seed(99 + rank)).cuda()
    step_ms = []
    for i in range(1 + args.steps):
        model.zero_grad(set_to_none=True)
        barrier_sync(world)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        loss = wt.fused_cross_entropy(model.forward_indices(d_idx), target)
        loss.backward()
        e1.record()
        torch.cuda.synchronize()
        if i > 0:
            step_ms.append(e0.elapsed_time(e1))
    step_t = max_over_ranks(sum(step_ms) / len(step_ms), world)
    train_step = {"ms_per_step": step_t, "frames_per_s": world * B * L / (step_t / 1e3), "loss": float(loss.detach()),
                  "grad_allreduce_bytes_per_step": red.bytes_reduced // max(1, 1 + len(step_ms)) if world > 1 else 0,
                  "grad_buckets_per_step": red.buckets // max(1, 1 + len(step_ms)) if world > 1 else 0,
                  "forward_blocks": getattr(rt, "last_block_mode", "ffma"), "backward_data": getattr(rt, "last_bwd_mode", "ffma"),
                  "scaling": "weak (B=8 per GPU)"}
    del loss
    model.zero_grad(set_to_none=True)
    if world > 1 and B % world == 0:
        # strong scaling: the SAME global batch of 8 sequences split over the ranks
        sidx = torch.randint(0, 256, (B, L), generator=torch.Generator().manual_seed(777))
        stgt = torch.randint(0, 256, (B, model.output_length), generator=torch.Generator().manual_seed(778))
        mine = dp.shard_batch(sidx, rank, world).to(torch.uint8).cuda()
        mine_t = dp.shard_batch(stgt, rank, world).reshape(-1).cuda()
        sms = []
        for i in range(1 + args.steps):
            model.zero_grad(set_to_none=True)
            barrier_sync(world)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            wt.fused_cross_entropy(model.forward_indices(mine), mine_t).backward()
            e1.record()
            torch.cuda.synchronize()
            if i > 0:
                sms.append(e0.elapsed_time(e1))
        st = max_over_ranks(sum(sms) / len(sms), world)
        train_step["strong"] = {"global_batch": B, "ms_per_step": st, "frames_per_s": B * L / (st / 1e3)}
        model.zero_grad(set_to_none=True)
        # correctness of the data-parallel step, visible to the driver: rank-averaged gradients of a small 256-channel net
        # on a sharded batch vs the single-process gradients of the whole batch (SURVEY.md section 8e)
        import wavenet_model as wmod
        kw = dict(layers=3, blocks=2, dilation_channels=256, residual_channels=256, skip_channels=256, end_channels=256,
                  classes=256, output_length=64, kernel_size=2, bias=True)
        torch.manual_seed(5)
        small = wmod.WaveNetModel(**kw).cuda()
        gi = torch.randint(0, 256, (2 * world, 300), generator=torch.Generator().manual_seed(31))
        gt = torch.randint(0, 256, (2 * world, 64), generator=torch.Generator().manual_seed(32))
        F.cross_entropy(small.forward_indices(gi.cuda()), gt.reshape(-1).cuda()).backward()
        whole = {k: v.grad.detach().clone() for k, v in small.named_parameters()}
        small.zero_grad(set_to_none=True)
        dp.make_data_parallel(small)
        F.cross_entropy(small.forward_indices(dp.shard_batch(gi, rank, world).cuda()),
                        dp.shard_batch(gt, rank, world).reshape(-1).cuda()).backward()
        err = max(float((v.grad - whole[k]).abs().max() / whole[k].abs().max().clamp_min(1e-30))
                  for k, v in small.named_parameters())
        train_step["ddp_grad_max_rel_err"] = max_over_ranks(err, world)
        small._runtime().grad_reducer = None
        del small, whole
    model._runtime().grad_reducer = None
    per_layer, start_b, head_b, flops = train_alg_bytes(model, B, L, dense_input=False)
    n_layers = len(per_layer)
    peak, peak_src = measured_peaks()
    ach = (sum(per_layer) / n_layers) / (block_ms / n_layers / 1e3) / 1e9
    tflops = flops / (block_ms / 1e3) / 1e12
    mode = fwd_mode
    if mode == "tb":
        tpeak, tsrc = measured_peaks("tensor")
        traffic, trsrc = captured_traffic("block_fused_kernel")
        roof = {"kernel": "block_fused_kernel (tcgen05 cta_group::2, bf16 hi/lo pairs; all blocks in one persistent launch)",
                "bound": "tensor", "achieved": tflops, "peak": tpeak, "unit": "TFLOP/s", "frac": tflops / tpeak,
                "traffic": traffic, "traffic_source": trsrc, "peak_source": tsrc,
                "launches_per_step": getattr(rt, "last_block_launches", n_layers),
                "avg_block_ms": block_ms / n_layers, "operand_split": "bf16x2",
                "mma_per_product": 3, "tensor_pipe_equiv_frac": 3 * tflops / tpeak,
                "hbm_achieved_gbs": ach, "hbm_peak_gbs": peak, "hbm_frac": ach / peak,
                "alg_bytes_per_block": sum(per_layer) / n_layers,
                "alg_bytes_per_frame": (sum(per_layer) + start_b + head_b) / (B * L)}
    elif mode == "tc":
        tpeak, tsrc = measured_peaks("tensor")
        prec = getattr(rt, "tc_precision", "tf32x3")
        mma_per_flop = 3 if prec == "bf16x2" else 6          # bf16-rate MMA equivalents per algorithmic FLOP
        roof = {"kernel": "frames_gemm_tc<GATE> + frames_gemm_tc<RES_SKIP> (tcgen05, " +
                          ("kind::f16 on bf16 hi/lo pairs" if prec == "bf16x2" else "kind::tf32, 3xTF32") + ", one block = 2 launches)",
                "bound": "tensor", "achieved": tflops, "peak": tpeak, "unit": "TFLOP/s", "frac": tflops / tpeak,
                # dram__bytes_read+write of the two launches of one block from the ncu --set full capture
                # profiles/prof_tc_block_r1_e.txt (layer of the cfg-3 forward, 3xTF32 variant: same activation traffic)
                "traffic": 128.15e6 + 85.84e6 + 363.67e6 + 189.49e6,
                "traffic_note": "per block (2 launches), ncu capture profiles/prof_tc_block_r1_e.txt; 1.67x the algorithmic "
                                "bytes because z is written by the first launch and read back by the second",
                "peak_source": tsrc, "launches_per_step": 2 * n_layers,
                "avg_block_ms": block_ms / n_layers, "operand_split": prec,
                "note": "achieved counts the algorithmic fp32 FLOPs once; fp32-class accuracy costs three MMAs per product "
                        f"(hi*hi + lo*hi + hi*lo) = {mma_per_flop} bf16-rate equivalents per FLOP with the {prec} split, so "
                        f"frac*{mma_per_flop} is the share of the measured tensor peak the kernel keeps busy",
                "tensor_pipe_equiv_frac": mma_per_flop * tflops / tpeak,
                "hbm_achieved_gbs": ach, "hbm_peak_gbs": peak, "hbm_frac": ach / peak,
                "alg_bytes_per_block": sum(per_layer) / n_layers,
                "alg_bytes_per_frame": (sum(per_layer) + start_b + head_b) / (B * L)}
    else:
        roof = {"kernel": "block_fwd_kernel<128> (fused residual block, exact fp32 FFMA)", "bound": "hbm",
                "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None,
                "peak_source": peak_src, "launches_per_step": n_layers, "avg_launch_ms": block_ms / n_layers,
                "alg_bytes_per_launch": sum(per_layer) / n_layers,
                "alg_bytes_per_frame": (sum(per_layer) + start_b + head_b) / (B * L),
                "tflops_fp32_achieved": tflops,
                "note": "exact-fp32 mode is bound by the fp32 FMA pipe, not by HBM (AI ~196 FLOP/B)"}
    return dict(metric="training-forward mu-law frames/sec", value=value, unit="frames/s", ms_per_step=ms / args.steps,
                clocks=clk, e2e=e2e, e2e_index_api={"value": world * B * L * e2e_steps / e2e_idx_s, "unit": "frames/s",
                                                   "h2d_bytes_per_step": int(idx_host.numel()),
                                                   "d2h_bytes_per_step": int(am.numel() * 8)},
                roofline=roof, train_step=train_step, fast_tf32=fast, dtype="f32", scaling="weak",
                config={"workload": "cfg3 forward: layers=10 blocks=5 ch=256, B=8 per GPU, L=16000, output_length=10885, "
                                    "uint8 index input resident in HBM", "block_kernels": mode, "global_batch": world * B, "seq_len": L,
                        "l2": "256 MiB buffer written between timed iterations (L2 flush)",
                        "parallelism": f"dp{world} (batch shards, no collective in forward)"},
                launches=args.steps * rt.launches_last_forward)


# ------------------------------------------------------------------------------------------------ cfg 5: deep 512-channel stack, bf16
CFG5_KW = dict(layers=10, blocks=8, dilation_channels=512, residual_channels=512, skip_channels=512, end_channels=512,
               classes=256, output_length=32000 - 8185 + 1, kernel_size=2, bias=False)
CFG5_L = 32000


def bench_train_cfg5(args, world, rank):
    """BASELINE.json configs[4]: layers=10, blocks=8, 512 channels, seq 32000, bf16 training; B = 1 sequence per GPU (the
    config names no batch).  Single-pass bf16 tensor-core operands, fp32 accumulation, fp32-class residual / skip streams."""
    import data_parallel as dp
    import wavenet_training as wt
    model = build_model(CFG5_KW).cuda()
    rt = model._runtime()
    rt.tc_precision = "bf16"
    L = CFG5_L
    idx = torch.randint(0, 256, (1, L), generator=torch.Generator().manual_seed(4321 + rank)).to(torch.uint8).cuda()
    target = torch.randint(0, 256, (model.output_length,), generator=torch.Generator().manual_seed(55 + rank)).cuda()
    flush = L2Flush()
    n = args.steps
    with torch.no_grad():
        for _ in range(2):
            model.forward_indices(idx)
        barrier_sync(world)
        evs, bevs = [], []
        for _ in range(n):
            flush()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            rt.block_events = (b0, b1)
            e0.record()
            model.forward_indices(idx)
            e1.record()
            evs.append((e0, e1)); bevs.append((b0, b1))
        rt.block_events = None
        barrier_sync(world)
        fwd_ms = max_over_ranks(sum(a.elapsed_time(b) for a, b in evs) / n, world)
        block_ms = sum(a.elapsed_time(b) for a, b in bevs) / n
    red = dp.make_data_parallel(model)
    step_ms = []
    for i in range(1 + n):
        model.zero_grad(set_to_none=True)
        barrier_sync(world)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        loss = wt.fused_cross_entropy(model.forward_indices(idx), target)
        loss.backward()
        e1.record()
        torch.cuda.synchronize()
        if i > 0:
            step_ms.append(e0.elapsed_time(e1))
    step_t = max_over_ranks(sum(step_ms) / len(step_ms), world)
    per_layer, start_b, head_b, flops = train_alg_bytes(model, 1, L, dense_input=False)
    tpeak, tsrc = measured_peaks("tensor")
    hpeak, _ = measured_peaks()
    tflops = flops / (block_ms / 1e3) / 1e12
    model._runtime().grad_reducer = None
    out = {"workload": "cfg5: layers=10 blocks=8 ch=512 (skip/end 512), B=1 per GPU, L=32000, output_length=23816, uint8 index input",
           "dtype": "bf16 operands / fp32 accumulate / fp32-class residual+skip", "metric": "training-forward mu-law frames/sec",
           "value": world * L / (fwd_ms / 1e3), "unit": "frames/s", "ms_per_step": fwd_ms,
           "train_step": {"ms_per_step": step_t, "frames_per_s": world * L / (step_t / 1e3), "loss": float(loss.detach()),
                          "grad_allreduce_bytes_per_step": red.bytes_reduced // (1 + n) if world > 1 else 0},
           "roofline": {"kernel": "block_fused_kernel<512, single-pass bf16>", "bound": "tensor", "achieved": tflops, "peak": tpeak,
                        "unit": "TFLOP/s", "frac": tflops / tpeak, "peak_source": tsrc, "avg_block_ms": block_ms / len(per_layer),
                        "hbm_frac": (sum(per_layer) / (block_ms / 1e3) / 1e9) / hpeak, "traffic": None},
           "parameters": model.parameter_count(), "scaling": "weak"}
    del loss
    return out


# ------------------------------------------------------------------------------------------------ CPU baseline
def cpu_generate(budget_s, temperature, threads):
    """samples/s of the CPU port at `threads` torch threads, on a sample sized to ~budget_s seconds."""
    from oracle import wavenet_oracle as O
    torch.set_num_threads(threads)
    spec = O.NetSpec(**GEN_KW)
    p = O.init_params(spec, seed=0)
    np.random.seed(0)
    # per-step cost is position independent, so a short run stands in for 16000 samples
    t0 = time.perf_counter()
    O.generate_fast(p, spec, 4, temperature=temperature)           # probe (also warms the allocator / thread pool)
    rate = 4 / (time.perf_counter() - t0)
    n = int(max(8, min(400, rate * budget_s)))
    t0 = time.perf_counter()
    O.generate_fast(p, spec, n, temperature=temperature)
    return n / (time.perf_counter() - t0), n


def cpu_generate_best(budget_s, temperature):
    """The reference leaves torch's thread count at its default (= all cores), which is a poor choice for these
    tiny matrix-vector ops; time 1, 8 and all threads and keep the fastest so the baseline is not a straw man."""
    cores = os.cpu_count() or 1
    res = {}
    for th in sorted({1, min(8, cores), cores}):
        res[th] = cpu_generate(budget_s, temperature, th)
    best = max(res, key=lambda k: res[k][0])
    note = ", ".join(f"{th} threads: {v[0]:.1f} samples/s ({v[1]} samples)" for th, v in res.items())
    return res[best][0], best, note


def cpu_train_forward(B, threads):
    from oracle import wavenet_oracle as O
    torch.set_num_threads(threads)
    spec = O.NetSpec(**GEN_KW)
    p = O.init_params(spec, seed=0)
    idx = torch.randint(0, 256, (B, TRAIN_L), generator=torch.Generator().manual_seed(1234))
    x = O.one_hot(idx, 256)
    with torch.no_grad():
        t0 = time.perf_counter()
        O.forward(p, spec, x)
        dt = time.perf_counter() - t0
    return B * TRAIN_L / dt


def cpu_train_step(threads):
    """frames/s of one forward + backward of the CPU port at B=1, L=16000 (autograd over the oracle; ~5 GB of host memory)."""
    import torch.nn.functional as F
    from oracle import wavenet_oracle as O
    torch.set_num_threads(threads)
    spec = O.NetSpec(**GEN_KW)
    p = {k: v.requires_grad_(True) for k, v in O.init_params(spec, seed=0).items()}
    idx = torch.randint(0, 256, (1, TRAIN_L), generator=torch.Generator().manual_seed(1234))
    x = O.one_hot(idx, 256)
    tgt = torch.randint(0, 256, (spec.output_length,), generator=torch.Generator().manual_seed(3))
    t0 = time.perf_counter()
    F.cross_entropy(O.forward(p, spec, x), tgt).backward()
    return TRAIN_L / (time.perf_counter() - t0)


def run_reference(args):
    """--impl reference: the CPU port of the reference (oracle/) on the host cores; rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    _, threads, note = cpu_generate_best(4.0, TEMPERATURE)
    vals, n_per_step = [], 0
    for i in range(args.warmup + args.steps):
        v, n_per_step = cpu_generate(6.0, TEMPERATURE, threads)
        if i >= args.warmup:
            vals.append(v)
    value = len(vals) / sum(1.0 / v for v in vals)
    sample = (f"~{n_per_step} samples per step, temperature=1.0 (per-sample cost is position independent); "
              f"thread sweep: {note}")
    print(json.dumps({
        "impl": "reference", "metric": "generate_fast samples/sec", "value": value, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * n_per_step / value,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": GEN_WORKLOAD, "parallelism": "1 CPU process (rank 0); per-sample cost is position independent, so each "
                   f"step times ~{n_per_step} samples instead of 16000"},
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


# ------------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="all", choices=["all", "generate", "train"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-batched", action="store_true", help="skip the 64-stream (cfg4) generation figure")
    ap.add_argument("--no-cfg5", action="store_true", help="skip the 512-channel bf16 deep-stack figures (cfg 5)")
    ap.add_argument("--variants", action="store_true", help="also time the other operand splits of the two-launch blocks")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the B200 path has no CPU fallback); use --impl reference for the CPU arm")
    world, rank, _ = dist_setup(args.gpus)
    dump = {} if args.dump_outputs and rank == 0 else None
    gen = bench_generate(args, world, rank, dump) if args.workload in ("all", "generate") else None
    train = bench_train(args, world, rank, dump) if args.workload in ("all", "train") else None
    cfg5 = None
    if train is not None and not args.no_cfg5:
        torch.cuda.empty_cache()
        cfg5 = bench_train_cfg5(args, world, rank)
        train["cfg5"] = cfg5
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, threads, note = cpu_generate_best(8.0, TEMPERATURE)
        cpu = {"value": v, "unit": "samples/s", "cores": threads, "kind": "port",
               "sample": "generate_fast samples for ~8 s per thread setting (position-independent per-sample cost), "
                         "temperature=1.0, torch CPU fp32 op-for-op port of the reference (oracle/wavenet_oracle.py); "
                         + note}
        threads = os.cpu_count() or 1
        if train is not None:
            res = {}
            for th in sorted({min(8, threads), min(32, threads), threads}):
                res[th] = cpu_train_forward(1, th)
            best = max(res, key=lambda k: res[k])
            if "train_step" in train:
                train["train_step"]["cpu_baseline"] = {
                    "value": cpu_train_step(best), "unit": "frames/s", "cores": best, "kind": "port",
                    "sample": "one forward + backward (torch autograd over the oracle port) at B=1, L=16000"}
            train["cpu_baseline"] = {"value": res[best], "unit": "frames/s", "cores": best, "kind": "port",
                                     "sample": "one no_grad forward of B=1, L=16000 one-hot input per thread setting (best kept): "
                                               + ", ".join(f"{k} threads: {v:.0f} frames/s" for k, v in res.items())}
    if rank == 0:
        primary = gen if gen is not None else train
        line = {
            "metric": "generate_fast samples/sec" if gen is not None else train["metric"],
            "value": primary["value"], "unit": "samples/s" if gen is not None else "frames/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": primary["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": gen["dtype"] if gen is not None else "f32", "data": "synthetic",
            "config": ({"workload": GEN_WORKLOAD,
                        "parallelism": f"{world} independent replicas (the sampling loop does not shard)",
                        "l2": "256 MiB buffer written between timed iterations (L2 flush)"}
                       if gen is not None else train["config"]),
            "clocks": primary["clocks"], "e2e": primary["e2e"], "gpu_launches": primary["launches"],
            "roofline": primary["roofline"],
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if gen is not None:
            line["argmax_samples_per_s"] = gen["argmax_samples_per_s"]
            if gen.get("batched") is not None:
                line["batched_64_streams"] = gen["batched"]
            if train is not None:
                line["train"] = train
        else:
            line.update({k: train[k] for k in ("train_step", "fast_tf32", "e2e_index_api", "cpu_baseline") if k in train})
        summ = {}
        if gen is not None:
            summ.update(gen_samples_per_s=gen["value"], gen_us_per_sample=gen["roofline"]["us_per_sample"],
                        gen_us_per_stage=gen["roofline"]["us_per_exchange_stage"])
            if gen.get("batched") is not None:
                summ["cfg4_64_streams_samples_per_s"] = gen["batched"]["value"]
        if train is not None:
            r = train["roofline"]
            summ.update(train_fwd_frames_per_s=train["value"], train_fwd_ms=train["ms_per_step"],
                        train_fwd_e2e_frames_per_s=train["e2e"]["value"], train_avg_block_ms=r.get("avg_block_ms", r.get("avg_launch_ms")),
                        train_tensor_pipe_equiv_frac=r.get("tensor_pipe_equiv_frac"), train_hbm_frac=r.get("hbm_frac", r.get("frac")),
                        train_step_ms=train["train_step"]["ms_per_step"],
                        train_step_frames_per_s=train["train_step"]["frames_per_s"])
            if "strong" in train["train_step"]:
                summ["train_step_strong_ms"] = train["train_step"]["strong"]["ms_per_step"]
            if "ddp_grad_max_rel_err" in train["train_step"]:
                summ["ddp_grad_max_rel_err"] = train["train_step"]["ddp_grad_max_rel_err"]
            if train.get("cfg5") is not None:
                summ.update(cfg5_fwd_ms=train["cfg5"]["ms_per_step"], cfg5_step_ms=train["cfg5"]["train_step"]["ms_per_step"],
                            cfg5_tensor_frac=train["cfg5"]["roofline"]["frac"])
        line["summary"] = summ
        if dump is not None:
            write_outputs(args.dump_outputs, dump)
        print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
