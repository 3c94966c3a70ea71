#!/usr/bin/env python
"""Benchmark of the UQ inference hot path (BASELINE.json metric: UQ samples x passes / sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload NAME]
                    [--dump-outputs DIR]

Workload (``configs[1]`` of BASELINE.json): binomial-options deep ensemble,
16 members x (5 -> 512 -> 512 -> 512 -> 1, Linear+BatchNorm1d+ReLU), 1 M synthetic samples,
bf16 tcgen05 mode.  One step = one ``model(x, return_ue=True)`` over the whole batch.
At N > 1 (one rank per GPU, launched by torchrun) the SAME job is sharded over the member axis
(strong scaling: 16 members in total, 16 / N per rank, each rank holding only its members'
weights): every rank reduces its members to per-sample (mean, M2) in the fused kernel and the
shards are combined reduce-scatter style over NCCL/NVLink (all-to-all of row slices, local Chan
merge, all-gather of the finished (mean, std) slices; ``distributed.KShard.combine``).

The JSON line follows the driver's contract: ``value`` is whole-job sample.members/s with inputs
resident in HBM; ``e2e`` is the same metric through the wrapper API with pinned HOST buffers
(H2D of x and D2H of mean/std inside the timed region); ``roofline`` is the fused kernel against
the measured bf16 tensor peak; ``cpu_baseline`` is the oracle port (the reference's torch-CPU
arithmetic) timed on a bounded sample on this box's host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOADS = {
    # name: (mode, d_in, hidden widths, d_out, members/passes, samples, dropout p)
    "ensemble16x512_1M": ("ensemble", 5, [512, 512, 512], 1, 16, 1 << 20, 0.0),
    "mcdropout100_binomial_10k": ("mc_dropout", 5, [128] * 6, 1, 100, 10000, 0.2),
    "deltauq32_binomial_4M": ("delta_uq", 5, [128] * 6, 1, 32, 1 << 22, 0.0),
    "mcdropout_1000x512_64k": ("mc_dropout", 5, [512] * 7, 1, 1000, 1 << 16, 0.2),
    # configs[3] of BASELINE.json (MC dropout, 1000 passes x 8-layer width-1024 MLP) on a
    # 64 k-sample slice of its 16 M samples, and the same net without dropout
    "mcdropout_1000x1024_64k": ("mc_dropout", 5, [1024] * 7, 1, 1000, 1 << 16, 0.2),
    "mcdropout_1000x1024_1M": ("mc_dropout", 5, [1024] * 7, 1, 1000, 1 << 20, 0.2),
    "ensemble8x1024_256k": ("ensemble", 5, [1024] * 7, 1, 8, 1 << 18, 0.0),
    # the binomial-options surrogate as a 32-member ensemble (same flops as deltauq32_binomial_4M)
    "ensemble32x128_4M": ("ensemble", 5, [128] * 6, 1, 32, 1 << 22, 0.0),
}
DEFAULT_WORKLOAD = "ensemble16x512_1M"
N_ROTATE = 8  # input buffers rotated per step so the working set exceeds the 126 MB L2
DUMP_BYTES = 64_000_000 - 4096  # --dump-outputs budget: 64 MB with room for the .npy headers


def kernel_name(widths, d_out):
    """Which fused kernel the library dispatches to (csrc/mlp_tc.cu:tc_forward)."""
    h = max(widths)
    bias = ", bias in the MMA" if d_out == 1 and os.environ.get("UQ_TC_BIAS_MMA", "1") == "1" else ""
    if h > 512:
        return "uq_mlp_tc3_kernel (CTA pairs, 64 rows per CTA%s)" % bias
    if h <= 128 and d_out == 1:
        return "uq_mlp_tc4_kernel (CTA pairs, 4 tile slots per CTA%s)" % bias
    return "uq_mlp_tc2_kernel (CTA pairs%s)" % bias


def flops_per_unit(d_in, widths, d_out):
    dims = [d_in] + list(widths) + [d_out]
    return 2 * sum(a * b for a, b in zip(dims[:-1], dims[1:]))


def mlp_arch(d_in, widths, d_out):
    arch, prev = [], d_in
    for w in widths:
        arch += [{"Linear": {"args": [prev, w]}}, {"BatchNorm1d": {"args": [w]}},
                 {"ReLU": {"inplace": True}}]
        prev = w
    arch.append({"Linear": {"args": [prev, d_out]}})
    return arch


def randomise_bn(net, seed):
    g = torch.Generator().manual_seed(seed)
    for m in net.modules():
        if isinstance(m, torch.nn.BatchNorm1d):
            m.running_mean.copy_(torch.randn(m.num_features, generator=g) * 0.1)
            m.running_var.copy_(torch.rand(m.num_features, generator=g) + 0.5)


def build_model(workload, member_offset=0, member_count=None):
    """Random-init model of the named architecture through the builder mirror (the reference's
    own construction path, model_builder.py:219-275); BN running stats randomised (seed 1+i).
    ``member_offset`` / ``member_count``: the slice of an ensemble's members one rank owns (member
    i is seeded 42 + i, as model_builder.py:229 does, whichever rank holds it)."""
    from nnueehcs_b200 import model_builder as mb
    mode, d_in, widths, d_out, k, n, p = WORKLOADS[workload]
    if mode == "ensemble":
        arch = mlp_arch(d_in, widths, d_out)
        k = k if member_count is None else member_count
        builder = mb.EnsembleModelBuilder(arch, {"num_models": k})
        model = builder.build()
        if member_offset:  # other ranks own other members: seeds 42 + offset + i
            for i in range(k):
                torch.manual_seed(42 + member_offset + i)
                model.models[i] = mb.build_network(arch)
        for i, net in enumerate(model.models):
            randomise_bn(net, 1 + member_offset + i)
    elif mode == "mc_dropout":
        torch.manual_seed(42)
        model = mb.MCDropoutModelBuilder(mlp_arch(d_in, widths, d_out),
                                         {"num_samples": k, "dropout_percent": p}).build()
        randomise_bn(model.model, 1)
    else:
        torch.manual_seed(42)
        model = mb.DeltaUQMLPModelBuilder(mlp_arch(d_in, widths, d_out),
                                          {"estimator": "std", "num_anchors": k,
                                           "anchored_batch_size": 4096}).build()
        randomise_bn(model.net, 1)
        model.anchors = torch.rand(k, d_in, generator=torch.Generator().manual_seed(2))
    model.eval()
    return model


def synth_x(n, d_in, seed):
    # binomial-options-shaped: 5 features min-max scaled to [0, 1] (data_utils.py:291-296)
    return torch.rand(n, d_in, generator=torch.Generator().manual_seed(seed))


# ------------------------------------------------------------------------------------------------
# CPU side: the oracle port (reference arithmetic on torch CPU)
# ------------------------------------------------------------------------------------------------

def cpu_forward_fn(workload, model):
    from oracle import uq_oracle
    mode, d_in, widths, d_out, k, n, p = WORKLOADS[workload]
    if mode == "ensemble":
        nets = list(model.models)
        return lambda x: uq_oracle.ensemble_forward(nets, x)
    if mode == "mc_dropout":
        return lambda x: uq_oracle.mc_dropout_forward(model.model, x, k, p)
    anchors = model.anchors
    return lambda x: uq_oracle.delta_uq_forward(model.net, x, anchors, k)


def time_cpu(workload, model, sample_n, steps, warmup):
    """(rate, seconds per step, (mean, std) of the last timed step)"""
    mode, d_in, widths, d_out, k, n, p = WORKLOADS[workload]
    fn = cpu_forward_fn(workload, model)
    x = synth_x(sample_n, d_in, 0)
    for _ in range(warmup):
        fn(x)
    t0 = time.perf_counter()
    for _ in range(steps):
        out = fn(x)
    dt = (time.perf_counter() - t0) / steps
    return sample_n * k / dt, dt, out


def cpu_sample_size(workload):
    mode, d_in, widths, d_out, k, n, p = WORKLOADS[workload]
    # a few seconds of CPU work per step (10-30 s for the whole bounded baseline run)
    target_flops = 1.2e12
    s = int(target_flops / (flops_per_unit(d_in, widths, d_out) * k))
    return max(256, min(n, 1 << (s.bit_length() - 1)))


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port, kind
    "port") on this box's host cores, same metric/config, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    # all the host threads it can use: torchrun exports OMP_NUM_THREADS=1 to every rank, which
    # would time the reference on one core (measured: 8.0e4 instead of 7.2e5 sample*members/s)
    try:
        host_threads = len(os.sched_getaffinity(0))
    except AttributeError:
        host_threads = os.cpu_count() or 1
    torch.set_num_threads(max(1, host_threads))
    wl = args.workload
    mode, d_in, widths, d_out, k, n, p = WORKLOADS[wl]
    model = build_model(wl)
    sample_n = cpu_sample_size(wl)
    steps, warmup = args.steps, max(1, min(args.warmup, 2))
    rate, dt, out = time_cpu(wl, model, sample_n, steps, warmup)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"mean": out[0], "std": out[1]})
    cores = torch.get_num_threads()
    line = {
        "impl": "reference", "metric": "uq_sample_passes_per_sec", "value": rate,
        "unit": "sample*members/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_dict(wl, 1, sample_note=f"{sample_n} of {n} samples per step"),
        "cpu_baseline": {"value": rate, "unit": "sample*members/s", "cores": cores,
                         "kind": "port",
                         "sample": f"{sample_n} samples x {k} members per step, {steps} steps, "
                                   f"torch {torch.__version__} CPU, os.cpu_count={os.cpu_count()}"},
        "e2e": {"value": rate, "unit": "sample*members/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)
    return 0


def config_dict(wl, n_gpus, sample_note=None):
    mode, d_in, widths, d_out, k, n, p = WORKLOADS[wl]
    cfg = {"workload": wl, "mode": mode, "arch": f"{d_in}->" + "->".join(map(str, widths)) + f"->{d_out}",
           "members_per_gpu": k / n_gpus, "members_total": k,
           "samples": n, "dropout_p": p,
           "parallelism": f"member-axis shards x{n_gpus} of the same job (strong scaling); per step "
                          "one all-to-all of (mean, M2) row slices, a local Chan merge and an "
                          "all-gather of the (mean, std) slices",
           "l2": f"inputs rotated over {N_ROTATE} device buffers (> 126 MB L2 with weights)"}
    if sample_note:
        cfg["cpu_sample"] = sample_note
    return cfg


def dump_outputs(out_dir, arrays):
    """--dump-outputs: each array of the last timed step as ``out_dir/<name>.npy`` in float32, so
    two builds run with the same arguments (hence the same seeded inputs) can be compared output
    for output.  Above DUMP_BYTES in all, every array keeps the same evenly strided rows."""
    import numpy as np
    arrays = {name: a.detach().float().cpu().numpy() for name, a in arrays.items()}
    stride = -(-sum(a.nbytes for a in arrays.values()) // DUMP_BYTES)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a[::stride]))


# ------------------------------------------------------------------------------------------------
# GPU side
# ------------------------------------------------------------------------------------------------

class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.proc = None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-i", str(self.gpu_index), "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in out.strip().splitlines():
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])), mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = sorted(sm)[len(sm) // 2:]  # samples under load dominate the upper half
        return {"sm_mhz": statistics.median(sm), "sm_mhz_under_load": statistics.median(busy),
                "sm_max_mhz": max(mx), "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return {"burst": d.get("bf16_tflops", 1590.0), "sustained": d.get("bf16_tflops_sustained", 1400.0),
                "hbm": d.get("hbm_gbs", 6650.0), "source": "MEASURED_PEAKS.json (of measured)"}
    return {"burst": 1590.0, "sustained": 1400.0, "hbm": 6650.0,
            "source": "B200_PROFILING.md fallback (of fallback)"}


def metric_kernel_lines(dev, peaks, n=50_000_000, steps=5):
    """BASELINE.json's metric also asks for the metric kernels' GB/s: ID-vs-OOD Wasserstein and
    KDE Jensen-Shannon over 50 M + 50 M synthetic uncertainty scores (configs[4] on one GPU),
    resident in HBM, timed with CUDA events around the public op; GB/s = the algorithmic 4 B per
    value (SURVEY 8d) over the call time, next to the measured HBM peak."""
    from nnueehcs_b200 import ops

    def gamma(shape, scale, seed):
        g = torch.Generator(device=dev).manual_seed(seed)
        u = torch.rand((shape, n), generator=g, device=dev).clamp_min_(1e-12)
        return (-torch.log(u)).sum(0).mul_(scale).contiguous()

    u, v = gamma(2, 0.05, 0), gamma(3, 0.08, 1)
    hbm = peaks.get("hbm")
    out = {}
    for name, fn, info, enqueue in (
            ("wasserstein_1d", lambda: ops.wasserstein_1d(u, v), lambda: ops.wasserstein_1d_info(u, v),
             lambda: ops.wasserstein_1d_async(u, v)),
            ("kde_jsd", lambda: ops.kde_jsd(u, v, 20000), lambda: ops.kde_jsd_info(u, v, 20000),
             lambda: ops.kde_jsd_async(u, v, 20000))):
        # device time per call with the host out of the loop: `steps` calls enqueued back to back
        # through the enqueue / finish API (uq_*_enqueue: memset + one launch each, no
        # synchronisation), one synchronisation at the end.  This is the kernel's launch duration
        # the roofline fraction refers to; "ms" below is what a caller of the synchronous op sees
        # (launch latency, the stream synchronisation and the Python / ctypes hop included).
        pend = [enqueue() for _ in range(2)]
        vals = [p.result() for p in pend]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        pend = [enqueue() for _ in range(2 * steps)]
        e1.record()
        torch.cuda.synchronize()
        ms_dev = e0.elapsed_time(e1) / (2 * steps)
        vals = [p.result() for p in pend]
        del pend
        for _ in range(3):   # warm-up of the synchronous op (its workspace comes from the allocator)
            val = fn()
        torch.cuda.synchronize()
        assert all(x == val for x in vals), (name, vals, val)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ops.reset_launch_count()
        e0.record()
        for _ in range(steps):
            val = fn()
        e1.record()
        torch.cuda.synchronize()
        launches = ops.launch_count() // steps
        ms = e0.elapsed_time(e1) / steps
        gbs = 2 * n * 4 / (ms * 1e-3) / 1e9
        gbs_dev = 2 * n * 4 / (ms_dev * 1e-3) / 1e9
        out[name] = {"values": 2 * n, "ms": ms, "values_per_s": 2 * n / (ms * 1e-3),
                     "algorithmic_GBps": gbs, "hbm_peak_GBps": hbm,
                     "frac_of_hbm_peak": gbs / hbm if hbm else None,
                     "ms_device": ms_dev, "algorithmic_GBps_device": gbs_dev,
                     "frac_of_hbm_peak_device": gbs_dev / hbm if hbm else None,
                     "device_timing": f"{2 * steps} calls enqueued back to back (uq_*_enqueue), one "
                                      "synchronisation at the end; results equal the synchronous "
                                      "calls' bit for bit",
                     "result": val,
                     "method": info()["method"], "gpu_launches_per_call": int(launches),
                     "data": "synthetic Gamma(2, 0.05) vs Gamma(3, 0.08) scores, float32, in HBM"}
    # scipy's own route (two radix sorts + a merge-path integral): the fallback of the binned
    # method and the engine of uq_score_metrics; and the sort on its own
    for name, fn in (("wasserstein_1d_sort", lambda: ops.wasserstein_1d(u, v, "sort")),
                     ("radix_sort_f32", lambda: ops.sort_f32(u))):
        for _ in range(2):
            val = fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            val = fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        nvals = 2 * n if name.startswith("wasserstein") else n
        out[name] = {"values": nvals, "ms": ms, "values_per_s": nvals / (ms * 1e-3),
                     "algorithmic_GBps": nvals * 4 / (ms * 1e-3) / 1e9, "hbm_peak_GBps": hbm,
                     "frac_of_hbm_peak": nvals * 4 / (ms * 1e-3) / 1e9 / hbm if hbm else None}
        if name.startswith("wasserstein"):
            out[name]["result"] = val
            out[name]["equals_binned"] = bool(abs(val - out["wasserstein_1d"]["result"])
                                              <= 1e-11 * abs(val))
        else:
            out[name]["sorted"] = bool((val[1:] >= val[:-1]).all().item())
        del val
    del u, v
    torch.cuda.empty_cache()
    return out


def parity_check(wl, packed_forward, x_dev, rows=4096):
    """bench.py checks its own output: the first ``rows`` rows of a forward against the CPU oracle
    (reference arithmetic), before anything is timed.  Returns the worst error of mean and std
    in the test-suite's units: fp32 in units of the 1e-5 tolerance (<= 1 passes), bf16 as a
    fraction of scale = max|mean| + max|std| (tests allow 1e-2)."""
    from oracle import uq_oracle  # the checker, never the thing measured
    mode, d_in, widths, d_out, k, n, p = WORKLOADS[wl]
    if mode != "ensemble":
        return None
    cpu_model = build_model(wl)
    xs = x_dev[:rows].cpu()
    ref_mean, ref_std = uq_oracle.ensemble_forward(list(cpu_model.models), xs)
    out = {}
    for prec, (mean, std) in packed_forward.items():
        mean, std = mean[:rows].double().cpu(), std[:rows].double().cpu()
        ms, ss = float(ref_mean.abs().max()), float(ref_std.abs().max())
        e_mean, e_std = (mean - ref_mean).abs(), (std - ref_std).abs()
        if prec == "bf16":
            out[prec] = {"max_err_of_scale": max(float(e_mean.max()), float(e_std.max())) / (ms + ss),
                         "allowed": 1e-2}
        else:
            tol_m = 1e-5 * ref_mean.abs() + 1e-5 * ms
            tol_s = 1e-5 * ref_std.abs() + 1e-5 * ms
            out[prec] = {"max_err_in_units_of_1e-5_tolerance":
                         max(float((e_mean / tol_m).max()), float((e_std / tol_s).max())),
                         "allowed": 1.0}
    out["rows"] = rows
    out["oracle"] = "oracle.uq_oracle.ensemble_forward (torch CPU, reference arithmetic)"
    return out


def gpu_eager_baseline(wl, dev, x, steps=2):
    """Informational: what a reference user has today on the same B200 -- the reference's own eager
    fp32 loop (models.py:103-107: stack([m(x) for m in models]), mean(0), std(0)) run by stock
    torch on the GPU (cuBLAS SGEMM, TF32 off).  Not the product path and not the target."""
    mode, d_in, widths, d_out, k, n, p = WORKLOADS[wl]
    if mode != "ensemble":
        return None
    model = build_model(wl).to(dev)
    nets = list(model.models)

    def fwd():
        with torch.no_grad():
            outputs = torch.stack([m(x) for m in nets])
            return outputs.mean(0), outputs.std(0)

    fwd()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fwd()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    del model, nets
    torch.cuda.empty_cache()
    return {"value": n * k / (ms * 1e-3), "unit": "sample*members/s", "ms_per_step": ms,
            "what": "stock torch eager fp32 EnsembleModel loop on the same GPU (cuBLAS; the "
                    "reference's models.py:103-107 as its authors run it on A100s)",
            "steps": steps}


def run_gpu(args):
    import torch.distributed as dist
    from nnueehcs_b200 import ops
    from nnueehcs_b200.distributed import KShard, split_range

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (no CPU fallback); use --impl reference "
                           "for the CPU baseline")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner on stdout when the first communicator comes up; stdout
        # carries exactly one JSON line, so the banner goes to stderr
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    wl = args.workload
    mode, d_in, widths, d_out, k, n, p = WORKLOADS[wl]
    precision = args.precision
    # strong scaling: the job (k members / passes / anchors over n samples) is fixed; an ensemble
    # rank builds and packs only the members it owns
    own_begin, own_count = split_range(k, world, rank) if mode == "ensemble" else (0, k)
    if mode == "ensemble" and own_count == 0:
        raise RuntimeError(f"{world} ranks but only {k} ensemble members")
    model = build_model(wl, member_offset=own_begin, member_count=own_count)
    model.to(dev)
    model.eval()
    model.uq_precision = precision
    shard = KShard() if world > 1 else None
    nets = (list(model.models) if mode == "ensemble" else
            [model.model] if mode == "mc_dropout" else [model.net])
    packed = model._packed(nets, dev)
    if precision == "bf16" and not packed.supports_bf16:
        raise RuntimeError(f"bf16 path unavailable: {packed.bf16_reason}")

    xs = [synth_x(n, d_in, s).to(dev) for s in range(N_ROTATE)]
    kw = {}
    if mode == "mc_dropout":
        kw = dict(dropout_p=p, dropout_active=True, seed=1234)
    if mode == "delta_uq":
        kw = dict(anchors=model.anchors.to(dev))

    def step(x, prec=precision):
        if shard is not None and mode == "ensemble":
            return shard.forward_owned(packed, x, mode, local_members=own_count, precision=prec,
                                       **kw)
        if shard is not None:
            return shard.forward(packed, x, mode, total_members=k, precision=prec, **kw)
        return packed.forward(x, mode, total_members=k, precision=prec, **kw)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- the bench verifies its own output before timing anything -----------------------------
    parity = None
    if mode == "ensemble":
        outs = {precision: step(xs[0])}
        if world == 1 and precision == "bf16" and packed.fp32_on_tensor_cores:
            outs["fp32"] = step(xs[0], "fp32")
        torch.cuda.synchronize()
        if rank == 0:
            parity = parity_check(wl, outs, xs[0])
            for prec, r in parity.items():
                if isinstance(r, dict):
                    worst = [v for key, v in r.items() if key.startswith("max_err")][0]
                    if not worst <= r["allowed"]:
                        raise RuntimeError(f"bench.py parity check failed ({prec}): {r}")
        del outs

    steps, warmup = args.steps, max(3, args.warmup)
    for i in range(warmup):
        out = step(xs[i % N_ROTATE])
    barrier()

    # ---- device-resident timing: CUDA events on the launching (current) stream -----------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
          for _ in range(steps)]
    ops.reset_launch_count()
    barrier()
    t_wall0 = time.perf_counter()
    e_begin, e_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e_begin.record()
    for i in range(steps):
        ev[i][0].record()
        out = step(xs[(warmup + i) % N_ROTATE])
        ev[i][1].record()
    e_end.record()
    barrier()
    wall = time.perf_counter() - t_wall0
    launches = ops.launch_count()
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:   # every rank holds the whole (mean, std)
        dump_outputs(args.dump_outputs, {"mean": out[0], "std": out[1]})
    total_ms = e_begin.elapsed_time(e_end)
    step_ms = [a.elapsed_time(b) for a, b in ev]
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    units_per_step = n * k          # the whole job, whatever the number of ranks
    value = units_per_step * steps / (total_ms * 1e-3)

    # ---- the fused kernel alone (K-sharded runs: forward without the exchange) -----------------
    kernel_ms = statistics.mean(step_ms)
    if shard is not None:
        slab = shard.new_slab(n * d_out, dev)
        fkw = dict(total_members=own_count) if mode == "ensemble" else \
            dict(zip(("member_begin", "member_count"), shard.split(k)), total_members=k)

        def fwd_only(x):
            packed.forward_into(x, mode, slab[0, :n * d_out].view(n, d_out),
                                slab[1, :n * d_out].view(n, d_out), precision=precision,
                                output="moments", **fkw, **kw)
        for i in range(2):
            fwd_only(xs[i])
        torch.cuda.synchronize()
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record()
        for i in range(steps):
            fwd_only(xs[(2 + i) % N_ROTATE])
        k1.record()
        torch.cuda.synchronize()
        kernel_ms = k0.elapsed_time(k1) / steps
        del slab

    # ---- end-to-end with pinned HOST buffers ---------------------------------------------------
    # N = 1: through the wrapper API.  N > 1: the samples live sharded in the ranks' host memory
    # (rank r holds rows [r n/N, (r+1) n/N)): every step each rank copies ITS rows host -> device,
    # one NCCL all-gather of x over NVLink gives every GPU all rows (the K axis is what is
    # sharded), the forward + combine run, and each rank copies ITS rows of (mean, std) back.
    model.uq_shard = None
    r_begin, r_count = split_range(n, world, rank)
    cap = -(-n // world)
    xh = [synth_x(n, d_in, s)[r_begin:r_begin + r_count].contiguous().pin_memory() for s in range(2)]
    mean_h = torch.empty((r_count, d_out), dtype=torch.float32).pin_memory()
    std_h = torch.empty((r_count, d_out), dtype=torch.float32).pin_memory()
    x_pad = torch.zeros((cap, d_in), dtype=torch.float32, device=dev) if world > 1 else None
    x_all = torch.empty((world * cap, d_in), dtype=torch.float32, device=dev) if world > 1 else None

    def e2e_step(xh_rows):
        if world > 1:
            x_pad[:r_count].copy_(xh_rows, non_blocking=True)
            dist.all_gather_into_tensor(x_all.view(-1), x_pad.view(-1))
            xd = x_all if n == world * cap else torch.cat(
                [x_all[q * cap:q * cap + split_range(n, world, q)[1]] for q in range(world)])
            mean, std = step(xd)
            mean_h.copy_(mean[r_begin:r_begin + r_count], non_blocking=True)
            std_h.copy_(std[r_begin:r_begin + r_count], non_blocking=True)
        else:
            xd = xh_rows.to(dev, non_blocking=True)
            with torch.no_grad():
                if mode == "mc_dropout":
                    torch.manual_seed(0)
                mean, std = model(xd, return_ue=True)
            mean_h.copy_(mean, non_blocking=True)
            std_h.copy_(std, non_blocking=True)
        torch.cuda.synchronize()

    e2e_steps = max(3, min(steps, 10))
    for i in range(2):
        e2e_step(xh[i % 2])
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        e2e_step(xh[i % 2])
    barrier()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    e2e_value = units_per_step * e2e_steps / e2e_s

    # ---- the 1e-5 parity mode on the same workload (N = 1 default line) ------------------------
    fp32_line = None
    if world == 1 and precision == "bf16" and not args.no_fp32_leg and \
            (wl == DEFAULT_WORKLOAD or args.fp32_leg):
        for i in range(3):
            step(xs[i], "fp32")
        torch.cuda.synchronize()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f_steps = max(3, min(steps, 8))
        f0.record()
        for i in range(f_steps):
            step(xs[(3 + i) % N_ROTATE], "fp32")
        f1.record()
        torch.cuda.synchronize()
        fp32_line = f0.elapsed_time(f1) / f_steps

    if rank == 0:
        peaks = measured_peaks()
        F = flops_per_unit(d_in, widths, d_out)
        timed_s = total_ms * 1e-3
        peak_kind = "sustained" if timed_s >= 2.0 else "burst"
        peak = peaks[peak_kind]
        # per-GPU rate of the fused kernel: a rank runs k / world of the members / passes
        k_rank = own_count if mode == "ensemble" else k / world
        achieved = F * n * k_rank / (kernel_ms * 1e-3) / 1e12
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as f:
                tj = json.load(f)
            traffic = tj.get(wl, {}).get(precision)
            traffic_src = tj.get("_source")

        def kernel_label(prec):
            if prec == "bf16":
                return kernel_name(widths, d_out)
            return ("uq_mlp_tcx_kernel (fp32 parity: scaled fp16 x 2 split on tcgen05, 3 MMAs per "
                    "K step)" if packed.fp32_on_tensor_cores else "sgemm_tn_kernel (fp32 CUDA cores)")

        line = {
            "metric": "uq_sample_passes_per_sec", "value": value, "unit": "sample*members/s",
            "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": total_ms / steps,
            "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None,
            "dtype": precision if precision == "bf16" else "f32", "data": "synthetic",
            "config": config_dict(wl, world),
            "e2e": {"value": e2e_value, "unit": "sample*members/s",
                    "h2d_bytes_per_step": n * d_in * 4, "d2h_bytes_per_step": 2 * n * d_out * 4,
                    "steps": e2e_steps,
                    "api": "model(x.to(device), return_ue=True) -> pinned host" if world == 1 else
                           "per rank: its rows of x pinned host -> device, NCCL all-gather of x, "
                           "KShard forward + combine, its rows of (mean, std) -> pinned host "
                           "(byte counts are the sums over the ranks)"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                         "peak_kind": peak_kind,
                         "peak_source": peaks["source"], "kernel": kernel_label(precision),
                         "flops_per_unit": F, "kernel_ms": kernel_ms,
                         "frac_of_sustained": achieved / peaks["sustained"]},
            "wall_s_timed_region": wall,
        }
        if parity is not None:
            line["parity_max_err"] = parity
        if world > 1:
            line["exchange_ms"] = total_ms / steps - kernel_ms
        if fp32_line is not None:
            a32 = F * n * k / (fp32_line * 1e-3) / 1e12
            line["roofline_fp32_parity"] = {
                "bound": "tensor", "achieved": a32, "peak": peaks["burst"], "unit": "TFLOP/s",
                "frac": a32 / peaks["burst"], "kernel": kernel_label("fp32"), "kernel_ms": fp32_line,
                "value": n * k / (fp32_line * 1e-3), "value_unit": "sample*members/s",
                "note": "algorithmic flops (what the reference executes) over the launch time; "
                        "the split issues 3 tensor-core MMAs per algorithmic one, so the tensor "
                        "pipe runs at 3x this fraction"}
        if world == 1 and wl == DEFAULT_WORKLOAD and not args.no_metric_kernels:
            line["metric_kernels"] = metric_kernel_lines(dev, peaks)
        if world == 1 and not args.no_cpu_baseline:
            sample_n = cpu_sample_size(wl)
            cpu_model = build_model(wl)
            rate, dt, _ = time_cpu(wl, cpu_model, sample_n, 2, 1)
            line["cpu_baseline"] = {
                "value": rate, "unit": "sample*members/s", "cores": torch.get_num_threads(),
                "kind": "port",
                "sample": f"{sample_n} of {n} samples x {k} members, 1 warm-up + 2 timed calls, "
                          f"{dt:.2f} s per call, os.cpu_count={os.cpu_count()}"}
            eager = gpu_eager_baseline(wl, dev, xs[0])
            if eager is not None:
                line["gpu_eager_baseline"] = eager
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--fp32-leg", action="store_true",
                    help="time the fp32 parity mode for a non-default workload as well")
    ap.add_argument("--no-fp32-leg", action="store_true",
                    help="skip timing the fp32 parity mode next to the bf16 line")
    ap.add_argument("--no-metric-kernels", action="store_true",
                    help="skip the Wasserstein / KDE-JS kernel timings added to the default line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the (mean, std) of the last timed step as DIR/mean.npy and "
                         "DIR/std.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
