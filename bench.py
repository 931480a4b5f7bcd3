#!/usr/bin/env python
"""bench.py -- BASELINE.json's headline metric: ResNet-50 (bin/nnc/imagenet.c v1d) fp32, N=256 per GPU, forward +
backward (+ the gradient allreduce for N>1, + the SGD commands), images/sec, on CCV_NNC_BACKEND_GPU_SM100.

  python bench.py --gpus 1 --steps K --warmup W            # this repo's arm
  python bench.py --impl reference --gpus N --steps K ...   # the reference's own CPU_REF path on the host cores
  torchrun --nproc-per-node N bench.py --gpus N ...         # one process per GPU, batch-sharded (weak scaling)

One JSON line on rank 0.  `value` is device-timed (CUDA events on the launching stream) with inputs resident in HBM;
`e2e` is the same step driven from pinned HOST buffers through the reference-facing command API (CMD_DATA_TRANSFER of
the input batch and labels in, the per-sample loss out), also device-timed.  Synthetic data, random-init weights.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# CPU_REF timing hygiene (must be in the environment before libgomp loads): threads pinned to cores and spinning between the
# thousands of small parallel regions of a step; the thread COUNT is set explicitly in reference_measure()
os.environ.setdefault("OMP_PROC_BIND", "true")
os.environ.setdefault("OMP_PLACES", "cores")
os.environ.setdefault("OMP_WAIT_POLICY", "active")

METRIC = "resnet50_fp32_n256_fwd_bwd_images_per_sec"
UNIT = "images/s"


def peaks():
    p = dict(hbm_gbs=6650.0, bf16_tflops=1590.0, source="fallback")
    try:
        m = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        p = dict(hbm_gbs=float(m["hbm_gbs"]), bf16_tflops=float(m["bf16_tflops"]), bf16_tflops_sustained=float(m.get("bf16_tflops_sustained", m["bf16_tflops"])), source="measured")
    except Exception:
        pass
    return p


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons while the timed region runs (B200_PROFILING.md recipe)."""

    def __init__(self, device):
        threading.Thread.__init__(self)
        self.daemon = True
        self.device, self.samples, self.reasons, self.stop_flag, self.max_mhz = device, [], set(), False, None

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.check_output(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + q, "--format=csv,noheader,nounits"], timeout=5).decode().strip().split(",")
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if v.strip().lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        return dict(sm_mhz=float(np.median(self.samples)) if self.samples else None, sm_max_mhz=self.max_mhz, reasons=sorted(self.reasons), samples=len(self.samples))


REF_SAMPLE_BATCH = 8   # images per CPU_REF step: pooling is issued per image (SURVEY.md 0.6), every other command sees the batch
REF_SAMPLE_STEPS = 5   # timed steps; the reported value is their median


def reference_measure(image, batch=REF_SAMPLE_BATCH, steps=REF_SAMPLE_STEPS, warmup=1):
    """ONE definition of the CPU number, used both by `--impl reference` and by the cpu_baseline object of the GPU arm:
    the identical ResNet-50 command list executed by the compiled, unmodified reference (oracle/_ref/libccv_ref.so,
    CCV_NNC_BACKEND_CPU_REF) on a bounded sample of the workload -- `batch` images of image x image per step, forward +
    backward + SGD -- with an explicit OpenMP thread count (one per physical core; an inherited OMP_NUM_THREADS, e.g. the 1
    torchrun exports, is overridden), one untimed step first (page faults, OpenMP pool start-up), median of `steps`."""
    from oracle import ref, ref_factory
    from ccv_b200 import resnet50
    if not ref.available():
        return None
    cores = ref.set_num_threads(ref.physical_cores())
    net = resnet50.Net(batch, image=image, classes=1000, global_batch=batch, factory=ref_factory.RefFactory())
    net.input.upload(np.random.RandomState(0).rand(batch, image, image, 3).astype(np.float32))
    net.labels.upload((np.arange(batch) % 1000).astype(np.int32))

    def step():
        ref_factory.run_nodes(net.fwd)
        ref_factory.run_nodes(net.bwd)
        ref_factory.run_nodes(net.opt)
    for _ in range(warmup):
        step()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
    dt = float(np.median(times))
    sample = ("ResNet-50 v1d fwd+bwd+SGD on CCV_NNC_BACKEND_CPU_REF (unmodified reference compiled into oracle/_ref), batch %d of %dx%d per step, "
              "%d OpenMP threads (one per physical core, set explicitly), %d warm-up + %d timed steps, median; per-step seconds: %s"
              % (batch, image, image, cores, warmup, steps, ", ".join("%.2f" % t for t in times)))
    return {"value": batch / dt, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample, "ms_per_step": dt * 1e3, "batch": batch, "steps": steps, "warmup": warmup,
            "spread": float((max(times) - min(times)) / dt)}


def reference_arm(args):
    """`--impl reference`: the reference's own CPU implementation of the path on the host cores.  Rank 0 only (the other
    ranks of a torchrun launch exit without work)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    m = reference_measure(args.image)
    if m is None:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libccv_ref.so not built (make -C oracle)"}))
        return
    print(json.dumps({"metric": METRIC, "value": m["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": m["steps"], "warmup": m["warmup"], "ms_per_step": m["ms_per_step"], "higher_is_better": True,
                      "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
                      "config": {"workload": "ResNet-50 v1d (bin/nnc/imagenet.c) fp32 NHWC fwd+bwd+SGD; bounded sample: batch %d per step on the host CPU" % m["batch"], "image": args.image},
                      "cpu_baseline": {k: m[k] for k in ("value", "unit", "cores", "kind", "sample")},
                      "e2e": {"value": m["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))


def cpu_baseline(image):
    """Reported next to the GPU number (rank 0, N=1): exactly the measurement `--impl reference` prints."""
    try:
        m = reference_measure(image)
        return None if m is None else {k: m[k] for k in ("value", "unit", "cores", "kind", "sample")}
    except Exception as e:  # the baseline must never take the benchmark down
        return {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": "unavailable: %r" % (e,)}


DTYPES = {"f32": 0x04000, "bf16": 0x80000, "f16": 0x20000}
MATH = {"f32": {-1: "tcgen05 kind::tf32, fp32 accumulate (TMA rounds operands to TF32); the dense layer 3xTF32", 0: "tcgen05 kind::tf32, fp32 accumulate (TMA rounds operands to TF32)",
                1: "3xTF32: three tcgen05 kind::tf32 MMAs on (hi, lo) operand splits, fp32 accumulate", 2: "CUDA-core fp32 FFMA"},
        "bf16": "tcgen05 kind::f16 (bf16 operands), fp32 accumulate in TMEM", "f16": "tcgen05 kind::f16 (fp16 operands), fp32 accumulate in TMEM"}


def to_bf16(a):
    u = np.ascontiguousarray(a, np.float32).view(np.uint32).astype(np.uint64)
    return (((u + 0x7FFF + ((u >> 16) & 1)) >> 16) & 0xFFFF).astype(np.uint16)


DUMP_SAMPLE = 1 << 21  # elements of each flat parameter / gradient buffer written by --dump-outputs (8 MB each in float32)


def _as_float32(t):
    """A tensor's contents as float32 (16-bit tensors are widened exactly)."""
    a = t.download()
    if a.dtype == np.uint16:  # bf16 bits
        return (a.astype(np.uint32) << 16).view(np.float32)
    return a.astype(np.float32)


def dump_outputs(out_dir, net):
    """What the last timed step handed back, as float32 .npy files: the per-sample loss, the logits and softmax probabilities
    of its forward pass, and a fixed seeded sample (the same indices every run) of the parameters after its SGD update and of
    the gradients its backward pass produced.  The model's inputs and initial weights are seeded, so two builds given the same
    arguments can be compared file by file."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": _as_float32(net.loss), "logits": _as_float32(net.logits), "probs": _as_float32(net.probs)}
    flats = [("params", net.w_flat), ("grads", net.g_flat)]
    if hasattr(net, "w_flat_b"):  # 16-bit model: the fp32 batch-norm parameters and their gradients live in buffers of their own
        flats += [("bn_params", net.w_flat_b), ("bn_grads", net.g_flat_b)]
    for name, t in flats:
        flat = _as_float32(t).reshape(-1)
        idx = np.sort(np.random.RandomState(0).choice(flat.size, min(DUMP_SAMPLE, flat.size), replace=False))
        arrays[name + "_sample"] = flat[idx]
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_model(args, dist, rank, world, local_rank, dtype="f32", algorithm=-1, per_op_path="", dump_dir=""):
    """One measured configuration of the ResNet-50 step: returns the JSON object (rank 0 fills roofline / per_op).  dump_dir:
    write the outputs of the last timed step there (dump_outputs)."""
    from ccv_b200 import nnc, resnet50
    device = local_rank
    dt = DTYPES[dtype]
    stream = nnc.Stream(device)
    net = resnet50.Net(args.batch, image=args.image, classes=1000, device=device, global_batch=args.batch * world, learn_rate=4e-5, algorithm=algorithm, dtype=dt)  # 0.4 * 0.0001: the first warm-up rate of bin/nnc/imagenet.c:296-312
    g_fb, g_opt = nnc.Graph(), nnc.Graph()
    # Gradient exchange (N > 1).  "overlap": COMM_ALLREDUCE nodes, one per gradient bucket, sit inside the backward graph on its
    # side stream, each right behind the node that completes its bucket, and are captured into the same CUDA graph -- the NCCL
    # kernels run under the remaining backward kernels.  "between": one allreduce command over the whole flat buffer between the
    # two CUDA graphs (round 1's scheme).
    in_graph = world > 1 and args.exchange == "overlap"
    if world > 1:
        from ccv_b200 import dp
        allreduce_between = dp.CommandAllreduce(net, dist, stream, rank, world)  # binds the NCCL communicator of this rank
    bwd_nodes, side = net.backward_with_exchange(args.buckets) if in_graph else (net.bwd, [])
    for cmd, hint, flags, ins, outs in net.fwd:
        g_fb.exec_new(cmd, hint, flags, ins, outs)
    for j, (cmd, hint, flags, ins, outs) in enumerate(bwd_nodes):
        idx = g_fb.exec_new(cmd, hint, flags, ins, outs)
        if j in side:
            g_fb.set_side_stream(idx)
    for cmd, hint, flags, ins, outs in net.opt:
        g_opt.exec_new(cmd, hint, flags, ins, outs)
    n_fused = 0 if args.no_fuse else g_fb.fuse() + g_opt.fuse()

    # synthetic batch in pinned host memory (for the e2e leg) and resident in HBM (for `value`); a 16-bit model takes a 16-bit batch
    rs = np.random.RandomState(1234 + rank)
    host_in = nnc.cpu_tensor([args.batch, args.image, args.image, 3], datatype=dt)
    host_lab = nnc.cpu_tensor([args.batch], datatype=nnc.CCV_32S)
    host_loss = nnc.cpu_tensor([args.batch])
    for t in (host_in, host_lab, host_loss):
        nnc.lib().ccv_nnc_tensor_pin_memory(t.ptr)
    img = rs.rand(args.batch, args.image, args.image, 3).astype(np.float32)
    host_in.upload(img if dtype == "f32" else to_bf16(img) if dtype == "bf16" else img.astype(np.float16))
    host_lab.upload(rs.randint(0, 1000, size=(args.batch,)).astype(np.int32))
    xfer = nnc.CMD_DATA_TRANSFER_FORWARD()
    assert nnc.cmd_exec(xfer, None, 0, [host_in, host_lab], [net.input, net.labels], stream) == 0
    stream.wait()

    # the single gradient exchange: ONE CCV_NNC_COMM_ALLREDUCE_FORWARD command of the backend over the flat gradient buffer(s)
    # (NCCL inside the library; torch.distributed only carries the communicator id, the barrier and the max-over-ranks time)
    allreduce = allreduce_between if world > 1 and not in_graph else None

    # eager pass: sizes workspaces, counts launches, checks every command returns success
    l0 = nnc.launch_count()
    if g_fb.run(stream) != 0 or g_opt.run(stream) != 0:
        raise SystemExit("bench.py: a command failed: %s" % nnc.lib().ccv_nnc_sm100_last_error())
    stream.wait()
    launches_per_step = nnc.launch_count() - l0
    first_loss = float(np.mean(net.loss.download()))
    use_graph = not args.no_cuda_graph
    if use_graph:
        cap_fb, cap_opt = g_fb.capture(stream), g_opt.capture(stream)

    def step():
        if use_graph:
            g_fb.replay(cap_fb, stream)
        else:
            g_fb.run(stream)
        if allreduce:
            allreduce()
        if use_graph:
            g_opt.replay(cap_opt, stream)
        else:
            g_opt.run(stream)

    def barrier():
        stream.wait()
        if dist is not None:
            dist.barrier()
        stream.wait()

    def timed(fn, steps):
        e0, e1 = nnc.Event(), nnc.Event()
        barrier()
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        ms = e0.elapsed_ms(e1)
        barrier()
        if dist is not None:
            import torch
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(device)
    sampler.start()
    ms = timed(step, args.steps)
    ms_per_step = ms / args.steps
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, net)

    # end to end: every step copies its batch from pinned host memory and reads the loss back, through the same public calls
    # (CMD_DATA_TRANSFER on stream contexts).  The copy of batch k+1 runs on a second stream context while step k computes
    # (stream signals order the two: lib/nnc/ccv_nnc.h:1041-1053); the compute stream then only does a device-to-device move of
    # the staged batch into the network's input tensor.  Steady state: one host-to-device copy and one loss read per step, all
    # inside the timed region; the first batch is staged before the clock starts, the prefetch of one extra batch is inside it.
    copy_stream = nnc.Stream(device)
    stage_in = nnc.gpu_tensor([args.batch, args.image, args.image, 3], datatype=dt, device=device)
    stage_lab = nnc.gpu_tensor([args.batch], datatype=nnc.CCV_32S, device=device)
    staged, consumed = nnc.Signal(device), nnc.Signal(device)

    def prefetch():
        consumed.wait(copy_stream)  # the previous staged batch has been moved into the network input
        nnc.cmd_exec(xfer, None, 0, [host_in, host_lab], [stage_in, stage_lab], copy_stream)
        staged.emit(copy_stream)

    def e2e_step():
        staged.wait(stream)
        nnc.cmd_exec(xfer, None, 0, [stage_in, stage_lab], [net.input, net.labels], stream)
        consumed.emit(stream)
        prefetch()  # next batch: overlaps this step's compute
        step()
        nnc.cmd_exec(xfer, None, 0, [net.loss], [host_loss], stream)
    consumed.emit(stream)
    prefetch()
    e2e_step()
    e2e_ms = timed(e2e_step, args.steps) / args.steps
    copy_stream.wait()
    sampler.stop_flag = True
    sampler.join()
    loss = float(np.mean(host_loss.download()))

    images_per_step = args.batch * world
    value = images_per_step / (ms_per_step * 1e-3)
    math = MATH[dtype][algorithm] if dtype == "f32" else MATH[dtype]
    exchange = ""
    if world > 1:
        exchange = ", %s over the flat %s gradient buffer%s" % (
            "%d COMM_ALLREDUCE commands (NCCL sum; one per gradient bucket, on the backward graph's side stream, overlapped with the rest of the backward pass)" % len(side) if in_graph else "one COMM_ALLREDUCE command (NCCL sum) between backward and SGD",
            "fp32" if dtype == "f32" else dtype, "" if dtype == "f32" else " (+ the small fp32 batch-norm gradient buffer, same NCCL group)")
    out = {"metric": METRIC if dtype == "f32" else METRIC.replace("fp32", dtype), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": dtype, "data": "synthetic",
           "config": {"workload": "ResNet-50 v1d (bin/nnc/imagenet.c:17-95) %s NHWC, per-GPU batch %d, %dx%d, fwd+bwd + nesterov SGD%s%s" % (
                          "fp32" if dtype == "f32" else dtype + " activations / filters / gradients, fp32 master weights + batch-norm parameters", args.batch, args.image, args.image,
                          "" if dtype == "f32" else " (mixed precision)", exchange),
                      "global_batch": images_per_step, "parallelism": "dp%d" % world, "tensor_core_math": math,
                      "cuda_graph": use_graph, "fused_pairs": n_fused, "first_step_loss": first_loss, "l2": "activations per step (>10 GB) exceed the 126 MB L2: no flush needed", "mean_loss": loss},
           "e2e": {"value": images_per_step / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(host_in.nbytes + host_lab.nbytes), "d2h_bytes_per_step": int(host_loss.nbytes), "ms_per_step": e2e_ms,
                   "pipeline": "batch k+1 is copied host->device on a second stream context while step k computes (stream signals); one pinned-host copy + one loss read per step inside the timed region"},
           "gpu_launches": int(launches_per_step * (args.steps * 2 + args.warmup + 2)), "gpu_launches_per_step": int(launches_per_step), "clocks": sampler.summary()}
    if rank == 0:
        # per-command profile (eager, CUDA events around every command) -> roofline of the dominant kernel
        pk = peaks()
        prof = profile_nodes(nnc, net, (g_fb, g_opt), stream, pk, dtype, algorithm)
        out["roofline"] = prof["roofline"]
        out["per_op"] = prof["summary"]
        if per_op_path:
            json.dump(prof, open(per_op_path, "w"), indent=1)
    for x in (g_fb, g_opt, net, stage_in, stage_lab, host_in, host_lab, host_loss, copy_stream, stream):
        x.free()
    return out


def run_sdpa_cfg5(args, steps=None, warmup=3):
    """BASELINE.json configs[4]: CCV_NNC_SCALED_DOT_PRODUCT_ATTENTION_FORWARD bf16 B=32 H=16 S=2048 D=128, non-causal and causal,
    scale 1/sqrt(128), through ccv_nnc_cmd_exec; q / k / v are the reference's i / count ramps (test/int/nnc/cublas.tests.c:2786-2794)
    rounded to bf16.  Per variant: device-timed (CUDA events) with the operands resident in HBM, and end to end from pinned host
    buffers (the three 268 MB operands in, the 268 MB result out, every step, inside the timed region).  steps: timed steps of
    every leg (None: 20 device-timed forwards, 5 end-to-end, 10 backwards, as measured next to the ResNet-50 step)."""
    from ccv_b200 import abi, nnc
    B, H, S, D = 32, 16, 2048, 128
    stream = nnc.Stream(0)
    pk = peaks()
    n = B * S * H * D
    ramp = to_bf16((np.arange(n, dtype=np.float64) / n).astype(np.float32)).reshape(B, S, H, D)
    dev = [nnc.gpu_tensor([B, S, H, D], datatype=abi.CCV_16BF) for _ in range(4)]
    host = [nnc.cpu_tensor([B, S, H, D], datatype=abi.CCV_16BF) for _ in range(4)]
    for t in host:
        nnc.lib().ccv_nnc_tensor_pin_memory(t.ptr)
    for t in host[:3]:
        t.upload(ramp)
    lse = nnc.gpu_tensor([B, H, S])
    grads = [nnc.gpu_tensor([B, S, H, D], datatype=abi.CCV_16BF) for _ in range(3)]
    xfer = nnc.CMD_DATA_TRANSFER_FORWARD()
    assert nnc.cmd_exec(xfer, None, 0, host[:3], dev[:3], stream) == 0
    sampler = ClockSampler(0)
    sampler.start()
    out = {}
    for causal in (0, 1):
        cmd = nnc._simple(abi.CCV_NNC_SCALED_DOT_PRODUCT_ATTENTION_FORWARD)
        cmd.info.scaled_dot_product_attention.scale = 1.0 / np.sqrt(D)
        cmd.info.scaled_dot_product_attention.is_causal = causal

        def fwd():
            assert nnc.cmd_exec(cmd, None, 0, dev[:3], [dev[3], lse], stream) == 0, nnc.lib().ccv_nnc_sm100_last_error()

        def e2e():
            nnc.cmd_exec(xfer, None, 0, host[:3], dev[:3], stream)
            fwd()
            nnc.cmd_exec(xfer, None, 0, [dev[3]], [host[3]], stream)
        res = {}
        for name, fn, reps in (("device", fwd, steps or 20), ("e2e", e2e, steps or 5)):
            for _ in range(warmup):
                fn()
            e0, e1 = nnc.Event(), nnc.Event()
            stream.wait()
            e0.record(stream)
            for _ in range(reps):
                fn()
            e1.record(stream)
            res[name] = e0.elapsed_ms(e1) / reps
        # backward (dq, dk, dv from dout, q, k, v and the forward's saved o / lse: inputs[9], inputs[10]); dout = the q ramp
        bcmd = nnc._simple(abi.CCV_NNC_SCALED_DOT_PRODUCT_ATTENTION_BACKWARD)
        bcmd.info.scaled_dot_product_attention.scale = 1.0 / np.sqrt(D)
        bcmd.info.scaled_dot_product_attention.is_causal = causal
        bcmd.info.scaled_dot_product_attention.deterministic = 1
        b_ins = [dev[0], None, None, dev[0], dev[1], dev[2], None, None, None, dev[3], lse]

        def bwd():
            assert nnc.cmd_exec(bcmd, None, 0, b_ins, grads, stream) == 0, nnc.lib().ccv_nnc_sm100_last_error()
        for _ in range(warmup):
            bwd()
        e0, e1 = nnc.Event(), nnc.Event()
        stream.wait()
        e0.record(stream)
        for _ in range(steps or 10):
            bwd()
        e1.record(stream)
        bms = e0.elapsed_ms(e1) / (steps or 10)
        bflops = 10.0 * B * H * S * S * D * (0.5 if causal else 1.0)  # the 5 GEMMs of the backward; the kernels issue 7 (S and dP twice)
        flops = 4.0 * B * H * S * S * D * (0.5 if causal else 1.0)
        byts = 4.0 * n * 2 + B * H * S * 4
        ms = res["device"]
        out["causal" if causal else "full"] = {
            "backward": {"ms": bms, "tflops": bflops / bms * 1e-9, "frac_of_bf16_peak": bflops / bms * 1e-9 / pk["bf16_tflops"], "algorithmic_flops": bflops,
                         "note": "fused deterministic tcgen05 backward (prep + dK/dV kernel + dQ kernel), 5-GEMM flop count"},
            "ms": ms, "tflops": flops / ms * 1e-9, "frac_of_bf16_peak": flops / ms * 1e-9 / pk["bf16_tflops"], "gbs": byts / ms * 1e-6, "frac_of_hbm_peak": byts / ms * 1e-6 / pk["hbm_gbs"],
            "algorithmic_flops": flops, "algorithmic_bytes": byts, "l2": "Q + K + V + O = 1.07 GB per launch: larger than the 126 MB L2",
            "e2e": {"ms": res["e2e"], "tflops": flops / res["e2e"] * 1e-9, "h2d_bytes_per_step": int(3 * n * 2), "d2h_bytes_per_step": int(n * 2)}}
    sampler.stop_flag = True
    sampler.join()
    out["clocks"] = sampler.summary()
    out["workload"] = "CCV_NNC_SCALED_DOT_PRODUCT_ATTENTION_FORWARD bf16 B=32 H=16 S=2048 D=128 (BASELINE.json configs[4]), tcgen05 flash-attention kernel, LSE written; `backward` = CCV_NNC_SCALED_DOT_PRODUCT_ATTENTION_BACKWARD on the same tensors"
    for t in dev + host + grads + [lse, stream]:
        t.free()
    return out


def run_reference_cnnp(args):
    """BASELINE.json configs[2] through the REFERENCE'S OWN public API: integration/cnnp_resnet50_bench.c builds the same ResNet-50 v1d
    with ccv_cnnp_* and trains it with ccv_cnnp_model_fit; linked against integration/_build/libccv_dropin.so every layer above the
    backend is the unmodified reference (model zoo, symbolic graph, autograd, memory planner, graph runner: one ccv_nnc_cmd_exec per node,
    no fusion pass, no CUDA graph) and every GPU command is served by CCV_NNC_BACKEND_GPU_SM100.  Runs as a child process after this
    process has finished its own measurements; whatever goes wrong there is reported as `unavailable`, never raised."""
    import subprocess
    exe = os.path.join(ROOT, "integration", "_build", "cnnp_resnet50_bench")
    if not os.path.exists(exe):
        return {"unavailable": "integration/_build/cnnp_resnet50_bench is not built (make -C integration; needs the reference sources)"}
    steps = max(1, min(int(args.steps), 5))
    cmd = [exe, "--device", "gpu", "--batch", str(args.batch), "--image", str(args.image), "--steps", str(steps), "--warmup", "2"]
    try:
        p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=150)
    except subprocess.TimeoutExpired:
        return {"unavailable": "timed out after 150 s"}
    except Exception as e:  # noqa: BLE001 -- a side measurement must not take the benchmark line down
        return {"unavailable": repr(e)[:300]}
    lines = [ln for ln in p.stdout.decode(errors="replace").splitlines() if ln.startswith("{")]
    if p.returncode != 0 or not lines:
        return {"unavailable": "exit %d: %s" % (p.returncode, p.stderr.decode(errors="replace").strip()[-400:])}
    try:
        r = json.loads(lines[-1])
    except ValueError:
        return {"unavailable": "unparsable output: " + lines[-1][:200]}
    r["note"] = ("the unmodified reference L2-L5 (ccv_cnnp_model_fit -> its symbolic graph / autograd / graph runner) on this backend as the only GPU "
                 "backend of the library; host-timed around ccv_nnc_stream_context_wait; inputs resident on the device")
    return r



def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="sm100")
    ap.add_argument("--batch", type=int, default=256, help="per-GPU batch (BASELINE: 256)")
    ap.add_argument("--image", type=int, default=224)
    ap.add_argument("--dtype", default="f32", choices=sorted(DTYPES), help="headline model dtype (the JSON line's own numbers); the other configurations ride along under `variants`")
    ap.add_argument("--algorithm", type=int, default=-1, help="fp32 contraction algorithm: -1 default (convolutions TF32, GEMM 3xTF32), 0 TF32, 1 3xTF32, 2 FFMA")
    ap.add_argument("--workload", default="resnet50", choices=["resnet50", "sdpa_cfg5"])
    ap.add_argument("--no-variants", action="store_true", help="only the headline configuration")
    ap.add_argument("--exchange", default="between", choices=["overlap", "between"], help="N > 1: one allreduce command between the backward and the optimizer graph (default), or bucketed allreduce nodes inside the backward graph on its side stream")
    ap.add_argument("--buckets", type=int, default=4, help="gradient buckets of the overlapped exchange")
    ap.add_argument("--no-cuda-graph", action="store_true")
    ap.add_argument("--no-fuse", action="store_true", help="run every reference command as its own kernel sequence (no peephole fusion)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--per-op", default="", help="write the per-command profile to this JSON file")
    ap.add_argument("--dump-outputs", default="", metavar="DIR", help="write what the last timed step of the headline configuration computed to DIR/<name>.npy (float32, about 18 MB)")
    args = ap.parse_args()
    if args.dump_outputs and (args.workload != "resnet50" or args.impl != "sm100"):
        ap.error("--dump-outputs writes the outputs of the resnet50 workload on this backend only")
    if args.impl == "reference":
        return reference_arm(args)
    args.warmup = max(args.warmup, 3)

    rank, world, local_rank = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from ccv_b200 import nnc
    nnc.init()
    if nnc.lib().ccv_nnc_device_count(nnc.CCV_STREAM_CONTEXT_GPU) <= 0:
        raise SystemExit("bench.py: no CUDA device and there is no CPU fallback (use --impl reference for the CPU_REF arm)")
    if args.workload == "sdpa_cfg5":
        if rank == 0:
            r = run_sdpa_cfg5(args, args.steps, args.warmup)
            full = r["full"]
            print(json.dumps({"metric": "sdpa_fwd_bf16_b32_h16_s2048_d128_tflops", "value": full["tflops"], "unit": "TFLOP/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": full["ms"], "higher_is_better": True,
                              "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": {"workload": r["workload"]},
                              "roofline": {"bound": "tensor", "achieved": full["tflops"], "peak": peaks()["bf16_tflops"], "unit": "TFLOP/s", "frac": full["frac_of_bf16_peak"], "traffic": None},
                              "e2e": {"value": full["e2e"]["tflops"], "unit": "TFLOP/s", "h2d_bytes_per_step": full["e2e"]["h2d_bytes_per_step"], "d2h_bytes_per_step": full["e2e"]["d2h_bytes_per_step"]},
                              "gpu_launches": 2 * (23 + 8), "sdpa": r, "clocks": r["clocks"]}))
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        return

    out = run_model(args, dist, rank, world, local_rank, args.dtype, args.algorithm, args.per_op, args.dump_outputs)
    if not args.no_variants:
        # the other BASELINE configurations, measured by the same code in the same process (same box, same clocks):
        #   bf16     configs[3] (ResNet-50 16-bit, batch-sharded): at N GPUs this IS configs[3]'s per-GPU shard of N x 256 images
        #   3xtf32   the fp32 model with fp32-grade (error-compensated) convolutions: what the <= 1e-3 whole-model parity is held on
        #   sdpa     configs[4] (N = 1 only: a single-op config, replicas add nothing)
        variants = {}
        for name, (dtype, algorithm) in (("bf16", ("bf16", -1)), ("fp32_3xtf32", ("f32", 1))):
            if dtype == args.dtype and algorithm == args.algorithm:
                continue
            v = run_model(args, dist, rank, world, local_rank, dtype, algorithm)
            variants[name] = {k: v[k] for k in ("metric", "value", "unit", "ms_per_step", "dtype", "config", "e2e", "gpu_launches_per_step", "clocks") if k in v}
            if "roofline" in v:
                variants[name]["roofline"], variants[name]["per_op"] = v["roofline"], v["per_op"]
        if world == 1 and rank == 0:
            variants["sdpa_cfg5"] = run_sdpa_cfg5(args)
            variants["reference_cnnp_resnet50"] = run_reference_cnnp(args)
        out["variants"] = variants
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(args.image)
        print(json.dumps(out))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


FUSED_NAMES = {1: "bn_relu_fwd", 2: "relu_bn_bwd", 3: "add_relu_fwd", 4: "add_relu_bwd", 5: "sgd", 7: "bn_fwd", 8: "bn_bwd"}


def node_cost(cmd, fused_kind, ins, outs):
    """(kind, algorithmic flops, algorithmic bytes) of one node, from its tensors (SURVEY.md 8d per-unit figures:
    contractions = 2 * M * N * K flops; everything else = the bytes it must read + write once)."""
    from ccv_b200 import abi
    nb = lambda t: 0 if t is None else t.nbytes
    if fused_kind == 6:  # convolution that also emits the batch-norm statistics: cost it as the convolution it is
        fused_kind, outs = 0, outs[:1]
    if fused_kind in (1, 7) and len(ins) == 6:  # batch norm reading those statistics: the small statistics tensor is not activation traffic
        ins = ins[:5]
    io = sum(nb(t) for t in ins) + sum(nb(t) for t in outs)
    if fused_kind:
        return FUSED_NAMES[fused_kind], 0.0, io
    c = cmd
    if c == abi.CCV_NNC_CONVOLUTION_FORWARD:
        n, p, q, k = outs[0].dims
        return "conv_fwd", 2.0 * n * p * q * k * ins[1].count / ins[1].dims[0], io
    if c == abi.CCV_NNC_CONVOLUTION_BACKWARD:
        n, p, q, k = ins[0].dims
        f = 2.0 * n * p * q * k * ins[2].count / ins[2].dims[0]
        return "conv_bwd", f * (2 if outs[0] is not None else 1), io
    if c == abi.CCV_NNC_GEMM_FORWARD:
        return "gemm_fwd", 2.0 * outs[0].count * ins[0].dims[-1], io
    if c == abi.CCV_NNC_GEMM_BACKWARD:
        return "gemm_bwd", 4.0 * ins[0].count * ins[1].dims[-1], io
    names = {abi.CCV_NNC_BATCH_NORM_FORWARD: "bn_fwd", abi.CCV_NNC_BATCH_NORM_BACKWARD: "bn_bwd", abi.CCV_NNC_RELU_FORWARD: "relu_fwd", abi.CCV_NNC_RELU_BACKWARD: "relu_bwd",
             abi.CCV_NNC_EWSUM_FORWARD: "ewsum", abi.CCV_NNC_MAX_POOL_FORWARD: "maxpool_fwd", abi.CCV_NNC_MAX_POOL_BACKWARD: "maxpool_bwd", abi.CCV_NNC_AVERAGE_POOL_FORWARD: "avgpool_fwd",
             abi.CCV_NNC_AVERAGE_POOL_BACKWARD: "avgpool_bwd", abi.CCV_NNC_SGD_FORWARD: "sgd", abi.CCV_NNC_SOFTMAX_FORWARD: "softmax", abi.CCV_NNC_SOFTMAX_BACKWARD: "softmax"}
    return names.get(c, "other"), 0.0, io


def profile_nodes(nnc, net, graphs, stream, pk, dtype="f32", algorithm=-1):
    """Every node of one step run on its own with CUDA events around it (best of 3), through the same runner."""
    by_ptr = dict((t.ptr, t) for t in net.tensors)
    rows = []
    for gph in graphs:
        ms = gph.profile(stream, 3)
        for (cmd, fk, ins, outs), t in zip(gph.nodes(), ms):
            kind, flops, nbytes = node_cost(cmd, fk, [by_ptr.get(p) for p in ins], [by_ptr.get(p) for p in outs])
            rows.append(dict(kind=kind, ms=t, flops=flops, bytes=nbytes))
    summary = {}
    for r in rows:
        s = summary.setdefault(r["kind"], dict(n=0, ms=0.0, flops=0.0, bytes=0.0))
        s["n"] += 1
        s["ms"] += r["ms"]
        s["flops"] += r["flops"]
        s["bytes"] += r["bytes"]
    # tensor peak of the math the contractions run in: bf16 / fp16 = the measured cuBLAS bf16 number; TF32 = half of it;
    # 3xTF32 = a third of the TF32 rate (three MMAs per product)
    tf32_peak = pk["bf16_tflops"] if dtype != "f32" else pk["bf16_tflops"] / 2.0 / (3.0 if algorithm == 1 else 1.0)
    peak_note = "bf16 cuBLAS burst peak" if dtype != "f32" else ("bf16 cuBLAS burst peak / 2 (TF32 tensor rate is half the bf16 rate)" + (" / 3 (3xTF32 issues three MMAs per product)" if algorithm == 1 else ""))
    for k, s in summary.items():
        if s["flops"] > 0:
            s["tflops"] = s["flops"] / (s["ms"] * 1e-3) / 1e12
            s["frac_of_tensor_peak"] = s["tflops"] / tf32_peak
        s["gbs"] = s["bytes"] / (s["ms"] * 1e-3) / 1e9
        s["frac_of_hbm_peak"] = s["gbs"] / pk["hbm_gbs"]
    tc = [r for r in rows if r["flops"] > 0]
    tc_flops, tc_ms = sum(r["flops"] for r in tc), sum(r["ms"] for r in tc)
    achieved = tc_flops / (tc_ms * 1e-3) / 1e12 if tc_ms > 0 else 0.0
    # every contraction command against ITS OWN bound, max(flops / tensor peak, algorithmic bytes / HBM peak): the 1x1 convolutions and the
    # stem move more bytes than they have flops for (half of the 110 convolution commands of ResNet-50 at N = 256 are HBM-bound)
    bound_ms = sum(max(r["flops"] / (tf32_peak * 1e12), r["bytes"] / (pk["hbm_gbs"] * 1e9)) for r in tc) * 1e3
    # DRAM bytes of the same launches from one ncu capture (tools/run_ncu_profiles.sh -> profiles/): all
    # contraction launches of one step, to be read against the algorithmic operand + result bytes of those commands
    traffic, traffic_note = None, None
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r02_contraction_traffic.json")))
        traffic, traffic_note = float(t["dram_bytes_per_step"]), "dram__bytes_read.sum + dram__bytes_write.sum over the %d contraction launches of one step (ncu, tools/run_ncu_profiles.sh -> profiles/r02_contraction_traffic.json)" % t["launches"]
    except Exception:
        pass
    if dtype != "f32" or algorithm == 1:
        traffic, traffic_note = None, None  # the committed ncu capture is of the fp32 / TF32 configuration
    roofline = {"bound": "tensor", "kernel": "umma_* (tcgen05 GEMM / implicit-GEMM convolution kernels; all convolution + GEMM commands of one step)", "achieved": achieved, "peak": tf32_peak, "unit": "TFLOP/s",
                "frac": achieved / tf32_peak, "traffic": traffic, "traffic_note": traffic_note, "algorithmic_bytes_per_step": sum(r["bytes"] for r in tc),
                "peak_source": "%s %s" % (pk["source"], peak_note),
                "launch_ms_total": tc_ms, "algorithmic_flops_per_step": tc_flops, "total_ms_all_commands": sum(r["ms"] for r in rows),
                "per_command_bound_ms": bound_ms, "frac_of_per_command_bound": bound_ms / tc_ms if tc_ms > 0 else None,
                "hbm_bound_commands": sum(1 for r in tc if r["bytes"] / (pk["hbm_gbs"] * 1e9) > r["flops"] / (tf32_peak * 1e12)), "contraction_commands": len(tc)}
    return dict(roofline=roofline, summary=summary, rows=rows)


if __name__ == "__main__":
    main()
