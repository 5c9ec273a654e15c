"""bench.py -- images/sec of the YOLOv6-S 640x640 bs32 inference hot path on N x B200 (BASELINE.json).

    python bench.py [--gpus N --steps K --warmup W] [--impl reference]
                    [--mode infer|train] [--model yolov6s] [--batch 32] [--size 640] [--no-extra]
                    [--dump-outputs DIR]

The default run prints ONE JSON line whose headline (`value`, `e2e`, `roofline`) is BASELINE.json's config 2 and which
also carries, under `modes`, the fp32-equivalent (bf16x3) precision mode with the measured bf16-vs-fp32 deviation on the
benchmark input, and under `configs` short measurements of the other GPU configurations of BASELINE.json: config 3
(YOLOv6-S bs32 training step), config 4 (YOLOv6-M training, 8 images per GPU, gradient all-reduce when N > 1) and
config 5 (YOLOv6-L6 1280x1280, 2 images per GPU).  `--mode train` makes the training step the headline instead.

One "step" = one batch through the whole hot path: stem -> backbone -> neck -> head -> decode
(sm_100a kernels via the C ABI) -> batched NMS (eval settings conf 0.03 / iou 0.65 / multi_label,
the settings of the reference's Evaler, core/evaler.py:118-134).  Per rank the batch is 32 images
(weak scaling: images are sharded across GPUs, no collective on this path -- SURVEY.md 8e).

JSON keys (see the task contract): value = device-resident throughput (CUDA events, max over ranks);
e2e = same metric through the public API from pinned HOST uint8 images incl. H2D and the D2H of the
detections; roofline = algorithmic conv FLOPs / measured conv-kernel time vs the measured bf16 peak;
cpu_baseline = the oracle (CPU restatement of the reference path) on a bounded sample of the workload.
`--impl reference` times that CPU path alone with all host threads.

`--dump-outputs DIR` writes, after the timed steps of the headline, what its last step computed as .npy files (rank 0):
inference: `detections.npy` float32 [n, 6] -- the per-image (x1, y1, x2, y2, conf, cls) rows `non_max_suppression` returns,
concatenated in image order -- and `counts.npy` float64 [batch], the rows per image; with CUDA graphs the last step's NMS
branch post-processes the batch before it (DetectStream), and those are its detections.  Training: `loss.npy` float64 [8],
what `TrainStep.run` returns.  Weights and inputs are seeded, so the same arguments give the same inputs on every run.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "images/sec YOLOv6-S 640 bs32"
GFLOP_PER_IMG = {"yolov6n": 11.316, "yolov6s": 44.967, "yolov6m": 85.087, "yolov6l6": 665.834}  # BASELINE.md section 2
NMS_KW = dict(conf_thres=0.03, iou_thres=0.65, multi_label=True, max_det=300)


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def load_keys(model):
    with open(os.path.join(ROOT, "tests", "golden", f"keys_{model}.json")) as f:
        return [(k, tuple(s)) for k, s in json.load(f)]


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons with nvidia-smi while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows if len(r) > 2 + i)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


def host_cores():
    """Host threads this process can really use: CPU affinity, capped by the cgroup CPU quota (a container
    that sees 128 logical CPUs but is throttled to a few would otherwise be timed oversubscribed)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:                       # cgroup v2
            quota, period = f.read().split()
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except (OSError, ValueError):
        try:                                                            # cgroup v1
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                quota = int(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                period = int(f.read())
            if quota > 0:
                n = max(1, min(n, quota // period))
        except (OSError, ValueError):
            pass
    return n


def pick_threads(step_one_image):
    """The thread count (<= host_cores()) at which the CPU path runs fastest on a 1-image probe -- the CPU arm
    gets its best configuration, not an oversubscribed one."""
    best, best_t = None, float("inf")
    cores = host_cores()
    for n in sorted({cores, min(cores, 64), min(cores, 32), min(cores, 16), min(cores, 8)}, reverse=True):
        torch.set_num_threads(n)
        step_one_image()
        t0 = time.perf_counter()
        step_one_image()
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best


def cpu_reference_step(sd, cfg, images, nms_kw):
    """The reference path restated on CPU (oracle): eval forward + NMS on `images` (NCHW fp32)."""
    from oracle import model as om
    from oracle import nms as onms
    with torch.no_grad():
        pred = om.forward(sd, cfg, images)
    return onms.non_max_suppression(pred.numpy(), **nms_kw)


def run_reference(args):
    """`--impl reference`: the reference's CPU implementation of the path (oracle port; /root/reference is
    not on the GPU box) on the host cores; rank 0 only."""
    rank, _, world = dist_env()
    if rank != 0:
        return
    from oracle import fabricate as fab
    from oracle import model as om
    from yolov6_b200.model import build_model          # only as the container of the seeded synthetic checkpoint
    from yolov6_b200.synth import randomize_            # (same weights as the GPU arm); nothing of it is timed
    sd = {k: v.detach() for k, v in randomize_(build_model(args.model, 80, torch.device("cpu")), seed=0).state_dict().items()}
    cfg = om.CONFIGS[args.model]
    sample = args.ref_batch
    x = fab.synthetic_images(sample, args.size, args.size, seed=0)
    cores = pick_threads(lambda: cpu_reference_step(sd, cfg, x[:1], NMS_KW))
    for _ in range(args.warmup_ref):
        cpu_reference_step(sd, cfg, x, NMS_KW)
    t0 = time.perf_counter()
    for _ in range(args.steps_ref):
        cpu_reference_step(sd, cfg, x, NMS_KW)
    dt = (time.perf_counter() - t0) / args.steps_ref
    val = sample / dt
    line = {"metric": METRIC, "value": val, "unit": "images/s", "n_gpus": world, "steps": args.steps_ref, "warmup": args.warmup_ref,
            "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "impl": "reference",
            "config": {"workload": f"{args.model} {args.size}x{args.size} inference + NMS (CPU oracle port of the reference path)",
                       "sample": f"batch {sample} per step", "nms": NMS_KW},
            "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "kind": "port",
                             "sample": f"{args.steps_ref} steps x batch {sample} at {args.size}x{args.size}"},
            "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def barrier(world):
    import torch.distributed as dist
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def timed(fn, steps, warmup, world, dev, farm=None):
    """W untimed steps, then exactly K steps between barrier + synchronize, CUDA events, max over ranks -> ms per step.
    farm: the steps run on the farm's own streams; the timing events bracket them through fence() / release()."""
    import torch.distributed as dist
    for i in range(warmup):
        fn(i)
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    if farm is not None:
        farm.release()         # no lane starts a timed step before e0
    for i in range(steps):
        fn(i)
    if farm is not None:
        farm.fence()           # e1 follows the last kernel of every lane
    e1.record()
    barrier(world)
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return ms.item() / steps


def load_peaks():
    pk_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk_path):
        with open(pk_path) as f:
            return json.load(f)
    return {}


def caller_detections(out, count, overflow):
    """The detections `non_max_suppression` would return for nms_batched's (out, count, overflow), as numpy arrays."""
    if int(overflow.item()):
        raise RuntimeError("non_max_suppression: more than 65536 near-identical candidate scores in one image")
    n = count.tolist()
    rows = torch.cat([out[b, :k] for b, k in enumerate(n)])
    return {"detections": rows.float().cpu().numpy(), "counts": torch.tensor(n, dtype=torch.float64).numpy()}


def dump_outputs(path, arrays):
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), a)


def bench_infer(model_name, B, S, steps, warmup, rank, world, dev, precision="bf16", e2e=True, roofline=True, graph=True,
                keep_outputs=False):
    """Forward + decode + batched NMS of `model_name` on B images of S x S per GPU.  Returns a dict of measurements
    (with keep_outputs, `_outputs`: the detections of the last timed step)."""
    from yolov6_b200.model import build_model
    from yolov6_b200.nms import nms_batched
    from yolov6_b200.pipeline import DetectFarm
    from yolov6_b200.synth import randomize_
    model = randomize_(build_model(model_name, 80, dev), seed=0)   # seeded synthetic checkpoint
    model.eval().set_precision(precision)
    eng = model.engine()
    g = torch.Generator().manual_seed(1 + rank)   # per-rank data like tools/train.py:104 seeds per rank
    host_u8 = [(torch.rand(B, 3, S, S, generator=g) * 255).to(torch.uint8).pin_memory() for _ in range(2)]
    dev_f32 = [h.to(dev).float() / 255 for h in host_u8]
    out = {"model": model_name, "batch_per_gpu": B, "size": S, "precision": precision}
    if graph:
        # steady state = one CUDA-graph launch per batch (yolov6_b200/pipeline.py); two pipelines with
        # separate static buffers alternate so that consecutive steps never reuse a cached input
        # (DetectStream: the graph of step i runs the network of batch i and, as a parallel branch, the NMS of batch i - 1)
        # DetectFarm: `lanes` such pipelines with their own buffers and streams, fed round-robin (independent batches)
        n_lanes = int(os.environ.get("YV6_FARM", "2"))
        stream_dev = DetectFarm(model, B, S, S, lanes=n_lanes, host_input=False, **NMS_KW)
        for ln in stream_dev.lanes:
            for i in range(2):
                ln.x_dev[i].copy_(dev_f32[i])

        def step_device(i):
            stream_dev.launch()
    else:
        last = {}

        def step_device(i):
            pred = eng.forward(dev_f32[i & 1])
            last["nms"] = nms_batched(pred, **NMS_KW)
    with torch.no_grad():
        ms_dev = timed(step_device, steps, warmup, world, dev, farm=stream_dev if graph else None)
        out["ms_per_step"] = ms_dev
        if keep_outputs:
            if graph:
                lane = stream_dev.lanes[(stream_dev.n - 1) % len(stream_dev.lanes)]
                res = lane.dev_step[1 - ((lane.steps - 1) & 1)]     # the NMS branch of the lane's last graph
            else:
                o, c, _, ov = last["nms"]
                res = (o, c, ov)
            out["_outputs"] = caller_detections(*res)
        out["value"] = world * B / (ms_dev * 1e-3)
        if e2e:
            if graph:
                stream_e2e = DetectFarm(model, B, S, S, lanes=n_lanes, host_input=True, **NMS_KW)   # H2D of batch i+1 overlaps the kernels of batch i
                for ln in stream_e2e.lanes:
                    for i in range(2):
                        ln.x_host[i].copy_(host_u8[i])

                def step_e2e(i):
                    stream_e2e.launch()            # H2D (u8, copy stream) -> graph: network(i) || NMS(i-1) -> D2H detections
            else:
                def step_e2e(i):
                    x = host_u8[i & 1].to(dev, non_blocking=True)
                    o, c, _, _ = nms_batched(eng.forward(x), **NMS_KW)
                    return o.cpu(), c.cpu()
            ms_e2e = timed(step_e2e, steps, warmup, world, dev, farm=stream_e2e if graph else None)
            out["e2e"] = {"value": world * B / (ms_e2e * 1e-3), "unit": "images/s", "ms_per_step": ms_e2e,
                          "h2d_bytes_per_step": B * 3 * S * S, "d2h_bytes_per_step": B * NMS_KW["max_det"] * 6 * 4 + B * 4}
        if roofline:
            conv_ms, conv_flop, n_conv = eng.profile_convs(dev_f32[0], steps=5)
            out["conv"] = {"ms": conv_ms, "flop": conv_flop, "launches": n_conv, "bytes_per_launch": eng.conv_bytes_per_launch(B, S, S)}
    out["launches_per_step"] = eng.launch_count(B, S, S) + (7 if 8400 * 80 > 65536 else 3)
    out["_model"], out["_input"] = model, dev_f32[0]
    return out


def precision_check(model, x, dev):
    """bf16 speed mode against the fp32-equivalent (bf16x3) mode on the benchmark input: max |a-b|/(1+|b|) over the
    [B, A, 85] predictions and the fraction of NMS output rows (box, score, class) that are identical."""
    from yolov6_b200.nms import nms_batched
    with torch.no_grad():
        model.set_precision("bf16")
        p16 = model.engine().forward(x).clone()
        o16, c16, _, _ = nms_batched(p16, **NMS_KW)
        model.set_precision("fp32")
        p32 = model.engine().forward(x).clone()
        o32, c32, _, _ = nms_batched(p32, **NMS_KW)
        err = float(((p16 - p32).abs() / (1 + p32.abs())).max())
        err_cls = float((p16[..., 5:] - p32[..., 5:]).abs().max())
        same, total, same_cls = 0, 0, 0
        c16, c32 = c16.tolist(), c32.tolist()
        for b in range(p16.shape[0]):
            n = min(c16[b], c32[b])
            total += max(c16[b], c32[b])
            same += int((o16[b, :n] == o32[b, :n]).all(-1).sum())
            # same detection = same class and boxes within a pixel, whatever the rank in the list
            same_cls += int(((o16[b, :n, 5] == o32[b, :n, 5]) & ((o16[b, :n, :4] - o32[b, :n, :4]).abs().max(-1).values < 1.0)).sum())
        model.set_precision("bf16")
    return {"max_rel_err_bf16_vs_fp32": err, "max_abs_err_scores": err_cls, "nms_rows_bit_identical_frac": same / max(total, 1),
            "nms_rows_same_class_and_box_within_1px_frac": same_cls / max(total, 1), "nms_rows": total,
            "tolerance_note": "north_star's 1e-4 is met by the fp32 mode (tests/test_gpu_model.py); bf16 is the speed mode"}


TRAIN_LOSS = {"yolov6n": dict(use_dfl=False, reg_max=0, iou_type="siou"), "yolov6s": dict(use_dfl=False, reg_max=0, iou_type="giou"),
              "yolov6m": dict(use_dfl=True, reg_max=16, iou_type="giou"), "yolov6l6": dict(use_dfl=True, reg_max=16, iou_type="giou")}


def bench_train(model_name, B, S, steps, warmup, rank, world, dev, graph=True, keep_outputs=False):
    """One training step of `model_name` on B images per GPU (BASELINE.json config 3 / 4): train-form forward, TAL
    assignment, VFL + IoU (+ DFL) loss, backward, gradient all-reduce over NCCL when world > 1; the optimizer (fused SGD +
    EMA) is timed separately and inside the end-to-end number."""
    from yolov6_b200.loss import ComputeLoss
    from yolov6_b200.model import build_model
    from yolov6_b200.optim import FusedSGDEMA
    from yolov6_b200.step import TrainStep
    from yolov6_b200.synth import synthetic_targets
    torch.manual_seed(0)                                  # same initial weights on every rank (DDP broadcasts rank 0's)
    model = build_model(model_name, 80, dev).train()      # random init of the architecture (initialize_biases etc.)
    strides = [int(v) for v in model.graph.strides]
    crit = ComputeLoss(fpn_strides=strides, num_classes=80, ori_img_size=S, warmup_epoch=0, **TRAIN_LOSS[model_name])
    opt = FusedSGDEMA(model, lr=0.01, momentum=0.937, weight_decay=5e-4)
    step = TrainStep(model, crit, B, S, S, in_dtype=torch.uint8, max_gt=64, optimizer=None, graph=graph)
    g = torch.Generator().manual_seed(1 + rank)           # tools/train.py:104 seeds per rank
    imgs = [(torch.rand(B, 3, S, S, generator=g) * 255).to(torch.uint8).pin_memory() for _ in range(2)]
    tgts = [synthetic_targets(B, seed=100 + 10 * rank + i).pin_memory() for i in range(2)]
    loss_host = torch.zeros(8, dtype=torch.float64).pin_memory()
    step.load(imgs[0], tgts[0])

    def step_device(i):
        step.run(epoch_num=0)

    def step_opt(i):
        opt.upload_hyper()
        opt.launch()

    def step_e2e(i):
        step.load(imgs[i & 1], tgts[i & 1])               # H2D: uint8 images + targets from pinned memory
        out = step.run(epoch_num=0)
        opt.upload_hyper()
        opt.launch()
        loss_host.copy_(out, non_blocking=True)           # D2H: loss / loss items

    ms_dev = timed(step_device, steps, warmup, world, dev)
    outputs = {"loss": step.state["out"].double().cpu().numpy()}
    first_loss = [float(v) for v in step.state["out"][:4].tolist()]
    ar_ms = step.sync.last_ms() if step.sync is not None else 0.0
    ms_opt = timed(step_opt, steps, 1, world, dev)
    ms_e2e = timed(step_e2e, steps, warmup, world, dev)
    model.mark_weights_changed()
    torch.cuda.synchronize()
    last_loss = [float(v) for v in loss_host[:4].tolist()]
    f, b = step.eng.launch_counts()
    nbytes = step.eng.flat.n_train * 4
    peaks = load_peaks()
    gflop_img = 3.0 * GFLOP_PER_IMG[model_name] * (S / (1280.0 if model_name == "yolov6l6" else 640.0)) ** 2
    achieved = gflop_img * 1e9 * B / (ms_dev * 1e-3) / 1e12
    peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
    res = {"model": model_name, "batch_per_gpu": B, "size": S, "value": world * B / (ms_dev * 1e-3), "unit": "images/s",
            "ms_per_step": ms_dev, "step": "train-form forward + TAL + VFL/GIoU" + ("/DFL" if TRAIN_LOSS[model_name]["use_dfl"] else "") +
            " loss + backward" + (" + gradient all-reduce" if world > 1 else ""),
            "optimizer_ms": ms_opt, "optimizer": "fused SGD-nesterov + weight decay + EMA, one kernel (yv6_sgd_ema_step)",
            "e2e": {"value": world * B / (ms_e2e * 1e-3), "unit": "images/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": B * 3 * S * S + int(tgts[0].numel()) * 4, "d2h_bytes_per_step": 64,
                    "includes": "H2D of uint8 images + targets, step, optimizer, D2H of the loss"},
            "allreduce": {"bytes_per_step": nbytes if world > 1 else 0, "buckets": len(step.eng.bucket_range), "dtype": "f32",
                          "ms_first_bucket_to_done": ar_ms, "world": world},
            "launches_per_step": 2 + f + b + 8, "graph": bool(graph),
            "loss_first_step": first_loss, "loss_after_training_steps": last_loss,
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                         "algorithmic_gflop_per_img": gflop_img,
                         "note": "3 x the deploy-form forward FLOPs (fwd + dgrad + wgrad), SURVEY.md 8d; the train form executes ~9 % more"}}
    if keep_outputs:
        res["_outputs"] = outputs
    return res


def free_cuda():
    import gc
    gc.collect()
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="infer", choices=["infer", "train"])
    ap.add_argument("--model", default="yolov6s")
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--size", type=int, default=None)
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--ref-batch", type=int, default=8)
    ap.add_argument("--steps-ref", type=int, default=3)
    ap.add_argument("--warmup-ref", type=int, default=1)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the fp32-mode leg and the other BASELINE configs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the headline computed to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    if args.size is None:
        args.size = 1280 if args.model == "yolov6l6" else 640
    if args.batch is None:
        args.batch = 32 if args.model != "yolov6l6" else 2
    if args.impl == "reference":
        return run_reference(args)

    rank, local_rank, world = dist_env()
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W = max(args.warmup, 3)
    use_graph = not args.no_graph
    B, S = args.batch, args.size
    sampler = ClockSampler(local_rank)
    sampler.start()
    peaks = load_peaks()
    peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
    short = max(5, min(args.steps, 20))

    if args.mode == "train":
        tr = bench_train(args.model, B, S, args.steps, W, rank, world, dev, graph=use_graph, keep_outputs=bool(args.dump_outputs))
        outputs = tr.pop("_outputs", None)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, outputs)
        sampler.stop_flag = True
        sampler.join(timeout=2)
        if rank == 0:
            line = {"metric": f"images/sec {args.model} {S} bs{B} training step", "value": tr["value"], "unit": "images/s", "n_gpus": world,
                    "steps": args.steps, "warmup": W, "ms_per_step": tr["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                    "vs_baseline": None, "dtype": "bf16 (fp32 master weights, fp32 accumulation)", "data": "synthetic",
                    "config": {"workload": f"{args.model} {S}x{S} bs{B}/GPU training step: {tr['step']}",
                               "targets": "synthetic COCO-shaped (Poisson(7.3) boxes per image)", "weights": "random init",
                               "parallelism": f"dp{world} image-sharded, one gradient all-reduce (sum) per step",
                               "l2": "activations (> 5 GB per step) exceed the 126 MB L2",
                               "launch": "CUDA graph segments (TrainStep)" if use_graph else "eager ctypes launches"},
                    "e2e": tr["e2e"], "gpu_launches": tr["launches_per_step"] * args.steps, "roofline": tr["roofline"],
                    "train": {k: v for k, v in tr.items() if k not in ("e2e", "roofline", "value", "unit", "ms_per_step")},
                    "clocks": sampler.summary()}
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---------------------------------------------------------------- inference headline (BASELINE.json config 2)
    main_r = bench_infer(args.model, B, S, args.steps, W, rank, world, dev, precision=args.precision, graph=use_graph,
                         keep_outputs=bool(args.dump_outputs))
    model, x0 = main_r.pop("_model"), main_r.pop("_input")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, main_r.pop("_outputs"))
    modes, check, extra = {}, None, {}
    if not args.no_extra:
        check = precision_check(model, x0, dev)
        other = "fp32" if args.precision == "bf16" else "bf16"
        del model
        free_cuda()
        r2 = bench_infer(args.model, B, S, short, 3, rank, world, dev, precision=other, e2e=False, roofline=False, graph=use_graph)
        r2.pop("_model"), r2.pop("_input")
        modes = {args.precision: {"value": main_r["value"], "ms_per_step": main_r["ms_per_step"]},
                 other: {"value": r2["value"], "ms_per_step": r2["ms_per_step"], "steps": short}}
        modes["note"] = "fp32 = bf16x3 split operands (fp32-equivalent products, fp32 accumulation): the mode that meets the 1e-4 bar"
        del r2
        free_cuda()
        # the other GPU configurations of BASELINE.json, per-GPU shard sizes, short runs
        try:
            t3 = bench_train("yolov6s", 32, 640, short, 3, rank, world, dev, graph=use_graph)
            extra["config3_yolov6s_bs32_train_step"] = t3
            free_cuda()
            t4 = bench_train("yolov6m", 8, 640, short, 3, rank, world, dev, graph=use_graph)
            extra["config4_yolov6m_bs8_per_gpu_train_step"] = t4
            free_cuda()
            r5 = bench_infer("yolov6l6", 2, 1280, short, 3, rank, world, dev, precision="bf16", e2e=True, roofline=True, graph=use_graph)
            r5.pop("_model"), r5.pop("_input")
            c5 = r5.pop("conv")
            r5["roofline"] = {"bound": "tensor", "achieved": c5["flop"] / (c5["ms"] * 1e-3) / 1e12, "peak": peak_tf, "unit": "TFLOP/s",
                              "frac": c5["flop"] / (c5["ms"] * 1e-3) / 1e12 / peak_tf, "conv_ms_per_step": c5["ms"], "launches_per_step": c5["launches"]}
            extra["config5_yolov6l6_1280_bs2_per_gpu_inference"] = r5
            free_cuda()
        except Exception as e:  # noqa: BLE001 -- the headline must survive a failure of an auxiliary measurement
            extra["error"] = f"{type(e).__name__}: {e}"
    sampler.stop_flag = True
    sampler.join(timeout=2)

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    conv = main_r["conv"]
    achieved_tf = conv["flop"] / (conv["ms"] * 1e-3) / 1e12
    traffic = None                # DRAM bytes per conv launch from the committed ncu capture (profiles/)
    for tname in ("r02_conv_traffic.json", "r01_conv_traffic.json"):
        tpath = os.path.join(ROOT, "profiles", tname)
        if os.path.exists(tpath):
            with open(tpath) as f:
                traffic = json.load(f).get("dram_bytes_per_launch")
            break
    line = {
        "metric": METRIC if (args.model, B, S) == ("yolov6s", 32, 640) else f"images/sec {args.model} {S} bs{B}",
        "value": main_r["value"], "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": W, "ms_per_step": main_r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16" if args.precision == "bf16" else "bf16x3 (fp32-equivalent)", "data": "synthetic",
        "config": {"workload": f"{args.model} {S}x{S} bs{B}/GPU inference: forward + decode + batched NMS",
                   "nms": NMS_KW, "weights": "seeded random (yolov6_b200/synth.py)", "parallelism": f"dp{world} image-sharded, no collective",
                   "l2": f"inputs ({B * 3 * S * S * 4 / 1e6:.0f} MB fp32 per batch, two alternating buffers) exceed the 126 MB L2"
                         if B * 3 * S * S * 4 > 126e6 else "two alternating input buffers; activations of one step exceed the 126 MB L2",
                   "launch": ("one CUDA graph per batch (pipeline.DetectStream): the graph of step i holds the network of batch i and, as a "
                              "parallel branch, the NMS of batch i-1 (head outputs double-buffered; every step runs one network and one NMS, "
                              "detections lag one step)") if use_graph else "eager ctypes launches",
                   "e2e_pipeline": "same graphs; the pinned-host -> device copy of batch i+1 runs on a copy stream under the kernels of batch i; "
                                   "the detections of batch i-1 are copied to pinned host memory inside the NMS branch of step i"},
        "e2e": main_r["e2e"],
        "gpu_launches": main_r["launches_per_step"] * args.steps,
        "roofline": {"bound": "tensor", "kernel": "yv6::conv_igemm_kernel", "achieved": achieved_tf, "peak": peak_tf,
                     "unit": "TFLOP/s", "frac": achieved_tf / peak_tf, "traffic": traffic,
                     "traffic_note": "bytes per conv_igemm launch, ncu dram__bytes_read+write averaged over the step's launches "
                                     f"(profiles/); algorithmic activation bytes per launch = {conv['bytes_per_launch']:.3e}",
                     "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback 1.4 PFLOP/s (B200_PROFILING.md)",
                     "frac_of_burst_peak": achieved_tf / float(peaks.get("bf16_tflops", 1661.3)),
                     "launches_per_step": conv["launches"], "conv_ms_per_step": conv["ms"], "algorithmic_gflop_per_step": conv["flop"] / 1e9,
                     "model_gflop_per_img": GFLOP_PER_IMG.get(args.model)},
        "clocks": sampler.summary(),
    }
    if modes:
        line["modes"] = modes
    if check:
        line["precision_check"] = check
    if extra:
        line["configs"] = extra
    if not args.no_cpu_baseline and world == 1:
        from oracle import model as om        # CPU-baseline leg: the checker, timed on the host cores
        from yolov6_b200.model import build_model
        from yolov6_b200.synth import randomize_
        sd = {k: v.detach().cpu() for k, v in randomize_(build_model(args.model, 80, torch.device("cpu")), seed=0).state_dict().items()}
        xs = torch.rand(args.ref_batch, 3, S, S, generator=torch.Generator().manual_seed(0))
        cores = pick_threads(lambda: cpu_reference_step(sd, om.CONFIGS[args.model], xs[:1], NMS_KW))
        t0 = time.perf_counter()
        for _ in range(args.steps_ref):
            cpu_reference_step(sd, om.CONFIGS[args.model], xs, NMS_KW)
        dt = (time.perf_counter() - t0) / args.steps_ref
        line["cpu_baseline"] = {"value": args.ref_batch / dt, "unit": "images/s", "cores": cores, "kind": "port",
                                "sample": f"{args.steps_ref} steps x batch {args.ref_batch} of the same workload (fp32 oracle: forward + NMS)"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
