#!/usr/bin/env python
"""bench.py -- CU-Net training-step throughput on B200 (images/sec), with roofline and CPU baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config cunet8|cunet2|cunet16|cunet8bin] [--scaling weak|strong] [--impl reference]
                    [--dump-outputs DIR]

One JSON line on stdout (rank 0).  A "step" is one full training step of the reference's train() loop
(cu-net.py:147-206) on one batch of synthetic input: forward, multi-loss MSE (+ fused landmark decode), backward,
[gradient allreduce], RMSprop.  `value` times it with the batch already resident in HBM; `e2e` times the same
step through the public Trainer API with pinned HOST buffers (H2D of image+heatmap and D2H of the loss inside the
timed region).  `--impl reference` times the reference's own algorithm on the host CPU cores (the oracle port of
models/cu_net.py) for the same config and metric.  `--dump-outputs DIR` writes what the last timed step computed as
DIR/<name>.npy (see step_outputs); the inputs and initial weights are seeded, so two builds can be compared output
for output: every timed step starts from the seeded model state (see the resident-input steps in main), so two runs
give bit-identical heads and landmarks, and loss, gradients and updated weights that differ only by the rounding of
the floating-point atomics that sum the gradients (RMSprop's first update, g / (sqrt(0.01 g^2) + eps), magnifies that
rounding on gradients near eps: on a B200 the weights of two runs differed by at most 3e-5 of their largest value).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CONFIGS = {
    # BASELINE.json configs[2] / [1] / [4]; batch = per-GPU batch (weak scaling, stated in the JSON line)
    "cunet8": dict(layer_num=8, order=1, loss_num=8, class_num=68, batch=24, dtype="bf16"),
    "cunet2": dict(layer_num=2, order=1, loss_num=2, class_num=68, batch=24, dtype="fp32"),
    "cunet16": dict(layer_num=16, order=1, loss_num=16, class_num=16, batch=16, dtype="bf16"),
    # BASELINE.json configs[3]: binary weights through the BinOp protocol of cu-net-prev-version-bin.py:163-191
    # (16 MPII joints, :48): binarize -> forward/backward -> restore -> fix gradients -> RMSprop, all inside the step
    "cunet8bin": dict(layer_num=8, order=1, loss_num=8, class_num=16, batch=24, dtype="bf16", quant="bin"),
}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        threading.Thread.__init__(self, daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([x.strip() for x in out.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=mx or None, reasons=sorted(reasons),
                    samples=len(sm))


def _cpu_step_fn(cfg, batch):
    import torch
    from oracle import cunet_oracle, synthetic
    state = cunet_oracle.init_state(cfg["class_num"], cfg["layer_num"], cfg["order"], seed=0)
    net = cunet_oracle.OracleCUNet(state, cfg["class_num"], cfg["layer_num"], cfg["order"], cfg["loss_num"])
    img, hm = synthetic.make_inputs(batch, cfg["class_num"], seed=0)
    params = net.parameters()
    sq = [torch.zeros_like(p) for p in params]

    def step():
        net.zero_grad()
        loss = cunet_oracle.multi_loss_mse(net(img), hm)
        loss.backward()
        grads = [p.grad if p.grad is not None else torch.zeros_like(p) for p in params]
        cunet_oracle.rmsprop_step(params, grads, sq, 2.5e-4)
    return step


def cpu_reference(cfg, sample_batch, iters, warmup=1):
    """The reference's algorithm (oracle port of models/cu_net.py + cu-net.py:175-183 loss/backward/RMSprop) on
    the host cores.  The thread count is the fastest of {16, 32, 64, all cores} (ascending, stops at the first slowdown) on a one-image CU-Net-2 probe
    step (oneDNN/ATen oversubscribe badly on 100+ core hosts for these small convolutions).
    Returns (images_per_sec, threads_used)."""
    import torch
    cores = os.cpu_count() or 1
    probe_cfg = dict(cfg, layer_num=2, loss_num=2)
    best, best_t = None, cores
    for t in sorted({min(cores, 16), min(cores, 32), min(cores, 64), cores}):   # ascending; stop once it gets slower
        torch.set_num_threads(t)
        fn = _cpu_step_fn(probe_cfg, 1)
        fn()
        t0 = time.perf_counter()
        fn()
        dt = time.perf_counter() - t0
        if best is None or dt < best:
            best, best_t = dt, t
        else:
            break
    torch.set_num_threads(best_t)
    step = _cpu_step_fn(cfg, sample_batch)
    times = []
    for it in range(warmup + iters):
        t0 = time.perf_counter()
        step()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    times.sort()
    return sample_batch / times[len(times) // 2], best_t


def _dump_state(state):
    """Initial weights -> a temp file for the oracle child process (the checker runs outside this process so that its
    CPU thread settings and memory stay out of the measured one)."""
    import tempfile
    import torch
    fd, path = tempfile.mkstemp(suffix=".pt", prefix="cunet_state0_")
    os.close(fd)
    torch.save(state, path)
    return path


def oracle_loss_main(cfg, batch):
    """Child mode: multi-loss MSE of the CPU oracle (train-mode BN, forward only) on the bench's rank-0 batch with the
    weights the B200 arm started from.  Test infrastructure used as the checker only."""
    import torch
    from oracle import cunet_oracle, synthetic
    path = os.environ["CUNET_STATE0"]
    state = torch.load(path, weights_only=False)
    os.unlink(path)
    torch.set_num_threads(min(os.cpu_count() or 1, 32))
    net = cunet_oracle.OracleCUNet(state, cfg["class_num"], cfg["layer_num"], cfg["order"], cfg["loss_num"])
    img, hm = synthetic.make_inputs(batch, cfg["class_num"], seed=0)
    with torch.no_grad():
        loss = cunet_oracle.multi_loss_mse(net(img), hm)
    _emit(dict(loss_oracle=float(loss)))
    return 0


PROBE_STEPS = 5         # eager steps whose probe-kernel times give the roofline median (not the timed steps)
DUMP_CAP = 4 << 20      # elements per dumped array: the three large ones stay under 48 MB of float32 together


def _sample(flat):
    """A 1-D device tensor whole, or DUMP_CAP of its elements at fixed seeded positions (the same for equal sizes)."""
    import torch
    if flat.numel() <= DUMP_CAP:
        return flat
    idx = torch.randint(flat.numel(), (DUMP_CAP,), generator=torch.Generator().manual_seed(0)).sort().values
    return flat[idx.to(flat.device)]


def step_outputs(net, eng):
    """What the last train_step() handed its caller, as host arrays: the loss it returned (float64), the decoded
    landmarks and the heads of that step, the model's state_dict after the update (flattened in state_dict order) and
    the gradients the update used (flattened in parameters() order); the last three are sampled by _sample."""
    import torch
    heads = torch.stack([h.float() for h in eng.head_outputs()]).flatten()
    state = torch.cat([v.detach().float().flatten() for v in net.state_dict().values()])
    grads = torch.cat([p.grad.float().flatten() for p in net.parameters()])
    out = dict(loss=eng.loss_value().view(1), preds=eng.preds.float(), heads=_sample(heads), state=_sample(state),
               grads=_sample(grads))
    return {k: v.cpu().numpy() for k, v in out.items()}


def op_bytes(eng, op, kind):
    """Algorithmic HBM bytes of one launch (DESIGN.md 'Kernels'): every operand read once, every result written once."""
    esz = 2 if eng.tdtype.itemsize == 2 else 4
    N = eng.N
    src = sum(N * t.res * t.res * t.C * esz for t, _ in op.srcs)
    out_rows = N * (op.res // 2 if op.pool else op.res) ** 2
    out = out_rows * op.out.C * (4 if op.out.fp32 else esz)
    if kind == "fwd":
        return src + out
    dy = out if op.out.fp32 else 2 * out          # batch-norm form reads G and T of the output
    if op.pool:
        dy += out_rows * op.out.C                 # argmax bytes
    if kind == "wgrad":
        return src + dy
    sched = {o.name: f for o, f in eng.plan.backward_schedule()}
    gacc = 0
    for (t, _), (acc, _) in zip(op.srcs, sched[op.name]):
        b = N * t.res * t.res * t.C * esz
        gacc += 2 * b if acc else b
    return src + dy + gacc


_OUT_FD = None


def _emit(obj):
    """The record line, on the process's original stdout."""
    data = (json.dumps(obj) + "\n").encode()
    if _OUT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_OUT_FD, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="cunet8", choices=sorted(CONFIGS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the config's)")
    ap.add_argument("--dtype", default="", choices=["", "bf16", "fp32"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: the config's batch per GPU (default); strong: the config's batch is the GLOBAL batch, "
                         "split over the GPUs like the reference's DataParallel does with --bs (cu-net.py:59,84)")
    ap.add_argument("--no-graph", action="store_true", help="launch eagerly instead of replaying CUDA graphs")
    ap.add_argument("--cpu-sample", type=int, default=8, help="images in the CPU-baseline sample step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-loss-check", action="store_true", help="skip the CPU-oracle loss of the first step")
    ap.add_argument("--oracle-loss", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the outputs of the last timed step to DIR/<name>.npy (rank 0, B200 arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    # stdout carries exactly ONE line, the JSON record: anything a library prints there (NCCL writes its version banner
    # to stdout at communicator creation) is sent to stderr instead
    global _OUT_FD
    sys.stdout.flush()
    _OUT_FD = os.dup(1)
    os.dup2(2, 1)
    cfg = dict(CONFIGS[args.config])
    if args.batch:
        cfg["batch"] = args.batch
    if args.dtype:
        cfg["dtype"] = args.dtype
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if max(args.warmup, 0) < 3:
        args.warmup = 3
    if args.scaling == "strong":
        if cfg["batch"] % world:
            raise SystemExit("--scaling strong needs the global batch %d to be divisible by %d GPUs" % (cfg["batch"], world))
        cfg["batch"] //= world
    workload = "CU-Net-%d order %d loss %d, %d classes, 256x256 -> 64x64 heatmaps, per-GPU batch %d, %s, train step%s" % (
        cfg["layer_num"], cfg["order"], cfg["loss_num"], cfg["class_num"], cfg["batch"], cfg["dtype"],
        ", binary weights (BinOp protocol)" if cfg.get("quant") == "bin" else "")

    if args.oracle_loss:
        return oracle_loss_main(cfg, cfg["batch"])

    # ------------------------------------------------------------------ reference arm (CPU, rank 0 only)
    if args.impl == "reference":
        if rank != 0:
            return 0
        if cfg.get("quant"):
            _emit(dict(impl="reference", unavailable="the CPU reference arm times the full-precision step only"))
            return 0
        ips, cores = cpu_reference(cfg, args.cpu_sample, args.steps, warmup=args.warmup)
        ref_workload = ("CU-Net-%d order %d loss %d, %d classes, 256x256 -> 64x64 heatmaps, train step on the host CPU: "
                        "%d-image sample batch, fp32 (torch CPU), %d threads -- bounded sample of the B200 arm's workload "
                        "(batch %d per GPU, %s)" % (cfg["layer_num"], cfg["order"], cfg["loss_num"], cfg["class_num"],
                                                    args.cpu_sample, cores, cfg["batch"], cfg["dtype"]))
        line = dict(impl="reference", metric="images_per_sec", value=ips, unit="images/s", n_gpus=args.gpus,
                    steps=args.steps, warmup=args.warmup, ms_per_step=1000.0 * args.cpu_sample / ips,
                    higher_is_better=True, scaling=args.scaling, vs_baseline=None, dtype="f32", data="synthetic",
                    config=dict(workload=ref_workload, sample_batch=args.cpu_sample, b200_arm_workload=workload),
                    cpu_baseline=dict(value=ips, unit="images/s", cores=cores, kind="port",
                                      sample="%d-image training step (fwd+MSE+bwd+RMSprop) of the same model, median of %d"
                                             % (args.cpu_sample, args.steps)),
                    e2e=dict(value=ips, unit="images/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
        _emit(line)
        return 0

    # ------------------------------------------------------------------ B200 arm
    import torch
    import __graft_entry__ as ge
    if not os.path.exists(ge.LIB):
        ge.build()
    from cunet_b200.models.cu_net import create_cu_net
    from cunet_b200.engine import Trainer
    from cunet_b200.utils import synthetic

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pg = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD
    torch.manual_seed(0)
    net = create_cu_net(4, 32, 128, cfg["class_num"], cfg["layer_num"], cfg["order"], cfg["loss_num"],
                        dtype=cfg["dtype"])
    B = cfg["batch"]
    quant = None
    if cfg.get("quant") == "bin":
        from cunet_b200.utils.quantize import BinOp
        net.engine(B, dev)                 # the quantizer needs the parameters in device storage
        quant = BinOp(net)
    tr = Trainer(net, B, lr=2.5e-4, device=dev, process_group=pg, world_size=world, use_graph=not args.no_graph,
                 quant=quant)
    if world > 1:
        import torch.distributed as dist
        dist.broadcast(tr.eng.params, 0)
    img, hm = synthetic.make_inputs(B, cfg["class_num"], seed=rank)
    img_h, hm_h = img.pin_memory(), hm.pin_memory()
    tr.load_batch(img_h, hm_h)
    torch.cuda.synchronize()
    # correctness guard (outside every timed region): the loss of the very first step, from the initial weights, is
    # reported next to the CPU oracle's loss on the same images and weights -- a wrong step can not score silently
    state0 = {k: v.detach().cpu().clone() for k, v in net.state_dict().items()} if rank == 0 else None

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, reset=None):
        """Device time of ``steps`` calls of fn.  With ``reset``, it is enqueued before every call and each call is
        bracketed by its own events, so the reset is not timed."""
        if reset is None:
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))]
        else:
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        if reset is None:
            evs[0][0].record()
            for _ in range(steps):
                fn()
            evs[0][1].record()
        else:
            for ev0, ev1 in evs:
                reset()
                ev0.record()
                fn()
                ev1.record()
        barrier()
        ms = sum(ev0.elapsed_time(ev1) for ev0, ev1 in evs)
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms

    # resident-input steps.  Every timed step is the same training step: it starts from the seeded initial model state
    # (Engine.save_state: weights, RMSprop state, BatchNorm running statistics and counters), copied back before it
    # and outside its timing.  The gradient sums use floating-point atomics, so a step from a given state is reproducible only to
    # rounding; chained steps would carry that rounding through RMSprop and bf16 activations into outputs that differ
    # from run to run.  From a fixed state, what the timed steps compute depends on the arguments only.
    state_init = tr.eng.save_state()
    loss_first = float(tr.train_step())
    for _ in range(args.warmup - 1):
        tr.train_step()
    sampler = ClockSampler(local)
    sampler.start()
    ms = timed(lambda: tr.train_step(), args.steps, reset=lambda: tr.eng.restore_state(state_init))
    sampler.stop_flag = True
    ms_per_step = ms / args.steps
    value = world * B / (ms_per_step / 1000.0)
    if args.dump_outputs and rank == 0:
        # before the steps below move the weights on
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in step_outputs(net, tr.eng).items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)

    # end-to-end steps: pinned host -> device copies and a device -> host read of the loss every step
    loss_host = torch.zeros(1, dtype=torch.float64).pin_memory()

    def e2e_step():
        # every step's inputs cross PCIe from pinned host memory: the copy of the NEXT step's batch is issued on the
        # copy stream right after this step's launch (Trainer.prefetch), so it overlaps the step's kernels; the
        # blocking loss read-back ends the step
        loss = tr.train_step()                     # consumes the batch staged by the previous prefetch
        tr.prefetch(img_h, hm_h)
        loss_host.copy_(loss.view(1), non_blocking=False)
    tr.prefetch(img_h, hm_h)
    for _ in range(2):
        e2e_step()
    ms_e2e = timed(e2e_step, args.steps) / args.steps
    e2e = world * B / (ms_e2e / 1000.0)
    tr._staged = None

    # ---- the reference's multi-GPU semantics (cu-net.py:59,84: --bs is the GLOBAL batch, scattered over the GPUs):
    # same model, same timing loop, the config's batch split over the ranks.  At N=1 it is the weak-scaling number.
    strong = None
    if args.scaling == "weak":
        gb = CONFIGS[args.config]["batch"] if not args.batch else args.batch
        if world == 1:
            strong = dict(global_batch=gb, per_gpu_batch=gb, value=value, unit="images/s", ms_per_step=ms_per_step)
        elif gb % world == 0:
            Bs = gb // world
            tr_s = Trainer(net, Bs, lr=2.5e-4, device=dev, process_group=pg, world_size=world,
                           use_graph=not args.no_graph, quant=quant)
            imgs, hms = synthetic.make_inputs(Bs, cfg["class_num"], seed=100 + rank)
            tr_s.load_batch(imgs.to(dev), hms.to(dev))
            for _ in range(args.warmup):
                tr_s.train_step()
            ms_s = timed(lambda: tr_s.train_step(), args.steps) / args.steps
            strong = dict(global_batch=gb, per_gpu_batch=Bs, value=gb / (ms_s / 1000.0), unit="images/s", ms_per_step=ms_s,
                          launches_per_step=tr_s.eng.launches_per_train_step(),
                          limit="launch-latency floor of the ~%d dependent launches per step (the kernels on <= 16x16 maps "
                                "are latency-bound whatever the batch), then the exposed ncclAllReduce of the %.1f MB fp32 "
                                "gradient bucket" % (tr_s.eng.launches_per_train_step(), 4e-6 * tr_s.eng.n_params))
            del tr_s

    if rank != 0:
        return 0

    # ---- the drop-in module API, timed literally as cu-net.py:171-183 drives it (N=1): net(img) -> multi-loss MSE in
    # torch -> loss.backward() -> torch.optim.RMSprop.step(), host buffers, H2D inside the timed region
    module_api = None
    if world == 1 and not cfg.get("quant"):
        opt_t = torch.optim.RMSprop(net.parameters(), lr=2.5e-4, alpha=0.99, eps=1e-8, momentum=0, weight_decay=0)
        net.train()

        def module_step():
            x, t = img_h.to(dev, non_blocking=True), hm_h.to(dev, non_blocking=True)
            out = net(x)
            loss = 0
            for o in out:
                d = (o - t) ** 2
                loss = loss + d.sum() / d.numel()
            opt_t.zero_grad()
            loss.backward()
            opt_t.step()
            loss_host.copy_(loss.detach().double().view(1), non_blocking=False)
        for _ in range(2):
            module_step()
        ms_m = timed(module_step, args.steps) / args.steps
        module_api = dict(value=B / (ms_m / 1000.0), unit="images/s", ms_per_step=ms_m,
                          path="net(img); loss.backward(); torch.optim.RMSprop.step() (cu-net.py:171-183), eager launches")
        net.bind_grads()

    # ---- roofline of the dominant kernel, measured live (eager launches bracketed by CUDA events)
    eng = tr.eng
    plan = eng.plan
    pk = peaks()
    probe_op = max(plan.ops, key=lambda o: (o.cin * o.cout * o.res * o.res, o.index))
    # large 1x1 ops run their backward as ONE fused dgrad+wgrad launch (csrc/conv_bwd1x1.cu): it is probed as "bwd"
    # with the bytes of the backward-data contract (G/T of the output, every source, every source gradient) -- the
    # filter gradient adds no HBM traffic of its own
    fused_bwd = eng.is_fused_1x1(probe_op)
    kinds = ["fwd", "bwd"] if fused_bwd else ["fwd", "dgrad", "wgrad"]
    eng.probes = {}
    evs = {}
    for k in kinds:
        prm = eng.call_index[(probe_op.name, "dgrad" if k == "bwd" else k)]
        evs[k] = [torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)]
        eng.probes[id(prm)] = evs[k]
    acc = {k: [] for k in kinds}
    for _ in range(PROBE_STEPS):
        tr._fwd_bwd()
        tr._opt()
        torch.cuda.synchronize()
        for k in kinds:
            acc[k].append(evs[k][0].elapsed_time(evs[k][1]))
    eng.probes = None
    roofs = {}
    for k in kinds:
        t_ms = sorted(acc[k])[len(acc[k]) // 2]
        by = op_bytes(eng, probe_op, "dgrad" if k == "bwd" else k)
        flops = 2.0 * eng.N * probe_op.res ** 2 * probe_op.cin * probe_op.cout * probe_op.taps * (2 if k == "bwd" else 1)
        roofs[k] = dict(kernel="conv_bwd1x1 (fused dgrad+wgrad)" if k == "bwd" else "conv_%s" % k, op=probe_op.name, us=1000.0 * t_ms, bytes=by,
                        achieved=by / (t_ms * 1e-3) / 1e9, peak=pk["hbm"], unit="GB/s",
                        frac=by / (t_ms * 1e-3) / 1e9 / pk["hbm"], tflops=flops / (t_ms * 1e-3) / 1e12)
    dom = roofs["bwd" if fused_bwd else "dgrad"]
    # DRAM traffic of the dominant kernel on this op: dram__bytes_read.sum + dram__bytes_write.sum of the committed
    # `ncu --set full` capture (profiles/traffic.json names the capture); not measurable from inside this process
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath) and cfg["dtype"] == "bf16":
        tj = json.load(open(tpath)).get("conv_bwd1x1" if fused_bwd else "conv_dgrad")
        if tj:
            # the capture is only quoted while the kernel source it was taken from is unchanged (sha1 of the .cu file)
            import hashlib
            src_file = os.path.join(ROOT, "cu-net_b200", "csrc", tj.get("kernel_file", "conv_dgrad_v2.cu"))
            sha = hashlib.sha1(open(src_file, "rb").read()).hexdigest() if os.path.exists(src_file) else None
            if tj.get("kernel_sha1") in (None, sha):
                traffic, traffic_src = tj["bytes"], tj["source"]
            else:
                traffic_src = "stale: %s changed since %s was captured" % (tj.get("kernel_file"), tj["source"])
    loss_oracle = None
    if not args.no_loss_check and not cfg.get("quant"):
        try:
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--oracle-loss", "--config", args.config,
                                  "--batch", str(B)] + (["--dtype", args.dtype] if args.dtype else []),
                                 input=None, capture_output=True, text=True, timeout=600,
                                 env=dict(os.environ, CUNET_STATE0=_dump_state(state0))).stdout
            loss_oracle = json.loads(out.strip().splitlines()[-1])["loss_oracle"]
        except Exception as exc:  # noqa: BLE001
            loss_oracle = "unavailable: %s" % type(exc).__name__
    train_gflop_img = (3.0 * plan.conv_flops_per_image() - 2.0 * 147 * 128 * 128 * 128) / 1e9
    tflops = value * train_gflop_img / 1e3
    line = dict(
        metric="images_per_sec", value=value, unit="images/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
        ms_per_step=ms_per_step, higher_is_better=True, scaling=args.scaling, vs_baseline=None,
        dtype="bf16" if cfg["dtype"] == "bf16" else "f32(3xtf32)", data="synthetic",
        config=dict(workload=workload, global_batch=world * B, parallelism="dp%d" % world,
                    l2="working set (~%.1f GB of activations per step) far exceeds the 126 MB L2; no flush needed"
                       % (sum(a.numel() * a.element_size() for a in eng.act.values()) / 1e9),
                    launch="cuda-graph replay" if not args.no_graph else "eager",
                    pdl="programmatic dependent launch between the conv kernels: %s"
                        % ("off" if os.environ.get("CUNET_PDL", "1") == "0" else "on")),
        e2e=dict(value=e2e, unit="images/s", ms_per_step=ms_e2e,
                 h2d_bytes_per_step=int(img_h.numel() * 4 + hm_h.numel() * 4), d2h_bytes_per_step=8,
                 path="Trainer.train_step() + Trainer.prefetch(img_host, heatmap_host): the next batch's H2D runs on a "
                      "copy stream under the current step, the loss read-back is blocking"),
        gpu_launches=int(eng.launches_per_train_step() * args.steps),
        loss_first_step=loss_first, loss_oracle=loss_oracle,
        loss_rel_err=(abs(loss_first - loss_oracle) / abs(loss_oracle)) if isinstance(loss_oracle, float) else None,
        strong_scaling=strong, e2e_module_api=module_api,
        roofline=dict(bound="hbm", achieved=dom["achieved"], peak=dom["peak"], unit="GB/s", frac=dom["frac"],
                      traffic=traffic, traffic_source=traffic_src, kernel=dom["kernel"], op=dom["op"], us_per_launch=dom["us"],
                      algorithmic_bytes=dom["bytes"], peak_source=pk["source"],
                      note="probe launches timed eagerly with CUDA events right after the timed region, median of "
                           "%d steps" % PROBE_STEPS),
        roofline_all=roofs,
        conv_flops=dict(train_gflop_per_image=train_gflop_img, achieved_tflops=tflops,
                        frac_of_bf16_sustained=tflops / pk["tf_sust"], peak_tflops=pk["tf_sust"]),
        clocks=sampler.summary(),
    )
    if not args.no_cpu_baseline and world == 1 and not cfg.get("quant"):
        # the reference arm in a child process: its thread settings stay out of this process and a pathological host
        # (oversubscribed cores) can only cost a bounded amount of time
        try:
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--config", args.config,
                                  "--cpu-sample", str(args.cpu_sample), "--steps", "3"] +
                                 (["--dtype", args.dtype] if args.dtype else []) +
                                 (["--batch", str(args.batch)] if args.batch else []),
                                 capture_output=True, text=True, timeout=240).stdout
            ref = json.loads(out.strip().splitlines()[-1])
            line["cpu_baseline"] = ref["cpu_baseline"]
        except Exception as exc:  # noqa: BLE001 -- report, never fail the GPU line because of the CPU baseline
            line["cpu_baseline"] = dict(value=None, unit="images/s", cores=None, kind="port",
                                        sample="unavailable: %s" % type(exc).__name__)
    _emit(line)
    return 0


if __name__ == "__main__":
    sys.exit(main())
