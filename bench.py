"""bench.py -- MoCo pretrain images/sec on N B200s (BASELINE.json metric), plus the kernel roofline.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # CPU arm: the UNMODIFIED reference train_moco (oracle/_ref) on host cores
    python bench.py --gpus 1 --steps 20 --warmup 5 --dump-outputs DIR    # + what the last timed step computed, as .npy

A step = one MoCo iteration (train.py:244-283): query encoder fwd, ShuffleBN permute, key encoder fwd,
un-shuffle, q.Queue^T + InfoNCE + dq, enqueue, backward, SGD step, EMA update -- ResNet-50, feat_dim 128,
batch 256/GPU, bf16 autocast, synthetic 224x224 images, random-init weights.
Workloads: N=1 -> BASELINE configs[1] (K=16384); N>1 -> configs[2] (K=65536, ShuffleBN over NVLink P2P) plus,
in the same JSON line, a multi-GPU parity block (run BEFORE the timed region; the run fails if it does), the
ShuffleBN permute timed alone and BASELINE configs[3] (K=131072 sharded over the ranks).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "MoCo pretrain images/sec (device-timed, max over ranks)"      # BASELINE.json:metric, same string in both arms


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="images per GPU")
    ap.add_argument("--arch", default="resnet50")
    ap.add_argument("--feat-dim", type=int, default=128)
    ap.add_argument("--nce-k", type=int, default=0, help="queue length (0: 16384 at 1 GPU, 65536 otherwise)")
    ap.add_argument("--nce-t", type=float, default=0.07)
    ap.add_argument("--memory-format", default="channels_last", choices=["channels_last", "contiguous"],
                    help="encoder activation layout (host PyTorch side)")
    ap.add_argument("--no-stress", action="store_true", help="skip the c5 roofline-stress microbench")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-bn-ab", action="store_true", help="N=1: skip the 5 steps timed with ATen's BatchNorm kernels")
    ap.add_argument("--cpu-sample-batch", type=int, default=16,
                    help="images per step of the CPU arm (a bounded sample of the 256-image batch)")
    ap.add_argument("--no-c1", action="store_true", help="reference arm: skip BASELINE configs[0] (R18, K=1024, N=32)")
    ap.add_argument("--no-sharded", action="store_true", help="N>1: skip the configs[3] sharded-queue block")
    ap.add_argument("--ddp-bucket-mb", type=int, default=25)
    ap.add_argument("--ddp-bf16", action="store_true", help="N>1: all-reduce gradients as bf16 (DDP compress hook)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="native arm: write what the last timed step computed to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


# dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed `ncu --set full`
# captures of this round (profiles/r2_*_ncu_metrics.csv; tools/gpu_lab.py op_c2 / op_c3 / op_c5 under ncu)
NCU_TRAFFIC_BYTES = {
    ("onepass", 256, 128, 16384): 4332544,                       # profiles/r2_head128_c2_ncu_metrics.csv
    ("onepass", 256, 128, 65536): 16915200,                      # profiles/r2_head128_c3_ncu_metrics.csv (0 B written: L2)
    ("onepass", 512, 256, 262144): 134541312 + 3316992,          # profiles/r2_head256_c5_ncu_metrics.csv
}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"hbm_gbs": d["hbm_gbs"], "tf_burst": d["bf16_tflops"], "tf_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU during the timed region (NVML)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, False, [], set(), None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksEventReasonHwSlowdown: "hw_slowdown",
                     nv.nvmlClocksEventReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     nv.nvmlClocksEventReasonSwThermalSlowdown: "sw_thermal_slowdown",
                     nv.nvmlClocksEventReasonSwPowerCap: "sw_power_cap"}
            while not self.stop_flag:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.1)
        except Exception as exc:       # NVML missing: report that instead of inventing clocks
            self.reasons.add(f"nvml_unavailable:{type(exc).__name__}")

    def result(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def default_k(world):
    return 16384 if world == 1 else 65536


def workload_name(args, K, world):
    return (f"{args.arch} feat_dim={args.feat_dim} K={K} batch={args.batch}/GPU bf16 "
            + ("(BASELINE configs[1])" if world == 1 else "(BASELINE configs[2], ShuffleBN P2P permute)"))


def config_block(args, K, world):
    """`config` of the JSON line -- identical in the native and the reference arm (same workload by construction)."""
    return {"workload": workload_name(args, K, world), "global_batch": args.batch * world,
            "parallelism": f"dp{world}", "temperature": args.nce_t,
            "l2": "native arm: inputs (308 MB/step) exceed L2, no explicit flush"}


def reference_job(arch, feat_dim, K, T, batch, steps, warmup, timeout=900):
    """The unmodified reference train_moco (oracle/ref_runner.py on oracle/_ref) in its OWN process: the shims
    (identity .cuda(), gloo group) must not leak into this one, and its thread pool starts clean."""
    env = dict(os.environ)
    for k in ("OMP_NUM_THREADS", "MKL_NUM_THREADS", "RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT",
              "GROUP_RANK", "LOCAL_WORLD_SIZE", "ROLE_RANK", "TORCHELASTIC_RUN_ID"):
        env.pop(k, None)                       # torchrun exports OMP_NUM_THREADS=1: the CPU arm uses every core
    env["CUDA_VISIBLE_DEVICES"] = ""
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "ref_runner.py"), "--arch", arch, "--feat-dim", str(feat_dim),
           "--nce-k", str(K), "--nce-t", str(T), "--batch", str(batch), "--steps", str(steps), "--warmup", str(warmup)]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env, cwd=ROOT)
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    if p.returncode != 0 or not lines:
        raise RuntimeError(f"reference CPU arm failed (rc={p.returncode}): {p.stderr[-2000:]}")
    return json.loads(lines[-1])


def cpu_baseline_block(r, extra=None):
    b = {"value": r["images_per_s"], "unit": "images/s", "cores": r["threads"], "kind": "reference",
         "sample": f"{r['warmup']} warm-up + {r['steps']} timed steps x {r['batch']} images of the UNMODIFIED reference "
                   f"train.train_moco (train.py:231-293, staged in oracle/_ref) -- {r['arch']}, feat_dim={r['feat_dim']}, "
                   f"K={r['K']}, fp32, gloo world 1, {r['threads']} host threads",
         "ms_per_step": r["ms_per_step"], "loss": r["loss"]}
    if extra:
        b.update(extra)
    return b


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    K = args.nce_k or default_k(world)
    steps, warmup = max(3, args.steps), max(3, args.warmup)
    r = reference_job(args.arch, args.feat_dim, K, args.nce_t, args.cpu_sample_batch, steps, warmup)
    extra = {}
    if not args.no_c1:
        # BASELINE configs[0] / SURVEY 8(d): the reference's own CPU-runnable case, full size (no sampling)
        c1 = reference_job("resnet18", 128, 1024, args.nce_t, 32, 10, 3)
        extra["c1"] = {"value": c1["images_per_s"], "unit": "images/s", "ms_per_step": c1["ms_per_step"],
                       "cores": c1["threads"], "workload": "BASELINE configs[0]: ResNet-18 feat_dim=128 K=1024 batch=32 "
                       "world 1, fp32, reference train_moco, 3 warm-up + 10 timed steps"}
    line = {
        "impl": "reference", "metric": METRIC, "value": r["images_per_s"], "unit": "images/s",
        "n_gpus": args.gpus, "steps": r["steps"], "warmup": r["warmup"], "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_block(args, K, world),
        "cpu_baseline": cpu_baseline_block(r, extra),
        "e2e": {"value": r["images_per_s"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def stress_roofline(peaks, dev):
    """BASELINE configs[4]: N=512, C=256, K=262144 -- the tensor-bound shape, hot-path kernels alone (queue 134 MB > L2).
    Default path = ONE sweep over the queue producing loss statistics AND dq (4NCK FLOP); the two-pass alternative
    (statistics kernel, then dq kernel that recomputes S: 6NCK FLOP executed, 4NCK credited) is timed beside it."""
    import torch
    import torch.nn.functional as F
    from moco_b200 import _lib
    lib = _lib.load()
    N, C, K, T = 512, 256, 262144, 0.07
    g = torch.Generator(device=dev).manual_seed(3)
    q = F.normalize(torch.randn(N, C, device=dev, generator=g), dim=1).bfloat16()
    k = F.normalize(torch.randn(N, C, device=dev, generator=g), dim=1).bfloat16()
    queue = F.normalize(torch.randn(K, C, device=dev, generator=g), dim=1).bfloat16()
    f32 = dict(dtype=torch.float32, device=dev)
    lse, lr, pr, lp, dq = torch.zeros(N, **f32), torch.zeros(N, **f32), torch.zeros(N, **f32), torch.zeros(2, **f32), torch.zeros(N, C, **f32)
    wsb = lib.moco_nce_workspace_bytes(N, C, K)
    ws = torch.zeros(wsb + 256, dtype=torch.uint8, device=dev)
    wp = ws.data_ptr() + (-ws.data_ptr()) % 256
    stream = torch.cuda.current_stream().cuda_stream
    iters = 20

    def timed_kernels(flags):
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(iters)]
        for e4 in ev:       # events must exist (be recorded once) before the library records into them; stop before
            for j in (1, 0, 3, 2):   # start, so a hook that never fires reads as a NEGATIVE interval
                e4[j].record()

        def call(i):
            if i >= 0:
                lib.moco_prof_set_events(1, ev[i][0].cuda_event, ev[i][1].cuda_event)
                lib.moco_prof_set_events(2, ev[i][2].cuda_event, ev[i][3].cuda_event)
            rc = lib.moco_nce_fwd(q.data_ptr(), k.data_ptr(), 1, queue.data_ptr(), N, C, K, 1.0 / T, None, lse.data_ptr(),
                                  lr.data_ptr(), pr.data_ptr(), lp.data_ptr(), dq.data_ptr(), wp, wsb, flags, stream)
            _lib.check(rc, "moco_nce_fwd")
        for _ in range(3):
            call(-1)
        for i in range(iters):
            call(i)
        lib.moco_prof_set_events(1, None, None)
        lib.moco_prof_set_events(2, None, None)
        torch.cuda.synchronize()
        return (sum(e[0].elapsed_time(e[1]) for e in ev) * 1e3 / iters, sum(e[2].elapsed_time(e[3]) for e in ev) * 1e3 / iters)

    _, us_one = timed_kernels(_lib.NCE_AUTO)                      # one-pass kernel reports on the DQ hook
    win = ctypes.c_float()
    lib.moco_prof_sweep_window(wp, 148, ctypes.byref(win), stream)
    us_stats, us_dq = timed_kernels(_lib.NCE_TWO_PASS)
    flops = 2.0 * N * C * (K + 1)                                 # per direction (SURVEY.md 8d): fwd = bwd = 2NC(K+1)
    bytes_ = K * C * 2 + 3 * N * C * 2 + 12 * N
    a = 2 * flops / (us_one * 1e-6) / 1e12
    return {
        "workload": "BASELINE configs[4]: N=512 feat_dim=256 K=262144 (hot-path kernels alone, queue 134 MB > L2)",
        "kernel": "nce_head256_kernel<FUSED> (one sweep on tcgen05: S=q.Queue^T, P=2^(S/T-m), O+=P.Queue, row sums; q half in "
                  "TMEM / half in smem, three S buffers) -> loss statistics + dq partials; the tail kernel finishes both",
        "bound": "tensor", "achieved": a, "peak": peaks["tf_burst"], "unit": "TFLOP/s", "frac": a / peaks["tf_burst"],
        "us_per_launch": us_one, "device_window_us": float(win.value),
        "algorithmic_flops": 2 * flops, "hbm_GBps": bytes_ / (us_one * 1e-6) / 1e9,
        "traffic": NCU_TRAFFIC_BYTES.get(("onepass", N, C, K)),
        "two_pass": {"stats_kernel_us": us_stats, "stats_TFLOPs": flops / (us_stats * 1e-6) / 1e12,
                     "stats_frac": flops / (us_stats * 1e-6) / 1e12 / peaks["tf_burst"],
                     "dq_kernel_us": us_dq, "dq_TFLOPs_executed": 2 * flops / (us_dq * 1e-6) / 1e12,
                     "sum_us": us_stats + us_dq,
                     "note": "statistics pass + dq pass (recomputes S): 6NCK executed for the same 4NCK of algorithmic work"},
    }


def shufflebn_block(x2, epoch, rank, world, dev, nhwc):
    """ShuffleBN forward permute (util.py:69-79 replacement) timed ALONE on this step's key batch: the whole call
    (publish into the peer-mapped staging buffer + signal barrier + P2P pull) and the pull kernel by itself.
    CUDA events on the launching stream, max over ranks.  Collective."""
    import torch
    import torch.distributed as dist
    from moco_b200 import _lib
    from moco_b200.util import DistributedShufle, ShuffleContext
    lib = _lib.load()
    n = x2.shape[0]
    iters = 10

    def timed_us(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1) / iters], device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms) * 1e3

    # the rows the step moves between GPUs (MoCoStep): the key crops as plain bf16 NHWC rows
    fwd_us = timed_us(lambda: DistributedShufle.forward_shuffle(x2, epoch, cast_dtype=torch.bfloat16, channels_last=nhwc))
    # the pull alone, on pre-staged data (bf16 rows = what crosses NVLink in the step)
    ctx = ShuffleContext.get()
    row_bytes = x2[0].numel() * 2
    buf = ctx._staging("bench_fwd", n * row_bytes)
    buf.tensor((n * row_bytes // 2,), torch.bfloat16).normal_()
    ctx.barrier()
    fwd_inds, _ = DistributedShufle.get_shuffle_ids(n * world, epoch, dev)
    src = DistributedShufle.get_local_id(fwd_inds).contiguous()
    out = torch.empty(n * row_bytes // 2, dtype=torch.bfloat16, device=dev)
    # the pull kernel exactly as forward_shuffle launches it (moco_shuffle_gather_sync: cross-GPU event folded in)
    gather_us = timed_us(lambda: ctx._pull(buf.table, n, src, row_bytes, out.data_ptr(), synced=True))
    ctx.barrier()
    remote = int(((src // n) != rank).sum().item())
    rr = torch.tensor([float(remote)], device=dev)
    dist.all_reduce(rr, op=dist.ReduceOp.MIN)
    return {"fwd_us": fwd_us, "gather_us": gather_us, "remote_rows": remote, "rows": n, "row_bytes": row_bytes,
            "row_layout": "bf16 NHWC [224, 224, 3]" if nhwc else "bf16 NCHW",
            "gather_GBps": n * row_bytes / (gather_us * 1e-6) / 1e9,
            "nvlink_GBps": remote * row_bytes / (gather_us * 1e-6) / 1e9,
            "nvlink_frac_of_900": remote * row_bytes / (gather_us * 1e-6) / 1e9 / 900.0,
            "note": "fwd_us = publish (crop+cast+layout into the peer-mapped staging buffer) + signal barrier + pull; "
                    "gather_us = the pull kernel alone; nvlink_GBps counts only rows that live on another GPU "
                    "(this rank's count; slowest rank's time)"}


def sharded_block(args, model, model_ema, opt, x1, x2, epoch, rank, world, dev, nhwc, peaks, timed):
    """BASELINE configs[3]: K = 131072 ring sharded over the ranks (ShardedMemoryMoCo), same step loop.
    Reports images/s of the whole step, the head alone (all exchanges + kernels) and the exchange steps."""
    import torch
    import torch.distributed as dist
    import torch.nn.functional as F
    from moco_b200.NCE import ShardedMemoryMoCo
    from moco_b200.train_step import MoCoStep
    N, C, T, Ksh = args.batch, args.feat_dim, args.nce_t, 131072
    smod = ShardedMemoryMoCo(C, Ksh, T).to(dev)
    step = MoCoStep(model, model_ema, smod, opt, channels_last=nhwc)
    steps = max(3, min(args.steps, 10))
    for _ in range(3):
        step(x1, x2, epoch)

    def loop(k):
        for _ in range(k):
            step(x1, x2, epoch)
    ms = timed(loop, steps)
    # head alone: forward_loss (q exchange, shard sweep, statistics exchange, merge, gradient exchange) + backward
    g = torch.Generator(device=dev).manual_seed(77 + rank)
    q = F.normalize(torch.randn(N, C, device=dev, generator=g), dim=1).requires_grad_(True)
    k = F.normalize(torch.randn(N, C, device=dev, generator=g), dim=1)
    k_all = torch.empty(N * world, C, device=dev)
    dist.all_gather_into_tensor(k_all, k)
    iters = 20

    def head(kk):
        for _ in range(kk):
            q.grad = None
            loss, _ = smod.forward_loss(q, k, k_all)
            loss.backward()
    head(3)
    smod.profile = []
    head(iters)
    prof, smod.profile = smod.profile, None
    torch.cuda.synchronize()
    parts = {}
    for name, e0, e1 in prof:
        parts[name] = parts.get(name, 0.0) + e0.elapsed_time(e1) * 1e3 / iters
    ms_head = timed(head, iters)
    flops = 4.0 * (N * world) * C * (Ksh // world)              # per rank: all W*N queries x its shard, fwd + bwd
    sweep = parts.get("shard_sweep_us")
    return {"workload": f"BASELINE configs[3]: K={Ksh} sharded /{world} ({Ksh // world} rows per rank), "
                        f"{N * world} queries per rank, same {args.arch} step",
            "value": N * world * steps / (ms * 1e-3), "unit": "images/s", "ms_per_step": ms / steps, "steps": steps,
            "head_us": ms_head * 1e3 / iters, "parts_us": parts,
            "shard_kernel": {"us": sweep, "algorithmic_flops": flops,
                             "TFLOPs": (flops / (sweep * 1e-6) / 1e12) if sweep else None,
                             "frac": (flops / (sweep * 1e-6) / 1e12 / peaks["tf_sustained"]) if sweep else None},
            "note": "parts_us: CUDA events around each stage of the head on the launching stream (exchanges = "
                    "publish + signal barrier + peer pull over NVLink; no NCCL on the data path)"}


def dump_outputs(path, loss, prob, model, model_ema, contrast, n_all):
    """What one MoCoStep call computed, as DIR/<name>.npy: the loss and prob it returned (float64 scalars) and the state
    it updated in place (float32) -- the n_all keys it enqueued (ring slots in write order), the query encoder's fc
    weight / bias after the SGD step and the EMA encoder's fc weight.  2.2 MB at the defaults.
    With --dump-outputs, run_native lets cuDNN pick the encoders' convolution algorithms by its heuristics instead of
    timing them (see run_native).  On a B200 (1000 W power limit), two runs at the default arguments wrote byte-identical
    files; the step ran about 3 % slower than with autotuned algorithms (7,763 vs 8,008 img/s).  Without the flag, two
    autotuned runs differed from each other by up to 2e-3 in the loss."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    rows = (torch.arange(n_all) + contrast.index - n_all) % contrast.queue_size
    net = model.module if hasattr(model, "module") else model
    arrays = {"loss": loss.double(), "prob": prob.double(), "enqueued_keys": contrast.memory[rows].float(),
              "fc_weight": net.fc.weight.float(), "fc_bias": net.fc.bias.float(), "ema_fc_weight": model_ema.fc.weight.float()}
    for name, t in arrays.items():
        np.save(os.path.join(path, name + ".npy"), t.detach().cpu().numpy())


def run_native(args):
    if args.dump_outputs:
        # cuDNN's autotuner times the candidate algorithms of every convolution and keeps the fastest; near-ties go either
        # way from run to run, and the algorithms round differently, so the training trajectory differs run to run.  The
        # heuristic choice (mode B: cuDNN's more accurate heuristics, read at the first convolution) does not depend on
        # timing, and cudnn.deterministic (set below) keeps it to algorithms without run-dependent accumulation order.
        os.environ.setdefault("TORCH_CUDNN_USE_HEURISTIC_MODE_B", "1")
    import torch
    import torch.distributed as dist
    from moco_b200 import _lib, encoders
    from moco_b200.NCE import MemoryMoCo
    from moco_b200.train_step import MoCoStep

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("bench.py --gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
        args.gpus = world
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (native arm) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()
    peaks = load_peaks()
    torch.backends.cudnn.benchmark = not args.dump_outputs          # autotuned algorithms unless outputs must reproduce
    torch.backends.cudnn.deterministic = bool(args.dump_outputs)
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.allow_tf32 = True

    N, C, T = args.batch, args.feat_dim, args.nce_t
    K = args.nce_k or default_k(world)

    # ---- multi-GPU parity, where the driver can see it (N > 1): ShuffleBN both directions + NHWC publish +
    #      dist_collect bit-exact against the oracle of util.py:47-111, three sharded-queue steps against the
    #      replicated oracle of Contrast.py:20-34.  Runs BEFORE the timed region; a failure fails the run.
    parity = None
    if world > 1:
        from tools.multi_gpu_check import correctness
        parity = correctness(rank, world, dev)
        if not parity["ok_all_ranks"]:
            if rank == 0:
                print(json.dumps({"metric": METRIC, "error": "multi-GPU parity check failed", "parity": parity}))
            dist.barrier()
            dist.destroy_process_group()
            sys.exit(1)

    torch.manual_seed(0)
    ctor = getattr(encoders, args.arch)
    mf = torch.channels_last if args.memory_format == "channels_last" else torch.contiguous_format
    model = ctor(low_dim=C).to(dev).to(memory_format=mf)
    model_ema = ctor(low_dim=C).to(dev).to(memory_format=mf)
    model_ema.load_state_dict(model.state_dict())
    contrast = MemoryMoCo(C, K, T).to(dev)
    opt = torch.optim.SGD(model.parameters(), lr=0.03 * N * world / 256, momentum=0.9, weight_decay=1e-4)
    ddp_cfg = None
    if world > 1:
        # library DDP as in train.py:198 (out of scope, host PyTorch); only its knobs are set: gradients live in the
        # bucket views (no grad->bucket copies), static graph (no per-step bucket rebuild checks)
        ddp_cfg = {"bucket_cap_mb": args.ddp_bucket_mb, "gradient_as_bucket_view": True, "static_graph": True,
                   "grad_comm_dtype": "bf16 (compress hook)" if args.ddp_bf16 else "f32"}
        model = torch.nn.parallel.DistributedDataParallel(
            model, device_ids=[local_rank], broadcast_buffers=False, bucket_cap_mb=args.ddp_bucket_mb,
            gradient_as_bucket_view=True, static_graph=True)
        if args.ddp_bf16:
            from torch.distributed.algorithms.ddp_comm_hooks import default_hooks
            model.register_comm_hook(None, default_hooks.bf16_compress_hook)
    nhwc = args.memory_format == "channels_last"
    step = MoCoStep(model, model_ema, contrast, opt, channels_last=nhwc)

    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    dev_inputs = torch.randn(N, 6, 224, 224, device=dev, generator=gen)           # dataset.py:31-33 layout
    host_inputs = [torch.empty(N, 6, 224, 224, pin_memory=True).copy_(dev_inputs) for _ in range(2)]
    epoch = 1

    def split(t):
        x1, x2 = torch.split(t, [3, 3], dim=1)                       # train.py:250 (views of the 6-channel batch)
        if nhwc:
            return x1, x2                 # MoCoStep reads the crops in place (moco_crop_to_nhwc_bf16)
        return (x1.contiguous(memory_format=mf), x2.contiguous())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn(steps)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    # ---- arm 1: inputs resident in HBM (308 MB per step > 126 MB L2)
    x1, x2 = split(dev_inputs)
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(args.steps)]
    for e4 in ev:
        for j in (1, 0, 3, 2):       # stop before start: a hook that never fires reads as a negative interval
            e4[j].record()

    def loop_resident(steps, profile=False):
        out = None
        for i in range(steps):
            if profile:
                lib.moco_prof_set_events(1, ev[i][0].cuda_event, ev[i][1].cuda_event)
                lib.moco_prof_set_events(2, ev[i][2].cuda_event, ev[i][3].cuda_event)
            out = step(x1, x2, epoch)
        return out

    loop_resident(args.warmup)
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = _lib.launches
    last = []
    ms_total = timed(lambda s: last.append(loop_resident(s, True)), args.steps)
    launches = _lib.launches - l0
    sampler.stop_flag = True
    sampler.join()
    if args.dump_outputs and rank == 0:          # before any further step changes the state
        dump_outputs(args.dump_outputs, *last[0], model, model_ema, contrast, N * world)
    lib.moco_prof_set_events(1, None, None)
    lib.moco_prof_set_events(2, None, None)
    win = ctypes.c_float()
    sc = next(iter(contrast._scratch.values()))
    lib.moco_prof_sweep_window(sc.ws_ptr, 148, ctypes.byref(win), torch.cuda.current_stream().cuda_stream)
    us_stats = sum(e[0].elapsed_time(e[1]) for e in ev) * 1e3 / args.steps
    us_dq = sum(e[2].elapsed_time(e[3]) for e in ev) * 1e3 / args.steps
    ms_step = ms_total / args.steps
    value = N * world * args.steps / (ms_total * 1e-3)

    # ---- arm 2: end to end through the public API with HOST inputs (pinned), H2D inside the timed region,
    #      next batch prefetched on a copy stream, loss + prob read back every step
    copy_stream = torch.cuda.Stream()
    bufs = [torch.empty_like(dev_inputs) for _ in range(2)]
    sink = []

    def loop_e2e(steps):
        main = torch.cuda.current_stream()
        with torch.cuda.stream(copy_stream):
            bufs[0].copy_(host_inputs[0], non_blocking=True)
        for i in range(steps):
            main.wait_stream(copy_stream)
            cur = bufs[i & 1]
            if i + 1 < steps:
                copy_stream.wait_stream(main)         # buffer (i+1)&1 was consumed by step i-1
                with torch.cuda.stream(copy_stream):
                    bufs[(i + 1) & 1].copy_(host_inputs[(i + 1) & 1], non_blocking=True)
            a, b = split(cur)
            loss, prob = step(a, b, epoch)
            sink.append((loss.item(), prob.item()))    # D2H read of the step's result (train.py:280-281)

    loop_e2e(max(2, args.warmup // 2))
    ms_e2e = timed(loop_e2e, args.steps)
    e2e_value = N * world * args.steps / (ms_e2e * 1e-3)
    h2d = N * 6 * 224 * 224 * 4
    final_loss = sink[-1][0]

    # ---- the same step with the encoders' BatchNorm -> add -> ReLU groups on ATen's kernels instead of this library's
    #      (moco_b200.bn.set_fused(False)): what csrc/bn_nhwc.cu is worth inside the step.  N = 1 only, 5 steps.
    encoder_bn = None
    if world == 1 and not args.no_bn_ab:
        from moco_b200 import bn as _bn
        _bn.set_fused(False)
        try:
            loop_resident(2)
            ms_aten = timed(loop_resident, 5) / 5
        finally:
            _bn.set_fused(True)
        loop_resident(1)
        # live HBM roofline of the BN kernels inside the step: CUDA events around every fused call of 2 extra steps
        # (kept out of the timed region above: 640 event records per step would perturb it)
        _bn._prof = []
        loop_resident(2)
        torch.cuda.synchronize()
        prof, _bn._prof = _bn._prof, None
        bn_bytes = sum(p[1] for p in prof) / 2
        bn_us = sum(p[2].elapsed_time(p[3]) for p in prof) * 1e3 / 2
        fwd_us = sum(p[2].elapsed_time(p[3]) for p in prof if p[0] == "bn_fwd") * 1e3 / 2
        n_bn = sum(1 for m in model.modules() if isinstance(m, _bn.BatchNormAct2d))
        encoder_bn = {
            "kernels": "bn_stats_kernel + bn_apply_kernel (forward, both encoders), bn_bwd_reduce_kernel + bn_bwd_apply_kernel "
                       "(backward, query encoder): training-mode BatchNorm with the residual add and ReLU folded in, bf16 NHWC",
            "layers_per_encoder": n_bn, "launches_per_step": 6 * n_bn,
            "ms_per_step": ms_step, "ms_per_step_aten_batchnorm": ms_aten, "step_speedup": ms_aten / ms_step,
            "roofline": {"bound": "hbm", "achieved": bn_bytes / (bn_us * 1e-6) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": bn_bytes / (bn_us * 1e-6) / 1e9 / peaks["hbm_gbs"], "peak_source": peaks["source"],
                         "algorithmic_bytes_per_step": bn_bytes, "us_per_step": bn_us, "forward_us_per_step": fwd_us,
                         "calls_per_step": len(prof) // 2,
                         "how": "CUDA events around every moco_bn_fwd_train / moco_bn_bwd call (2 launches each) of 2 extra "
                                "steps; bytes = 2 B x elements x (statistics 1 + apply 2 [+1 residual]) forward, "
                                "(reduce 2 [+1 mask] + apply 3 [+1 mask] [+1 d residual]) backward"},
            "note": "ATen arm = nn.BatchNorm2d's own bf16 channels_last kernels + separate add and ReLU passes, everything "
                    "else identical (same MoCoStep, same head kernels); profiles/ has the per-kernel ncu captures"}

    shufflebn = sharded = None
    if world > 1:
        # the one NCCL collective of the step (library DDP, out of scope): the bucketed gradient all-reduce, timed alone
        n_params = sum(p.numel() for p in model.parameters())
        gbuf = torch.zeros(n_params, dtype=torch.bfloat16 if args.ddp_bf16 else torch.float32, device=dev)

        def allreduce(k):
            for _ in range(k):
                dist.all_reduce(gbuf)
        allreduce(2)
        ar_ms = timed(allreduce, 5) / 5
        ddp_cfg["limiting_collective"] = {
            "what": "DDP gradient all-reduce (NCCL, overlapped with backward inside the step)", "bytes": gbuf.numel() * gbuf.element_size(),
            "alone_us": ar_ms * 1e3, "busbw_GBps": 2 * (world - 1) / world * gbuf.numel() * gbuf.element_size() / (ar_ms * 1e-3) / 1e9}
        del gbuf
        shufflebn = shufflebn_block(x2, epoch, rank, world, dev, nhwc)
        if not args.no_sharded:
            sharded = sharded_block(args, model, model_ema, opt, x1, x2, epoch, rank, world, dev, nhwc, peaks, timed)

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # dominant hot-path kernel inside the step: the one-pass kernel (T = 0.07 -> MOCO_NCE_AUTO takes one sweep);
    # algorithmic work per launch = forward 2NC(K+1) + backward 2NC(K+1) FLOP (SURVEY.md 8d), queue read once
    flops = 4.0 * N * C * (K + 1)
    bytes_ = K * C * 2 + 3 * N * C * 2 + 12 * N
    one_pass = us_stats <= 0.0                        # the statistics-kernel hook never fired
    us_main = us_dq if one_pass else us_stats + us_dq
    a_tf = flops / (us_main * 1e-6) / 1e12
    roofline = {
        "kernel": ("nce_head128_kernel<FUSED>: one sweep over the queue on tcgen05 (q staged in-kernel, S = q.Queue^T, "
                   "P = 2^(S/T - m), O += P.Queue, row sums) -> loss statistics + dq partials" if one_pass else
                   "nce_stats_kernel + nce_head128_kernel (two-pass)") + ", timed inside the step",
        "bound": "tensor", "achieved": a_tf, "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
        "frac": a_tf / peaks["tf_sustained"], "peak_source": peaks["source"] + ", sustained bf16",
        "us_per_launch": us_main, "algorithmic_flops": flops, "algorithmic_bytes": bytes_,
        "device_window_us": float(win.value),
        "device_window_note": "first CTA entry -> last CTA exit of the last sweep kernel on the device clock (%globaltimer): "
                              "what the CTAs took; us_per_launch (CUDA events around the single kernel, which breaks its "
                              "programmatic-dependent-launch overlap) also contains ~4.5 us of grid launch and ~2 us of completion",
        "hbm_GBps": bytes_ / (us_main * 1e-6) / 1e9, "hbm_frac": bytes_ / (us_main * 1e-6) / 1e9 / peaks["hbm_gbs"],
        "traffic": NCU_TRAFFIC_BYTES.get(("onepass", N, C, K)),
        "note": f"ideal time for this shape is {flops / (peaks['tf_sustained'] * 1e12) * 1e6:.1f} us "
                f"({flops / 1e9:.2f} GFLOP, {bytes_ / 1e6:.1f} MB): {-(-K // 128 * ((N + 127) // 128) // 148)} 128-row tile(s) per CTA, "
                "so launch + prologue + one pipeline fill + the split-K partials dominate; roofline_stress (N=1 runs) is "
                "the tensor-bound shape of BASELINE configs[4]",
    }
    line = {
        "metric": METRIC, "value": value, "unit": "images/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "cudnn_algorithms": "heuristic (reproducible outputs)" if args.dump_outputs else "autotuned",
        "config": config_block(args, K, world),
        "clocks": sampler.result(),
        "e2e": {"value": e2e_value, "unit": "images/s", "ms_per_step": ms_e2e / args.steps,
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 8},
        "gpu_launches": launches,
        "roofline": roofline,
        "final_loss": final_loss,
    }
    if parity is not None:
        line["parity"] = {"shufflebn": parity["shufflebn"], "sharded": parity["sharded_queue"],
                          "max_err": parity["max_err"], "world": world,
                          "what": "ShuffleBN fwd/bwd + NHWC publish + dist_collect bit-exact vs the oracle of util.py:47-111; "
                                  "3 sharded-queue steps vs the replicated oracle of Contrast.py:20-34 (all ranks)"}
        line["ddp"] = ddp_cfg
    if encoder_bn is not None:
        line["encoder_bn"] = encoder_bn
    if shufflebn is not None:
        line["shufflebn"] = shufflebn
    if sharded is not None:
        line["sharded"] = sharded
    if world == 1 and not args.no_stress:
        line["roofline_stress"] = stress_roofline(peaks, dev)
    if world == 1 and not args.no_cpu_baseline:
        r = reference_job(args.arch, C, K, T, args.cpu_sample_batch, 5, 3)
        line["cpu_baseline"] = cpu_baseline_block(r)
    print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_native(a)
