#!/usr/bin/env python
"""bench.py -- persons/s of the simple-HRNet hot path (network forward + argmax decode) on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|reference-cuda]
                  [--config w48|w32|poseresnet50] [--dump-outputs DIR]
  (N > 1: launched by torchrun, one rank per GPU; crops sharded by batch, one NCCL all-gather of joints)
  --dump-outputs DIR: after the timed steps, the joints [B,17,3] (y, x, confidence) the last timed step returned are
  written to DIR/joints.npy (float32).  Weights and inputs are seeded, so two builds run with the same arguments can be
  compared output for output.

One "step" = one pass of the hot path over one batch of synthetic crops.  Default config = BASELINE.json configs[2],
the one the metric is quoted on: HRNet-W48 @ 384x288, 17 joints, 64 persons per GPU, random-init weights
(oracle.make_state_dict, seed 0), inputs torch.randn at the model boundary.  `--config w32` / `poseresnet50` are
BASELINE configs[1] / [4] (HRNet-W32 256x192 batch 32, PoseResNet-50 256x192 batch 64).
  value : whole-job persons/s, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e   : same metric from pinned HOST uint8 crops to HOST joints through HostPipeline (double-buffered
          hrnet_forward_host_u8_async): every step's H2D and D2H copies are inside the timed region; the blocking
          one-call-per-step figure is reported next to it (sync_call_value)
  roofline     : the dominant kernel class (HRNet: the stage-4 3x3 implicit-GEMM branch convs on tcgen05) timed alone
                 with CUDA events, algorithmic FLOPs / time vs the measured dense bf16 peak (burst: the timed pass is
                 tens of milliseconds long)
  cpu_baseline : the reference's CPU path on this box's host cores -- the UNMODIFIED reference class from oracle/_ref
                 (kind "reference") when it is installed, else the oracle port (kind "port"); thread count calibrated
                 at the timed batch, worker process pinned to the cores of as few NUMA nodes as possible
`--impl reference` times that CPU implementation as the reference arm (same metric / config); `--impl reference-cuda`
is an informative second bar: the unmodified reference on the same GPU through its own CUDA/cuDNN path (SURVEY 8f4).
Prints ONE JSON line on rank 0.
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
sys.dont_write_bytecode = True      # the tree may be read-only: nothing is written or cached there

J = 17
CONFIGS = {
    # GFLOP per person = 2 * MACs of every conv (SURVEY.md section 8d, forward-hook tally of the reference modules)
    "w48": dict(arch="hrnet", c=48, H=384, W=288, batch=64, gflop=70.613, name="HRNet-W48 384x288",
                baseline="BASELINE.json configs[2] (headline)", s4_gflop=27.519),
    "w32": dict(arch="hrnet", c=32, H=256, W=192, batch=32, gflop=15.290, name="HRNet-W32 256x192",
                baseline="BASELINE.json configs[1]", s4_gflop=5.436),
    "poseresnet50": dict(arch="poseresnet", c=50, H=256, W=192, batch=64, gflop=10.853, name="PoseResNet-50 256x192",
                         baseline="BASELINE.json configs[4]", s4_gflop=None),
}


def metric_name(cfg):
    return f"persons/sec {cfg['name']} (forward + argmax decode)"


# ------------------------------------------------------------------------------------------------ CPU worker (child)
def numa_cpu_order():
    """Logical CPUs ordered node by node (physical cores first when sibling lists are available)."""
    nodes = []
    base = "/sys/devices/system/node"
    try:
        for d in sorted(os.listdir(base), key=lambda s: int(s[4:]) if s.startswith("node") and s[4:].isdigit() else 1 << 30):
            if not (d.startswith("node") and d[4:].isdigit()):
                continue
            cpus = []
            for part in open(os.path.join(base, d, "cpulist")).read().strip().split(","):
                if "-" in part:
                    a, b = part.split("-"); cpus += list(range(int(a), int(b) + 1))
                elif part:
                    cpus.append(int(part))
            nodes.append(cpus)
    except Exception:
        nodes = []
    allowed = sorted(os.sched_getaffinity(0))
    if not nodes:
        return allowed
    order = [c for n in nodes for c in n if c in set(allowed)]
    return order or allowed


def cpu_worker(argv):
    """Child process: `bench.py --cpu-worker <config> <threads> <n> <warmup> <steps>`.  Pins itself BEFORE importing
    torch (every OpenMP worker inherits the mask), runs the reference's CPU path and prints one JSON line."""
    key, threads, n, warm, steps = argv[0], int(argv[1]), int(argv[2]), int(argv[3]), int(argv[4])
    cfg = CONFIGS[key]
    order = numa_cpu_order()
    pinned = False
    if threads < len(order):
        try:
            os.sched_setaffinity(0, order[:threads]); pinned = True
        except Exception:
            pass
    os.environ["OMP_NUM_THREADS"] = str(threads)
    os.environ["MKL_NUM_THREADS"] = str(threads)
    import numpy as np
    import tempfile
    import torch
    torch.set_num_threads(threads)
    from oracle import hrnet_oracle as O
    from oracle.install_ref import import_reference
    spec = O.hrnet_param_spec(cfg["c"], J) if cfg["arch"] == "hrnet" else O.poseresnet_param_spec(cfg["c"], J)
    sd = O.make_state_dict(spec, seed=0, bn="default")
    H, W = cfg["H"], cfg["W"]
    crops = np.random.default_rng(0).integers(0, 256, (n, H, W, 3), dtype=np.uint8)
    ref = import_reference()
    if ref is not None:
        kind = "reference"
        with tempfile.TemporaryDirectory() as td:
            ck = os.path.join(td, "w.pth"); torch.save(sd, ck)
            import contextlib, io
            with contextlib.redirect_stdout(io.StringIO()):          # the reference prints its device line
                m = ref[0](cfg["c"], J, ck, model_name="HRNet" if cfg["arch"] == "hrnet" else "PoseResNet",
                           resolution=(H, W), multiperson=False, max_batch_size=n, device=torch.device("cpu"))
        run = lambda: m.predict(crops)                               # unmodified SimpleHRNet.predict (SimpleHRNet.py:174-210)
        what = "unmodified reference SimpleHRNet(..., device=cpu).predict(uint8 crops): resize/cvtColor/transform + model + numpy decode"
    else:
        kind = "port"
        fwd = O.hrnet_forward if cfg["arch"] == "hrnet" else O.poseresnet_forward
        boxes = np.repeat(np.asarray([[0, 0, W, H]], dtype=np.float32), n, axis=0)
        run = lambda: O.decode_joints(fwd(sd, O.preprocess(crops, (H, W))).numpy(), boxes)
        what = "oracle port of the reference CPU path (same aten ops + numpy decode)"
    ts = []
    for i in range(warm + steps):
        t0 = time.perf_counter()
        run()
        if i >= warm:
            ts.append(time.perf_counter() - t0)
    print(json.dumps({"kind": kind, "what": what, "threads": threads, "pinned": pinned, "n": n, "times": ts,
                      "torch": torch.__version__, "ncpu": os.cpu_count()}), flush=True)


def run_cpu_child(key, threads, n, warm, steps, timeout=900):
    cmd = [sys.executable, os.path.abspath(__file__), "--cpu-worker", key, str(threads), str(n), str(warm), str(steps)]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout)
        line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
        return json.loads(line)
    except Exception as e:   # noqa: BLE001
        return {"error": repr(e)[:200]}


def cpu_arm(key, warm, steps, n):
    """Best thread count at the TIMED batch (one warm-up + one timed rep per candidate), then the timed run."""
    ncpu = os.cpu_count() or 1
    # 16 / 32 / 64 threads (a socket's worth at most): every hardware thread of a big host is far slower (oneDNN
    # oversubscribed: 123 s for a 4-person forward on 128 threads in round 1), so it is not even tried
    cands = sorted({min(t, ncpu) for t in (16, 32, 64)})
    calib = {}
    for t in cands:
        r = run_cpu_child(key, t, n, 1, 1, timeout=300)
        if "times" in r:
            calib[t] = round(r["times"][0], 3)
    best = min(calib, key=calib.get) if calib else min(16, ncpu)
    r = run_cpu_child(key, best, n, warm, steps)
    return best, calib, r


# ------------------------------------------------------------------------------------------------ helpers (parent)
def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tflops=d.get("bf16_tflops", 1590.0), tflops_sustained=d.get("bf16_tflops_sustained", 1400.0),
                    hbm=d.get("hbm_gbs", 6650.0), source="measured (MEASURED_PEAKS.json)")
    return dict(tflops=1590.0, tflops_sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


def load_traffic():
    """ncu dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernels, extracted from the committed
    `ncu --set full` capture (profiles/r02_traffic.json, written by tools/ncu_traffic.py); None if no capture exists."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            try:
                d = json.load(open(p)); d["file"] = "profiles/" + name
                return d
            except Exception:
                pass
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        import numpy as np
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], None, [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1]); pw.append(float(r[2]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(pw) if pw else None}


def make_weights(cfg):
    from oracle import hrnet_oracle as O
    spec = O.hrnet_param_spec(cfg["c"], J) if cfg["arch"] == "hrnet" else O.poseresnet_param_spec(cfg["c"], J)
    return O.make_state_dict(spec, seed=0, bn="default")


# ------------------------------------------------------------------------------------------------ reference arms
def run_reference(args, cfg, rank):
    """The reference's own CPU implementation of the path on the box's host cores (rank 0 only)."""
    if rank != 0:
        return
    n = 16                               # bounded sample of the config's batch (W48: ~1-2 s per step on a big host)
    threads, calib, r = cpu_arm(args.config, args.warmup, args.steps, n)
    if "times" not in r:
        print(json.dumps({"impl": "reference", "unavailable": f"CPU worker failed: {r.get('error')}"}), flush=True)
        return
    ts = r["times"]
    total = float(sum(ts))
    v = n * len(ts) / total
    sample = (f"{n} persons x {len(ts)} steps of the {cfg['batch']}-person workload, {r['what']}, torch {r['torch']} CPU, "
              f"{threads} of {r['ncpu']} threads (pinned node by node: {r['pinned']}; fastest at the timed batch of "
              f"{{threads: s per step}} {calib})")
    out = {"impl": "reference", "metric": metric_name(cfg), "value": v, "unit": "persons/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(ts),
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"{cfg['name']}, 17 joints, forward + argmax decode on the host CPU (fp32), bounded sample "
                                  f"of {n} persons per step ({cfg['baseline']})",
                      "per_gpu_batch": cfg["batch"], "sample_per_step": n},
           "cpu_baseline": {"value": v, "unit": "persons/s", "cores": threads, "kind": r["kind"], "sample": sample},
           "e2e": {"value": v, "unit": "persons/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)


def run_reference_cuda(args, cfg, rank):
    """Informative second bar (SURVEY 8f4): the unmodified reference on this GPU through its own CUDA path
    (SimpleHRNet.py:123-142: nn.DataParallel + cuDNN, fp32), plus the bare model in fp32 / fp16."""
    if rank != 0:
        return
    import contextlib, io, tempfile
    import numpy as np
    import torch
    from oracle.install_ref import import_reference
    ref = import_reference()
    if ref is None or not torch.cuda.is_available():
        print(json.dumps({"impl": "reference-cuda", "unavailable": "reference not installed in oracle/_ref or no GPU"}), flush=True)
        return
    sd = make_weights(cfg)
    H, W, n = cfg["H"], cfg["W"], cfg["batch"]
    dev = torch.device("cuda:0")
    with tempfile.TemporaryDirectory() as td:
        ck = os.path.join(td, "w.pth"); torch.save(sd, ck)
        with contextlib.redirect_stdout(io.StringIO()):
            m = ref[0](cfg["c"], J, ck, model_name="HRNet" if cfg["arch"] == "hrnet" else "PoseResNet", resolution=(H, W),
                       multiperson=False, max_batch_size=n, device=dev)
    crops = [np.random.default_rng(i).integers(0, 256, (n, H, W, 3), dtype=np.uint8) for i in range(2)]
    for i in range(args.warmup):
        m.predict(crops[i % 2])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(args.steps):
        m.predict(crops[i % 2])
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    v = n * args.steps / dt
    bare = {}
    net = ref[1](cfg["c"], J) if cfg["arch"] == "hrnet" else ref[2](cfg["c"], J)
    net.load_state_dict(sd)
    for name, dtype in (("fp32", torch.float32), ("fp16", torch.float16)):
        mod = net.to(dev).to(dtype).eval()
        xs = [torch.randn(n, 3, H, W, device=dev, dtype=dtype) for _ in range(3)]
        with torch.no_grad():
            for i in range(3):
                mod(xs[i % 3])
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(args.steps):
                mod(xs[i % 3])
            e1.record(); torch.cuda.synchronize()
        bare[name] = {"ms_per_step": round(e0.elapsed_time(e1) / args.steps, 3),
                      "persons_per_s": round(n * args.steps / (e0.elapsed_time(e1) / 1e3), 1)}
    out = {"impl": "reference-cuda", "metric": metric_name(cfg), "value": round(v, 2), "unit": "persons/s", "n_gpus": 1,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * dt / args.steps, 3), "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"{cfg['name']}, {n} persons per step, unmodified reference SimpleHRNet(device=cuda:0).predict "
                                  "(host resize/cvtColor/transform, DataParallel + cuDNN fp32 forward, D2H of heat-maps, numpy decode)",
                      "per_gpu_batch": n},
           "bare_model": bare,
           "e2e": {"value": round(v, 2), "unit": "persons/s", "h2d_bytes_per_step": n * 3 * H * W * 4,
                   "d2h_bytes_per_step": n * J * (H // 4) * (W // 4) * 4},
           "note": "informative: cuDNN library path of the reference on the same B200; never replaces the CPU reference arm"}
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------------------ our arm
def main():
    if len(sys.argv) > 1 and sys.argv[1] == "--cpu-worker":
        cpu_worker(sys.argv[2:])
        return
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-cuda"])
    ap.add_argument("--config", default="w48", choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernel-roofline", action="store_true")
    ap.add_argument("--flags", type=int, default=0, help="HRNET_FLAG_* plan flags (experiments)")
    ap.add_argument("--tune", default="", help="HRNET_TUNE_* overrides, e.g. 0=400,1=250 (experiments)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the joints of the last timed step to DIR/joints.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3)
    cfg = CONFIGS[args.config]

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, cfg, rank)
        return
    if args.impl == "reference-cuda":
        run_reference_cuda(args, cfg, rank)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from simple_hrnet_b200 import B200Engine, HostPipeline, ShardedPredictor, load_library, shard_range

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product path has no CPU fallback)")
    load_library(build_if_missing=False)     # the library build() made; bench never compiles into the tree
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    peaks = load_peaks()
    H, W, PB = cfg["H"], cfg["W"], cfg["batch"]
    is_hrnet = cfg["arch"] == "hrnet"

    sd = make_weights(cfg)
    tune = {int(k): int(v) for k, v in (kv.split("=") for kv in args.tune.split(",") if kv)}
    eng = B200Engine(cfg["arch"], cfg["c"], J, (H, W), PB, dev, flags=args.flags, tune=tune)
    eng.load_state_dict(sd)
    B = PB * world
    lo, hi = shard_range(B, world, rank)
    # three rotating input buffers; the activations a step streams through HBM evict the 126 MB L2 many times over
    # between two reads of the same input

    def make_inputs(r):
        g = torch.Generator().manual_seed(1000 + r)
        a, b = shard_range(B, world, r)
        return [torch.randn(b - a, 3, H, W, generator=g).to(dev) for _ in range(3)], g
    xs, gen = make_inputs(rank)
    pred = ShardedPredictor(lambda imgs, out: eng.forward_decode(imgs, joints_out=out), J, dev)

    def run_steps(first, count):
        """`count` steps; returns the joints [B,17,3] of the last one.  Multi-GPU: pipelined form -- step i's all-gather
        runs on a side stream while step i+1's forward computes; every step's result is consumed one step later."""
        if world == 1:
            out = None
            for i in range(first, first + count):
                out = pred.predict_joints(B, xs[i % 3])
            return out
        prev = None
        for i in range(first, first + count):
            h = pred.submit(B, xs[i % 3])
            if prev is not None:
                pred.result(prev)
            prev = h
        return pred.result(prev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    run_steps(0, args.warmup)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    joints = run_steps(0, args.steps)
    e1.record()
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    per_rank_ms = None
    if world > 1:
        allms = torch.zeros(world, device=dev)
        dist.all_gather_into_tensor(allms, ms)
        per_rank_ms = [round(float(v) / args.steps, 4) for v in allms.tolist()]
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    clocks = sampler.stop() if rank == 0 else None
    value = B * args.steps / (ms_total / 1e3)
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "joints.npy"), joints.cpu().numpy().astype(np.float32))

    # ---- multi-GPU correctness of the gathered result (outside the timed region): every rank recomputes the shard of
    # rank (r+1) % world from that rank's seed and compares it bit for bit with its slice of the gathered joints
    gather_check = None
    if world > 1:
        nb = (rank + 1) % world
        a, b = shard_range(B, world, nb)
        xn, _ = make_inputs(nb)
        jn, _, _ = eng.forward_decode(xn[(args.steps - 1) % 3])
        own, _, _ = eng.forward_decode(xs[(args.steps - 1) % 3])
        ok = torch.equal(joints[a:b], jn) and torch.equal(joints[lo:hi], own)
        flag = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        gather_check = "ok" if int(flag.item()) == 1 else "MISMATCH"
        del xn

    # ---- e2e: the reference-facing call with HOST buffers, H2D + D2H inside the timed region
    e2e_steps = max(3, args.steps // 2)
    if is_hrnet:
        # uint8 BGR crops at network resolution in pinned host memory -> joints in host memory
        xh = [torch.randint(0, 256, (hi - lo, H, W, 3), generator=gen, dtype=torch.uint8).pin_memory() for _ in range(2)]
        xh_np = [t.numpy() for t in xh]
        sync_call = lambda i: eng.forward_host_u8(xh_np[i % 2])
        h2d = (hi - lo) * 3 * H * W          # uint8 images; normalisation runs in the stem kernel
    else:
        xh = [torch.randn(hi - lo, 3, H, W, generator=gen).pin_memory() for _ in range(2)]
        xh_np = [t.numpy() for t in xh]
        sync_call = lambda i: eng.forward_host(xh_np[i % 2])
        h2d = (hi - lo) * 3 * H * W * 4      # fp32 NCHW (the uint8 entry point is HRNet-only)
    d2h = (hi - lo) * J * 3 * 4 + (hi - lo) * J * 4

    def consume(jh):
        if world > 1:   # the gathered result is what a multi-GPU caller receives
            buf = torch.empty(B, J, 3, device=dev)
            buf[lo:hi].copy_(torch.from_numpy(jh), non_blocking=True)
            dist.all_gather_into_tensor(buf, buf[lo:hi])
            buf.cpu()
    for i in range(3):
        sync_call(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        consume(sync_call(i)[0])
    barrier()
    e2e_s = torch.tensor([time.perf_counter() - t0], device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_sync_value = B * e2e_steps / float(e2e_s.item())
    e2e_value, e2e_call = e2e_sync_value, "one blocking host-buffer call per step (hrnet_forward_host)"
    if is_hrnet:
        # the serving loop a throughput user runs: HostPipeline double-buffers two engines that share the device weights, so
        # batch i+1's H2D copy and batch i-1's D2H copy overlap batch i's forward; every step's copies are inside the timed region
        pipe = HostPipeline(eng, depth=2)
        for jh in pipe.run(xh[i % 2] for i in range(4)):
            consume(jh)
        barrier()
        t0 = time.perf_counter()
        for jh in pipe.run(xh[i % 2] for i in range(e2e_steps)):
            consume(jh)
        barrier()
        e2e_s = torch.tensor([time.perf_counter() - t0], device=dev)
        if world > 1:
            dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
        e2e_value = B * e2e_steps / float(e2e_s.item())
        e2e_call = ("HostPipeline.run (hrnet_forward_host_u8_async on 2 engines sharing the weights): pinned uint8 BGR crops "
                    f"[n,{H},{W},3] -> H2D -> forward + decode -> D2H joints, batch i+1's copy overlaps batch i's forward")

    # ---- dominant kernel class, timed live with one CUDA event pair per kernel (hrnet_profile_ops: serial pass over the
    # plan's ops, inputs = real activations; a branch chain is one kernel: its time is split evenly over its 8 convs)
    roofline, breakdown = None, None
    if rank == 0 and not args.no_kernel_roofline:
        ops, desc = eng.profile_ops(xs[0], iters=5)
        n = PB
        cls_t, cls_f, cls_n = {}, {}, {}
        per_branch = {}
        chained = {i for ch in desc.get("chains", []) for i in ch["ops"]}
        for oi, (name, op, us) in enumerate(ops):
            flop = 0.0
            if op["kind"] == 1:
                tin = desc["tensors"][op["in"]]
                s = op["stride"]
                oh, ow = (tin["H"], tin["W"]) if op["pad"] >= 100 else (tin["H"] // s, tin["W"] // s)
                flop = 2.0 * n * oh * ow * op["k"] ** 2 * op["cin"] * op["cout"]
                if ".branches." in name:
                    cls = name.split(".")[0] + " 3x3 branch convs"
                    if name.startswith("stage4."):
                        kern = ("chain:" if oi in chained else "") + ("patch" if op["use_patch"] else "im2col")
                        key = (op["cin"], f"{tin['H']}x{tin['W']}", kern)
                        pb = per_branch.setdefault(key, [0.0, 0.0, 0])
                        pb[0] += us; pb[1] += flop; pb[2] += 1
                elif "fuse_layers" in name:
                    cls = "exchange-unit convs (1x1 up, 3x3 s2 down)"
                elif name.startswith("layer1") and is_hrnet:
                    cls = "layer1 bottlenecks"
                elif name.startswith("deconv"):
                    cls = "transposed convs (4 sub-pixel phases each)"
                elif name.startswith("layer"):
                    cls = "ResNet bottlenecks"
                else:
                    cls = "stem conv2 + transitions"
            else:
                cls = {0: "stem conv1 (hi/lo-split tcgen05)", 2: "exchange-unit sum", 3: "head 1x1", 4: "argmax decode",
                       5: "max pool", 6: "stem 7x7"}[op["kind"]]
            cls_t[cls] = cls_t.get(cls, 0.0) + us
            cls_f[cls] = cls_f.get(cls, 0.0) + flop
            cls_n[cls] = cls_n.get(cls, 0) + 1
        tot = sum(cls_t.values())
        breakdown = {"serial_total_us": round(tot, 1), "classes": {
            k: {"us": round(v, 1), "share": round(v / tot, 4), "ops": cls_n[k],
                "tflops": round(cls_f[k] / v / 1e6, 1) if cls_f[k] else None} for k, v in sorted(cls_t.items(), key=lambda kv: -kv[1])}}
        if is_hrnet:
            k4 = "stage4 3x3 branch convs"
            ach = cls_f[k4] / cls_t[k4] / 1e6
            nchain = sum(1 for ch in desc.get("chains", []) if ops[ch["ops"][0]][0].startswith("stage4."))
            what = (f"stage-4 3x3 s1 branch convs, N={n}: 96 convs" +
                    (f" issued as {nchain} branch-chain kernels (conv_chain_patch_kernel C<=96, conv_chain_igemm_kernel above; "
                     "8 convs per launch, each chain timed alone on the whole GPU with a CUDA event pair" if nchain else
                     " (conv3x3_patch_tc_kernel / conv_igemm_tc_kernel), each timed with a CUDA event pair") +
                    " inside a serial pass of the whole network); achieved = algorithmic conv FLOPs / summed kernel time")
            launches = nchain if nchain else cls_n[k4]
        else:
            k4 = "all convolutions"
            t4 = sum(v for k, v in cls_t.items() if cls_f[k]); f4 = sum(cls_f.values())
            cls_t[k4], cls_f[k4] = t4, f4
            ach = f4 / t4 / 1e6
            what = f"all tensor-core convs of the network, N={n}, each timed with a CUDA event pair inside a serial pass"
            launches = sum(v for k, v in cls_n.items() if cls_f.get(k))
        # traffic: DRAM bytes (ncu dram__bytes_read.sum + dram__bytes_write.sum) of ONE launch of the dominant kernel class =
        # the four concurrent branch-chain kernels of stage4.0 (the unit `achieved` is timed on); details in traffic_detail
        tdet = load_traffic()
        tnum = None
        if tdet and is_hrnet:
            ch = [k for k in tdet.get("kernels", []) if "conv_chain" in k.get("kernel", "") and k.get("traffic") is not None]
            if len(ch) >= 4:
                tnum = int(sum(k["traffic"] for k in ch[:4]))
        roofline = {"kernel": what.replace("each chain timed alone on the whole GPU with a CUDA event pair",
                                           "the chains of a module launched together on their in-forward grids and timed with one CUDA event pair"),
                    "bound": "tensor", "achieved": round(ach, 1), "peak": peaks["tflops"], "unit": "TFLOP/s",
                    "frac": round(ach / peaks["tflops"], 4),
                    "frac_of_sustained_peak": round(ach / peaks["tflops_sustained"], 4), "traffic": tnum, "traffic_detail": tdet,
                    "peak_source": peaks["source"] + ", burst figure (the per-op timing pass lasts tens of milliseconds at boost clocks)",
                    "launches": launches, "us_total": round(cls_t[k4], 1),
                    "per_branch": [{"C": k[0], "map": k[1], "kernel": k[2], "convs": v[2], "us_per_conv": round(v[0] / v[2], 2),
                                    "tflops": round(v[1] / v[0] / 1e6, 1), "frac_of_burst_peak": round(v[1] / v[0] / 1e6 / peaks["tflops"], 4)}
                                   for k, v in sorted(per_branch.items())]}

    # ---- CPU baseline on this box's host cores (rank 0, N=1 only), bounded sample
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ncpu_n = 16
        threads, calib, r = cpu_arm(args.config, 1, 2, ncpu_n)
        if "times" in r:
            v = ncpu_n * len(r["times"]) / sum(r["times"])
            cpu = {"value": round(v, 3), "unit": "persons/s", "cores": threads, "kind": r["kind"],
                   "sample": f"{ncpu_n} persons x {len(r['times'])} reps (after warm-up) of the {PB}-person workload, {r['what']}, "
                             f"{threads} of {r['ncpu']} threads (pinned node by node: {r['pinned']}; fastest at the timed batch of "
                             f"{{threads: s}} {calib}), rep times {[round(t, 2) for t in r['times']]} s"}
        else:
            cpu = {"value": None, "unit": "persons/s", "cores": 0, "kind": "port", "sample": f"CPU worker failed: {r.get('error')}"}

    if rank == 0:
        step_tflops = cfg["gflop"] * value / 1e3
        out = {"metric": metric_name(cfg), "value": round(value, 2), "unit": "persons/s", "n_gpus": world, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": round(ms_total / args.steps, 4), "higher_is_better": True,
               "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
               "config": {"workload": f"{cfg['name']}, 17 joints, {PB} persons per GPU per step, fp16 NHWC activations "
                                      f"with fp32 accumulate, random-init weights (seed 0), torch.randn inputs ({cfg['baseline']})",
                          "global_batch": B, "per_gpu_batch": PB, "parallelism": f"dp{world}",
                          "l2": "3 rotating input buffers; a step streams far more activation bytes through HBM than the 126 MB L2 holds",
                          "collective": ("one NCCL all_gather_into_tensor of joints [B,17,3] f32 per step, issued on a side stream behind "
                                         "that step's decode so that it overlaps the next step's forward (two rotating gather "
                                         "buffers, results consumed one step later)") if world > 1 else "none"},
               "clocks": clocks,
               "e2e": {"value": round(e2e_value, 2), "unit": "persons/s", "h2d_bytes_per_step": h2d,
                       "d2h_bytes_per_step": d2h, "steps": e2e_steps, "call": e2e_call,
                       "sync_call_value": round(e2e_sync_value, 2),
                       "sync_call": "one blocking host-buffer call per step (no overlap)"},
               "gpu_launches": eng.launch_count * args.steps,
               "launches_per_forward": eng.launch_count,
               "step_flops": {"tflops": round(step_tflops, 1), "per_gpu_tflops": round(step_tflops / world, 1),
                              "per_gpu_persons_per_s": round(value / world, 1),
                              "frac_of_burst_peak": round(step_tflops / world / peaks["tflops"], 4),
                              "frac_of_sustained_peak": round(step_tflops / world / peaks["tflops_sustained"], 4),
                              "gflop_per_person": cfg["gflop"]},
               "roofline": roofline, "layer_breakdown": breakdown, "cpu_baseline": cpu}
        if gather_check is not None:
            out["gather_check"] = gather_check
            # every rank's own device time per step: the reported step time is the slowest rank's (the ranks only meet in
            # the pipelined all-gather, so a spread here is GPU-to-GPU variation, not communication)
            out["ms_per_step_per_rank"] = per_rank_ms
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
