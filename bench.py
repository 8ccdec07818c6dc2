#!/usr/bin/env python
"""bench.py — MeshNet hot-path benchmark (BASELINE.json metric: SMPL meshes/sec at B=256 per B200).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--mode fwd|train] [--batch 256] [--precision fp16x3|fp32]
    python bench.py --impl reference ...     # the reference algorithm on the host cores (oracle port)
    python bench.py --elide-padding 0|1|2    # ablation of the padding-vertex elision (default: library default = 1)
    python bench.py --dump-outputs DIR       # also write the last timed step's outputs as DIR/<name>.npy
    torchrun --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Workload (BASELINE.json configs[1]): batch 256 synthetic H36M 17-joint poses [256,17,5] ~ N(0,1),
full coarse-to-fine MeshNet forward (eval mode, randomised BatchNorm running stats, random-init
weights under torch.manual_seed(123)) on a synthetic 6890-vertex genus-0 mesh whose hierarchy has the
real SMPL level sizes 12288/6144/.../96 (mesh seed 2; SMPL's topology is licence-gated, SURVEY F10).
One "step" = one forward over one batch of 256 poses per GPU; N GPUs = N independent shards of a
256*N batch (weak scaling, no data-path collective).  The same line carries a `train` object: the
training step of configs[2]/[4] at the same N — forward+backward with an L1 loss to random targets at
B=256 per GPU plus the single NCCL all-reduce of the flat gradient (the path's only exchange step,
SURVEY.md §8e), device-timed, max over ranks, with the all-reduce's own device time — so the driver's
1/2/4/8 runs also record the north-star multi-GPU configuration.  `--mode train` makes that step the
headline instead (and `--train-steps 0` skips the train object).

Printed JSON (one line, rank 0): see the task contract — `value` is device-timed whole-job meshes/s
with inputs resident in HBM; `e2e` is the same metric through the C-ABI host entry point
(p2m_meshnet_forward_host: pinned host poses in, host meshes out, copies inside the timed region);
`roofline` describes the dominant kernel (the V=12288, 128->128 Chebyshev conv) from CUDA-event
timings taken live; `cpu_baseline` is the CPU oracle on the host cores on a bounded sample.
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

import numpy as np  # noqa: E402
import torch  # noqa: E402

MESH = dict(n_vertex=6890, seed=2, levels=9)
WORKLOAD = "configs[1]: B=256 H36M-17 poses -> full MeshNet forward (eval), SMPL-size hierarchy 12288..96"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mode", default="fwd", choices=["fwd", "train"])
    ap.add_argument("--batch", type=int, default=256, help="poses per GPU per step")
    ap.add_argument("--precision", default="fp16x3", choices=["fp16x3", "fp32"])
    ap.add_argument("--cpu-sample", type=int, default=24, help="meshes in the cpu_baseline sample (0 = skip)")
    ap.add_argument("--no-graph", action="store_true", help="do not replay the forward from a CUDA graph")
    ap.add_argument("--elide-padding", type=int, default=-1, choices=[-1, 0, 1, 2],
                    help="ablation: p2m_debug_set_elide_padding level (-1 = library default)")
    ap.add_argument("--train-steps", type=int, default=5,
                    help="timed steps of the `train` object of a forward run (0 = skip it)")
    ap.add_argument("--ref-sample", type=int, default=32, help="--impl reference: meshes per step (bounded sample)")
    ap.add_argument("--mesh", default="smpl", choices=["smpl", "mano"],
                    help="smpl: 6890-vertex SMPL-size hierarchy (default, BASELINE configs[1,2,4]); "
                         "mano: 778-vertex MANO-size hierarchy 1088..68, 21 joints (configs[3], use --batch 1024)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (fwd: the meshes; "
                         "train: the loss and every parameter's gradient); at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(path, arrays):
    """--dump-outputs: one .npy per output array, float32 as computed.  The inputs are seeded, so two builds run with
    the same arguments can be compared file by file.  Above DUMP_BYTES in all, every array keeps the same share of its
    leading-axis rows (e.g. whole meshes), picked by a fixed seed."""
    os.makedirs(path, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    keep = min(1.0, DUMP_BYTES / max(total, 1))
    rng = np.random.default_rng(0)
    for name, a in arrays.items():
        if keep < 1.0 and a.ndim > 0:
            a = a[np.sort(rng.choice(a.shape[0], max(1, int(a.shape[0] * keep)), replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d["bf16_tflops"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        """Launch the sampler (nvidia-smi needs ~1 s to print its first line) and wait for the first sample."""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
            t0 = time.time()
            while not self.lines and time.time() - t0 < 5.0:
                time.sleep(0.02)
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def mark(self):
        self.t_begin = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        t_end = time.time()
        time.sleep(0.12)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        inside = [ln for (t, ln) in self.lines if getattr(self, "t_begin", 0) - 0.05 <= t <= t_end + 0.12]
        for ln in (inside or [ln for (_, ln) in self.lines[-3:]]):
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_problem(mesh="smpl"):
    from pose2mesh_release_b200 import graph as pg

    if mesh == "mano":
        face = pg.synthetic_sphere_faces(778, 1)
        _, graph_L, _, perm_rev = pg.build_coarse_graphs(face, 21, pg.MANO_SKELETON, pg.MANO_HORI_CONN, levels=6)
        return graph_L, perm_rev
    face = pg.synthetic_sphere_faces(MESH["n_vertex"], MESH["seed"])
    _, graph_L, _, perm_rev = pg.build_coarse_graphs(face, 17, pg.H36M_SKELETON, pg.H36M_FLIP_PAIRS,
                                                     levels=MESH["levels"])
    return graph_L, perm_rev


def randomize_bn_(sd, seed=7):
    g = torch.Generator().manual_seed(seed)
    for k in sorted(sd):
        if not k.startswith("bn."):
            continue
        t = sd[k]
        if k.endswith(".weight") or k.endswith(".running_var"):
            t.copy_(torch.rand(t.shape, generator=g) + 0.5)
        elif k.endswith(".bias") or k.endswith(".running_mean"):
            t.copy_(torch.randn(t.shape, generator=g) * 0.1)
    return sd


def best_thread_count(fn):
    """All host threads the port can USE: torch's CPU sparse / permute kernels slow down when
    oversubscribed (128 threads on this box run 2.5x slower than 8), so probe a few pool sizes on a tiny
    sample and keep the fastest.  Returns the chosen thread count (reported as `cores`)."""
    total = os.cpu_count() or 1
    best, best_t = total, None
    for n in sorted({min(total, c) for c in (8, 16, 32, 64, total)}):
        torch.set_num_threads(n)
        with torch.no_grad():
            fn()
            t0 = time.perf_counter()
            fn()
            dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best


def cpu_port_meshes_per_s(graph_L, sample, threads=None):
    """The reference algorithm on the host cores: the CPU oracle (a port; /root/reference does not
    exist on the GPU box).  Eval forward on `sample` meshes, 1 small warm-up + 1 timed pass."""
    from oracle import meshnet_oracle as mo

    laps = mo.laplacians_to_torch(graph_L)
    torch.manual_seed(123)
    sd = mo.randomize_bn_(mo.init_state_dict(5, 3, [m.shape[0] for m in laps], False), seed=7)
    g = torch.Generator().manual_seed(0)
    x = torch.randn(sample, 17, 5, generator=g)
    used = best_thread_count(lambda: mo.forward(sd, laps, x[:min(8, sample)], training=False))
    with torch.no_grad():
        mo.forward(sd, laps, x[:2], training=False)
        t0 = time.perf_counter()
        mo.forward(sd, laps, x, training=False)
        dt = time.perf_counter() - t0
    return sample / dt, dt, used


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (the oracle port: /root/reference does not
    exist on the GPU box) on the host threads it can use; each step is a bounded sample of the 256-pose batch.
    Nothing of the product is imported here — the hierarchy comes from oracle.graph_oracle — so that the arm's process
    never maps libp2m_b200.so."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import graph_oracle as go
    from oracle import meshnet_oracle as mo

    face = go.synthetic_sphere_faces(MESH["n_vertex"], MESH["seed"])
    _, graph_L, _, _ = go.build_coarse_graphs(face, 17, go.H36M_SKELETON, go.H36M_FLIP_PAIRS, levels=MESH["levels"])
    laps = mo.laplacians_to_torch(graph_L)
    torch.manual_seed(123)
    sd = mo.randomize_bn_(mo.init_state_dict(5, 3, [m.shape[0] for m in laps], False), seed=7)
    sample = max(1, min(args.ref_sample, args.batch))
    g = torch.Generator().manual_seed(1000)
    x = torch.randn(sample, 17, 5, generator=g)
    cores = best_thread_count(lambda: mo.forward(sd, laps, x[:min(8, sample)], training=False))
    with torch.no_grad():
        for _ in range(args.warmup):
            mo.forward(sd, laps, x[:2], training=False)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            mo.forward(sd, laps, x, training=False)
        dt = time.perf_counter() - t0
    v = sample * args.steps / dt
    assert not any("libp2m_b200" in ln for ln in open("/proc/self/maps")), "reference arm mapped the product library"
    line = {"impl": "reference", "metric": "SMPL meshes/sec", "value": v, "unit": "meshes/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "batch_per_gpu": args.batch, "global_batch": args.batch,
                       "mesh": "synthetic genus-0, 6890 verts, seed 2", "levels": [int(m.shape[0]) for m in graph_L],
                       "precision": "fp32 (torch CPU kernels)",
                       "sample": f"each step = {sample} of the {args.batch} meshes of a batch (bounded sample; the "
                                 "per-mesh cost of the eval forward does not depend on the batch size)"},
            "cpu_baseline": {"value": v, "unit": "meshes/s", "cores": cores, "kind": "port", "host_cores": os.cpu_count(),
                             "sample": f"{args.steps} x {sample} meshes, eval forward, CPU oracle (torch CPU kernels)"},
            "e2e": {"value": v, "unit": "meshes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


_REAL_STDOUT = None


def emit(line: dict):
    """The ONE JSON line of the contract goes to the real stdout; everything libraries print (NCCL's version
    banner, torch warnings) was diverted to stderr by capture_stdout()."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def capture_stdout():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def measure_train(model, x_host, dev, B, world, rank, steps, warmup, flush, barrier, outputs=None):
    """configs[2]/[4]: forward + backward (L1 loss to random targets, train-mode BatchNorm, B per GPU) + the single
    all-reduce of the flat gradient.  Device-timed per step (CUDA events), max over ranks; the all-reduce is also
    timed on its own (events around the collective: it runs after backward on the same stream, i.e. fully exposed).
    If `outputs` is a dict, it receives the last timed step's loss and reduced gradients (host float32 arrays)."""
    import torch.distributed as dist

    from pose2mesh_release_b200.dist import DataParallelStep

    model.train()
    dp = DataParallelStep(model)
    x = x_host.to(dev)
    tgt = torch.randn(B, model.num_vertices, 3, generator=torch.Generator().manual_seed(7 + rank)).to(dev)

    def launch(ev=None):
        dp.zero_grad()
        loss = (model(x) - tgt).abs().mean()
        loss.backward()
        if ev is not None:
            ev[0].record()
        dp.reduce_gradients()
        if ev is not None:
            ev[1].record()
        return loss

    for _ in range(max(warmup, 3)):
        launch()
    barrier()
    from pose2mesh_release_b200 import _lib

    _lib.load().p2m_launch_count_reset()
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(steps)]
    for i in range(steps):
        flush.zero_()
        evs[i][0].record()
        loss = launch(evs[i][2:])
        evs[i][1].record()
    barrier()
    launches = int(_lib.load().p2m_launch_count())
    if outputs is not None:
        outputs["loss"] = loss.detach().float().cpu().numpy()
        outputs.update({"grad." + k: p.grad.detach().float().cpu().numpy() for k, p in model.named_parameters()})
    step_ms = sum(e[0].elapsed_time(e[1]) for e in evs)
    ar_ms = sum(e[2].elapsed_time(e[3]) for e in evs)
    t = torch.tensor([step_ms, ar_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    step_ms, ar_ms = float(t[0].item()) / steps, float(t[1].item()) / steps
    # end to end: host poses in, host loss out, wall clock
    t0 = time.perf_counter()
    for _ in range(steps):
        xs = x_host.to(dev, non_blocking=True)
        dp.zero_grad()
        loss = (model(xs) - tgt).abs().mean()
        loss.backward()
        dp.reduce_gradients()
        loss.item()
    dt = time.perf_counter() - t0
    tt = torch.tensor([dt], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    grad_bytes = int(dp.flat.grad.numel() * 4)
    return {"metric": "SMPL meshes/sec (fwd+bwd train step, one gradient all-reduce)", "value": B * world / (step_ms * 1e-3),
            "unit": "meshes/s", "ms_per_step": step_ms, "steps": steps, "batch_per_gpu": B, "global_batch": B * world,
            "gpu_launches": launches, "gpu_launches_per_step": launches // max(steps, 1),
            "allreduce_ms": ar_ms if world > 1 else 0.0, "allreduce_bytes": grad_bytes if world > 1 else 0,
            "allreduce": (f"one NCCL all_reduce(SUM) of the flat fp32 gradient ({grad_bytes / 1e6:.1f} MB) + 1/world scale per "
                          "step, issued after backward on the same stream (exposed time = allreduce_ms)") if world > 1
                         else "single GPU: no collective",
            "allreduce_busbw_GBps": (2.0 * (world - 1) / world * grad_bytes / (ar_ms * 1e-3) * 1e-9) if world > 1 and ar_ms > 0 else None,
            "e2e": {"value": B * world * steps / float(tt.item()), "unit": "meshes/s",
                    "h2d_bytes_per_step": int(x_host.numel() * 4), "d2h_bytes_per_step": 4}}


def main():
    args = parse()
    capture_stdout()
    if args.impl == "reference":
        return run_reference(args)

    import torch.distributed as dist

    from pose2mesh_release_b200 import _lib
    from pose2mesh_release_b200.meshnet import Pose2Mesh

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU port")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"   # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()

    graph_L, perm_rev = build_problem(args.mesh)
    n_joint = 21 if args.mesh == "mano" else 17
    torch.manual_seed(123)
    model = Pose2Mesh(5, 3, graph_L, joint_set="mano" if args.mesh == "mano" else "human36")
    model.load_state_dict(randomize_bn_({k: v.clone() for k, v in model.state_dict().items()}))
    model = model.to(dev).set_precision(args.precision)
    if args.elide_padding >= 0:
        model._hier.set_debug(local, elide_padding=args.elide_padding)
    B = args.batch
    g = torch.Generator().manual_seed(1000 + rank)
    x_host = torch.randn(B, n_joint, 5, generator=g).pin_memory()
    x = x_host.to(dev)
    hbm_gbs, bf16_tf, peak_src = measured_peaks()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if args.mode == "train":
        # the training step as the headline (profiles/: bench.py --mode train)
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
            sampler.mark()
        outputs = {} if args.dump_outputs and rank == 0 else None
        tr = measure_train(model, x_host, dev, B, world, rank, args.steps, args.warmup, flush, barrier, outputs)
        clocks = sampler.stop() if rank == 0 else None
        if rank == 0:
            emit({"metric": "SMPL meshes/sec (fwd+bwd train step)", "value": tr["value"], "unit": "meshes/s", "n_gpus": world,
                  "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": tr["ms_per_step"],
                  "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                  "dtype": "f32 (tcgen05 fp16x3 split, fp32 accumulate)" if args.precision == "fp16x3" else "f32",
                  "data": "synthetic",
                  "config": {"workload": "configs[2]/[4]: B=256/GPU fwd+bwd, L1 loss, train-mode BatchNorm, one NCCL "
                                         "all-reduce of the flat gradient" if args.mesh == "smpl" else
                                         "configs[3]: MANO-size hierarchy 1088..68, 21 joints, forward+backward, L1 loss",
                             "batch_per_gpu": B, "global_batch": B * world, "levels": [int(m.shape[0]) for m in graph_L],
                             "precision": args.precision, "parallelism": f"dp{world} (single all-reduce per step)",
                             "l2": "256 MiB buffer written between timed iterations (outside the event pairs)"},
                  "e2e": tr["e2e"], "gpu_launches": tr["gpu_launches"], "gpu_launches_per_step": tr["gpu_launches_per_step"],
                  "clocks": clocks, "train": tr})
            if outputs is not None:
                dump_outputs(args.dump_outputs, outputs)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    step_graph = None
    model.eval()

    def step():
        with torch.no_grad():
            return model(x)

    launch, y_static = step, None
    if not args.no_graph:
        # replay the ~100-launch forward from a CUDA graph (the library only enqueues on the current stream)
        try:
            side = torch.cuda.Stream()
            with torch.cuda.stream(side):
                step()
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                y_static = step()  # the graph's output tensor: every replay rewrites it
            torch.cuda.synchronize()
            step_graph, launch = graph, graph.replay
        except Exception as e:  # keep the bench alive; say so in the JSON
            sys.stderr.write(f"[bench] CUDA graph capture failed ({e}); running eagerly\n")
            torch.cuda.synchronize()
            step_graph, launch = None, step

    for _ in range(max(args.warmup, 3)):
        launch()
    barrier()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    lib.p2m_launch_count_reset()
    barrier()
    sampler.mark()
    for i in range(args.steps):
        flush.zero_()               # evict L2 between timed iterations (not timed)
        evs[i][0].record()
        y_last = launch()
        evs[i][1].record()
    barrier()
    launches_eager = lib.p2m_launch_count()
    clocks = sampler.stop() if rank == 0 else None
    outputs = None
    if args.dump_outputs and rank == 0:
        outputs = {"meshes": (y_static if step_graph is not None else y_last).float().cpu().numpy()}
    total_ms = sum(a.elapsed_time(b) for a, b in evs)
    t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    value = B * world * args.steps / (total_ms * 1e-3)

    # kernel launches per step: counted by the library while the step was captured / run eagerly
    if step_graph is not None:
        lib.p2m_launch_count_reset()
        with torch.no_grad():
            model(x)
        torch.cuda.synchronize()
        per_step_launches = lib.p2m_launch_count()
    else:
        per_step_launches = launches_eager // max(args.steps, 1)

    # ---- end to end through the C-ABI host entry point, wall clock: pinned host poses in, host vertices out.  The call
    # is p2m_meshnet_forward_vertices_host: the callers' gather pred[:, perm_reverse[:6890]] (lib/core/base.py:130,201)
    # is fused into the head layer, so what travels back is what the reference's callers keep of a mesh.
    n_real = MESH["n_vertex"] if args.mesh == "smpl" else 778
    y_host = torch.empty((B, n_real, 3), dtype=torch.float32).pin_memory()
    for _ in range(2):
        model.forward_host(x_host, out=y_host, perm_reverse=perm_rev, n_vertex=n_real)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        model.forward_host(x_host, out=y_host, perm_reverse=perm_rev, n_vertex=n_real)   # synchronises its stream
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    tt = torch.tensor([dt], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    e2e = {"value": B * world * args.steps / float(tt.item()), "unit": "meshes/s",
           "h2d_bytes_per_step": int(x_host.numel() * 4), "d2h_bytes_per_step": int(y_host.numel() * 4),
           "call": "p2m_meshnet_forward_vertices_host (fused perm_reverse gather: [B, 6890, 3] back to the host)"}

    # ---- roofline of the dominant kernel: per-layer CUDA events inside the eval forward
    roofline, layers = None, None
    if rank == 0:
        model.eval()
        hier = model._hier
        hier.set_profiling(local, True)
        info = hier.layer_info(local)
        acc = np.zeros(len(info))
        reps = 5
        with torch.no_grad():
            for _ in range(reps):
                flush.zero_()
                model(x)
                acc += np.array(hier.layer_times_ms(local))
        hier.set_profiling(local, False)
        acc /= reps
        layers = []
        for li, (d, ms) in enumerate(zip(info, acc)):
            byt = 4.0 * d["V"] * (d["fin"] + d["fout"]) * B
            fl = (2.0 * d["V"] * 3 * d["fin"] * d["fout"]) * B
            layers.append({"layer": li, "V": d["V"], "fin": d["fin"], "fout": d["fout"], "ms": round(float(ms), 4),
                           "GBps": round(byt / ms * 1e-6, 1), "TFLOPs": round(fl / ms * 1e-9, 1)})
        dom = [i for i, d in enumerate(info) if d["V"] == info[-1]["V"] and d["fin"] == 128 and d["fout"] == 128]
        nnz0 = int(graph_L[0].nnz)
        if dom:
            ms = float(np.mean([acc[i] for i in dom]))
            d = info[dom[0]]
            byt = 4.0 * d["V"] * (d["fin"] + d["fout"]) * B          # SURVEY §8(d): 4*V*(Fin+Fout) per mesh
            fl = (2.0 * d["V"] * 3 * d["fin"] * d["fout"] + 2.0 * (2 * nnz0 * d["fin"]) + 2.0 * d["V"] * d["fin"]) * B
            ach = byt / (ms * 1e-3) * 1e-9
            traffic, traffic_src = None, None
            tpath = os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")
            if os.path.exists(tpath) and args.precision == "fp16x3":
                with open(tpath) as fh:
                    tj = json.load(fh)
                if (tj["V"], tj["fin"], tj["fout"]) == (d["V"], d["fin"], d["fout"]):
                    traffic = tj["layer_dram_bytes"] * B / tj["batch"]   # DRAM bytes scale with the batch
                    traffic_src = tj["source"] + "; T1 pass + conv kernel + plain GEMM of one layer"
            roofline = {"bound": "hbm", "kernel": f"cheb conv V={d['V']} {d['fin']}->{d['fout']} K=3 (layers {dom}): "
                                                  "k_cheb_t1 + k_cheb_conv_umma<128,3,2> (connected rows) + its plain-GEMM "
                                                  "mode (representatives of the isolated rows)",
                        "achieved": ach, "peak": hbm_gbs, "unit": "GB/s", "frac": ach / hbm_gbs, "traffic": traffic,
                        "traffic_source": traffic_src,
                        "ms_per_launch": ms, "algorithmic_bytes": byt, "algorithmic_flops": fl,
                        "tensor_TFLOPs": fl / (ms * 1e-3) * 1e-12, "tensor_frac_of_bf16_peak": fl / (ms * 1e-3) * 1e-12 / bf16_tf,
                        "peak_source": peak_src,
                        "note": "achieved = SURVEY 8(d) algorithmic bytes 4*V*(Fin+Fout)*B with the padded V the reference "
                                "computes / measured layer time (CUDA events inside the library, mean of the layers listed; "
                                "includes the weight pack launches, <1%); the eval forward computes each class of identical "
                                "isolated (padding) rows once, see DESIGN.md 4.1; precision " + args.precision}

    cpu_baseline = None
    if rank == 0 and args.cpu_sample > 0 and args.mode == "fwd" and args.mesh == "smpl":
        v, dt, used = cpu_port_meshes_per_s(graph_L, args.cpu_sample)
        cpu_baseline = {"value": v, "unit": "meshes/s", "cores": used, "kind": "port", "host_cores": os.cpu_count(),
                        "sample": f"{args.cpu_sample} meshes, eval forward, CPU oracle (torch CPU kernels), {dt:.1f} s; "
                                  f"thread count = fastest of 8/16/32/64/all"}

    used_graph = step_graph is not None
    train = None
    if args.train_steps > 0 and args.mesh == "smpl":
        del step_graph, launch
        train = measure_train(model, x_host, dev, B, world, rank, args.train_steps, 3, flush, barrier)

    if rank == 0:
        line = {
            "metric": "SMPL meshes/sec" if args.mode == "fwd" else "SMPL meshes/sec (fwd+bwd train step)",
            "value": value, "unit": "meshes/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 (tcgen05 fp16x3 split, fp32 accumulate)" if args.precision == "fp16x3" else "f32",
            "data": "synthetic",
            "config": {"workload": ("configs[3]: MANO-size hierarchy 1088..68 (778 verts), 21 joints, "
                                    + ("forward (eval)" if args.mode == "fwd" else "forward+backward, L1 loss"))
                       if args.mesh == "mano" else WORKLOAD if args.mode == "fwd" else
                       "configs[2]/[4]: B=256/GPU fwd+bwd, L1 loss, train-mode BatchNorm, one NCCL all-reduce of the flat gradient",
                       "batch_per_gpu": B, "global_batch": B * world,
                       "mesh": "synthetic genus-0, 778 verts, seed 1 (MANO-size)" if args.mesh == "mano"
                       else "synthetic genus-0, 6890 verts, seed 2",
                       "levels": [int(m.shape[0]) for m in graph_L], "precision": args.precision,
                       "parallelism": f"dp{world} (independent shards, no data-path collective)" if args.mode == "fwd"
                       else f"dp{world} (single all-reduce per step)",
                       "l2": "256 MiB buffer written between timed iterations (outside the event pairs)",
                       "cuda_graph": used_graph},
            "e2e": e2e, "gpu_launches": int(per_step_launches * args.steps), "gpu_launches_per_step": int(per_step_launches),
            "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu_baseline, "train": train, "layers": layers,
        }
        emit(line)
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
