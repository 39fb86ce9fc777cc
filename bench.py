#!/usr/bin/env python
"""bench.py — DDPM 256x256 denoising steps/sec @ 1.2 % edit (BASELINE.json metric), B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|reference-cuda] [--ratio 0.012]
                    [--path fused|modules] [--no-flush] [--dump-outputs DIR]

One "step" = one SPARSE forward of the DDPM U-Net on the edited latent with pre-filled caches —
what the reference's Runner.profile times (reference diffusion/runner.py:214-245).  Workload =
BASELINE.json configs[1]: DDPM 256x256, 1.2 % centred-square edit, random-init (deterministic)
weights, synthetic inputs, fp16.

Multi-GPU (⑤): independent edits, one per GPU (weak scaling).  Rank 0 runs the dense pass on the
original image; its caches are sent ONCE with NCCL broadcast before the step loop; there is no
collective on the per-step path.  value = edits-steps/s summed over ranks, time = max over ranks.

Timing: W untimed steps, then K timed steps, each bracketed by CUDA events on the launching
stream, with an L2 flush (256 MiB write) between steps outside the event brackets; the whole
region sits between barrier + synchronize.  e2e = the same step through the public API with
host buffers: pinned H2D copy of x_t and D2H copy of eps inside every timed step.

Our arm drives the reference's UNMODIFIED model file (baseline/_ref/diffusion/models/ddpm_arch/sige_fused_unet.py, a
verbatim copy made by baseline/build_ref.py) on this repository's `sige` package through its public call
`model(x, t)`; in sparse mode SIGEModel runs that forward as a fused step (sige_b200.fused).  When baseline/_ref did
not travel, the in-tree restatement of the same architecture (sige_b200.workloads.ddpm) is used and
`config.model_file` says so.

--impl reference: the reference itself — its python package, its sige.cpu OpenMP kernels + oneDNN conv — on this
box's host cores (baseline/run_reference.py in a child process), rank 0 only.
--impl reference-cuda: the reference itself on the SAME GPU — its python package, its sige.cuda kernels recompiled for
sm_100a + cuDNN, fp32 — i.e. what a user of the reference gets on a B200 today.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)


_T0 = time.time()


def log(msg):
    sys.stderr.write("[bench %7.1fs] %s\n" % (time.time() - _T0, msg))
    sys.stderr.flush()


def _env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-cuda"])
    ap.add_argument("--ratio", type=float, default=0.012)
    ap.add_argument("--workload", default="ddpm", choices=["ddpm", "sd", "gaugan"],
                    help="ddpm = BASELINE.json's metric (default).  sd / gaugan = the reference's secondary consumers at full size "
                         "(configs[2]: SD v1 U-Net, 64x64 latent, B = 2, 15 %% mask; configs[3]: SPADE generator 512x1024, 3 %% label edit), "
                         "the reference's own unmodified model files on this repo's sige.nn: a secondary line, one GPU")
    ap.add_argument("--edits", type=int, default=1, help="independent edits of the same original image per GPU, batched in one fused step "
                                                         "(each with its own mask; weights are read once per step)")
    ap.add_argument("--total-edits", type=int, default=0, help="BASELINE.json configs[4]: a FIXED batch of edits sharded over the GPUs "
                                                               "(strong scaling); overrides --edits with total/world per GPU")
    ap.add_argument("--dtype", default="fp16", choices=["fp16", "bf16"])
    ap.add_argument("--path", default="fused", choices=["fused", "modules"],
                    help="fused = model(x, t) as a traced, fused, graph-captured step (the default behaviour of SIGEModel); "
                         "modules = the eager sige.nn operator modules, graph-captured")
    ap.add_argument("--model", default="auto", choices=["auto", "reference", "intree"],
                    help="reference = the reference's unmodified model file from baseline/_ref on this repo's sige.nn; "
                         "intree = sige_b200.workloads.ddpm (same architecture, same weights)")
    ap.add_argument("--no-flush", action="store_true", help="do not flush L2 between timed steps")
    ap.add_argument("--cpu-steps", type=int, default=20, help="timed steps of the cpu_baseline leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-reference-cuda", action="store_true", help="skip the reference's own CUDA path (sige.cuda for sm_100a + cuDNN) timed beside ours on GPU 0")
    ap.add_argument("--threads", type=int, default=0, help="(reference arm) torch/OpenMP threads; 0 = sweep")
    ap.add_argument("--_cpu-child", dest="_cpu_child", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--no-tc5", action="store_true", help="engine: use the mma.sync kernel everywhere (default: tcgen05/TMEM/TMA kernel where the geometry allows)")
    ap.add_argument("--no-producer-preop", action="store_true", help="engine: apply GroupNorm affine + SiLU in every gather (reference order) instead of once in the producer's epilogue")
    ap.add_argument("--dense-stem", action="store_true", help="engine: evaluate conv_in on the whole image even when only the active tiles are read")
    ap.add_argument("--no-fused-attention", action="store_true", help="engine: torch matmul/softmax instead of the fused attention-core kernel")
    ap.add_argument("--no-fuse-shortcut", action="store_true", help="engine: keep the 1x1 shortcut convs as separate launches")
    ap.add_argument("--no-pdl", action="store_true", help="engine: plain stream order between fused layers (default: programmatic dependent launch)")
    ap.add_argument("--ksplit", type=int, default=0, help="engine: force the split-K factor (0 = auto)")
    ap.add_argument("--no-graph", action="store_true", help="launch the step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--ncu", action="store_true",
                    help="profiling aid: after warm-up run one eager step between cudaProfilerStart/Stop and exit "
                         "(use with `ncu --profile-from-start off`); prints no bench line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned to its caller as DIR/<name>.npy (float32, "
                         "at most 64 MB in all: a larger output is cut to a fixed, seeded sample); the inputs are seeded, so two "
                         "builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes this repository's outputs (--impl ours)")
    if args.dump_outputs and args.ncu:
        ap.error("--ncu runs no timed steps: there is nothing for --dump-outputs to write")
    return args


def dump_outputs(directory, arrays, limit=64 * 10 ** 6):
    """Write each array as directory/<name>.npy in float32.  When the arrays together exceed `limit` bytes, each one is
    replaced by the same fixed, seeded sample of its flattened elements (in index order), in proportion to its size."""
    import numpy as np

    os.makedirs(directory, exist_ok=True)
    arrays = {k: np.ascontiguousarray(v, dtype=np.float32) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > limit:
            keep = a.size * (limit - 4096 * len(arrays)) // total
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(directory, name + ".npy"), a)
    log("outputs of the last timed step written to %s: %s" % (directory, ", ".join(sorted(arrays))))


# ------------------------------------------------------------------------------------------
# clocks sampling (NVML) during the timed region
# ------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.interval = float(os.environ.get("SIGE_BENCH_SAMPLE_S", "0.01"))       # NVML polling period
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:  # noqa: BLE001
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
            "hw_power_brake": getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80),
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(self.interval)

    def start(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()

    def stop(self):
        self._stop.set()
        if self._thr is not None:
            self._thr.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------
# reference arm / cpu baseline (oracle/ is imported ONLY here)
# ------------------------------------------------------------------------------------------
def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001
        return os.cpu_count() or 1


def _reference_child(backend: str, ratio: float, steps: int, warmup: int, threads: int, timeout: float, extra=()):
    """One run of baseline/run_reference.py (the reference's own python + native backend) in a clean child process."""
    import subprocess

    sys.path.insert(0, os.path.join(REPO, "baseline"))
    import loader

    env = loader.reference_env(threads)
    if backend == "cpu":
        env["CUDA_VISIBLE_DEVICES"] = ""
        if host_cores() > 32:   # many-core host: keep torch's and the reference kernels' OpenMP runtimes from spinning against each other
            env.update(OMP_WAIT_POLICY="PASSIVE", GOMP_SPINCOUNT="0")
    cmd = [sys.executable, os.path.join(REPO, "baseline", "run_reference.py"), "--backend", backend, "--steps", str(steps), "--warmup", str(warmup),
           "--ratio", str(ratio)] + (["--threads", str(threads)] if threads else []) + list(extra)
    out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=timeout)
    if out.returncode != 0:
        raise RuntimeError("reference child failed: %s" % out.stderr.strip().splitlines()[-1:] )
    return json.loads(out.stdout.strip().splitlines()[-1])


def cpu_reference_legacy(ratio: float, steps: int, warmup: int, threads: int):
    """Fallback when baseline/_ref did not travel: the in-tree model graph on the reference's CPU kernels (oracle/_ref)
    or the oracle port, in THIS process (call from a process that has not touched CUDA)."""
    import torch

    from oracle.cpu_runtime import ddpm_cpu_sparse_step
    from sige_b200.workloads.ddpm import DDPMConfig

    step, kind = ddpm_cpu_sparse_step(DDPMConfig(), ratio, threads=threads or host_cores())
    try:
        for _ in range(warmup):
            step()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        dt = time.perf_counter() - t0
    finally:
        step.close()
    return {"steps_per_s": steps / dt, "ms_per_step": 1e3 * dt / steps, "threads": torch.get_num_threads(), "kind": kind}


def cpu_reference_subprocess(ratio: float, steps: int, warmup: int, timeout: int = 170, threads: int = 0):
    """The reference's CPU flow on this box's host cores: a short thread sweep (all host cores is not the fastest on a
    100+-core host for this small workload), then the winning count re-timed on the full `steps`."""
    sys.path.insert(0, os.path.join(REPO, "baseline"))
    import loader

    cores = host_cores()
    budget = time.time() + timeout
    if not loader.available():
        import subprocess

        env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--_cpu-child", "--threads", str(threads or min(cores, 32)),
                              "--steps", str(steps), "--warmup", str(warmup), "--ratio", str(ratio)], env=env, capture_output=True, text=True, timeout=timeout)
        r = json.loads(out.stdout.strip().splitlines()[-1])
        return {"value": r["steps_per_s"], "unit": "steps/s", "cores": r["threads"], "host_cores": cores, "kind": r["kind"] if r["kind"] == "port" else "reference",
                "timed_steps": steps, "ms_per_step": r["ms_per_step"],
                "sample": "%d sparse DDPM-256 steps @%.1f%% edit, in-tree model graph on %s + oneDNN conv, fp32 (baseline/_ref absent)" % (steps, 100 * ratio, r["kind"])}
    cands = [threads] if threads else sorted({c for c in (cores, 64, 32, 16, 8) if c <= cores}, reverse=True)
    tried, best_t, best_v = [], None, 0.0
    for th in cands:
        if len(cands) == 1:
            best_t = th
            break
        left = budget - time.time()
        if left < 40:
            break
        try:
            r = _reference_child("cpu", ratio, max(3, steps // 4), 1, th, min(left - 20, 60))
        except Exception as e:  # noqa: BLE001
            tried.append({"threads": th, "error": type(e).__name__})
            continue
        tried.append({"threads": th, "steps_per_s": r["steps_per_s"]})
        if r["steps_per_s"] > best_v:
            best_t, best_v = th, r["steps_per_s"]
    if best_t is None:
        raise RuntimeError("cpu reference leg failed: %r" % (tried,))
    r = _reference_child("cpu", ratio, steps, warmup, best_t, max(30.0, budget - time.time()))
    return {"value": r["steps_per_s"], "unit": "steps/s", "cores": r["threads"], "host_cores": cores, "kind": "reference", "timed_steps": r["steps"],
            "warmup": r["warmup"], "ms_per_step": r["ms_per_step"], "thread_sweep": tried,
            "sample": "%d sparse DDPM-256 steps @%.1f%% edit after %d warm-up: the reference's own python (sige.nn, sige_fused_unet.py) + its sige.cpu "
                      "OpenMP kernels + oneDNN conv, fp32, %d threads (best of the sweep)" % (r["steps"], 100 * ratio, r["warmup"], r["threads"])}


def workload_name(ratio: float) -> str:
    """The same workload label on every arm (BASELINE.json configs[1] at the default ratio)."""
    return ("DDPM U-Net 256x256 (ch128, mult 1-1-2-2-4-4), %.1f%% centred-square edit (%d px), sparse step, random-init weights"
            % (100 * ratio, int(round((ratio ** 0.5) * 256))))


def run_reference(args):
    rank = _env_int("RANK", 0)
    if rank != 0:
        return
    if args._cpu_child:
        print(json.dumps(cpu_reference_legacy(args.ratio, max(1, args.steps), max(1, args.warmup), args.threads)), flush=True)
        return
    warm = max(1, min(args.warmup, 5))
    # the time limit grows with --steps (a few seconds per step is ample for the host-core flow), so every step asked for is timed
    r = cpu_reference_subprocess(args.ratio, args.steps, warm, timeout=170 + 5 * args.steps, threads=args.threads)
    line = {
        "impl": "reference", "metric": "DDPM 256x256 denoising steps/sec @1.2% edit", "value": r["value"], "unit": "steps/s",
        "n_gpus": args.gpus, "steps": r["timed_steps"], "warmup": r.get("warmup", warm), "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.ratio), "device": "cpu",
                   "edits_per_gpu": 0, "parallelism": "the reference's CPU flow on the host cores (rank 0 only)"},
        "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "host_cores", "kind", "sample", "thread_sweep") if k in r},
        "e2e": {"value": r["value"], "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_reference_cuda(args):
    """The reference's own CUDA path (sige.cuda for sm_100a + cuDNN, fp32, its unmodified python) on GPU 0 of this box."""
    rank = _env_int("RANK", 0)
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(REPO, "baseline"))
    import loader

    if not loader.available(cuda=True):
        print(json.dumps({"impl": "reference-cuda", "unavailable": "baseline/_ref/sige/cuda.so absent (run baseline/build_ref.py where /root/reference exists)"}), flush=True)
        return
    steps, warm = max(1, args.steps), max(3, args.warmup)
    r = _reference_child("cuda", args.ratio, steps, warm, 0, 600)
    line = {
        "impl": "reference-cuda", "metric": "DDPM 256x256 denoising steps/sec @1.2% edit", "value": r["steps_per_s"], "unit": "steps/s",
        "n_gpus": 1, "steps": r["steps"], "warmup": r["warmup"], "ms_per_step": r["ms_per_step"], "device_ms_per_step": r["device_ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (cuDNN TF32 allowed: %s — torch default)" % r["tf32"], "data": "synthetic",
        "config": {"workload": workload_name(args.ratio), "device": r["gpu"], "path": "reference sige.nn + sige.cuda (sm_100a rebuild) + cuDNN, eager, NCHW",
                   "timing": "the reference's Runner.profile protocol: synchronize after every forward, wall clock"},
        "e2e": {"value": r["steps_per_s"], "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------
def build_model(cfg, which: str):
    """(model, label): the reference's unmodified model file on this repo's sige.nn when baseline/_ref is present."""
    import warnings

    from sige_b200.workloads.ddpm import SIGEDDPMUNet, init_deterministic

    sys.path.insert(0, os.path.join(REPO, "baseline"))
    import loader

    use_ref = which == "reference" or (which == "auto" and loader.available())
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        if use_ref:
            model = loader.reference_ddpm_on_this_repo(cfg)
            label = "baseline/_ref/diffusion/models/ddpm_arch/sige_fused_unet.py (the reference's file, unmodified) on this repo's sige.nn"
        else:
            model = SIGEDDPMUNet(cfg)
            label = "sige_b200/workloads/ddpm.py (in-tree restatement of the same architecture; baseline/_ref absent)"
        model = init_deterministic(model, seed=0).eval()
    return model, label


def run_ours(args):
    import torch
    import torch.distributed as dist

    from sige_b200 import ops
    from sige_b200.masks import downsample_mask
    from sige_b200.workloads.ddpm import DDPMConfig, synthetic_inputs

    rank, world, local = _env_int("RANK", 0), _env_int("WORLD_SIZE", 1), _env_int("LOCAL_RANK", 0)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    distributed = world > 1
    if distributed:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    dtype = torch.float16 if args.dtype == "fp16" else torch.bfloat16
    cfg = DDPMConfig()
    torch.backends.cudnn.benchmark = True

    path = args.path
    model, model_label = build_model(cfg, args.model if path == "fused" else "intree")
    # fused: the reference's own flow — fp32 model, fp32 dense pass on the original image (untimed, as in the reference's
    # Runner.profile) — with the sparse steps on the fp16/bf16 tensor-core path (set_fused(dtype=...)).
    # modules: a half, channels-last model through the eager operator modules (in-tree model only: the reference's model
    # file computes its time embedding in fp32 and cannot run its dense pass in half).
    io_dtype = torch.float32 if path == "fused" else dtype
    model = model.to(dev).to(io_dtype)
    if path != "fused":
        model = model.to(memory_format=torch.channels_last)
    # every rank edits the SAME original image with its OWN edits (edit seed = global edit number; edits after the first of a
    # rank are moved to other places of the image so that the batch does not share tiles)
    n_edits = args.edits
    if args.total_edits:
        if args.total_edits % world:
            raise SystemExit("--total-edits must be a multiple of the number of GPUs")
        n_edits = args.total_edits // world
    if n_edits > 1 and path != "fused":
        raise SystemExit("a batch of independent edits runs as a fused step only")
    x0 = None
    edit_x, edit_masks = [], []
    for e in range(n_edits):
        ge = rank * n_edits + e
        x0, x1e, mask_e, t = synthetic_inputs(cfg, args.ratio, seed=0, edit_seed=ge)
        if e > 0:
            g = torch.Generator().manual_seed(1000 + ge)
            shift = tuple(int(v) for v in torch.randint(-96, 97, (2,), generator=g))
            mask_e = torch.roll(mask_e, shift, (0, 1))
            x1e = x0 + torch.roll(x1e - x0, shift, (2, 3))
        edit_x.append(x1e)
        edit_masks.append(mask_e)
    x1 = torch.cat(edit_x, 0)
    x0d = x0.to(dev).to(io_dtype)
    td = t.to(dev)

    log("model built (%s); dense pass on the original image" % model_label)
    with torch.no_grad():
        model.set_mode("full")
        model(x0d, td)                       # every rank records shapes; rank 0's caches are authoritative
        if distributed:
            from sige_b200.parallel import broadcast_caches

            torch.cuda.synchronize()
            t_b = time.perf_counter()
            nbytes = broadcast_caches(model, src=0)
            torch.cuda.synchronize()
            bcast_ms = 1e3 * (time.perf_counter() - t_b)     # one-off, outside the per-step path: reported, not part of `value`
        else:
            nbytes, bcast_ms = 0, 0.0
        if n_edits == 1:
            model.set_masks(downsample_mask(edit_masks[0].to(dev), min_res=8))
        else:
            from sige_b200.masks import stack_mask_pyramids

            model.set_masks(stack_mask_pyramids([downsample_mask(m.to(dev), min_res=8) for m in edit_masks]))
        model.set_mode("sparse")

    log("masks set; building the step (path=%s, %d edit(s) per GPU)" % (path, n_edits))
    x_host = x1.to(io_dtype).contiguous().pin_memory()
    x_dev = x_host.to(dev)
    out_host = torch.empty((n_edits, cfg.out_ch, cfg.image_size, cfg.image_size), dtype=io_dtype).pin_memory()
    use_graph = not (args.no_graph or args.ncu)

    if path == "fused":
        model.set_fused(True, dtype=dtype, use_graph=use_graph, pdl=not args.no_pdl, ksplit=args.ksplit, tc5=not args.no_tc5, producer_preop=not args.no_producer_preop,
                        fuse_shortcut=not args.no_fuse_shortcut, fused_attention=not args.no_fused_attention, sparse_stem=not args.dense_stem)
        with torch.no_grad():
            model(x_dev, td)                 # first sparse call: trace -> lower -> capture
        runner = model.fused_step
        if runner is None:
            raise SystemExit("bench.py: the model did not run as a fused step")
        log("fused step: %d fused conv launches, %d steps, eager nodes: %s" % (len(runner.fused), len(runner.steps), runner.eager_nodes or "none"))

        def step(x):
            return model(x, td)              # the public call: copy-in, graph replay, copy-out
    else:
        from sige_b200.graphs import GraphedStep

        model.set_fused(False)
        runner = GraphedStep(model, x_dev, td, use_graph=use_graph)

        def step(x):
            if x is not runner.x:
                runner.x.copy_(x, non_blocking=True)
            return runner.replay()
    launches_per_step = runner.launches_per_step

    flush = None if args.no_flush else torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream()

    if args.ncu:
        with torch.no_grad():
            for _ in range(max(3, args.warmup)):
                step(x_dev)
            torch.cuda.synchronize()
            torch.cuda.profiler.start()
            if flush is not None:
                flush.fill_(1)
            step(x_dev)                      # one step is the unit of every committed capture; ncu replays each kernel ~40 times under --set full
            torch.cuda.synchronize()
            torch.cuda.profiler.stop()
        log("profiled 1 eager step (%d launches of our kernels per step)" % launches_per_step)
        return

    def timed_steps(k, e2e):
        total = 0.0
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(k)]
        with torch.no_grad():
            for i in range(k):
                if flush is not None:
                    flush.fill_(i & 0xFF)
                evs[i][0].record(stream)
                if e2e:
                    x = x_host.to(dev, non_blocking=True)       # this step's input arrives from pinned host memory
                    out = step(x)
                    out_host.copy_(out, non_blocking=True)      # ... and its result goes back
                else:
                    out = step(x_dev)
                evs[i][1].record(stream)
                if e2e:
                    evs[i][1].synchronize()      # the caller consumes eps before issuing the next step
        torch.cuda.synchronize()
        for a, b in evs:
            total += a.elapsed_time(b)
        return total                         # milliseconds of device time over k steps

    def region(k, e2e):
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()
        ms = timed_steps(k, e2e)
        torch.cuda.synchronize()
        if distributed:
            tt = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms = float(tt.item())
            dist.barrier()
        return ms

    log("runner ready: %d launches of our kernels per step; warm-up" % launches_per_step)
    region(max(3, args.warmup), False)
    log("timing %d steps (device-resident), then %d steps end-to-end" % (args.steps, args.steps))
    sampler = ClockSampler(local)
    sampler.start()
    ms = region(args.steps, False)
    ms_e2e = region(args.steps, True)
    clocks = sampler.stop()
    if args.dump_outputs:
        # out_host holds eps of the last end-to-end step: what a caller of the public call receives
        dump_outputs(args.dump_outputs, {"eps" if world == 1 else "eps_rank%d" % rank: out_host.numpy()}, limit=64 * 10 ** 6 // world)

    value = world * n_edits * args.steps / (ms / 1e3)            # denoising steps of ONE edit per second, summed over edits and GPUs
    e2e_value = world * n_edits * args.steps / (ms_e2e / 1e3)

    log("timed: %.3f ms/step resident, %.3f ms/step e2e; roofline + cpu baseline" % (ms / args.steps, ms_e2e / args.steps))
    roof = None
    cpu = None
    if rank == 0:
        try:
            from sige_b200 import roofline

            if path == "fused":
                fused_opts = dict(model.__dict__.get("_fused_options", {}))
                roof = roofline.measure_in_graph(model, (x_dev, td), fused_opts, flush)
                iso = roofline.measure_engine(runner, flush)          # the same launches one at a time, cold L2, launch latency included
                roof["isolated_cold"] = {k: iso[k] for k in ("achieved", "frac", "avg_launch_us", "note")}
            else:
                roof = roofline.measure_dominant_kernel(model, dtype, flush)
        except Exception as e:  # noqa: BLE001
            import traceback

            roof = {"error": repr(e), "trace": traceback.format_exc()[-1500:]}
        log("roofline done")
        ref_cuda = None
        if world == 1 and n_edits == 1 and not args.no_reference_cuda:
            # the reference's OWN CUDA path on this GPU, same inputs (after our timed regions: the GPU is idle)
            try:
                sys.path.insert(0, os.path.join(REPO, "baseline"))
                import loader

                if loader.available(cuda=True):
                    r = _reference_child("cuda", args.ratio, 50, 10, 0, 300)
                    ref_cuda = {"value": r["steps_per_s"], "unit": "steps/s", "ms_per_step": r["ms_per_step"], "steps": r["steps"], "warmup": r["warmup"],
                                "what": "the reference's unmodified python + sige.cuda (its kernels rebuilt for sm_100a) + cuDNN, fp32 (TF32 convs: torch default), "
                                        "eager, its Runner.profile protocol (synchronize after every forward)",
                                "speedup_of_this_line": value / r["steps_per_s"]}
                else:
                    ref_cuda = {"unavailable": "baseline/_ref/sige/cuda.so absent"}
            except Exception as e:  # noqa: BLE001
                ref_cuda = {"error": repr(e)}
        if world == 1 and not args.no_cpu_baseline:
            try:
                cpu = cpu_reference_subprocess(args.ratio, args.cpu_steps, 2)
                cpu.pop("ms_per_step", None)
            except Exception as e:  # noqa: BLE001
                cpu = {"error": repr(e)}
        line = {
            "metric": "DDPM 256x256 denoising steps/sec @1.2% edit", "value": value, "unit": "steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong" if args.total_edits else "weak", "vs_baseline": None, "dtype": "f16" if dtype == torch.float16 else "bf16", "data": "synthetic",
            "config": {
                "workload": workload_name(args.ratio), "model_file": model_label,
                "path": path + (" (model(x, t) -> SIGEModel fused step: traced, lowered, CUDA graph; fp32 model + fp32 I/O, %s arithmetic)" % args.dtype if path == "fused" else ""),
                "edits_per_gpu": n_edits, "total_edits": n_edits * world,
                "parallelism": "edits sharded %d/GPU (batched in one fused step), caches broadcast once (%d bytes, %.1f ms over NCCL, outside the timed region), no per-step collective" % (n_edits, nbytes, bcast_ms),
                "l2": "flushed (256 MiB write) between timed steps" if flush is not None else "not flushed",
                "timing": "per-step CUDA events on the launching stream, max over ranks",
            },
            "e2e": {"value": e2e_value, "unit": "steps/s", "h2d_bytes_per_step": x_host.numel() * x_host.element_size(),
                    "d2h_bytes_per_step": out_host.numel() * out_host.element_size(), "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches_per_step * args.steps,
            "clocks": clocks,
            "roofline": roof,
            "cpu_baseline": cpu,
            "reference_cuda": ref_cuda,
        }
        print(json.dumps(line), flush=True)
    if distributed:
        dist.barrier()
        dist.destroy_process_group()


def run_consumer(args):
    """Secondary line: the reference's SD U-Net / GauGAN generator (unmodified model files, full size) — the reference's own
    CUDA path, this repo's exact fp32 operator modules and the fused fp16 step, on the same GPU, same inputs, with the
    parity of the two latter against the former."""
    import tempfile

    import numpy as np
    import torch

    sys.path.insert(0, os.path.join(REPO, "baseline"))
    import consumers
    import loader
    from sige.utils import dilate_mask, downsample_mask

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    dtype = torch.float16 if args.dtype == "fp16" else torch.bfloat16
    ref = None
    if loader.available(cuda=True):
        dump = os.path.join(tempfile.mkdtemp(prefix="sige_ref_"), "ref.npz")
        r = _reference_child("cuda", args.ratio, args.steps, 3, 0, 900 + 5 * args.steps, extra=["--workload", args.workload])      # stock settings (TF32 convs): the timing
        _reference_child("cuda", args.ratio, 1, 1, 0, 900, extra=["--workload", args.workload, "--no-tf32", "--dump", dump])         # exact fp32: the parity target
        ref = (r, np.load(dump))
        log("reference CUDA path: %.2f ms/step" % r["ms_per_step"])
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False      # our dense pass: exact fp32, like the parity target
    net = (consumers.build_sd("full") if args.workload == "sd" else consumers.build_gaugan("full")).to(dev)
    run = (lambda fused: consumers.run_sd(net, downsample_mask, device=dev, fused=fused, size="full")) if args.workload == "sd" else \
          (lambda fused: consumers.run_gaugan(net, downsample_mask, dilate_mask, device=dev, fused=fused, size="full"))
    full0, out_mod = run(lambda n: n.set_fused(False))
    sparse_args = tuple(v.to(dev) for v in (consumers.sd_inputs("full") if args.workload == "sd" else consumers.gaugan_inputs("full")))
    sparse_args = (sparse_args[1], sparse_args[3], sparse_args[4]) if args.workload == "sd" else (sparse_args[1],)

    def timed(k):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(k)]
        with torch.no_grad():
            for i in range(k):
                evs[i][0].record()
                out = net(*sparse_args)
                evs[i][1].record()
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in evs) / k, out

    timed(3)
    ms_mod, out_mod = timed(args.steps)
    net.set_fused(True, dtype=dtype)
    t0 = time.time()
    with torch.no_grad():
        net(*sparse_args)
    compile_s = time.time() - t0
    step = net.fused_step
    timed(3)
    ms_fused, out_fused = timed(args.steps)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"out": out_fused.float().cpu().numpy()})

    def rel(a, b):
        return float(np.abs(a - b).max() / np.abs(b).max())

    parity = None
    if ref is not None:
        want = ref[1]["sparse_out"]
        parity = {"dense_pass_vs_reference_cuda": rel(full0.float().cpu().numpy(), ref[1]["full0_out"]),
                  "fp32_modules_vs_reference_cuda": rel(out_mod.float().cpu().numpy(), want),
                  "fused_%s_vs_reference_cuda" % args.dtype: rel(out_fused.float().cpu().numpy(), want)}
    from collections import Counter

    name = {"sd": "Stable Diffusion v1 U-Net (859.5 M params), 64x64 latent (512x512 image), B = 2, 15 % square mask",
            "gaugan": "GauGAN SPADE generator (ngf 64, 'more' up-sampling), 512x1024, 2.98 % label edit"}[args.workload]
    line = {
        "metric": "%s sparse steps/sec" % args.workload, "value": 1e3 / ms_fused, "unit": "steps/s", "n_gpus": 1, "ms_per_step": ms_fused,
        "steps": args.steps, "warmup": 3,
        "higher_is_better": True, "dtype": "f16" if dtype == torch.float16 else "bf16", "data": "synthetic (random-init weights)",
        "config": {"workload": name, "model_file": "the reference's unmodified model file (baseline/_ref) on this repo's sige.nn",
                   "path": ("model(...) as a fused step: %d fused conv launches + %d sige_sparse_attention + %d sige_spade_modulate launches + %d recorded torch calls in one CUDA graph"
                            % (len(step.fused), step.low.sparse_attention_calls, step.low.spade_calls, len(step.eager_nodes))) if step else "eager"},
        "eager_fp32_modules_ms_per_step": ms_mod,
        "reference_cuda_ms_per_step": None if ref is None else ref[0]["ms_per_step"],
        "speedup_vs_reference_cuda": None if ref is None else ref[0]["ms_per_step"] / ms_fused,
        "parity": parity, "compile_seconds": compile_s,
        "eager_node_kinds": dict(Counter(step.eager_nodes).most_common(12)) if step else None,
    }
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    if args.workload != "ddpm" and args.impl == "ours":
        run_consumer(args)
        return
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "reference-cuda":
        run_reference_cuda(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
