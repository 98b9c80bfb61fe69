#!/usr/bin/env python
"""bench.py -- the hot path's headline measurement (contract: see DESIGN.md "Measurement").

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, libodevit.so)
    python bench.py --impl reference --gpus N ...            # reference arm: CPU PyTorch path (oracle port)

A "step" is one optimizer step of ODE-ViT CE training on one synthetic batch: patch embed ->
fixed-grid solve of the vector field (the hot path, libodevit.so) -> head -> cross-entropy ->
backward (reverse sweep through the solver) -> [gradient all-reduce] -> clip 1.0 -> AdamW.
Workload at N=1 = BASELINE.json configs[1] (the C100 shape of SURVEY section 8: 224 px, patch 16,
D=768, H=12, mlp_ratio 1, 10 registers, N=207 tokens, Euler over 24 grid points, 64 images per
GPU), weak scaling over N.  One JSON line on stdout (rank 0).

    python bench.py --steps K --dump-outputs DIR   # also write the last timed step's outputs as DIR/<name>.npy

The inputs and the initial weights are seeded, so two builds run with the same arguments can be compared output for
output (see `dump_outputs`).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

C100 = dict(img_size=224, patch_size=16, num_classes=100, embed_dim=768, num_heads=12, mlp_ratio=1.0, emulate_depth=12,
            time_interval=1.0, num_eval_steps=24, solver="euler", register_tokens=10)
C10 = dict(img_size=32, patch_size=4, num_classes=10, embed_dim=192, num_heads=3, mlp_ratio=4.0, emulate_depth=12,
           time_interval=1.0, num_eval_steps=5, solver="rk4", register_tokens=4)
WORKLOADS = {
    # BASELINE.json configs[1]; YAML experiment_vit_edo.yaml solver/batch, SURVEY 8 "C100" shape.  THE default (driver) line.
    "c100": dict(kind="train", cfg=C100, batch=64, cpu_sample_batch=64,
                 name="ODE-ViT C100-shape CE training (224px p16 D768 H12 r1 R10 N207, euler T=24)"),
    # the CIFAR-10 model at a throughput batch
    "c10": dict(kind="train", cfg=C10, batch=512, cpu_sample_batch=64,
                name="ODE-ViT CIFAR-10 CE training (32px p4 D192 H3 r4 R4 N69, rk4 T=5)"),
    # BASELINE.json configs[0]: RK4 (3/8) forward+backward, batch 8 -- the reference's own CPU-runnable case
    "c10b8": dict(kind="train", cfg=C10, batch=8, cpu_sample_batch=8,
                  name="ODE-ViT CIFAR-10 fwd+bwd step (32px p4 D192 H3 r4 R4 N69, rk4 T=5), batch 8"),
    # BASELINE.json configs[2]: distillation step (random-init ViT-B/16 teacher, 7M student r=4, Euler T=36, MSE + L1 + JaSMin)
    "distill": dict(kind="train", cfg=dict(C100, mlp_ratio=4.0, num_eval_steps=36), batch=64, cpu_sample_batch=4, distill=True,
                    name="ODE-ViT distillation step (ViT-B/16 teacher no-grad + 7M student 224px D768 r4 N207 euler T=36; "
                         "MSE full path + L1 attention mass + JaSMin k=2)"),
    # BASELINE.json configs[3]: S3.8M-shape inference (registers + positional encoding on them), Euler T=36
    "infer": dict(kind="infer", cfg=dict(C100, num_eval_steps=36, pos_embed_register_tokens=True), batch=1024, cpu_sample_batch=8,
                  name="ODE-ViT S3.8M-shape inference (224px p16 D768 H12 r1 R10 N207, euler T=36)"),
    # BASELINE.json configs[4]: solver-step sweep on the CIFAR-10 student, inference
    "sweep": dict(kind="sweep", cfg=C10, batch=512, cpu_sample_batch=64,
                  name="ODE-ViT CIFAR-10 student solver-step sweep (euler/rk4 x 4..64 steps over [0,1]), inference"),
}
STAGES = {"euler": 1, "midpoint": 2, "rk4": 4}


def field_flops_fwd(cfg) -> float:
    """SURVEY 8(d): forward FLOPs of one field evaluation for one image = 8ND^2 + 4rND^2 + 4N^2D."""
    D = cfg["embed_dim"]
    N = (cfg["img_size"] // cfg["patch_size"]) ** 2 + 1 + cfg["register_tokens"]
    hid = int(D * cfg["mlp_ratio"])
    return 8.0 * N * D * D + 4.0 * N * D * hid + 4.0 * N * N * D


def class_flops(cfg, B) -> dict:
    """Algorithmic FLOPs of ONE launch of each GEMM-shaped kernel class (B images per launch)."""
    D = cfg["embed_dim"]
    N = (cfg["img_size"] // cfg["patch_size"]) ** 2 + 1 + cfg["register_tokens"]
    hid = int(D * cfg["mlp_ratio"])
    M = B * N
    g_in, g_out, att = 2.0 * M * D * (3 * D + hid), 2.0 * M * D * (D + hid), 2.0 * B * N * N * D
    return {"gemm_in_qkv_fc1": g_in, "gemm_out_rk": g_out, "attn_qk": att, "attn_pv": att,
            "fused_attn": 2 * att, "fused_attn_export": 2 * att,
            # backward = 2 x forward (SURVEY 8d): dq, dk, dv and dP = 4 products; the on-chip recomputation of S is a
            # fifth one the kernel EXECUTES but that does not count as algorithmic work (`EXECUTED_FLOPS_RATIO`)
            "fused_attn_bwd": 4 * att, "bwd_gemm_doh": g_out, "bwd_gemm_g2": g_out, "bwd_attn": att,
            "bwd_gemm_dx": g_in, "bwd_gemm_g1": g_in}


EXECUTED_FLOPS_RATIO = {"fused_attn_bwd": 5.0 / 4.0}   # executed / algorithmic, for classes that recompute on chip


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU every 100 ms while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons = index, threading.Event(), [], set()
        self.max_mhz, self.ok = None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:  # noqa: BLE001 -- NVML missing: report clocks as unavailable
            self.nv = None

    def run(self):
        if not self.ok or os.environ.get("ODEVIT_BENCH_NO_SAMPLER"):
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                 nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake"}
        while not self.stop_flag.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            self.stop_flag.wait(0.1)

    def result(self):
        self.stop_flag.set()
        if self.is_alive():
            self.join(2.0)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def synthetic_batch(cfg, B, seed_off=0):
    """SURVEY 8(d): pixel_values ~ N(0,1) (seed 1234), labels uniform (seed 1235), on the host."""
    S, C = cfg["img_size"], cfg["num_classes"]
    px = torch.randn(B, 3, S, S, generator=torch.Generator().manual_seed(1234 + seed_off))
    lb = torch.randint(0, C, (B,), generator=torch.Generator().manual_seed(1235 + seed_off))
    return px, lb


DUMP_BUDGET_BYTES = 64 * 10**6


def host_arrays(prefix, obj):
    """{name: float32 host array} of every floating-point tensor in `obj` (a tensor or nested dicts of them)."""
    if torch.is_tensor(obj):
        return {prefix: obj.detach().float().cpu().numpy()} if obj.is_floating_point() else {}
    out = {}
    if isinstance(obj, dict):
        for k, v in obj.items():
            out.update(host_arrays(f"{prefix}.{k}" if prefix else str(k), v))
    return out


def dump_outputs(out_dir, arrays):
    """Writes every array as out_dir/<name>.npy in float32, DUMP_BUDGET_BYTES in all.  When the arrays are larger than
    that, each array above a common element count is replaced by a sample of that many of its flattened elements: the
    same positions (seeded, in ascending order) in every run, so that dumps of two builds still compare element for
    element."""
    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_BUDGET_BYTES // 4 - 32 * len(arrays)         # in elements; an .npy header is 128 bytes
    sizes = sorted(a.size for a in arrays.values())
    cap = None
    for i, n in enumerate(sizes):                             # largest cap with sum(min(size, cap)) <= left
        if n > left // (len(sizes) - i):
            cap = left // (len(sizes) - i)
            break
        left -= n
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float32)
        if cap is not None and a.size > cap:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the CPU PyTorch path (oracle port of the reference's modules)
# ------------------------------------------------------------------------------------------------
# YAML experiment_classification_edo_distillation.yaml:9-23
DISTILL_TRAINER = dict(mse_full_path=True, use_distillation=True, use_supervision=True, use_mse_loss=True,
                       temperature=3.0, jasmin_k=2, lambda_param=0.5, curriculum=True, patience_factor=0.5)


def build_hf_teacher():
    """Random-init DINO-shape ViT-B/16 (there is no network for checkpoints), eager attention as the reference sets it."""
    from transformers import ViTConfig, ViTForImageClassification
    torch.manual_seed(1)
    return ViTForImageClassification(ViTConfig(num_labels=100, attn_implementation="eager")).eval()


def cpu_reference_step_factory(wl, B):
    """One step of the workload on the host cores through the oracle port (test infrastructure, used here as the timed
    CPU baseline only): training step, distillation step, or a no-grad forward."""
    cfg = wl["cfg"]
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import odevit_oracle as orc
    sd = orc.reference_like_init(cfg, cfg["num_classes"], seed=0)
    px, lb = synthetic_batch(cfg, B)
    if wl["kind"] != "train":
        def fwd():
            with torch.no_grad():
                return float(orc.vit_ode_forward(sd, cfg, px)["logits"].sum())
        return fwd
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    opt = torch.optim.AdamW(list(params.values()), lr=1e-4, weight_decay=5e-2)
    if wl.get("distill"):
        from odevit_b200.loss_trainer import ImageDistilTrainer   # plain PyTorch loss code (no CUDA in it)

        class OracleStudent(torch.nn.Module):
            def __init__(self):
                super().__init__()
                self.ps = torch.nn.ParameterList([torch.nn.Parameter(v) for v in params.values()])

            def forward(self, pixel_values, labels=None, **kw):
                return orc.vit_ode_forward(dict(zip(params.keys(), self.ps)), cfg, pixel_values, labels=labels, **kw)
        student = OracleStudent()
        opt = torch.optim.AdamW(student.parameters(), lr=1e-4, weight_decay=5e-2)
        trainer = ImageDistilTrainer(teacher_model=build_hf_teacher(), student_model=student, optimizer=opt, **DISTILL_TRAINER)
        return lambda: float(trainer({"pixel_values": px}, lb, epoch=0)["loss"].detach())

    def step():
        opt.zero_grad(set_to_none=True)
        out = orc.vit_ode_forward(params, cfg, px, labels=lb)
        out["loss"].backward()
        torch.nn.utils.clip_grad_norm_(list(params.values()), 1.0)
        opt.step()
        return float(out["loss"].detach())

    return step


def time_cpu_reference(wl, B, steps, warmup):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    step = cpu_reference_step_factory(wl, B)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    return B / dt, dt, cores


def metric_of(wl):
    return {"train": "train_images_per_sec", "infer": "inference_images_per_sec", "sweep": "field_evals_per_sec"}[wl["kind"]]


def workload_config(wl, B, world, precision):
    """The `config` object of the JSON line -- the SAME object on both arms (the reference arm runs this workload)."""
    return {"workload": wl["name"], "per_gpu_batch": B, "global_batch": B * world, "parallelism": f"dp{world}",
            "precision_mode": precision,
            "l2_note": "working set per step (trajectory + stage buffers) is far larger than the 126 MB L2"}


def run_reference(args, wl):
    """Reference arm: the reference's CPU PyTorch path (oracle port; /root/reference does not exist on the GPU box and
    the reference is not pip-installable) on the host cores, on OUR arm's workload/config/metric.  Each step is a bounded
    sample of `cpu_sample_batch` images (the default c100 workload: the full per-GPU batch, 64)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg, Bs = wl["cfg"], wl["cpu_sample_batch"]
    B_full = args.batch or wl["batch"]
    Bs = min(Bs, B_full)
    if wl["kind"] == "sweep":
        cfg = dict(cfg, solver="rk4", num_eval_steps=65)
        wl = dict(wl, cfg=cfg)
    ips, dt, cores = time_cpu_reference(wl, Bs, args.steps, max(1, args.warmup))
    nfe = (cfg["num_eval_steps"] - 1) * STAGES[cfg["solver"]]
    value = ips * nfe if wl["kind"] == "sweep" else ips
    unit = "field_evals/s" if wl["kind"] == "sweep" else "img/s"
    sample = (f"{Bs} images per step of the same model/grid on {cores} host threads "
              f"(workload batch {B_full} per GPU; {'the full batch' if Bs == B_full else 'bounded sample'})")
    line = {
        "impl": "reference", "metric": metric_of(wl), "value": value, "unit": unit,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": max(1, args.warmup), "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(wl, B_full, 1 if args.gpus < 1 else args.gpus, args.precision),
        "device": "cpu", "sample_batch": Bs,
        "field_evals_per_sec": ips * nfe,
        "cpu_baseline": {"value": value, "unit": unit, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
class Ranks:
    """Process-group plumbing shared by every workload kind: one process per GPU, NCCL when WORLD_SIZE > 1."""

    def __init__(self):
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device (odevit_b200 has no CPU path; use --impl reference)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self._saved_stdout_fd = None
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            # stdout carries ONE JSON line: whatever NCCL logs (its version banner at WARN, the NVLS lines at INFO) goes
            # to stderr
            os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
            # ... and so does anything a native library prints to file descriptor 1 (the bundled NCCL writes its
            # "NCCL version" banner there even with NCCL_DEBUG unset): fd 1 points at stderr until the JSON line
            sys.stdout.flush()
            self._saved_stdout_fd = os.dup(1)
            os.dup2(2, 1)
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, ms: float) -> float:
        t = torch.tensor([ms], device=self.dev)
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    def emit(self, line: dict):
        if self.rank == 0 and line:
            if self._saved_stdout_fd is not None:
                sys.stdout.flush()
                os.dup2(self._saved_stdout_fd, 1)
            print(json.dumps(line), flush=True)
        if self.world > 1:
            dist.destroy_process_group()


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        return {}


def run_ours(args, wl):
    import odevit_b200 as ob
    from odevit_b200 import _lib
    from odevit_b200.dp import FlatGradAllReduce

    rk = Ranks()
    rank, local, world, dev = rk.rank, rk.local, rk.world, rk.dev

    cfg, B = wl["cfg"], args.batch or wl["batch"]
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    torch.manual_seed(0)
    model = ob.ViTNeuralODE(**cfg).to(dev).train()      # the reference's own init (:494-513), dropout 0
    model.precision = args.precision
    params = [p for p in model.parameters() if p.requires_grad]
    initial_params = [p.detach().clone() for p in params] if args.dump_outputs else None
    opt = torch.optim.AdamW(params, lr=1e-4, weight_decay=5e-2, fused=True, capturable=True)
    reducer = FlatGradAllReduce(params)

    px_h, lb_h = synthetic_batch(cfg, B, seed_off=rank)
    px_h, lb_h = px_h.pin_memory(), lb_h.pin_memory()
    px_d, lb_d = px_h.to(dev), lb_h.to(dev)
    last = {}          # what the latest step returned (under graph replay: the captured step's output buffers)

    if wl.get("distill"):
        # the reference's trainer (loss_trainer.py:305-372 -> odevit_b200.loss_trainer) around the frozen teacher, whose
        # encoder runs through the library too (odevit_b200.ViTTeacher)
        teacher = ob.ViTTeacher(build_hf_teacher().to(dev), precision=args.precision, attention_maps="last")
        trainer = ob.ImageDistilTrainer(teacher_model=teacher, student_model=model, optimizer=opt, **DISTILL_TRAINER)

        def loss_fn(m, px, lb):
            out = trainer.loss_only({"pixel_values": px}, lb, epoch=0)
            last["logits"] = out["student_output"]["logits"].detach()   # not its autograd graph: that would keep the step's tape alive
            return out["loss"]
    else:
        def loss_fn(m, px, lb):
            out = m(px, labels=lb)
            last["logits"] = out["logits"].detach()   # not its autograd graph: that would keep the step's tape alive
            return out["loss"]

    def step(px, lb):
        opt.zero_grad(set_to_none=True)
        loss = loss_fn(model, px, lb)
        loss.backward()
        if not os.environ.get("ODEVIT_BENCH_SKIP_ALLREDUCE"):   # diagnosis only: never set by the driver
            reducer()
        torch.nn.utils.clip_grad_norm_(params, 1.0, foreach=True)
        opt.step()
        return loss.detach()

    barrier = rk.barrier

    def timed_once(fn, k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms) / k

    repeats_log = {}

    def timed(fn, k, tag):
        """EXACTLY k steps between barrier + synchronize, max over ranks -- taken `args.repeats` times, the
        MEDIAN region is reported and every region is listed in the JSON line (`timed_regions_ms_per_step`):
        the hosts of this pool show sporadic multi-millisecond CPU stalls that land in a 5-step region."""
        vals = [timed_once(fn, k) for _ in range(max(1, args.repeats))]
        repeats_log[tag] = [round(v, 3) for v in vals]
        return sorted(vals)[len(vals) // 2]

    import gc
    for _ in range(args.warmup):
        step(px_d, lb_d)
    # The timed steps replay ONE CUDA graph of forward + backward (then all-reduce, clipping, AdamW eagerly):
    # ~1200 launches per step leave sub-microsecond gaps that a replay closes.  Same kernels, same work; the
    # per-class roofline region below stays eager (it brackets every launch with events).
    stepper, launch_mode, graph_launches, graph_logits = None, "eager", 0, None
    if not args.no_graph and not args.quick:
        try:
            from odevit_b200.graphs import GraphedTrainStep
            ob.reset_launch_count()
            # forward + backward in the graph; all-reduce, clipping and AdamW eager after the replay, at every N
            stepper = GraphedTrainStep(model, opt, (px_d, lb_d), clip=1.0, warmup=1, capture_optimizer=False, loss_fn=loss_fn,
                                       grad_hook=(reducer if world > 1 and not os.environ.get("ODEVIT_BENCH_SKIP_ALLREDUCE") else None))
            graph_launches = ob.launch_count() // 2       # one warm-up step + the captured one
            graph_logits = last["logits"]                 # the capture was the last forward: every replay rewrites it
            launch_mode = "cuda_graph_replay (forward+backward; all-reduce/clip/AdamW eager)"
        except Exception as e:  # noqa: BLE001
            import traceback
            traceback.print_exc(file=sys.stderr)
            stepper, launch_mode = None, f"eager (graph capture failed: {type(e).__name__}: {str(e)[:120]})"
            torch.cuda.synchronize()

    def fast_step(px, lb):
        if stepper is None:
            last["loss"] = step(px, lb)
        else:
            last["loss"], last["logits"] = stepper(px, lb), graph_logits
        return last["loss"]
    # per-class event pairs are created here, outside the timed region (cudaEventCreate can stall)
    ob.reset_launch_count()
    step(px_d, lb_d)
    torch.cuda.synchronize()
    _lib.profile_reserve((args.steps * max(1, args.repeats) + 1) * (ob.launch_count() + 64))
    gc.collect()
    gc.disable()       # no collector pauses inside the timed regions (re-enabled below)
    sampler = ClockSampler(local)
    sampler.start()
    # ---- end to end: host buffers in, loss out, every step.  Every step's inputs are copied from pinned host
    # memory inside the timed region; the copy of step k+1 is enqueued on a side stream before step k computes
    # (odevit_b200.dp.HostBatchPrefetcher), and the loss is read back (a host sync) every step.
    from odevit_b200.dp import HostBatchPrefetcher
    feeder = HostBatchPrefetcher(dev)

    def e2e_region(k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        feeder.submit(px_h, lb_h)
        for i in range(k):
            slot, (px, lb) = feeder.take()
            if i + 1 < k:
                feeder.submit(px_h, lb_h)
            loss = fast_step(px, lb)
            feeder.release(slot)
            float(loss.item())
        e1.record()
        barrier()
        return rk.max_over_ranks(e0.elapsed_time(e1)) / k

    # ---- the device-resident number ("value": K steps, inputs resident, no per-class event pairs in the stream) and
    # the end-to-end number alternate, region by region, so that the pair sees the same clocks / power state
    ob.reset_launch_count()
    if not args.quick:
        e2e_region(1)
        ob.reset_launch_count()
    vals_v, vals_e = [], []
    dumped = None
    for r in range(max(1, args.repeats)):
        if args.dump_outputs and r == max(1, args.repeats) - 1:
            # The weight gradients are summed with float atomics, so their last bits vary from run to run, and AdamW's
            # early updates (~lr * sign(g)) turn that into weight differences that grow step after step.  The dumped
            # region therefore starts from the seeded weights and a fresh AdamW state (in place: the captured graph
            # keeps these addresses): its first step has the same inputs in every run; with --steps above 1, the
            # later steps inherit the rounding of the atomics again.
            with torch.no_grad():
                for p, p0 in zip(params, initial_params):
                    p.copy_(p0)
                for state in opt.state.values():
                    for t in state.values():
                        if torch.is_tensor(t):
                            t.zero_()
            torch.cuda.synchronize()
        vals_v.append(timed_once(lambda: fast_step(px_d, lb_d), args.steps))
        if args.dump_outputs and rank == 0 and r == max(1, args.repeats) - 1:
            # the last headline step: its loss and logits, the gradients it left and the weights after its AdamW update
            # (copied now: the regions below keep training the same model)
            dumped = host_arrays("", {"loss": last["loss"], "logits": last["logits"]})
            for n, p in model.named_parameters():
                if p.requires_grad:
                    dumped.update(host_arrays(f"param.{n}", p))
                    if p.grad is not None:
                        dumped.update(host_arrays(f"grad.{n}", p.grad))
        if not args.quick:
            vals_e.append(e2e_region(args.steps))
    repeats_log["value"] = [round(v, 3) for v in vals_v]
    repeats_log["e2e"] = [round(v, 3) for v in vals_e]
    ms_step = sorted(vals_v)[len(vals_v) // 2]
    ms_e2e = sorted(vals_e)[len(vals_e) // 2] if vals_e else float("nan")
    launches = ob.launch_count() // (max(1, args.repeats) * (1 if args.quick else 2))     # per timed region of K steps
    if stepper is not None:
        launches = graph_launches * args.steps                # kernel nodes replayed (counted while capturing)
    # ---- the same K steps once more with an event pair around every launch (2 x ~1200 event records per
    # step cost ~4 % of the step): per-class kernel times for the roofline lines, in their own timed region
    _lib.profile_enable(True)
    ms_prof = timed(lambda: step(px_d, lb_d), args.steps, "value_with_kernel_events")
    prof = {k: (v[0] / max(1, args.repeats), v[1] // max(1, args.repeats)) for k, v in _lib.profile_read().items()}
    _lib.profile_enable(False)
    clocks = sampler.result()

    # ---- kernel-only forward (inference) of the same batch: field evaluations per second
    model.eval()
    with torch.no_grad():
        if args.quick:
            ms_inf = float("nan")
        else:
            for _ in range(2):
                model(px_d)
            ms_inf = timed(lambda: model(px_d), max(2, args.steps), "inference")
    model.train()
    # ---- the same step with the shipped YAML's dropout (experiment_vit_edo.yaml:53-55: 0.3 on the attention map, after
    # out_proj, after GELU and after fc2), replayed as a CUDA graph: the mask seed lives in device memory and a 1-thread
    # kernel inside the captured step advances it (every replay draws new masks).  An extra key, not the headline.
    ms_drop = None
    if not args.quick and not wl.get("distill") and stepper is not None and world == 1:
        try:
            from odevit_b200.graphs import GraphedTrainStep
            torch.manual_seed(0)
            model_d = ob.ViTNeuralODE(**dict(cfg, attn_drop=0.3, proj_drop=0.3, mlp_drop=0.3)).to(dev).train()
            model_d.precision = args.precision
            opt_d = torch.optim.AdamW([p for p in model_d.parameters() if p.requires_grad], lr=1e-4, weight_decay=5e-2,
                                      fused=True, capturable=True)
            step_d = GraphedTrainStep(model_d, opt_d, (px_d, lb_d), clip=1.0, warmup=2, capture_optimizer=False)
            for _ in range(2):
                step_d(px_d, lb_d)
            ms_drop = timed(lambda: step_d(px_d, lb_d), args.steps, "value_dropout_0.3")
            del step_d, opt_d, model_d
        except Exception as e:  # noqa: BLE001
            ms_drop = f"failed: {type(e).__name__}: {str(e)[:100]}"
    gc.enable()

    nfe = (cfg["num_eval_steps"] - 1) * STAGES[cfg["solver"]]
    ips = world * B / (ms_step * 1e-3)
    ips_e2e = world * B / (ms_e2e * 1e-3)
    step_flops = 3.0 * B * nfe * field_flops_fwd(cfg)

    # ---- roofline of the dominant kernel class (largest share of device time in the timed region)
    peaks = load_peaks()
    tensor_peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
    peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if peaks else "fallback 1.4 PF sustained"
    cf = class_flops(cfg, B)
    traffic = {}
    for name in ("r02_traffic.json", "r01_traffic.json"):   # DRAM bytes per launch from the committed `ncu --set full` captures
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", name)))
            break
        except Exception:  # noqa: BLE001
            pass
    traffic_ok = (args.workload == "c100" and B == wl["batch"] and args.precision == "bf16")
    total_ms = sum(v[0] for v in prof.values()) or 1.0
    shares = {k: round(v[0] / total_ms, 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}
    roofline = None
    gemm_classes = [(k, v) for k, v in prof.items() if k in cf]
    if gemm_classes:
        k, (ms, n) = max(gemm_classes, key=lambda kv: kv[1][0])
        achieved = cf[k] / (ms / n * 1e-3) / 1e12
        roofline = {"kernel": k, "bound": "tensor", "achieved": achieved, "peak": tensor_peak, "unit": "TFLOP/s",
                    "frac": achieved / tensor_peak,
                    "traffic": traffic.get(k) if traffic_ok else None, "peak_source": peak_src,
                    "avg_launch_us": ms / n * 1e3, "launches": n, "share_of_kernel_time": shares.get(k),
                    "flop_count": "algorithmic (SURVEY 8d: forward 4N^2D / 2MNK, backward 2x forward)",
                    "executed_tflops": achieved * EXECUTED_FLOPS_RATIO.get(k, 1.0)}

    # every GEMM-shaped class against the tensor-pipe peak (the `roofline` object is the largest of them)
    roofline_tensor = {}
    for k, (ms, n) in prof.items():
        if k in cf:
            tf = cf[k] / (ms / n * 1e-3) / 1e12
            roofline_tensor[k] = {"achieved": round(tf, 1), "frac": round(tf / tensor_peak, 4), "unit": "TFLOP/s",
                                  "avg_launch_us": round(ms / n * 1e3, 2)}
    # ---- HBM-bound row kernels: algorithmic bytes per launch / measured launch time
    hbm_peak = float(peaks.get("hbm_gbs", 6500.0))
    D_, T_ = cfg["embed_dim"], cfg["num_eval_steps"]
    N_ = (cfg["img_size"] // cfg["patch_size"]) ** 2 + 1 + cfg["register_tokens"]
    act_b = 2 if args.precision == "bf16" else 4
    class_bytes = {"center_rows": B * N_ * D_ * (4 + act_b),       # read the fp32 state row, write xc
                   "fd_curvature": T_ * B * N_ * D_ * 4}           # read the trajectory once
    roofline_hbm = {}
    for k, nbytes in class_bytes.items():
        if k in prof:
            ms, n = prof[k]
            gbs = nbytes / (ms / n * 1e-3) / 1e9
            roofline_hbm[k] = {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s",
                               "frac": gbs / hbm_peak, "avg_launch_us": ms / n * 1e3, "launches": n,
                               "algorithmic_bytes": nbytes, "traffic": traffic.get(k) if traffic_ok else None}

    if rank == 0:
        cpu_baseline = None
        if world == 1 and not args.no_cpu_baseline and not args.quick:
            cb = min(wl["cpu_sample_batch"], B)
            c_ips, c_dt, cores = time_cpu_reference(wl, cb, 3, 1)
            cpu_baseline = {"value": c_ips, "unit": "img/s", "cores": cores, "kind": "port",
                            "sample": f"{cb} images per step of the same model/grid ({'the full per-GPU batch' if cb == B else 'bounded sample'}), "
                                      "3 steps after 1 warm-up"}
        line = {
            "metric": "train_images_per_sec", "value": ips, "unit": "img/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "ms_per_step_with_kernel_events": ms_prof,
            "higher_is_better": True,
            "repeats": max(1, args.repeats), "timed_regions_ms_per_step": repeats_log,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "f32",
            "data": "synthetic",
            "config": workload_config(wl, B, world, args.precision),
            "field_evals_per_sec": ips * nfe,
            "train_tflops_algorithmic": step_flops * world / (ms_step * 1e-3) / 1e12,
            "ms_per_step_dropout_0.3": ms_drop,
            "inference_images_per_sec": world * B / (ms_inf * 1e-3),
            "inference_field_evals_per_sec": world * B * nfe / (ms_inf * 1e-3),
            "e2e": {"value": ips_e2e, "unit": "img/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": px_h.numel() * 4 + lb_h.numel() * 8, "d2h_bytes_per_step": 4},
            "gpu_launches": launches, "launch_mode": launch_mode,
            "clocks": clocks,
            "roofline": roofline,
            "roofline_tensor": roofline_tensor,
            "roofline_hbm": roofline_hbm,
            "kernel_time_shares": shares,
            "kernel_avg_us": {k: round(v[0] / v[1] * 1e3, 2) for k, v in prof.items()},
            "kernel_launches_per_step": {k: v[1] // args.steps for k, v in prof.items()},
            "cpu_baseline": cpu_baseline,
            "grad_allreduce_bytes": reducer.bucket_bytes if world > 1 else 0,
        }
        if dumped is not None:
            dump_outputs(args.dump_outputs, dumped)
        rk.emit(line)
    else:
        rk.emit({})


def run_infer(args, wl):
    """Workload kinds "infer" (BASELINE config 4: one grid, large batch) and "sweep" (config 5: euler / rk4 x 4..64 steps
    on the CIFAR-10 student): no-grad forward of the drop-in module, batch-sharded replicas, NO collective on the data
    path.  A "step" is one forward over the per-GPU batch.  The headline point (`value`, `e2e`, `roofline`) is the
    workload's grid for "infer" and (rk4, 64 steps) for "sweep"; every sweep point is listed under `sweep`."""
    import odevit_b200 as ob
    from odevit_b200 import _lib
    from odevit_b200.dp import HostBatchPrefetcher
    rk = Ranks()
    rank, world, dev = rk.rank, rk.world, rk.dev
    cfg, B = wl["cfg"], args.batch or wl["batch"]
    sweep = wl["kind"] == "sweep"
    points = [(s_, n_) for s_ in ("euler", "rk4") for n_ in (4, 8, 16, 32, 64)] if sweep else [(cfg["solver"], cfg["num_eval_steps"] - 1)]
    px_h, _ = synthetic_batch(cfg, B, seed_off=rank)
    px_h = px_h.pin_memory()
    px_d = px_h.to(dev)
    peaks = load_peaks()
    tensor_peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
    hbm_peak = float(peaks.get("hbm_gbs", 6500.0))

    def build(solver, steps):
        torch.manual_seed(0)
        m = ob.ViTNeuralODE(**dict(cfg, solver=solver, num_eval_steps=steps + 1)).to(dev).eval()
        m.precision = args.precision
        return m

    def region(fn, k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        rk.barrier()
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        rk.barrier()
        return rk.max_over_ranks(e0.elapsed_time(e1)) / k

    import gc
    sampler = ClockSampler(rk.local)
    sampler.start()
    rows, regions_log = [], {}
    head = None
    last = {}

    def forward():
        last["out"] = model(px_d)

    with torch.no_grad():
        for solver, steps in points:
            model = build(solver, steps)
            nfe = steps * STAGES[solver]
            for _ in range(max(3, args.warmup)):
                model(px_d)
            gc.collect()
            vals = sorted(region(forward, args.steps) for _ in range(max(1, args.repeats)))
            ms = vals[len(vals) // 2]
            tf = world * B * nfe * field_flops_fwd(cfg) / (ms * 1e-3) / 1e12
            rows.append({"solver": solver, "steps": steps, "ms_per_step": round(ms, 4), "img_per_s": world * B / ms * 1e3,
                         "field_evals_per_sec": world * B * nfe / ms * 1e3, "algorithmic_tflops": round(tf, 1),
                         "frac_of_tensor_peak": round(tf / world / tensor_peak, 4)})
            regions_log[f"{solver}_{steps}"] = [round(v, 4) for v in vals]
            head = (model, solver, steps, nfe, ms)
        model, solver, steps, nfe, ms_step = head
        # the last timed forward is the headline point's (the last point)
        dumped = host_arrays("", last["out"]) if args.dump_outputs and rank == 0 else None
        # ---- end to end for the headline point: pinned host images in (prefetched one step ahead), logits out
        feeder = HostBatchPrefetcher(dev)
        out_h = torch.empty(B, cfg["num_classes"], dtype=torch.float32).pin_memory()

        def e2e_region(k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            rk.barrier()
            e0.record()
            feeder.submit(px_h)
            for i in range(k):
                slot, (px,) = feeder.take()
                if i + 1 < k:
                    feeder.submit(px_h)
                logits = model(px)["logits"]
                feeder.release(slot)
                out_h.copy_(logits, non_blocking=True)
                torch.cuda.current_stream().synchronize()
            e1.record()
            rk.barrier()
            return rk.max_over_ranks(e0.elapsed_time(e1)) / k
        e2e_region(1)
        vals_e = sorted(e2e_region(args.steps) for _ in range(max(1, args.repeats)))
        ms_e2e = vals_e[len(vals_e) // 2]
        regions_log["e2e"] = [round(v, 4) for v in vals_e]
        # ---- per-class kernel times of the headline point (event pairs around every launch)
        ob.reset_launch_count()
        model(px_d)
        torch.cuda.synchronize()
        launches_per_step = ob.launch_count()
        _lib.profile_reserve((args.steps + 1) * (launches_per_step + 16))
        _lib.profile_enable(True)
        ms_prof = region(lambda: model(px_d), args.steps)
        prof = _lib.profile_read()
        _lib.profile_enable(False)
    clocks = sampler.result()
    total_ms = sum(v[0] for v in prof.values()) or 1.0
    shares = {k: round(v[0] / total_ms, 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}
    cf = class_flops(dict(cfg, solver=solver, num_eval_steps=steps + 1), B)
    cf["resident_solve"] = B * nfe * field_flops_fwd(cfg)      # the whole solve of the batch is ONE launch
    roofline, roofline_tensor = None, {}
    for k, (ms, n) in prof.items():
        if k in cf:
            tf = cf[k] / (ms / n * 1e-3) / 1e12
            roofline_tensor[k] = {"achieved": round(tf, 1), "frac": round(tf / tensor_peak, 4), "unit": "TFLOP/s",
                                  "avg_launch_us": round(ms / n * 1e3, 2)}
    gemm_classes = [(k, v) for k, v in prof.items() if k in cf]
    if gemm_classes:
        k, (ms, n) = max(gemm_classes, key=lambda kv: kv[1][0])
        achieved = cf[k] / (ms / n * 1e-3) / 1e12
        roofline = {"kernel": k, "bound": "tensor", "achieved": achieved, "peak": tensor_peak, "unit": "TFLOP/s",
                    "frac": achieved / tensor_peak, "traffic": None,
                    "peak_source": "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if peaks else "fallback 1.4 PF sustained",
                    "avg_launch_us": ms / n * 1e3, "launches": n, "share_of_kernel_time": shares.get(k),
                    "note": ("the on-chip-state solver touches HBM for x0, one trajectory row per step and the weights only "
                             "(DRAM throughput ~2 %): it is reported against the TENSOR peak, not the HBM roofline"
                             if k == "resident_solve" else "algorithmic FLOPs (SURVEY 8d)")}
    D_, T_ = cfg["embed_dim"], steps + 1
    N_ = (cfg["img_size"] // cfg["patch_size"]) ** 2 + 1 + cfg["register_tokens"]
    roofline_hbm = {}
    for k, nbytes in {"center_rows": B * N_ * D_ * (4 + (2 if args.precision == "bf16" else 4)), "fd_curvature": T_ * B * N_ * D_ * 4}.items():
        if k in prof:
            ms, n = prof[k]
            gbs = nbytes / (ms / n * 1e-3) / 1e9
            roofline_hbm[k] = {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                               "avg_launch_us": ms / n * 1e3, "launches": n, "algorithmic_bytes": nbytes}
    if rank != 0:
        rk.emit({})
        return
    ips, ips_e2e = world * B / (ms_step * 1e-3), world * B / (ms_e2e * 1e-3)
    unit = "field_evals/s" if sweep else "img/s"
    scale = nfe if sweep else 1
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        cb = min(wl["cpu_sample_batch"], B)
        c_ips, c_dt, cores = time_cpu_reference(dict(wl, cfg=dict(cfg, solver=solver, num_eval_steps=steps + 1)), cb, 2, 1)
        cpu_baseline = {"value": c_ips * scale, "unit": unit, "cores": cores, "kind": "port",
                        "sample": f"{cb} images per forward of the headline point ({solver}, {steps} steps), 2 calls after 1 warm-up"}
    line = {
        "metric": metric_of(wl), "value": ips * scale, "unit": unit, "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms_step, "ms_per_step_with_kernel_events": ms_prof, "higher_is_better": True,
        "repeats": max(1, args.repeats), "timed_regions_ms_per_step": regions_log,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
        "config": dict(workload_config(wl, B, world, args.precision), headline_point=f"{solver}, {steps} steps",
                       collectives="none (replicas)"),
        "inference_images_per_sec": ips, "field_evals_per_sec": ips * nfe,
        "algorithmic_tflops": world * B * nfe * field_flops_fwd(cfg) / (ms_step * 1e-3) / 1e12,
        "e2e": {"value": ips_e2e * scale, "unit": unit, "ms_per_step": ms_e2e, "h2d_bytes_per_step": px_h.numel() * 4,
                "d2h_bytes_per_step": out_h.numel() * 4},
        "gpu_launches": launches_per_step * args.steps, "launch_mode": "eager",
        "clocks": clocks, "roofline": roofline, "roofline_tensor": roofline_tensor, "roofline_hbm": roofline_hbm,
        "kernel_time_shares": shares,
        "kernel_avg_us": {k: round(v[0] / v[1] * 1e3, 2) for k, v in prof.items()},
        "cpu_baseline": cpu_baseline,
    }
    if sweep:
        line["sweep"] = rows
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped)
    rk.emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c100", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the workload's)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--repeats", type=int, default=3,
                    help="timed regions of K steps each; the median one is reported, all are listed")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of the CUDA-graph replay of the step")
    ap.add_argument("--quick", action="store_true",
                    help="profiling helper (ncu launch lists): only the device-resident timed region, any warm-up count; "
                         "its JSON line is not a bench value")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (training: loss, logits, gradients and the updated "
                         "weights; inference: the forward's outputs) as DIR/<name>.npy, float32, at most 64 MB in all. "
                         "Training: the last headline region (and every region after it) then starts from the seeded "
                         "weights and a fresh AdamW state, so that the dump is comparable between runs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.quick:
        args.repeats = 1
    if args.impl == "ours" and not args.quick:
        args.warmup = max(3, args.warmup)
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, wl)
    elif wl["kind"] == "train":
        run_ours(args, wl)
    else:
        run_infer(args, wl)


if __name__ == "__main__":
    main()
