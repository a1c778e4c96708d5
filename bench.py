#!/usr/bin/env python
"""Benchmark of the DINO-Soft loss hot path (fwd + bwd), BASELINE.json's metric.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

N = 1 (default): global batch B = 32768 (BASELINE config 3's batch, which fits one B200 because the
B x B logits are never materialised), D = 512, DINO dim 768, MLP projection head, text-symmetric soft
term.  N > 1 (launched by torchrun): the same global batch sharded by row block (strong scaling),
one NCCL all-gather of the packed bf16 embeddings per step.

One JSON line is printed by rank 0.  `value` = samples/s with inputs resident in HBM; `e2e` = the same
metric through the module with pinned HOST inputs (H2D inside the timed region, loss read back);
`roofline` = the dominant tile kernel against the measured bf16 tensor peak; `cpu_baseline` = the reference's
own loss.py (staged as oracle/_ref/loss.py by oracle/make_ref.py; the oracle port only if that copy is absent,
and `kind` says which) timed on this box's host cores on a bounded sample; `gpu_eager_baseline` = the same
reference code run eagerly on this B200 under bf16 autocast (cuBLAS + ATen element-wise kernels), the comparator
SURVEY.md 2a names.  `--impl reference` times only the CPU reference.

Other BASELINE configs: `--batch 4096` (config 2), `--clip-dim 768 --dino-dim 1024 --no-head --batch 65536`
under torchrun with 8 ranks (config 4).

`--dump-outputs DIR` writes what the last timed step returned on rank 0 (the loss terms and the gradients of the
image / text features, the logit scale and the head parameters) as DIR/<name>.npy in float32.  The inputs are
seeded, so two builds run with the same arguments can be compared array for array.
"""
from __future__ import annotations

import argparse
import ctypes as C
import importlib.util
import json
import os
import statistics
import subprocess
import sys
import threading
import time
import types

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the tree as it found it (it may be read-only)

METRIC = "dino_soft_loss_fwd_bwd_samples_per_sec"
GLOBAL_B, D_CLIP, D_DINO = 32768, 512, 768
KERNEL_NAMES = ["fwd_clip_i2t", "fwd_clip_t2i", "fwd_soft", "bwd_clip_image", "bwd_clip_text",
                "bwd_student", "bwd_text", "bwd_build_g_clip", "bwd_build_g_soft"]
NK = len(KERNEL_NAMES)
LOSS_ARGS = dict(use_projection=True, projection_type="mlp", lambda_soft=0.5, soft_mode="kl_teacher",
                 soft_dino_to_text=True, text_lambda=0.5, text_student_temp=0.02, teacher_temp=0.15,
                 lambda_original=1.0, lambda_weighted=0.0)


def load_reference_module():
    """The reference's own loss.py staged under oracle/_ref (None if it was never staged)."""
    spec = importlib.util.spec_from_file_location("dsoft_make_ref", os.path.join(ROOT, "oracle", "make_ref.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    try:
        return mod.load_reference()
    except Exception as e:  # checksum mismatch etc.: say so, fall back to the port
        print(f"[bench] oracle/_ref unusable: {e}", file=sys.stderr)
        return None


def load_oracle():
    spec = importlib.util.spec_from_file_location("dinosoft_oracle", os.path.join(ROOT, "oracle", "dinosoft_oracle.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules["dinosoft_oracle"] = mod
    spec.loader.exec_module(mod)
    return mod


def synth(seed, rows, D, Dd, device, clustered=True):
    """SURVEY.md 8(d) synthetic inputs: clustered embeddings, image/text L2-normalised, DINO raw."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    K = max(rows // 16, 2)
    cid = torch.randint(0, K, (rows,), generator=g)

    def make(d, scale=1.0):
        cent = torch.randn(K, d, generator=g)
        return (cent[cid] + 0.5 * torch.randn(rows, d, generator=g)) * scale

    img = torch.nn.functional.normalize(make(D), dim=-1)
    txt = torch.nn.functional.normalize(make(D), dim=-1)
    dino = make(Dd, 3.0)
    r = lambda x: x.to(torch.bfloat16).to(torch.float32)
    return r(img).to(device), r(txt).to(device), r(dino).to(device)


# --------------------------------------------------------------------------------------------------
# reference timing (CPU, and eagerly on the GPU)
# --------------------------------------------------------------------------------------------------
USE_HEAD = True


def cpu_port_step(oracle, img, txt, dino, head, scale, cfg):
    """One fwd+bwd of the oracle port (fp32, torch CPU ops, all host threads): only used when oracle/_ref is absent."""
    im = img.clone().requires_grad_(True)
    tx = txt.clone().requires_grad_(True)
    sc = torch.tensor(scale, requires_grad=True)
    pp = None if head is None else {k: v.clone().requires_grad_(True) for k, v in head.items()}
    student = None if pp is None else oracle.mlp_head(im, pp, "mlp")
    out = oracle.rank_loss(im, tx, sc, dino, student, cfg, rank=0)
    out["total_loss"].backward()
    return float(out["total_loss"].detach())


class ReferenceRunner:
    """fwd+bwd of the reference loss (or the port) on `device` for a batch of B rows of the bench workload."""

    def __init__(self, B, device, autocast=False):
        self.ref = load_reference_module()
        self.kind = "reference" if self.ref is not None else "port"
        self.device, self.autocast, self.B = device, autocast, B
        torch.manual_seed(0)
        self.img, self.txt, self.dino = synth(4321, B, D_CLIP, D_DINO, device)
        self.args = types.SimpleNamespace(**dict(LOSS_ARGS, use_projection=USE_HEAD))
        self.scale = 14.2857
        if self.ref is not None:
            self.loss = self.ref.ClipLossWithDINOEnhancements(local_loss=False, gather_with_grad=False,
                                                              cache_labels=False, rank=0, world_size=1)
            if USE_HEAD:
                self.loss.init_proj(D_CLIP, D_DINO, device, "mlp")
        else:
            self.oracle = load_oracle()
            H = (D_CLIP + D_DINO) // 2
            self.head = None
            if USE_HEAD:
                l0, l1 = torch.nn.Linear(D_CLIP, H), torch.nn.Linear(H, D_DINO)
                self.head = {"w0": l0.weight.detach(), "b0": l0.bias.detach(), "w1": l1.weight.detach(),
                             "b1": l1.bias.detach()}
            self.cfg = self.oracle.OracleConfig(lambda_soft=0.5, soft_mode="kl_teacher", soft_dino_to_text=True,
                                                text_lambda=0.5, text_student_temp=0.02, teacher_temp=0.15)

    def step(self):
        if self.ref is None:
            return cpu_port_step(self.oracle, self.img, self.txt, self.dino, self.head, self.scale, self.cfg)
        im = self.img.clone().requires_grad_(True)
        tx = self.txt.clone().requires_grad_(True)
        sc = torch.tensor(self.scale, device=self.device, requires_grad=True)
        if self.loss.image_to_dino_proj is not None:
            for p in self.loss.image_to_dino_proj.parameters():
                p.grad = None
        if self.autocast:
            with torch.autocast("cuda", dtype=torch.bfloat16):
                out = self.loss(im, tx, sc, self.dino, self.args, output_dict=True)
        else:
            out = self.loss(im, tx, sc, self.dino, self.args, output_dict=True)
        out["total_loss"].backward()
        return out["total_loss"].detach()


def time_cpu_reference(sample_B, iters, warmup=1):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    run = ReferenceRunner(sample_B, "cpu")
    for _ in range(warmup):
        run.step()
    times = []
    for _ in range(iters):
        t0 = time.perf_counter()
        float(run.step())
        times.append(time.perf_counter() - t0)
    return times, cores, run.kind


def time_gpu_eager(B, device, iters=5, warmup=2):
    """The reference loss.py itself on the GPU: eager PyTorch under bf16 autocast, CUDA-event timed."""
    run = ReferenceRunner(B, device, autocast=True)
    if run.ref is None:
        return None
    for _ in range(warmup):
        run.step()
    torch.cuda.synchronize()
    times = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run.step()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    del run
    torch.cuda.empty_cache()
    return statistics.median(times)


REF_SAMPLE_B = 4096


def sample_note(kind, B, cores):
    what = ("the reference's own src/open_clip/loss.py (oracle/_ref/loss.py, unmodified)" if kind == "reference"
            else "the oracle port of the reference loss (oracle/_ref not staged)")
    return (f"{what}: B={B} rows of the bench workload per step (D={D_CLIP}, Dd={D_DINO}, "
            f"{'MLP head, ' if USE_HEAD else ''}text-symmetric), fp32 torch CPU ops, {cores} threads.  The full "
            f"B={GLOBAL_B} step needs ~40 GiB of fp32 B x B intermediates and minutes per step on a CPU; cost per "
            f"sample grows linearly with B, so samples/s at B={GLOBAL_B} is about {B}/{GLOBAL_B} of this figure")


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    times, cores, kind = time_cpu_reference(REF_SAMPLE_B, args.steps, max(args.warmup, 1))
    total = sum(times)
    value = REF_SAMPLE_B * len(times) / total
    # one larger sample to show the O(B^2) growth the note claims (3 steps)
    big_times, _, _ = time_cpu_reference(2 * REF_SAMPLE_B, 3, 1)
    big = 2 * REF_SAMPLE_B / statistics.median(big_times)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.gpus),
        "sample_batch": REF_SAMPLE_B,
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": cores, "kind": kind,
                         "sample": sample_note(kind, REF_SAMPLE_B, cores),
                         "median_ms_per_step": 1e3 * statistics.median(times),
                         "samples_per_s_at_2x_sample": big,
                         "extrapolated_to_global_batch": value * REF_SAMPLE_B / GLOBAL_B},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(n):
    head = "MLP projection head" if USE_HEAD else "no projection head"
    packed_mb = GLOBAL_B * (2 * D_CLIP + (D_DINO if USE_HEAD else 0) + D_DINO) * 2 / 1e6
    return {
        "workload": f"DINO-Soft loss fwd+bwd, global batch {GLOBAL_B}, D={D_CLIP}, DINOv2 dim {D_DINO}, {head}, "
                    f"text-symmetric soft term, logit_scale=14.2857",
        "global_batch": GLOBAL_B, "local_batch": GLOBAL_B // n, "D": D_CLIP, "Dd": D_DINO,
        "parallelism": f"row-block x{n}" if n > 1 else "single GPU",
        "l2": (f"inputs larger than L2 (packed bf16 embeddings {packed_mb:.0f} MB + fp16 gradient operands)"
               if packed_mb > 126 else
               f"L2 flushed between steps by the step's own logit-gradient matrices "
               f"({2e-6 * GLOBAL_B * GLOBAL_B / n:.0f} MB per matrix; packed embeddings {packed_mb:.0f} MB)"),
    }


def load_ncu_traffic():
    """DRAM bytes (read + write) per launch from the tracked ncu --set full summary of THIS workload
    (profiles/ncu_traffic.csv: kernel,dram_bytes,source,git_sha); {} if the file is absent."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.csv")
    out = {}
    try:
        for ln in open(path):
            f = [x.strip() for x in ln.split(",")]
            if len(f) >= 2 and not ln.startswith("#") and f[0] != "kernel":
                out[f[0]] = float(f[1])
    except OSError:
        pass
    return out


DUMP_ROWS = 4096  # rows kept of a per-sample gradient: 8 MB at D = 512 (the full one is 64 MB at B = 32768)
DUMP_MAX_BYTES = 64_000_000


def snapshot_outputs(out, leaves):
    """Host float32 copies of what the caller of a step receives: the loss terms of `out` and the gradients of the
    (name, tensor) `leaves`.  A gradient with more than DUMP_ROWS rows keeps a fixed seeded sample of its rows, in
    ascending order, so that two runs keep the same rows."""
    arrays = {k: out[k] for k in ("total_loss", "classic_loss", "soft_loss", "weighted_loss") if k in out}
    for name, t in leaves:
        g = t.grad
        if g is None:
            continue
        if g.dim() > 0 and g.shape[0] > DUMP_ROWS:
            rows = torch.randperm(g.shape[0], generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values
            g = g[rows.to(g.device)]
        arrays["grad_" + name] = g
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs, more than {DUMP_MAX_BYTES}")
    return arrays


def write_outputs(directory, arrays):
    import numpy as np

    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


# --------------------------------------------------------------------------------------------------
# clocks sampler
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def mark(self):
        """Index of the next sample: brackets the timed region inside a sampler that is already running (the
        nvidia-smi process needs ~0.1 s to start, longer than a whole timed region on 8 GPUs)."""
        return len(self.lines)

    def stop(self, first=0, last=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        last = len(self.lines) if last is None else last
        window = self.lines[first:last]
        if not window:  # region shorter than one sampling period: the samples around it
            window = self.lines[max(0, first - 1):last + 1]
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in window:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            try:
                pw.append(float(f[2]))
            except ValueError:
                pass
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w": statistics.median(pw) if pw else None, "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    import dinosoft_b200 as pkg
    from dinosoft_b200 import _cabi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA sm_100 device (no CPU fallback for the product path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    stdout_fd = None
    if world > 1:
        # NCCL prints its version banner to stdout (fd 1) when the communicator is created; stdout must carry the
        # JSON line only, so fd 1 points at stderr until the line is printed
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        sys.stdout.flush()
        stdout_fd = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
    assert GLOBAL_B % world == 0
    b = GLOBAL_B // world
    lib = _cabi.lib()
    # started before the inputs are generated: nvidia-smi needs ~0.1 s to come up, longer than a whole timed
    # region on 8 GPUs; mark() brackets the timed region in its sample stream
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    img, txt, dino = synth(1234 + rank, b, D_CLIP, D_DINO, dev)
    larg = types.SimpleNamespace(**dict(LOSS_ARGS, use_projection=USE_HEAD))
    loss = pkg.ClipLossWithDINOEnhancements(local_loss=True, gather_with_grad=True, rank=rank, world_size=world)
    torch.manual_seed(99)
    params = []
    if USE_HEAD:
        loss.init_proj(D_CLIP, D_DINO, dev, "mlp")
        params = list(loss.image_to_dino_proj.parameters())
    scale = torch.tensor(14.2857, device=dev, requires_grad=True)
    img.requires_grad_(True)
    txt.requires_grad_(True)

    def zero_grads():
        img.grad = txt.grad = scale.grad = None
        for p in params:
            p.grad = None

    def step(im, tx, dn):
        # the reference calls the loss inside torch.autocast (open_clip_train/train.py:285): the projection
        # head runs in bf16 on cuBLAS; the fused loss kernels are unaffected (bf16 operands, fp32 math)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = loss(im, tx, scale, dn, larg, output_dict=True)
        out["total_loss"].backward()
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # --graph: forward and backward replay CUDA graphs (dinosoft_b200.make_graphed, the package's public helper for
    # the launch-bound small-batch regime); the per-kernel pass below stays eager (it needs the host-side recorder)
    # Default (neither --graph nor --no-graph): eager, except on ONE GPU when the step is bound by the host (a block of
    # at most 2^28 similarity entries: config 2, 0.8 ms of Python / ctypes enqueue against 0.35 ms of kernels).  With
    # several ranks --graph also works (NCCL collectives are captured: 2 GPUs 7.07-7.26 ms against 7.36-7.65 ms eager)
    # but is opt-in: only the 2-GPU capture has been run.
    eager_step = step
    use_graph = args.graph or (not args.no_graph and world == 1 and float(b) * GLOBAL_B <= 2.0 ** 28)
    graph_note = None
    if use_graph:
        try:
            zero_grads()
            ref_loss = float(eager_step(img, txt, dino)["total_loss"].detach())
            gstep = pkg.make_graphed(loss, larg, img, txt, scale, dino, autocast_dtype=torch.bfloat16)

            def graph_step(im, tx, dn):
                t, c, s = gstep(im, tx, scale, dn)
                t.backward()
                return {"total_loss": t, "classic_loss": c, "soft_loss": s}

            zero_grads()
            got_loss = float(graph_step(img, txt, dino)["total_loss"].detach())
            if not abs(got_loss - ref_loss) <= 1e-5 * abs(ref_loss):
                raise RuntimeError(f"graph replay gives loss {got_loss}, eager {ref_loss}")
            step = graph_step
        except Exception as exc:  # capture refused (e.g. a collective that cannot be captured): time the eager path
            use_graph = False
            graph_note = f"graph capture failed, eager step timed: {type(exc).__name__}: {exc}"[:300]
            print("[bench] " + graph_note, file=sys.stderr)
            torch.cuda.synchronize()

    # ---- warm-up
    for _ in range(max(args.warmup, 3)):
        zero_grads()
        step(img, txt, dino)
    barrier()

    # ---- timed region: resident inputs
    clk_first = sampler.mark()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    h0 = time.perf_counter()
    for _ in range(args.steps):
        zero_grads()
        out = step(img, txt, dino)
    e1.record()
    host_ms = (time.perf_counter() - h0) * 1e3  # host time to enqueue the loop (diagnostic: host-bound if ~ ms)
    barrier()
    ms = e0.elapsed_time(e1)
    if os.environ.get("DSOFT_BENCH_REPEAT"):
        print(f"[bench] rank {rank}: headline {ms / args.steps:.4f} ms/step, host enqueue {host_ms / args.steps:.4f} "
              "ms/step", file=sys.stderr)
    final_loss = float(out["total_loss"].detach())
    dumped = None
    if args.dump_outputs and rank == 0:  # before the passes below overwrite the gradients
        leaves = [("image", img), ("text", txt), ("logit_scale", scale)]
        if USE_HEAD:
            leaves += [("head_" + n.replace(".", "_"), p) for n, p in loss.image_to_dino_proj.named_parameters()]
        dumped = snapshot_outputs(out, leaves)

    # ---- per-kernel pass (same inputs, same loop, clocks still sampled): the product launches the independent
    # tile kernels of a pass on forked streams so they fill each other's last wave; CUDA events around a kernel
    # that shares the GPU do not give its own duration, so the recorder serialises the launches and this pass
    # is timed separately from the headline above
    prof_steps = max(1, min(args.steps, 10))
    lib.dsoft_profile_enable(1)
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    p0.record()
    for _ in range(prof_steps):
        zero_grads()
        eager_step(img, txt, dino)
    p1.record()
    barrier()
    ms_serial = p0.elapsed_time(p1)
    clocks = sampler.stop(clk_first, sampler.mark()) if rank == 0 else None
    ms_sum = (C.c_double * NK)()
    cnt = (C.c_int * NK)()
    _cabi.check(lib.dsoft_profile_read(ms_sum, cnt, NK), "dsoft_profile_read")
    lib.dsoft_profile_enable(0)
    ms_again = None
    if os.environ.get("DSOFT_BENCH_REPEAT"):  # diagnostic: the headline loop once more, after the profiled pass
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        r0.record()
        for _ in range(args.steps):
            zero_grads()
            step(img, txt, dino)
        r1.record()
        barrier()
        ms_again = r0.elapsed_time(r1) / args.steps
        print(f"[bench] headline loop repeated after the profiled pass: {ms_again:.4f} ms/step", file=sys.stderr)

    # ---- e2e: pinned host inputs -> H2D -> module -> loss scalars back to the host, every step
    h_img = img.detach().cpu().pin_memory()
    h_txt = txt.detach().cpu().pin_memory()
    h_dino = dino.detach().cpu().pin_memory()
    h2d_bytes = (h_img.numel() + h_txt.numel() + h_dino.numel()) * 4
    del p0, p1
    host_out = torch.empty(3, dtype=torch.float32).pin_memory()

    # double-buffered device staging: the H2D copy of step n+1 is issued on a side stream before step n runs
    # (what train.py's `.to(device, non_blocking=True)` from the pinned DINO table achieves, train.py:280),
    # so every step still pays its own 235 MB of host->device traffic inside the timed region
    copy_stream = torch.cuda.Stream(device=dev)
    stage_bufs = [[torch.empty_like(t, device=dev) for t in (h_img, h_txt, h_dino)] for _ in range(2)]
    stage_evt = [torch.cuda.Event() for _ in range(2)]

    def issue_h2d(slot):
        with torch.cuda.stream(copy_stream):
            for d, h in zip(stage_bufs[slot], (h_img, h_txt, h_dino)):
                d.copy_(h, non_blocking=True)
            stage_evt[slot].record(copy_stream)

    e2e_count = [0]

    def e2e_step():
        n = e2e_count[0]
        e2e_count[0] += 1
        issue_h2d((n + 1) % 2)  # prefetch the next step's inputs
        torch.cuda.current_stream().wait_event(stage_evt[n % 2])
        zero_grads()
        im = stage_bufs[n % 2][0].requires_grad_(True)
        tx = stage_bufs[n % 2][1].requires_grad_(True)
        dn = stage_bufs[n % 2][2]
        o = step(im, tx, dn)
        host_out.copy_(torch.stack([o["total_loss"].detach(), o["classic_loss"].detach(), o["soft_loss"].detach()]),
                       non_blocking=True)
        torch.cuda.current_stream().synchronize()  # the training loop reads the loss every step (train.py:354)
        im.requires_grad_(False)
        tx.requires_grad_(False)
        im.grad = tx.grad = None
        return float(host_out[0])

    ms_e2e = float("nan")
    if not args.no_e2e:
        issue_h2d(0)
        for _ in range(2):
            e2e_step()
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(args.steps):
            e2e_step()
        f1.record()
        barrier()
        ms_e2e = f0.elapsed_time(f1)

    if world > 1:
        t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = float(t[0]), float(t[1])

    if rank == 0:
        from dinosoft_b200.loss import _cuda_backend

        plan = next(iter(_cuda_backend._plans.values()))
        alg = (C.c_double * NK)()
        exe = (C.c_double * NK)()
        _cabi.check(lib.dsoft_plan_kernel_flops(plan.handle, alg, exe, NK), "dsoft_plan_kernel_flops")
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_burst = peaks.get("bf16_tflops")
        peak_sust = peaks.get("bf16_tflops_sustained")
        peak_src = "MEASURED_PEAKS.json (bf16_tflops_sustained: kernels timed inside a long step)"
        if not peak_sust:
            peak_sust, peak_burst, peak_src = 1400.0, 1590.0, "fallback (B200_PROFILING.md: 1.59 PF burst / ~1.4 PF sustained)"
        kern = {}
        for k, name in enumerate(KERNEL_NAMES):
            if cnt[k] == 0:
                continue
            avg_ms = ms_sum[k] / cnt[k]
            kern[name] = {"ms": round(avg_ms, 4), "alg_tflops": round(alg[k] / avg_ms / 1e9, 1),
                          "exec_tflops": round(exe[k] / avg_ms / 1e9, 1), "launches": cnt[k]}
        # DRAM bytes (read + write) per launch: loaded from the tracked ncu summary of the default workload
        default_workload = (GLOBAL_B == 32768 and world == 1 and D_CLIP == 512 and D_DINO == 768 and USE_HEAD)
        ncu_traffic = load_ncu_traffic() if default_workload else {}
        # dominant kernel = the longest launch that carries algorithmic FLOPs (the logit-gradient kernels of
        # the two-phase backward only recompute similarity tiles: SURVEY 8(d) counts those products once, in
        # the forward; their executed FLOPs are in `kernels`)
        dom = max((n for n in kern if alg[KERNEL_NAMES.index(n)] > 0), key=lambda n: kern[n]["ms"])
        dk = KERNEL_NAMES.index(dom)
        dom_ms = ms_sum[dk] / cnt[dk]
        achieved = alg[dk] / dom_ms / 1e9
        tile_ms = sum(ms_sum[k] for k in range(NK)) / prof_steps
        step_ms = ms / args.steps
        step_alg_tflops = plan.flops / step_ms / 1e9  # this rank's algorithmic FLOPs / step time
        cpu_baseline = None
        gpu_eager = None
        if world == 1 and not args.no_cpu_baseline:
            sb = min(REF_SAMPLE_B, GLOBAL_B)
            cpu_times, cores, kind = time_cpu_reference(sb, 5, 1)
            med = statistics.median(cpu_times)
            cpu_baseline = {
                "value": sb / med, "unit": "samples/s", "cores": cores, "kind": kind,
                "sample": sample_note(kind, sb, cores) + "; 1 warm-up + 5 timed fwd+bwd, median",
                "extrapolated_to_global_batch": sb / med * sb / GLOBAL_B}
            # the comparator SURVEY 2a names: the same reference code, eager on this GPU under bf16 autocast
            gpu_eager = {"impl": "reference loss.py, eager PyTorch, torch.autocast(bf16), CUDA events, median of 5",
                         "runs": []}
            for eb in (8192, 16384):
                if eb > GLOBAL_B:
                    continue
                try:
                    ems = time_gpu_eager(eb, dev)
                except torch.cuda.OutOfMemoryError:
                    ems = None
                    torch.cuda.empty_cache()
                if ems is not None:
                    gpu_eager["runs"].append({"batch": eb, "ms_per_step": round(ems, 3),
                                              "samples_per_s": round(eb / ems * 1e3, 1),
                                              "extrapolated_to_global_batch": round(eb / ems * 1e3 * eb / GLOBAL_B, 1)})
            if not gpu_eager["runs"]:
                gpu_eager = None
        launches_per_step = plan.launches_fwd + plan.launches_bwd  # pack, scalars, norms, tiles, finalize ...
        line = {
            "metric": METRIC, "value": GLOBAL_B * args.steps / (ms / 1e3), "unit": "samples/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": step_ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": dict(workload_config(world), graphed=bool(use_graph),
                           **({"graph_note": graph_note} if graph_note else {})),
            "backward_impl": ("two-phase: fp16 logit-gradient matrices + M=256xN=256 gradient GEMMs"
                              + (", symmetric shortcuts (world 1)" if world == 1 else "")
                              if plan.shape.flags & _cabi.DSOFT_F_GMAT else
                              "fused: logit gradients stay in shared memory"),
            "clocks": clocks,
            "e2e": None if args.no_e2e else {
                "value": GLOBAL_B * args.steps / (ms_e2e / 1e3), "unit": "samples/s",
                "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 12, "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches_per_step * args.steps,
            "roofline": {"bound": "tensor", "kernel": dom, "achieved": round(achieved, 1), "peak": peak_sust,
                         "unit": "TFLOP/s", "frac": round(achieved / peak_sust, 4),
                         "traffic": ncu_traffic.get(dom),
                         "peak_source": peak_src, "peak_burst": peak_burst,
                         "executed_tflops": kern[dom]["exec_tflops"],
                         "executed_frac": round(kern[dom]["exec_tflops"] / peak_sust, 4),
                         "note": "achieved = algorithmic FLOPs of this launch (SURVEY 8d: each distinct product "
                                 "once, Gram symmetry not discounted, tile recompute not counted) / its CUDA-event "
                                 "duration; a launch that exploits the symmetry executes about half of them, so frac "
                                 "can exceed 1: executed_frac is the utilisation of the launch, step_roofline the "
                                 "figure for the whole step"},
            "step_roofline": {"algorithmic_tflops_per_gpu": round(step_alg_tflops, 1),
                              "frac_of_sustained_peak": round(step_alg_tflops / peak_sust, 4),
                              "frac_of_burst_peak": round(step_alg_tflops / peak_burst, 4) if peak_burst else None,
                              "serial_ms_per_step": round(ms_serial / prof_steps, 4),
                              "tile_kernel_ms_per_serial_step": round(tile_ms, 4),
                              "tile_kernel_share_of_serial_step": round(tile_ms / (ms_serial / prof_steps), 4),
                              "note": "per-kernel durations come from a second pass of the same loop with the "
                                      "tile kernels launched serially (dsoft_profile_enable); the headline "
                                      "ms_per_step launches them on forked streams"},
            "kernels": kern,
            "cpu_baseline": cpu_baseline,
            "gpu_eager_baseline": gpu_eager,
            "loss": final_loss,
        }
        if dumped is not None:
            write_outputs(args.dump_outputs, dumped)
        if stdout_fd is not None:
            sys.stdout.flush()
            os.dup2(stdout_fd, 1)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
        if use_graph:
            # graphs that captured NCCL kernels are still alive: destroying the communicator under them blocked the
            # exit for minutes (2 GPUs, torch 2.11 / NCCL 2.28); everything is flushed, leave without destructors
            sys.stdout.flush()
            sys.stderr.flush()
            os._exit(0)
        dist.destroy_process_group()


def main():
    global GLOBAL_B, D_CLIP, D_DINO, USE_HEAD
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer leg (profiling runs)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU port timing (profiling runs)")
    ap.add_argument("--batch", type=int, default=32768, help="global batch (default: BASELINE's 32768)")
    ap.add_argument("--clip-dim", type=int, default=512, help="CLIP embedding dim D (config 4: 768)")
    ap.add_argument("--dino-dim", type=int, default=768, help="DINOv2 feature dim (config 4: 1024)")
    ap.add_argument("--no-head", action="store_true", help="student = image features (no projection head)")
    ap.add_argument("--graph", action="store_true",
                    help="replay the loss forward / backward as CUDA graphs (dinosoft_b200.make_graphed); default: "
                         "only where the step is host-bound (per-rank block <= 2^28 similarity entries)")
    ap.add_argument("--no-graph", action="store_true", help="always time the eager step")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss terms and gradients of the last timed step as DIR/<name>.npy (float32; "
                         f"gradients with more than {DUMP_ROWS} rows keep a fixed seeded sample of rows)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    GLOBAL_B, D_CLIP, D_DINO, USE_HEAD = args.batch, args.clip_dim, args.dino_dim, not args.no_head
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
