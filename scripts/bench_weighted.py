"""Step time of the weighted CE branch (lambda_weighted > 0) on the default soft / text / MLP-head workload.

One process per GPU, like bench.py's multi-GPU lines:

    python scripts/bench_weighted.py                                   # 1 GPU
    torchrun --nproc_per_node 8 scripts/bench_weighted.py              # 8 GPUs, weighted_scope="global"

The global batch (default 32768) is split over the ranks.  Four arms run alternately in one process:
lambda_weighted = 0 (the branch off), 0.5 with weight_text_symmetry on, 0.5 with it off - these three under the
module's default backward choice (`DSOFT_GMAT=auto`: two-phase for weighted plans) - and 0.5 with symmetry on the
fused backward (`loss.GMAT = "never"` around that arm).  --arms picks a subset, e.g.

    python scripts/bench_weighted.py --batch 196608 --arms base,weighted_sym_fused --steps 2 --warmup 1 --rounds 2

Every arm's shape is warmed up first; then each round times every arm over --steps eager fwd+bwd steps with CUDA
events (rank 0's events, after a barrier), and --rounds rounds give the spread.  Rank 0 prints one JSON line per
world size with the median / min / max step ms and samples/s of every arm, the overhead of each weighted arm over the
baseline, the peak of torch.cuda.max_memory_allocated over the arm's timed steps, and the card name and power limit
read in the same call.  Writes nothing into the tree.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import types

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True

LOSS_ARGS = dict(use_projection=True, projection_type="mlp", lambda_soft=0.5, soft_mode="kl_teacher",
                 soft_dino_to_text=True, text_lambda=0.5, text_student_temp=0.02, teacher_temp=0.15,
                 lambda_original=1.0, rho=0.1, c_clip=1.0)
# name, lambda_weighted, weight_text_symmetry, loss.GMAT during the arm
ARMS = (("base", 0.0, False, "auto"), ("weighted_sym", 0.5, True, "auto"), ("weighted_nosym", 0.5, False, "auto"),
        ("weighted_sym_fused", 0.5, True, "never"))


def card(index):
    try:
        out = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:  # the timing itself does not depend on it
        return {"error": repr(e)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--batch", type=int, default=32768)
    ap.add_argument("--clip-dim", type=int, default=512)
    ap.add_argument("--dino-dim", type=int, default=768)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--arms", default=",".join(n for n, *_ in ARMS), help="comma-separated subset of the arms")
    a = ap.parse_args()
    want = a.arms.split(",")
    unknown = set(want) - {n for n, *_ in ARMS}
    if unknown:
        raise SystemExit(f"unknown arms {sorted(unknown)}")
    arms = [arm for arm in ARMS if arm[0] in want]

    from gpu_util import synth
    import dinosoft_b200 as pkg
    from dinosoft_b200 import loss as loss_mod

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench_weighted.py needs a CUDA sm_100 device")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert a.batch % world == 0
    b = a.batch // world
    img, txt, dino = synth(1234 + rank, b, a.clip_dim, a.dino_dim, device=dev)
    loss = pkg.ClipLossWithDINOEnhancements(local_loss=True, gather_with_grad=True, rank=rank, world_size=world,
                                            weighted_scope="global")
    torch.manual_seed(99)
    loss.init_proj(a.clip_dim, a.dino_dim, dev, "mlp")
    scale = torch.tensor(14.2857, device=dev, requires_grad=True)
    img.requires_grad_(True)
    txt.requires_grad_(True)
    params = list(loss.image_to_dino_proj.parameters())

    def step(larg):
        img.grad = txt.grad = scale.grad = None
        for p in params:
            p.grad = None
        loss_mod.GMAT = larg.gmat  # read by the forward when it picks the backward form
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = loss(img, txt, scale, dino, larg, output_dict=True)
        out["total_loss"].backward()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    largs = {n: types.SimpleNamespace(**dict(LOSS_ARGS, lambda_weighted=lw, weight_text_symmetry=ws, gmat=gm))
             for n, lw, ws, gm in arms}
    for n, *_ in arms:  # warm-up of every shape
        for _ in range(a.warmup):
            step(largs[n])
    barrier()
    ms = {n: [] for n, *_ in arms}
    peak = {n: 0 for n, *_ in arms}
    for _ in range(a.rounds):
        for n, *_ in arms:
            barrier()
            torch.cuda.reset_peak_memory_stats(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.steps):
                step(largs[n])
            e1.record()
            barrier()
            ms[n].append(e0.elapsed_time(e1) / a.steps)
            peak[n] = max(peak[n], torch.cuda.max_memory_allocated(dev))
    loss_mod.GMAT = "auto"
    if rank == 0:
        res = {"metric": "weighted_ce_step", "gpus": world, "global_batch": a.batch, "D": a.clip_dim,
               "Dd": a.dino_dim, "head": "mlp", "steps": a.steps, "rounds": a.rounds, "card": card(local_rank),
               "arms": {}}
        base = statistics.median(ms["base"]) if "base" in ms else None
        for n, lw, ws, gm in arms:
            med = statistics.median(ms[n])
            res["arms"][n] = {"lambda_weighted": lw, "weight_text_symmetry": ws, "gmat": gm,
                              "step_ms_median": round(med, 4),
                              "step_ms_min": round(min(ms[n]), 4), "step_ms_max": round(max(ms[n]), 4),
                              "samples_per_s": round(a.batch / (med / 1e3), 1),
                              "overhead_vs_base": None if base is None else round(med / base - 1.0, 4),
                              "peak_allocated_gib": round(peak[n] / 2 ** 30, 2)}
        print(json.dumps(res), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
