"""DistillClipLoss on one GPU: `DistillClipLoss` (dsoft_distill_forward / _backward) against open_clip's
DistillClipLoss recipe run eagerly on the same GPU under bf16 autocast (four [B, B] logit matrices, softmax /
log_softmax, CE, autograd).

    python scripts/bench_distill.py                             # writes profiles/r09_bench_distill.json
    python scripts/bench_distill.py --batches 16384 --rounds 3 --out /tmp/d.json

Per batch B (a ViT-B student, D = --dim, against a ViT-L teacher, Dt = --tdim; unit-norm features, every caption near
its image, the student correlated with the teacher; s = 14.29, s_t = 100), the two arms run forward + backward of
contrastive + distill alternately in one process: --rounds rounds of --iters timed steps each after one warm-up step,
CUDA events around each round; the reported time is the median over rounds of the per-step time.  --module-only
batches run the module alone.  Per arm: peak torch.cuda.max_memory_allocated above the inputs and the largest
difference to the other arm (losses relative, gradients as max error over max magnitude).  The module's per-kernel
split comes from the library's profile slots in a separate pass.  A cell that did not run (out of memory) says "not
measured" and why.  The card name and power limit are read in the same run.

Arithmetic (not measured): this design executes 2 B^2 (5 D + 3 Dt) FLOP per step (forward: both products per
direction; G: both products once; two gradient GEMMs), the eager recipe 2 B^2 (6 D + 2 Dt) (four logit products, four
gradient products).
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

S, ST = 14.29, 100.0
PROFILE_SLOTS = {"forward_image_rows": 0, "forward_text_rows": 1, "gemm_image_rows": 3, "gemm_text_rows": 4,
                 "g_kernel": 7}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:  # noqa: BLE001 - the numbers stay usable, the card line says why it is missing
        return {"name": torch.cuda.get_device_name(0), "error": repr(e)}


def upstream_loss(img, txt, scale, dimg, dtxt, dscale):
    """open_clip DistillClipLoss.forward at world size 1 (get_logits of student and teacher, CE, dist_loss)."""
    lpi = scale * img @ txt.T
    lpt = scale * txt @ img.T
    dpi = dscale * dimg @ dtxt.T
    dpt = dscale * dtxt @ dimg.T
    labels = torch.arange(img.shape[0], device=img.device)
    contrastive = (F.cross_entropy(lpi, labels) + F.cross_entropy(lpt, labels)) / 2
    dist = lambda t, s: -(t.softmax(dim=1) * s.log_softmax(dim=1)).sum(dim=1).mean(dim=0)  # noqa: E731
    distill = (dist(dpi, lpi) + dist(dpt, lpt)) / 2
    return contrastive, distill


def make_inputs(B, D, Dt, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    dimg = F.normalize(torch.randn(B, Dt, device="cuda", generator=g), dim=-1)
    dtxt = F.normalize(dimg + 4.0 * torch.randn(B, Dt, device="cuda", generator=g) / Dt ** 0.5, dim=-1)
    proj = torch.randn(Dt, D, device="cuda", generator=g) / Dt ** 0.5  # the student sees a projection of the teacher
    img = F.normalize(dimg @ proj + 0.5 * torch.randn(B, D, device="cuda", generator=g) / D ** 0.5, dim=-1)
    txt = F.normalize(dtxt @ proj + 0.5 * torch.randn(B, D, device="cuda", generator=g) / D ** 0.5, dim=-1)
    return img, txt, dimg, dtxt


def run_arm(arm, mod, leaves, teacher, iters):
    """iters forward + backward steps; returns (ms per step, losses, grads, peak bytes above the start)."""
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        for t in leaves:
            t.grad = None
        if arm == "module":
            c, d = mod(leaves[0], leaves[1], leaves[2], *teacher)
        else:
            with torch.autocast("cuda", dtype=torch.bfloat16):
                c, d = upstream_loss(leaves[0], leaves[1], leaves[2], *teacher)
        (c + d).backward()
    e1.record()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    return (e0.elapsed_time(e1) / iters, (float(c.detach()), float(d.detach())),
            [t.grad.detach().clone() for t in leaves], peak)


def kernel_split(lib, mod, leaves, teacher, iters):
    """Mean ms per step of the module's kernels, from the library's profile slots (a separate, recorded pass)."""
    n = 16
    ms, cnt = (C.c_double * n)(), (C.c_int * n)()
    lib.dsoft_profile_enable(1)
    lib.dsoft_profile_read(ms, cnt, n)  # clears
    for _ in range(iters):
        for t in leaves:
            t.grad = None
        c, d = mod(leaves[0], leaves[1], leaves[2], *teacher)
        (c + d).backward()
    torch.cuda.synchronize()
    lib.dsoft_profile_read(ms, cnt, n)
    lib.dsoft_profile_enable(0)
    return {k: round(ms[v] / iters, 3) for k, v in PROFILE_SLOTS.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="16384,32768,65536")
    ap.add_argument("--module-only", default="131072")
    ap.add_argument("--dim", type=int, default=512)
    ap.add_argument("--tdim", type=int, default=768)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_bench_distill.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_distill needs a CUDA device")
    import dinosoft_b200 as pkg
    from dinosoft_b200 import _cabi

    result = {"card": card(), "dim": a.dim, "teacher_dim": a.tdim, "s": S, "s_t": ST, "rounds": a.rounds,
              "iters": a.iters, "rows": []}
    mod = pkg.DistillClipLoss()
    lib = _cabi.lib()
    batches = [(int(x), False) for x in a.batches.split(",") if x] + \
              [(int(x), True) for x in a.module_only.split(",") if x]
    for B, module_only in batches:
        img, txt, dimg, dtxt = make_inputs(B, a.dim, a.tdim)
        leaves = [img.clone().requires_grad_(True), txt.clone().requires_grad_(True),
                  torch.tensor(S, device="cuda", requires_grad=True)]
        teacher = (dimg, dtxt, torch.tensor(ST, device="cuda"))
        arms = {}
        for arm in ("module",) if module_only else ("module", "upstream_eager_bf16"):
            try:
                run_arm(arm, mod, leaves, teacher, 1)  # warm-up
                arms[arm] = {"ms": []}
            except torch.cuda.OutOfMemoryError as e:
                arms[arm] = {"not_measured": "out of memory: " + str(e).split("\n")[0][:200]}
            torch.cuda.empty_cache()
        outs = {}
        for _ in range(a.rounds):
            for arm, rec in arms.items():
                if "not_measured" in rec:
                    continue
                ms, losses, grads, peak = run_arm(arm, mod, leaves, teacher, a.iters)
                rec["ms"].append(ms)
                rec["peak_bytes"] = max(rec.get("peak_bytes", 0), peak)
                outs[arm] = (losses, grads)
                torch.cuda.empty_cache()
        row = {"B": B}
        if module_only:
            row["upstream_eager_bf16"] = {"ms": "not measured", "reason": "module-only batch"}
        for arm, rec in arms.items():
            if "not_measured" in rec:
                row[arm] = {"ms": "not measured", "peak_GiB": "not measured", "reason": rec["not_measured"]}
                continue
            med = statistics.median(rec["ms"])
            row[arm] = {"ms": round(med, 3), "ms_rounds": [round(x, 3) for x in rec["ms"]],
                        "peak_GiB": round(rec["peak_bytes"] / 2 ** 30, 2)}
        if "ms" in arms.get("module", {}):
            row["module"]["kernel_ms"] = kernel_split(lib, mod, leaves, teacher, a.iters)
        if len(outs) == 2:
            (l0, g0), (l1, g1) = outs["module"], outs["upstream_eager_bf16"]
            diff = {"contrastive_rel": abs(l0[0] - l1[0]) / abs(l1[0]), "distill_rel": abs(l0[1] - l1[1]) / abs(l1[1])}
            for name, x, y in zip(("d_image", "d_text", "d_scale"), g0, g1):
                y = y.float()
                diff[name] = float((x.float() - y).abs().max() / y.abs().max().clamp_min(1e-30))
            row["max_difference_module_vs_upstream"] = diff
        else:
            row["max_difference_module_vs_upstream"] = "not measured (one arm did not run)"
        result["rows"].append(row)
        print(json.dumps(row), flush=True)
        del img, txt, dimg, dtxt, leaves, teacher, outs
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["card"]))


if __name__ == "__main__":
    main()
