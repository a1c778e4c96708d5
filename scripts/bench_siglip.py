"""SigLIP loss on one GPU: `SigLipLoss` (dsoft_siglip_forward / _backward) against open_clip's SigLipLoss recipe run
eagerly on the same GPU under bf16 autocast (logits, labels matrix, logsigmoid, autograd).

    python scripts/bench_siglip.py                              # writes profiles/r08_bench_siglip.json
    python scripts/bench_siglip.py --batches 16384 --rounds 3 --out /tmp/s.json

Per batch B (D = --dim, unit-norm features with every caption near its image, s = 10, beta = -10), the two arms run
forward + backward alternately in one process: --rounds rounds of --iters timed steps each after one warm-up step,
CUDA events around each round; the reported time is the median over rounds of the per-step time.  Per arm: peak
torch.cuda.max_memory_allocated above the inputs, executed TFLOP/s (6 B^2 D: the logit product and the two gradient
products; neither arm recomputes), and the largest difference to the other arm (loss relative, gradients as max error
over max magnitude).  A cell that did not run (out of memory) says "not measured" and why.  The card name and power
limit are read in the same run.
"""
import argparse
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

S, BETA = 10.0, -10.0


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:  # noqa: BLE001 - the numbers stay usable, the card line says why it is missing
        return {"name": torch.cuda.get_device_name(0), "error": repr(e)}


def upstream_loss(img, txt, scale, bias):
    """open_clip SigLipLoss at world size 1 (_loss: get_logits, get_ground_truth, -logsigmoid(labels*logits).sum()/n)."""
    logits = scale * img @ txt.T
    logits += bias
    n = img.shape[0]
    labels = -torch.ones((n, n), device=img.device, dtype=img.dtype)
    labels = 2 * torch.eye(n, device=img.device, dtype=img.dtype) + labels
    return -F.logsigmoid(labels * logits).sum() / n


def make_inputs(B, D, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    img = F.normalize(torch.randn(B, D, device="cuda", generator=g), dim=-1)
    txt = F.normalize(img + 4.0 * torch.randn(B, D, device="cuda", generator=g) / D ** 0.5, dim=-1)
    return img, txt


def run_arm(arm, mod, leaves, iters):
    """iters forward + backward steps; returns (ms per step, loss, grads, peak bytes above the start)."""
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        for t in leaves:
            t.grad = None
        if arm == "module":
            loss = mod(*leaves)
        else:
            with torch.autocast("cuda", dtype=torch.bfloat16):
                loss = upstream_loss(*leaves)
        loss.backward()
    e1.record()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    return e0.elapsed_time(e1) / iters, float(loss.detach()), [t.grad.detach().clone() for t in leaves], peak


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="16384,32768,65536,131072")
    ap.add_argument("--dim", type=int, default=512)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_bench_siglip.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_siglip needs a CUDA device")
    import dinosoft_b200 as pkg

    result = {"card": card(), "dim": a.dim, "s": S, "beta": BETA, "rounds": a.rounds, "iters": a.iters, "rows": []}
    mod = pkg.SigLipLoss()
    for B in [int(x) for x in a.batches.split(",")]:
        img, txt = make_inputs(B, a.dim)
        leaves = [img.clone().requires_grad_(True), txt.clone().requires_grad_(True),
                  torch.tensor(S, device="cuda", requires_grad=True),
                  torch.tensor(BETA, device="cuda", requires_grad=True)]
        flops = 6.0 * B * B * a.dim
        arms = {}
        for arm in ("module", "upstream_eager_bf16"):
            try:
                run_arm(arm, mod, leaves, 1)  # warm-up
                arms[arm] = {"ms": []}
            except torch.cuda.OutOfMemoryError as e:
                arms[arm] = {"not_measured": "out of memory: " + str(e).split("\n")[0][:200]}
            torch.cuda.empty_cache()
        outs = {}
        for _ in range(a.rounds):
            for arm, rec in arms.items():
                if "not_measured" in rec:
                    continue
                ms, loss, grads, peak = run_arm(arm, mod, leaves, a.iters)
                rec["ms"].append(ms)
                rec["peak_bytes"] = max(rec.get("peak_bytes", 0), peak)
                outs[arm] = (loss, grads)
                torch.cuda.empty_cache()
        row = {"B": B}
        for arm, rec in arms.items():
            if "not_measured" in rec:
                row[arm] = {"ms": "not measured", "peak_GiB": "not measured", "tflops_executed": "not measured",
                            "reason": rec["not_measured"]}
                continue
            med = statistics.median(rec["ms"])
            row[arm] = {"ms": round(med, 3), "ms_rounds": [round(x, 3) for x in rec["ms"]],
                        "peak_GiB": round(rec["peak_bytes"] / 2 ** 30, 2),
                        "tflops_executed": round(flops / (med * 1e-3) / 1e12, 1)}
        if len(outs) == 2:
            (l0, g0), (l1, g1) = outs["module"], outs["upstream_eager_bf16"]
            diff = {"loss_rel": abs(l0 - l1) / abs(l1)}
            for name, x, y in zip(("d_image", "d_text", "d_scale", "d_bias"), g0, g1):
                y = y.float()
                diff[name] = float((x.float() - y).abs().max() / y.abs().max().clamp_min(1e-30))
            row["max_difference_module_vs_upstream"] = diff
        else:
            row["max_difference_module_vs_upstream"] = "not measured (one arm did not run)"
        result["rows"].append(row)
        print(json.dumps(row), flush=True)
        del img, txt, leaves, outs
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["card"]))


if __name__ == "__main__":
    main()
