"""Retrieval metrics on one GPU: `clip_metrics` (dsoft_retrieval_ranks, no logit matrix) against the open_clip
get_clip_metrics recipe (full logit matrix + torch.argsort in both directions).

    python scripts/bench_retrieval.py                      # writes profiles/r07_bench_retrieval.json
    python scripts/bench_retrieval.py --pools 1000x5000 --dtypes bf16 --out /tmp/r.json

Pools are N_img x N_txt with unit-norm random features of width --dim; a non-square pool gives every image
N_txt / N_img captions (t(j) = j mod N_img) and the argsort recipe then takes the first positive in each ranking,
which is get_clip_metrics itself for square pools.  Arms per pool and input dtype:

  * kernel        clip_metrics (host checks, operand split, ranks, metric reduction), host clock around a synchronised
                  call, median of --reps after one warm-up call;
  * argsort_gpu   logits on the GPU, torch.argsort on the GPU (where the matrix and the index tensors fit);
  * argsort_host  logits and argsort on the host, as get_clip_metrics does after `.cpu()` (pools up to --host-max
                  pairs only).

Each arm records its peak torch.cuda.max_memory_allocated above what the inputs hold, and the number of ranks in
which it differs from the kernel's (near-ties of the fp32 logits).  An arm that runs out of memory or is skipped is
reported as "not measured" with the reason.  The card name and power limit are read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:  # noqa: BLE001 - the numbers stay usable, the card line says why it is missing
        return {"name": torch.cuda.get_device_name(0), "error": repr(e)}


def make_pool(n_img, n_txt, dim, dtype, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    img = torch.nn.functional.normalize(torch.randn(n_img, dim, device="cuda", generator=g), dim=-1)
    t = torch.arange(n_txt, device="cuda") % n_img
    # noise of norm 4: positive scores ~0.24, five to six standard deviations of the negatives' (~dim^-1/2)
    txt = torch.nn.functional.normalize(img[t] + 4.0 * torch.randn(n_txt, dim, device="cuda", generator=g) / dim ** 0.5,
                                        dim=-1)
    return img.to(dtype), txt.to(dtype), (None if n_img == n_txt else t)


def argsort_ranks(img, txt, t):
    """The get_clip_metrics recipe on whatever device the features are: fp32 logits, argsort per direction, position
    of the first positive."""
    n_img, n_txt = img.shape[0], txt.shape[0]
    logits = img.float() @ txt.float().t()
    t = torch.arange(n_txt, device=img.device) if t is None else t.to(img.device)
    ranking = torch.argsort(logits, dim=1, descending=True)
    rank_img = (t[ranking] == torch.arange(n_img, device=img.device)[:, None]).int().argmax(1)
    del ranking
    ranking = torch.argsort(logits.t(), dim=1, descending=True)
    rank_txt = (ranking == t[:, None]).int().argmax(1)
    return rank_img, rank_txt


def timed(fn, reps, warmup=1):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        times.append((time.perf_counter() - t0) * 1e3)
    return out, times


def run_arm(fn, reps, warmup):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    try:
        out, times = timed(fn, reps, warmup)
    except torch.OutOfMemoryError as e:
        torch.cuda.empty_cache()
        return None, {"status": "not measured", "reason": f"out of memory: {str(e).splitlines()[0]}"}
    peak = torch.cuda.max_memory_allocated() - base
    return out, {"status": "measured", "ms_median": statistics.median(times), "ms_min": min(times),
                 "ms_max": max(times), "reps": len(times), "peak_alloc_bytes": int(peak)}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--pools", default="1000x5000,5000x25000,32768x32768,131072x131072")
    ap.add_argument("--dtypes", default="bf16,fp32")
    ap.add_argument("--dim", type=int, default=512)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--argsort-reps", type=int, default=3)
    ap.add_argument("--host-max", type=float, default=5e6, help="largest pool (pairs) timed on the host")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_bench_retrieval.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_retrieval.py needs a CUDA device")
    import dinosoft_b200 as pkg
    from dinosoft_b200.retrieval import metrics_from_ranks

    dtypes = {"bf16": torch.bfloat16, "fp32": torch.float32}
    res = {"card": card(), "dim": args.dim, "torch": torch.__version__, "rows": []}
    for spec in args.pools.split(","):
        n_img, n_txt = (int(x) for x in spec.lower().split("x"))
        for dname in args.dtypes.split(","):
            img, txt, t = make_pool(n_img, n_txt, args.dim, dtypes[dname])
            row = {"pool": f"{n_img}x{n_txt}", "dtype": dname, "n_img": n_img, "n_txt": n_txt,
                   "logit_matrix_bytes": 4 * n_img * n_txt}
            ranks = pkg.retrieval_ranks(img, txt, t)
            _, row["kernel"] = run_arm(lambda: pkg.clip_metrics(img, txt, text_image=t), args.reps, 1)
            row["metrics"] = metrics_from_ranks(*ranks)
            ref, row["argsort_gpu"] = run_arm(lambda: argsort_ranks(img, txt, t), args.argsort_reps, 1)
            if ref is not None:
                row["argsort_gpu"]["ranks_differing"] = int((ref[0] != ranks[0]).sum() + (ref[1] != ranks[1]).sum())
            del ref
            torch.cuda.empty_cache()
            if n_img * n_txt <= args.host_max:
                hi, ht, hm = img.cpu(), txt.cpu(), (None if t is None else t.cpu())
                t0 = time.perf_counter()
                href = argsort_ranks(hi, ht, hm)
                row["argsort_host"] = {"status": "measured", "ms": (time.perf_counter() - t0) * 1e3, "reps": 1,
                                       "ranks_differing": int((href[0] != ranks[0].cpu()).sum()
                                                              + (href[1] != ranks[1].cpu()).sum())}
            else:
                row["argsort_host"] = {"status": "not measured", "reason": f"pool above --host-max {args.host_max:g}"}
            print(json.dumps(row), flush=True)
            res["rows"].append(row)
            del img, txt, t, ranks
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"card": res["card"], "out": args.out}))


if __name__ == "__main__":
    main()
