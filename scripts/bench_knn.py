"""kNN classification on one GPU: `knn_classify` (dsoft_knn_topk, no N_query x N_key matrix) against DINO's chunked
`knn_classifier` recipe (fp32 `mm` of the L2-normalised features per query chunk, `topk`, weighted vote).

    python scripts/bench_knn.py                                   # writes profiles/r10_bench_knn.json
    python scripts/bench_knn.py --pools 2000x20000 --dtypes bf16 --rounds 2 --out /tmp/k.json

Features are clustered synthetic data: 1000 unit-norm class centres plus Gaussian noise of norm 4.5, labels uniform
(top-1 roughly 40 % at 100 train features per class).  Per pool and
input dtype both arms run at k in --ks (the kernel arm takes one top-k at max(k) for all of them, as knn_classify
does; the recipe arm runs once per k, as DINO's eval does), alternating in one process after one warm-up call each.
Reported per arm: the median and all round times (host clock around a synchronised call), the peak
torch.cuda.max_memory_allocated above the inputs, and the accuracies; the difference of the accuracies between the
arms is recorded.  A separate pass under torch.profiler splits the kernel arm's device time into the tile pass
(dsoft_fwd_kernel), the merge (knn_merge_kernel) and everything else.  The card name, power limit and maximum SM clock
are read in the same run.
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
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True

DTYPES = {"bf16": torch.bfloat16, "fp32": torch.float32}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:  # noqa: BLE001 - the numbers stay usable, the card line says why it is missing
        return {"name": torch.cuda.get_device_name(0), "error": repr(e)}


def make_pool(n_test, n_train, dim, classes, seed=0, noise=4.5):
    g = torch.Generator(device="cuda").manual_seed(seed)
    centres = torch.nn.functional.normalize(torch.randn(classes, dim, device="cuda", generator=g), dim=1)
    ytr = torch.randint(0, classes, (n_train,), device="cuda", generator=g)
    yte = torch.randint(0, classes, (n_test,), device="cuda", generator=g)
    xtr = torch.empty(n_train, dim, device="cuda")
    for r0 in range(0, n_train, 1 << 18):  # in pieces: the noise of the whole set would double the peak
        r1 = min(r0 + (1 << 18), n_train)
        xtr[r0:r1] = centres[ytr[r0:r1]] + noise * torch.randn(r1 - r0, dim, device="cuda", generator=g) / dim ** 0.5
    xte = centres[yte] + noise * torch.randn(n_test, dim, device="cuda", generator=g) / dim ** 0.5
    return xtr, ytr, xte, yte


def recipe(xtr, ytr, xte, yte, k, T, classes, chunk_rows=500):
    """DINO's knn_classifier: fp32 normalised features, one [chunk, N_train] score matrix per query chunk."""
    from knn_ref import dino_knn_classifier

    ntr = torch.nn.functional.normalize(xtr.float(), dim=1)
    nte = torch.nn.functional.normalize(xte.float(), dim=1)
    chunks = max(1, xte.shape[0] // chunk_rows)
    top1, top5 = dino_knn_classifier(ntr, ytr, nte, yte, k, T, num_classes=classes, chunk=chunks)
    return {f"knn_top1@{k}": top1, f"knn_top5@{k}": top5}


def timed_call(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, (time.perf_counter() - t0) * 1e3, torch.cuda.max_memory_allocated() - base


def profile_split(fn):
    """Device time of the kernel arm by kernel family, from one call under torch.profiler."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    split = {"tile_pass_ms": 0.0, "merge_ms": 0.0, "other_device_ms": 0.0}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if t <= 0:
            continue
        key = ("tile_pass_ms" if "dsoft_fwd_kernel" in ev.key else
               "merge_ms" if "knn_merge_kernel" in ev.key else "other_device_ms")
        split[key] += t / 1e3
    return split


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pools", default="10000x100000,50000x1281167", help="N_test x N_train, comma separated")
    ap.add_argument("--dtypes", default="bf16,fp32")
    ap.add_argument("--ks", default="10,20")
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--classes", type=int, default=1000)
    ap.add_argument("--T", type=float, default=0.07)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_bench_knn.json"))
    args = ap.parse_args()
    import dinosoft_b200 as pkg

    ks = [int(x) for x in args.ks.split(",")]
    result = {"card": card(), "dim": args.dim, "classes": args.classes, "T": args.T, "ks": ks,
              "rounds": args.rounds, "timing": "host clock around a synchronised call, median of the rounds; the "
              "two arms alternate after one warm-up call each", "pools": []}
    print(json.dumps(result["card"]))
    for pool in args.pools.split(","):
        n_test, n_train = [int(x) for x in pool.split("x")]
        for dname in args.dtypes.split(","):
            dtype = DTYPES[dname]
            xtr, ytr, xte, yte = make_pool(n_test, n_train, args.dim, args.classes, seed=n_train)
            xtr, xte = xtr.to(dtype), xte.to(dtype)
            torch.cuda.empty_cache()

            def kernel():
                return pkg.knn_classify(xtr, ytr, xte, yte, k=ks, T=args.T, num_classes=args.classes)

            def dino():
                out = {}
                for k in ks:
                    out.update(recipe(xtr, ytr, xte, yte, k, args.T, args.classes))
                return out

            entry = {"pool": pool, "dtype": dname, "flop_per_product": 2.0 * n_test * n_train * args.dim,
                     "products": 1 if dtype == torch.bfloat16 else 3}
            arms = {"kernel": kernel, "dino_recipe": dino}
            times = {a: [] for a in arms}
            peak = {a: 0 for a in arms}
            acc = {}
            for a, fn in arms.items():  # warm-up
                acc[a], _, peak[a] = timed_call(fn)
            for _ in range(args.rounds):
                for a, fn in arms.items():
                    acc[a], ms, pk = timed_call(fn)
                    times[a].append(round(ms, 3))
                    peak[a] = max(peak[a], pk)
            for a in arms:
                entry[a] = {"median_ms": round(statistics.median(times[a]), 3), "rounds_ms": times[a],
                            "peak_extra_mib": round(peak[a] / 2 ** 20, 1), "accuracy": acc[a]}
            entry["speedup"] = round(entry["dino_recipe"]["median_ms"] / entry["kernel"]["median_ms"], 2)
            entry["accuracy_difference"] = {key: acc["kernel"][key] - acc["dino_recipe"][key] for key in acc["kernel"]}
            entry["kernel_device_split"] = {k: round(v, 3) for k, v in profile_split(kernel).items()}
            tile_s = entry["kernel_device_split"]["tile_pass_ms"] / 1e3
            entry["tile_pass_pflops"] = round(entry["flop_per_product"] * entry["products"] / tile_s / 1e15, 3)
            print(json.dumps(entry))
            result["pools"].append(entry)
            del xtr, ytr, xte, yte
            torch.cuda.empty_cache()
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
