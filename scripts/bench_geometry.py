"""Embedding geometry on one GPU: `embedding_geometry` / `image_text_geometry` (dsoft_geometry, no N x N matrix) against
Wang & Isola's pdist recipe and a chunked torch recipe on the same GPU.

    python scripts/bench_geometry.py                      # writes profiles/r11_bench_geometry.json
    python scripts/bench_geometry.py --cases one_flickr_img --rounds 2 --out /tmp/g.json

Cases (Flickr30k-sized pools, ImageNet-sized train set; features are clustered synthetic data, 1000 unit centres plus
Gaussian noise of norm 0.8, fp32 unless stated):
  one_flickr_img   one set 31 783 x 512: kernel, pdist recipe, chunked recipe
  one_flickr_txt   one set 158 915 x 512: kernel, chunked recipe (the pdist recipe fails to launch at this size)
  one_imagenet     one set 1 281 167 x 768 bf16: kernel only (the pdist recipe needs 8.2e11 fp32 distances, 3.3 TB
                   per intermediate, and the chunked recipe would take of the order of minutes per call)
  two_flickr       two sets 31 783 images x 158 915 captions (5 per image, caption map): kernel, chunked recipe
All arms compute uniformity at t = 2 and (except pdist) a 100-bin histogram over [-1, 1]; the two-set arms compute the
positive and negative histograms and the alignment at alpha = 2.  Arms alternate in one process after one warm-up call
each; reported per arm: the median and all round times (host clock around a synchronised call), the peak
torch.cuda.max_memory_allocated above the inputs, and the results.  A separate pass under torch.profiler gives the
kernel arm's tile-pass time (dsoft_fwd_kernel) and its rate 2 pairs K / time (K = d for bf16, 3 d for the split of
fp32 inputs).  The card name, power limit and maximum SM clock are read in the same run.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

T, BINS, ALPHA = 2.0, 100, 2.0
CASES = {
    "one_flickr_img": dict(n=31783, d=512, dtype="fp32", arms=["kernel", "pdist", "chunked"]),
    # torch.pdist does not run at this size: its launch fails with "CUDA error: invalid configuration argument"
    # (1.26e10 distances), before any memory limit is reached; that arm is recorded, not timed
    "one_flickr_txt": dict(n=158915, d=512, dtype="fp32", arms=["kernel", "chunked"],
                           note={"pdist": "fails: torch.pdist raises 'CUDA error: invalid configuration argument' "
                                          "at 158 915 rows (its launch grid), so it was not timed"}),
    "one_imagenet": dict(n=1281167, d=768, dtype="bf16", arms=["kernel"]),
    "two_flickr": dict(n_img=31783, n_txt=158915, d=512, dtype="fp32", arms=["kernel", "chunked"]),
}
DTYPES = {"bf16": torch.bfloat16, "fp32": torch.float32}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:  # noqa: BLE001 - the numbers stay usable, the card line says why it is missing
        return {"name": torch.cuda.get_device_name(0), "error": repr(e)}


def pool(n, d, dtype, seed, centres=None):
    g = torch.Generator(device="cuda").manual_seed(seed)
    if centres is None:
        centres = torch.nn.functional.normalize(torch.randn(1000, d, device="cuda", generator=g), dim=1)
    x = torch.empty(n, d, device="cuda", dtype=dtype)
    for r0 in range(0, n, 1 << 18):  # in pieces: the noise of the whole set would double the peak
        r1 = min(r0 + (1 << 18), n)
        x[r0:r1] = (centres[torch.randint(0, centres.shape[0], (r1 - r0,), device="cuda", generator=g)]
                    + 0.8 * torch.randn(r1 - r0, d, device="cuda", generator=g) / d ** 0.5).to(dtype)
    return x, centres


def pdist_recipe(x):
    """Wang & Isola's uniform_loss as written, fp32 on F.normalize'd rows."""
    xn = torch.nn.functional.normalize(x.float(), dim=-1)
    return {"uniformity": float(torch.pdist(xn, p=2).pow(2).mul(-T).exp().mean().log())}


def _histc(c):
    return torch.histc(c, BINS, -1.0, 1.0).to(torch.int64), (c < -1.0).sum(), (c > 1.0).sum()


def chunked_recipe(x, block=4096):
    """Row blocks of the fp32 cosine matrix (upper triangle): the exp sum in fp64, histc plus the out-of-range counts."""
    xn = torch.nn.functional.normalize(x.float(), dim=-1)
    n = xn.shape[0]
    esum = torch.zeros((), dtype=torch.float64, device="cuda")
    hist = torch.zeros(BINS, dtype=torch.int64, device="cuda")
    out = torch.zeros(2, dtype=torch.int64, device="cuda")
    for i0 in range(0, n, block):
        c = xn[i0:i0 + block] @ xn[i0:].t()
        c = c[torch.ones_like(c, dtype=torch.bool).triu_(1)]
        esum += torch.exp(2 * T * (c - 1)).sum(dtype=torch.float64)
        h, lo, hi = _histc(c)
        hist += h
        out += torch.stack([lo, hi])
    return {"uniformity": math.log(float(esum) / (n * (n - 1) // 2)), "hist_sum": int(hist.sum()),
            "below": int(out[0]), "above": int(out[1])}


def chunked_two(img, txt, tmap, block=8192):
    a = torch.nn.functional.normalize(img.float(), dim=-1)
    b = torch.nn.functional.normalize(txt.float(), dim=-1)
    pos = (a[tmap] * b).sum(1)
    neg = torch.zeros(BINS, dtype=torch.int64, device="cuda")
    for j0 in range(0, b.shape[0], block):
        c = a @ b[j0:j0 + block].t()
        mask = torch.ones_like(c, dtype=torch.bool)
        mask[tmap[j0:j0 + block], torch.arange(c.shape[1], device="cuda")] = False
        neg += _histc(c[mask])[0]
    return {"alignment": float((2 - 2 * pos).clamp_min(0).pow(ALPHA / 2).mean()),
            "pos_hist_sum": int(_histc(pos)[0].sum()), "neg_hist_sum": int(neg.sum())}


def timed(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    try:
        out = fn()
    except torch.OutOfMemoryError as e:
        torch.cuda.synchronize()
        return {"error": "out of memory: " + str(e).split("\n")[0]}, None, torch.cuda.max_memory_allocated() - base
    torch.cuda.synchronize()
    return out, (time.perf_counter() - t0) * 1e3, torch.cuda.max_memory_allocated() - base


def tile_time_ms(fn):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    us = sum(e.device_time_total for e in prof.key_averages() if "dsoft_fwd_kernel" in e.key)
    return us / 1e3


def summary(res):
    out = {}
    for k, v in res.items():
        if isinstance(v, torch.Tensor):
            out[k + "_sum"] = int(v.sum())
        else:
            out[k] = v
    return out


def run_case(name, spec, rounds, pkg):
    dtype = DTYPES[spec["dtype"]]
    d = spec["d"]
    if "n" in spec:
        x, _ = pool(spec["n"], d, dtype, 1)
        pairs = spec["n"] * (spec["n"] - 1) // 2
        fns = {"kernel": lambda: summary(pkg.embedding_geometry(x, t=T, bins=BINS)),
               "pdist": lambda: pdist_recipe(x), "chunked": lambda: chunked_recipe(x)}
        shape = {"n": spec["n"], "d": d}
    else:
        img, centres = pool(spec["n_img"], d, dtype, 1)
        tmap = torch.arange(spec["n_txt"], device="cuda") // 5
        txt = (img.float()[tmap] + 0.8 * torch.randn(spec["n_txt"], d, device="cuda") / d ** 0.5).to(dtype)
        pairs = spec["n_img"] * spec["n_txt"]
        fns = {"kernel": lambda: summary(pkg.image_text_geometry(img, txt, tmap, bins=BINS, alpha=ALPHA)),
               "chunked": lambda: chunked_two(img, txt, tmap)}
        shape = {"n_img": spec["n_img"], "n_txt": spec["n_txt"], "d": d, "captions_per_image": 5}
    arms = {a: {"ms": [], "peak_bytes_above_inputs": 0, "result": None} for a in spec["arms"]}
    dead = set()
    for r in range(rounds + 1):  # round 0 warms up every arm
        for a in spec["arms"]:
            if a in dead:
                continue
            out, ms, peak = timed(fns[a])
            arms[a]["result"] = out
            arms[a]["peak_bytes_above_inputs"] = max(arms[a]["peak_bytes_above_inputs"], peak)
            if ms is None:
                dead.add(a)
                continue
            if r:
                arms[a]["ms"].append(round(ms, 3))
            print(f"[{name}] {a} round {r}: {ms if ms is not None else 'OOM'} ms", flush=True)
    for a, v in arms.items():
        v["median_ms"] = statistics.median(v["ms"]) if v["ms"] else "not measured"
    k = d if dtype == torch.bfloat16 else 3 * d
    tile_ms = tile_time_ms(fns["kernel"])
    return {"case": name, **shape, **({"note": spec["note"]} if "note" in spec else {}), "dtype": spec["dtype"], "pairs": pairs, "arms": arms, "tile_pass_ms": tile_ms,
            "tile_pass_pflops": 2.0 * pairs * k / (tile_ms * 1e-3) / 1e15, "K": k}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default=",".join(CASES))
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11_bench_geometry.json"))
    args = ap.parse_args()
    import dinosoft_b200 as pkg

    report = {"card": card(), "t": T, "bins": BINS, "alpha": ALPHA, "rounds": args.rounds, "cases": []}
    for name in args.cases.split(","):
        report["cases"].append(run_case(name, CASES[name], args.rounds, pkg))
        torch.cuda.empty_cache()
        with open(args.out, "w") as f:
            json.dump(report, f, indent=1)
    print(json.dumps(report["card"]))


if __name__ == "__main__":
    main()
