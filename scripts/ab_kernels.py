"""A/B of kernel variants selected by environment switches that libdsoft.so reads at plan creation
(DSOFT_CLIP_SYM, DSOFT_SYM_W, ...), in ONE process on one GPU so that both arms see the same
board, clocks and power state.  Arms alternate `--rounds` times; per arm: whole-step time (forked streams) and the
serial per-kernel times of the recorder (dsoft_profile_enable).

  python scripts/ab_kernels.py DSOFT_CLIP_SYM=0 DSOFT_CLIP_SYM=1 [--batch 32768] [--steps 10] [--rounds 3]
"""
import argparse
import ctypes as C
import json
import os
import sys
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("arms", nargs="+", help="VAR=value[,VAR=value...] per arm")
    ap.add_argument("--batch", type=int, default=32768)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    import dinosoft_b200 as pkg
    from dinosoft_b200 import _cabi
    from dinosoft_b200 import loss as loss_mod

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lib = _cabi.lib()
    img, txt, dino = bench.synth(1234, a.batch, bench.D_CLIP, bench.D_DINO, dev)
    larg = types.SimpleNamespace(**dict(bench.LOSS_ARGS, use_projection=True))
    loss = pkg.ClipLossWithDINOEnhancements(local_loss=True, gather_with_grad=True)
    torch.manual_seed(99)
    loss.init_proj(bench.D_CLIP, bench.D_DINO, dev, "mlp")
    params = list(loss.image_to_dino_proj.parameters())
    scale = torch.tensor(14.2857, device=dev, requires_grad=True)
    img.requires_grad_(True)
    txt.requires_grad_(True)

    def step():
        img.grad = txt.grad = scale.grad = None
        for p in params:
            p.grad = None
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = loss(img, txt, scale, dino, larg, output_dict=True)
        out["total_loss"].backward()
        return out

    def timed(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(n):
            out = step()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n, float(out["total_loss"].detach())

    res = {arm: {"step_ms": [], "kernels": []} for arm in a.arms}
    switches = {kv.split("=")[0] for arm in a.arms for kv in arm.split(",")}
    base_env = {k: os.environ.get(k) for k in switches}
    for rnd in range(a.rounds):
        for arm in a.arms:
            for k, v in base_env.items():  # a switch an arm does not name keeps the caller's value
                if v is None:
                    os.environ.pop(k, None)
                else:
                    os.environ[k] = v
            for kv in arm.split(","):
                k, v = kv.split("=")
                os.environ[k] = v
            be = loss_mod._cuda_backend
            if be is not None:
                be._plans.clear()  # the switches are read when a plan is created
            for _ in range(3):
                step()
            ms, lv = timed(a.steps)
            lib.dsoft_profile_enable(1)
            timed(a.steps)
            ms_sum = (C.c_double * bench.NK)()
            cnt = (C.c_int * bench.NK)()
            _cabi.check(lib.dsoft_profile_read(ms_sum, cnt, bench.NK), "dsoft_profile_read")
            lib.dsoft_profile_enable(0)
            kern = {n: round(ms_sum[i] / max(cnt[i], 1), 4) for i, n in enumerate(bench.KERNEL_NAMES) if cnt[i]}
            res[arm]["step_ms"].append(round(ms, 4))
            res[arm]["kernels"].append(kern)
            res[arm]["loss"] = lv
            print(f"[ab] round {rnd} {arm}: {ms:.3f} ms/step loss={lv:.6f} {kern}", file=sys.stderr, flush=True)
    out = {}
    for arm, r in res.items():
        ks = r["kernels"][0].keys()
        out[arm] = {"step_ms_min": min(r["step_ms"]), "step_ms": r["step_ms"], "loss": r["loss"],
                    "kernel_ms_min": {k: min(x[k] for x in r["kernels"]) for k in ks}}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
