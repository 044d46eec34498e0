#!/usr/bin/env python
"""Cost of the coordinate gradient (ENF_FLAG_GRAD_X): the same backward with and without dx, alternated.

    python tools/grad_x_cost.py [--configs ns64,sw192,ihc] [--runs 3] [--steps 20] [--warmup 5] [--out FILE]

Per config (bench.py's CONFIGS, tensor-core precision, one shared coordinate grid as in bench.py) and per mode, `runs`
runs of `steps` training steps after warm-up, the two modes alternating run by run.  Timed per step, with CUDA events:
the whole backward (`out.backward`, from after the forward to the end of the last gradient), and the fused pair backward
kernels (prep + A + B + C, the library's enf_profile_collect ring).  Prints one JSON line per config plus the card's name
and power limit read in the same run; medians and [min, max] over the runs of the per-run mean step."""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, plim = (s.strip() for s in q.split(","))
        return {"name": name, "power_limit": plim}
    except Exception as e:            # the measurement stands without it, but says so
        return {"name": None, "power_limit": None, "error": repr(e)}


def measure(cfg_name, runs, steps, warmup):
    import torch
    import enf_pde_b200 as E
    from bench import CONFIGS
    from enf_pde_b200.latents import make_coords
    cfg = CONFIGS[cfg_name]
    dev = torch.device("cuda", 0)
    lib = E.load_library()
    inv = E.get_ca_invariant(types.SimpleNamespace(invariant_type=cfg["invariant_type"], num_in=cfg["num_in"]))
    nef = E.EquivariantCrossAttentionNeF(cfg["d"], cfg["H"], 0, cfg["O"], cfg["L"], inv, inv, "rff", cfg["freq"], True,
                                         cfg["window"], precision="bf16")
    gen = torch.Generator().manual_seed(1234)
    B, Z = cfg["B"], cfg["Z"]
    p_h, a_h, s_h = E.init_latents(inv, B, Z, cfg["L"], polar_grid=cfg["polar_grid"])
    p_h = p_h + 0.02 * torch.randn(p_h.shape, generator=gen)
    a_h = a_h + 0.1 * torch.randn(a_h.shape, generator=gen)
    x = make_coords(inv, cfg["grid"]).contiguous().to(dev)
    C = x.shape[0]
    variables = nef.init(0, x[None], p_h.to(dev), a_h.to(dev), s_h.to(dev))
    leaves = [t.requires_grad_(True) for t in E.params_to_leaves(variables)]
    p, a, s = (t.to(dev).requires_grad_(True) for t in (p_h, a_h, s_h))
    cot = torch.randn(B, C, cfg["O"], generator=gen).to(dev) / (B * C)
    sig = s if cfg["window"] else None

    def step(with_dx, ev):
        for t in leaves + [p, a, s]:
            t.grad = None
        xx = x.detach().requires_grad_(with_dx)
        out = nef.apply(variables, xx[None].expand(B, -1, -1), p, a, sig)
        ev[0].record()
        out.backward(cot)
        ev[1].record()
        return xx.grad

    res = {True: [], False: []}
    pairs = {True: [], False: []}
    buf = (ctypes.c_float * 256)()
    for mode in (False, True):
        for _ in range(warmup):
            step(mode, [torch.cuda.Event(enable_timing=True) for _ in range(2)])
    torch.cuda.synchronize()
    for r in range(runs):
        for mode in ((False, True) if r % 2 == 0 else (True, False)):
            evs = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(steps)]
            lib.enf_profile_enable(1)
            for i in range(steps):
                dx = step(mode, evs[i])
            torch.cuda.synchronize()
            n = lib.enf_profile_collect(1, buf, 256)
            lib.enf_profile_enable(0)
            assert n == steps, n
            assert (dx is not None) == mode
            res[mode].append(sum(e0.elapsed_time(e1) for e0, e1 in evs) / steps)
            pairs[mode].append(sum(buf[i] for i in range(n)) / n)
    summ = lambda v: {"median": round(statistics.median(v), 4), "min": round(min(v), 4), "max": round(max(v), 4)}
    bw0, bw1 = statistics.median(res[False]), statistics.median(res[True])
    pk0, pk1 = statistics.median(pairs[False]), statistics.median(pairs[True])
    return {"config": cfg_name, "B": B, "C": C, "Z": Z, "d": cfg["d"], "H": cfg["H"], "steps_per_run": steps, "runs": runs,
            "backward_ms": {"without_dx": summ(res[False]), "with_dx": summ(res[True])},
            "pair_backward_ms": {"without_dx": summ(pairs[False]), "with_dx": summ(pairs[True])},
            "backward_overhead_pct": round(100 * (bw1 - bw0) / bw0, 3),
            "pair_backward_overhead_pct": round(100 * (pk1 - pk0) / pk0, 3),
            "runs_ms": {"backward_without_dx": res[False], "backward_with_dx": res[True],
                        "pairs_without_dx": pairs[False], "pairs_with_dx": pairs[True]}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="ns64,sw192,ihc")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("grad_x_cost.py measures on a CUDA device; there is none")
    lines = [{"card": card()}] + [measure(c, args.runs, args.steps, args.warmup) for c in args.configs.split(",")]
    for l in lines:
        print(json.dumps(l))
    if args.out:
        with open(args.out, "a") as f:
            for l in lines:
                f.write(json.dumps(l) + "\n")


if __name__ == "__main__":
    main()
