#!/usr/bin/env python
"""Training-step cost of num_heads on the tensor-core path: bf16 (tcgen05 pair kernels, head groups beyond two heads) against
the fp32 pair kernels on the same description, alternated.

    python tools/heads_cost.py [--cases ns64:2,3,4/plane64:2,3,4/ihc:3,4] [--runs 3] [--steps 10] [--fp32-steps 3]
                               [--warmup 2] [--out FILE]

Per case (bench.py's CONFIGS with num_heads overridden; one shared coordinate grid as in bench.py) and per precision,
`runs` runs of `steps` fwd + bwd steps with every weight gradient after warm-up, the two precisions alternating run by run.
Timed per step with CUDA events from before the forward to after the backward, and separately the fused pair kernels of the
forward (every head group) and of the backward (prep, kernels A per head group, B, C; the library's enf_profile_collect
ring).  Prints one JSON line per case plus the card's name and power limit read in the same run; medians and [min, max]
over the runs of the per-run mean step."""
import argparse
import ctypes
import json
import os
import statistics
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from grad_x_cost import card  # noqa: E402


def measure(cfg_name, H, runs, steps, fp32_steps, warmup):
    import torch
    import enf_pde_b200 as E
    from enf_pde_b200 import _lib
    from bench import CONFIGS
    from enf_pde_b200.latents import make_coords
    cfg = CONFIGS[cfg_name]
    dev = torch.device("cuda", 0)
    lib = E.load_library()
    inv = E.get_ca_invariant(types.SimpleNamespace(invariant_type=cfg["invariant_type"], num_in=cfg["num_in"]))
    nefs = {prec: E.EquivariantCrossAttentionNeF(cfg["d"], H, 0, cfg["O"], cfg["L"], inv, inv, "rff", cfg["freq"], True,
                                                 cfg["window"], precision=prec) for prec in ("bf16", "fp32")}
    gen = torch.Generator().manual_seed(1234)
    B, Z = cfg["B"], cfg["Z"]
    p_h, a_h, s_h = E.init_latents(inv, B, Z, cfg["L"], polar_grid=cfg["polar_grid"])
    p_h = p_h + 0.02 * torch.randn(p_h.shape, generator=gen)
    a_h = a_h + 0.1 * torch.randn(a_h.shape, generator=gen)
    x = make_coords(inv, cfg["grid"]).contiguous().to(dev)
    C = x.shape[0]
    variables = nefs["bf16"].init(0, x[None], p_h.to(dev), a_h.to(dev), s_h.to(dev))
    leaves = [t.requires_grad_(True) for t in E.params_to_leaves(variables)]
    p, a, s = (t.to(dev).requires_grad_(True) for t in (p_h, a_h, s_h))
    cot = torch.randn(B, C, cfg["O"], generator=gen).to(dev) / (B * C)
    sig = s if cfg["window"] else None
    desc = _lib.EnfDesc(B=B, C=C, Z=Z, d=cfg["d"], H=H, L=cfg["L"], O=cfg["O"], Dx=cfg["num_in"],
                        invariant_kind=_lib.INVARIANT_KINDS[cfg["invariant_type"]], use_window=int(cfg["window"]), precision=1, flags=0)
    dispatch = _lib.dispatch(desc)
    assert dispatch == (True, True), dispatch            # the bf16 arm runs the tcgen05 kernels, not the fp32 fallback

    def step(prec, ev):
        for t in leaves + [p, a, s]:
            t.grad = None
        ev[0].record()
        out = nefs[prec].apply(variables, x[None].expand(B, -1, -1), p, a, sig)
        out.backward(cot)
        ev[1].record()

    res = {"bf16": [], "fp32": []}
    pf = {"bf16": [], "fp32": []}
    pb = {"bf16": [], "fp32": []}
    launches = {}
    buf = (ctypes.c_float * 256)()
    for prec in ("bf16", "fp32"):
        for _ in range(warmup):
            step(prec, [torch.cuda.Event(enable_timing=True) for _ in range(2)])
        launches[prec] = E.last_launch_counts()
    torch.cuda.synchronize()
    for r in range(runs):
        for prec in (("bf16", "fp32") if r % 2 == 0 else ("fp32", "bf16")):
            n_steps = steps if prec == "bf16" else fp32_steps
            evs = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(n_steps)]
            lib.enf_profile_enable(1)
            for i in range(n_steps):
                step(prec, evs[i])
            torch.cuda.synchronize()
            nf = lib.enf_profile_collect(0, buf, 256)
            pf[prec].append(sum(buf[i] for i in range(nf)) / nf)
            nb = lib.enf_profile_collect(1, buf, 256)
            pb[prec].append(sum(buf[i] for i in range(nb)) / nb)
            lib.enf_profile_enable(0)
            assert nf == n_steps and nb == n_steps, (nf, nb)
            res[prec].append(sum(e0.elapsed_time(e1) for e0, e1 in evs) / n_steps)
    summ = lambda v: {"median": round(statistics.median(v), 3), "min": round(min(v), 3), "max": round(max(v), 3)}
    return {"config": cfg_name, "B": B, "C": C, "Z": Z, "d": cfg["d"], "H": H, "runs": runs,
            "steps_per_run": {"bf16": steps, "fp32": fp32_steps},
            "step_ms": {k: summ(v) for k, v in res.items()},
            "pair_fwd_ms": {k: summ(v) for k, v in pf.items()},
            "pair_bwd_ms": {k: summ(v) for k, v in pb.items()},
            "speedup_bf16_over_fp32": round(statistics.median(res["fp32"]) / statistics.median(res["bf16"]), 2),
            "launches_fwd_bwd": launches,
            "runs_ms": {"step": res, "pair_fwd": pf, "pair_bwd": pb}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="ns64:2,3,4/plane64:2,3,4/ihc:3,4")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--fp32-steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("heads_cost.py measures on a CUDA device; there is none")
    cases = [(c.split(":")[0], int(h)) for c in args.cases.split("/") for h in c.split(":")[1].split(",")]
    lines = [{"card": card()}]
    for name, H in cases:
        lines.append(measure(name, H, args.runs, args.steps, args.fp32_steps, args.warmup))
        print(json.dumps(lines[-1]), flush=True)
    print(json.dumps(lines[0]))
    if args.out:
        with open(args.out, "a") as f:
            for l in lines:
                f.write(json.dumps(l) + "\n")


if __name__ == "__main__":
    main()
