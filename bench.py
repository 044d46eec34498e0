#!/usr/bin/env python
"""Benchmark of the ENF steerable cross-attention hot path (forward + backward), BASELINE.json's metric.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config ns64] [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic fields: `nef.apply` (fused cross
attention + decode MLP) followed by the full reverse pass (latent gradients dp, da, dsigma AND all
weight gradients) for an MSE loss against synthetic targets.  Prints ONE JSON line (rank 0).

  value     device-timed throughput, inputs resident in HBM                [coord-queries / s, whole job]
  e2e       same, through the public API from pinned HOST buffers, H2D of the step's inputs and D2H of
            loss + latent gradients inside the timed region
  roofline  the dominant kernel (fused pair backward): algorithmic FLOP / live CUDA-event kernel time,
            against the measured dense bf16 tensor peak (MEASURED_PEAKS.json)
  cpu_baseline  the oracle (PyTorch-CPU fp32 restatement of the reference graph; JAX is not installable in
            this image) timed on this box's host cores on a bounded sample of the same workload

N > 1 (torchrun, one process per GPU): fields shard across ranks with no data-path collective (weak scaling,
per-rank batch fixed); the outer-loop weight gradients are all-reduced with NCCL inside the timed step.
  --scaling strong      the config's global batch is SPLIT over the ranks (total work fixed)
  --partition queries   every rank takes all fields and a slice of the coordinate queries (SURVEY 8e fallback for fewer
                        fields than ranks); latent gradients join the weight gradients in the all-reduce
  --forward-only        validation / visualisation roll-out (SURVEY 8f-2): `nef.apply` under no_grad over --fields signals
  --recompute           bounded-memory training (ENF_FLAG_RECOMPUTE), chunk size --chunk-fields
"""
import argparse
import ctypes
import json
import math
import os
import sys
import threading
import time
import types

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "coord-queries/sec (ENF cross-attn fwd+bwd)"
UNIT = "queries/s"

# BASELINE.json configs (SURVEY.md section 8d).  configs[1] (ns64) is the one the metric is quoted on.
CONFIGS = {
    "plane64": dict(label="2D planar heat diffusion 64x64, 25 latents", invariant_type="ponita", num_in=2, d=64, H=2, L=16, O=1,
                    B=32, grid=(64, 64), Z=25, freq=(0.05, 0.01), window=True, polar_grid=None),
    "ns64": dict(label="2D Navier-Stokes 64x64 vorticity, 64 latents, batch 32 fields", invariant_type="rel_pos_periodic",
                 num_in=2, d=128, H=2, L=16, O=1, B=32, grid=(64, 64), Z=64, freq=(0.05, 0.1), window=True, polar_grid=None),
    "sphere": dict(label="spherical diffusion 128x64 lat-lon, 18 latents", invariant_type="polar_periodic", num_in=2, d=16, H=2,
                   L=4, O=1, B=8, grid=(128, 64), Z=18, freq=(0.01, 0.01), window=False, polar_grid=(6, 3)),
    "sw192": dict(label="shallow water 192x96 sphere, 144 latents", invariant_type="latitude_periodic", num_in=2, d=128, H=2,
                  L=32, O=3, B=4, grid=(192, 96), Z=144, freq=(0.05, 0.2), window=True, polar_grid=(16, 9)),
    "ihc": dict(label="3D IHC ball 64x40x40 coords, 256 latents", invariant_type="ball", num_in=3, d=32, H=3, L=32, O=1,
                B=1, grid=(64, 40, 40), Z=256, freq=(0.2, 0.5), window=True, polar_grid=None),
}


def flops_per_pair(cfg, I):
    d, H = cfg["d"], cfg["H"]
    alg = 2 * I * d + (6 + 6 * H) * d * d + 4 * H * d          # SURVEY 8d contract figure (after the survey's folds)
    ref = 2 * I * d + (10 + 10 * H) * d * d                     # reference graph as written
    return alg, ref


def flops_per_query_tail(cfg):
    d, H, O = cfg["d"], cfg["H"], cfg["O"]
    return 2 * H * d * d + 6 * (H * d) ** 2 + 2 * H * d * d + 2 * d * d + 2 * d * O


def pipe_times(cfg, I, pairs, queries, peaks, passes=3.0, sm_mhz=1965.0):
    """Seconds each pipe needs for one step at 100 % (SURVEY 8d): tensor (contract FLOP / measured dense 16-bit peak), MUFU
    ((2+H) d transcendentals per pair and pass-pair, 16 / clk / SM), fp32 FMA (the element-wise epilogue work, ~(40+20H) d flop
    per pair forward, 256 flop / clk / SM).  passes: 3 = fwd + bwd, 1 = forward only."""
    f_alg, _ = flops_per_pair(cfg, I)
    d, H = cfg["d"], cfg["H"]
    clk = sm_mhz * 1e6
    tensor = passes * (f_alg * pairs + flops_per_query_tail(cfg) * queries) / (peaks["bf16_sustained"] * 1e12)
    mufu = (2.0 if passes > 1 else 1.0) * (2 + H) * d * pairs / (16 * 148 * clk)      # x2 for fwd + bwd (SURVEY 8d)
    fma = passes * (40 + 20 * H) * d * pairs / (256 * 148 * clk)
    return {"tensor": tensor, "mufu": mufu, "fma": fma}


FP32_FMA_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12        # 74.4: 128 fp32 FMA lanes / SM / clk at the measured max SM clock


def read_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            pk = json.load(f)
        return dict(bf16_sustained=pk.get("bf16_tflops_sustained", 1400.0), bf16_burst=pk.get("bf16_tflops", 1590.0),
                    hbm=pk.get("hbm_gbs", 6650.0), source="measured (MEASURED_PEAKS.json)")
    return dict(bf16_sustained=1400.0, bf16_burst=1590.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


DUMP_BYTES = 64 << 20           # --dump-outputs: everything one run writes, .npy headers included


def dump_outputs(out_dir, arrays):
    """--dump-outputs: each named tensor -> out_dir/<name>.npy, float64 kept, every other dtype as float32, so that two builds
    can be compared output for output.  When the tensors hold more than DUMP_BYTES together, each keeps the same fraction of its
    elements: the flattened tensor at sorted indices drawn from a generator seeded with 0, the same sample for the same shapes."""
    import numpy as np
    import torch
    arrays = {k: v.detach() for k, v in arrays.items() if v is not None}
    size = lambda t: t.numel() * (8 if t.dtype == torch.float64 else 4)
    keep = min(1.0, (DUMP_BYTES - 256 * len(arrays)) / max(1, sum(size(t) for t in arrays.values())))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        if keep < 1.0:
            n = t.numel()
            idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:int(n * keep)].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        t = t if t.dtype == torch.float64 else t.float()
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())
    print(f"bench.py: wrote {len(arrays)} arrays to {out_dir}" + (f" (a seeded sample of {keep:.3g} of each)" if keep < 1.0 else ""),
          file=sys.stderr)


class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU during the timed region (NVML, 10 ms period)."""

    def __init__(self, index):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._thr = None

    def _run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                     "hw_power_brake": 0x80, "sync_boost": 0x10, "applications_clocks_setting": 0x2}
            while not self._stop.is_set():
                self.samples.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                try:
                    mask = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    mask = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for n, bit in names.items():
                    if mask & bit:
                        self.reasons.add(n)
                self._stop.wait(0.01)
        except Exception as e:          # noqa: BLE001
            self.reasons.add(f"sampler_error:{type(e).__name__}")

    def __enter__(self):
        self._thr = threading.Thread(target=self._run, daemon=True)
        self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._thr.join(timeout=2)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ---------------------------------------------------------------------------------------------------------
# CPU leg: the oracle on host cores (cpu_baseline / --impl reference)
# ---------------------------------------------------------------------------------------------------------

def cpu_leg(cfg, steps, warmup, budget_s=25.0):
    """budget_s: stop after this many seconds once two steps are timed (None: time all `steps`)."""
    import torch
    from oracle import enf_ref as R
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ocfg = R.EnfConfig(num_in=cfg["num_in"], num_hidden=cfg["d"], num_heads=cfg["H"], num_out=cfg["O"], latent_dim=cfg["L"],
                       invariant_type=cfg["invariant_type"], embedding_freq_multiplier=cfg["freq"],
                       use_gaussian_window=cfg["window"])
    # bounded sample of the same workload: same Z, d, H, invariant; fewer fields and queries (the unfused graph
    # materialises ~20 (B,C,Z,2Hd) fp32 tensors; the reference itself sub-samples to 512..10000 queries per step)
    Bs = min(cfg["B"], 2)
    per_pair_bytes = 4 * 2 * cfg["H"] * cfg["d"] * 24
    Cs = int(max(64, min(512, (3 << 30) // (per_pair_bytes * cfg["Z"] * Bs))))
    dt = torch.float32
    params = R.nef_init(ocfg, seed=0, dtype=dt)
    p, a, sigma = R.init_latents(ocfg, Bs, cfg["Z"], polar_grid=cfg["polar_grid"], dtype=dt, jitter=0.02)
    coords = R.make_coords(ocfg, cfg["grid"], dtype=dt)
    g = torch.Generator().manual_seed(0)
    idx = torch.randperm(coords.shape[0], generator=g)[:Cs]
    x = coords[idx][None].expand(Bs, -1, -1)
    y = torch.randn(Bs, Cs, cfg["O"], generator=g, dtype=dt)

    def step():
        P = R.tree_map(lambda t: t.detach().requires_grad_(True), params)
        pp, aa, ss = p.clone().requires_grad_(True), a.clone().requires_grad_(True), sigma.clone().requires_grad_(True)
        out = R.nef_apply(ocfg, P, x, pp, aa, ss)
        loss = ((out - y) ** 2).mean()
        loss.backward()
        return float(loss.detach())

    for _ in range(max(1, min(warmup, 2))):
        step()
    times = []
    t_start = time.perf_counter()
    for i in range(steps):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
        if budget_s is not None and time.perf_counter() - t_start > budget_s and i >= 1:
            break
    tot = sum(times)
    return dict(value=Bs * Cs * len(times) / tot, unit=UNIT, cores=cores, kind="port",
                sample=f"{Bs} fields x {Cs} queries x {cfg['Z']} latents per step (same d,H,invariant), {len(times)} steps, "
                       f"PyTorch-CPU fp32 restatement of the reference graph with autograd (JAX not installable here)",
                ms_per_step=1e3 * tot / len(times), steps=len(times))


# ---------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------

def reference_probe():
    """BASELINE.md section 4: prefer the real reference (JAX CPU backend) when it can be imported -- from the environment or
    from a driver-provided install under baseline/_ref -- else the oracle port.  Returns (kind, why)."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if os.path.isdir(ref_dir) and ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    try:
        import jax      # noqa: F401
        import flax     # noqa: F401
    except Exception as e:      # noqa: BLE001
        return "port", f"jax/flax not importable here ({type(e).__name__}); timing the PyTorch-CPU restatement (oracle/enf_ref.py)"
    if not os.path.isdir("/root/reference") and not os.path.isdir(os.path.join(ref_dir, "enf")):
        return "port", "jax present but the reference sources are not on this box; timing the oracle port"
    return "reference", "jax importable: the reference modules could be timed on JAX_PLATFORMS=cpu"


def ode_line(args):
    """`--ode`: one call of the latent ODE model (PonitaODEGen, ponita_ode_g.py) forward + vector-Jacobian product with all weight
    gradients -- the model evaluation the ODE phase takes per solver stage (pde_trainer.py:299,328) -- at the Navier-Stokes
    experiment's sizes: 64 latents, hidden 128, 3 layers, basis 64, degree 3 (340 tensor-power features of the 4 periodic
    invariants), 32 latent sets (= 8 signals x 4 time steps).  Not the headline metric: a row of SURVEY 8f."""
    import torch
    import enf_pde_b200 as E
    from oracle import enf_ref as R
    from oracle import ode_ref as O
    assert torch.cuda.is_available(), "bench.py --ode needs a CUDA device"
    dev = torch.device("cuda", 0)
    B, Z, L = args.fields or 32, 64, 16
    ocfg = O.OdeConfig(invariant_type="rel_pos_periodic", num_in=2, num_hidden=128, num_layers=3, latent_dim=L, basis_dim=64, degree=3,
                       widening_factor=2)
    inv = E.get_sa_invariant(types.SimpleNamespace(invariant_type="rel_pos_periodic", num_in=2))
    model = E.PonitaODEGen(128, 3, L, 1, inv, 64, 3, 2)
    gen = torch.Generator().manual_seed(7)
    p_h = torch.as_tensor(R.init_positions_grid(B, Z, 2), dtype=torch.float32) + 0.02 * torch.randn(B, Z, 2, generator=gen)
    a_h = 1.0 + 0.3 * torch.randn(B, Z, L, generator=gen)
    cp_h, ca_h = torch.randn(B, Z, 2, generator=gen), torch.randn(B, Z, L, generator=gen)
    variables = model.init(0, (p_h,), device=dev)
    leaves = R.tree_flatten(variables["params"])
    for t in leaves.values():
        t.requires_grad_(True)
    pin = lambda t: t.pin_memory()
    p_pin, a_pin, cp_pin, ca_pin = map(pin, (p_h, a_h, cp_h, ca_h))
    out_pin = torch.empty(B, Z, 2 + L).pin_memory()
    p_d, a_d, cp_d, ca_d = (t.to(dev) for t in (p_h, a_h, cp_h, ca_h))
    last = {}           # --dump-outputs: model output and latent gradients of the latest device-resident step

    def step(e2e):
        if e2e:
            pp, aa = p_pin.to(dev, non_blocking=True).requires_grad_(True), a_pin.to(dev, non_blocking=True).requires_grad_(True)
            cp, ca = cp_pin.to(dev, non_blocking=True), ca_pin.to(dev, non_blocking=True)
        else:
            pp, aa, cp, ca = p_d.detach().requires_grad_(True), a_d.detach().requires_grad_(True), cp_d, ca_d
        for t in leaves.values():
            t.grad = None
        dp, da, _ = model.apply(variables, (pp, aa, None))
        ((dp * cp).sum() + (da * ca).sum()).backward()
        if e2e:
            out_pin.copy_(torch.cat([pp.grad, aa.grad], -1), non_blocking=True)
        elif args.dump_outputs:
            last.update(dp_dt=dp.detach(), da_dt=da.detach(), grad_p=pp.grad, grad_a=aa.grad)

    def timed(e2e):
        for _ in range(max(3, args.warmup)):
            step(e2e)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            step(e2e)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.steps

    with ClockSampler(0) as sampler:
        ms = timed(False)
        if args.dump_outputs:       # the end-to-end steps rebind, not overwrite, these gradients
            outputs = {**last, **{"grad_" + k.replace("/", "."): t.grad for k, t in leaves.items()}}
        ms_e2e = timed(True)
    clocks = sampler.summary()
    n, m, F, Hd, Bd, NL, W = B * Z * Z, B * Z, ocfg.poly_dim, 128, 64, 3, 256
    flop_fwd = 2.0 * n * (F * Hd + Hd * Bd + NL * (Bd * Hd + Hd)) + 2.0 * m * (L * Hd + NL * 2 * Hd * W + Hd * (L + 2))
    peak = 148 * 128 * 2 * 1.965e9 / 1e12            # fp32 FMA peak of one B200, TFLOP/s (no measured figure in MEASURED_PEAKS.json)
    ach = 3 * flop_fwd / (ms * 1e-3) / 1e12
    # CPU baseline: the oracle restatement in fp32 on the host cores, same sizes, bounded sample
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    Bs = min(B, 4)
    params32 = O.ode_init(ocfg, seed=0, dtype=torch.float32, readout_scale=1e6)

    def cpu_step():
        P = R.tree_map(lambda t: t.detach().requires_grad_(True), params32)
        pp, aa = p_h[:Bs].clone().requires_grad_(True), a_h[:Bs].clone().requires_grad_(True)
        dp, da = O.ponita_ode(ocfg, P, pp, aa)
        ((dp * cp_h[:Bs]).sum() + (da * ca_h[:Bs]).sum()).backward()

    cpu = None
    if not args.no_cpu_baseline:
        cpu_step()
        t0, k = time.perf_counter(), 0
        while k < 3 or (time.perf_counter() - t0 < 10.0 and k < 50):
            cpu_step(); k += 1
        cpu = {"value": Bs * k / (time.perf_counter() - t0), "unit": "latent sets/s", "cores": cores, "kind": "port",
               "sample": f"{Bs} latent sets x 64 latents per step, {k} steps, PyTorch-CPU fp32 restatement (oracle/ode_ref.py) with autograd"}
    line = {"metric": "latent-ODE model evaluations/sec (PonitaODEGen fwd+bwd)", "value": B / (ms * 1e-3), "unit": "latent sets/s", "n_gpus": 1,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "latent ODE model at config_navier_stokes.yaml `node:` sizes", "B": B, "Z": Z, "hidden": Hd, "layers": NL,
                       "basis": Bd, "degree": 3, "poly_features": F, "invariant": "rel_pos_periodic (self-attention variant)",
                       "l2": "working set (pair-row activations, %.0f MB) > 126 MB L2" % (model_ws_mb(model, p_d, a_d))},
            "roofline": {"bound": "fp32-fma", "kernel": "enf_gemm_kernel (pair-row Dense layers) + ode_* kernels", "achieved": ach, "peak": peak,
                         "unit": "TFLOP/s", "frac": ach / peak, "traffic": None, "peak_source": "nominal fp32 FMA rate (148 SMs x 128 lanes x 2 x 1.965 GHz)",
                         "algorithmic_flop_per_step": 3 * flop_fwd},
            "cpu_baseline": cpu, "clocks": clocks,
            "e2e": {"value": B / (ms_e2e * 1e-3), "unit": "latent sets/s", "h2d_bytes_per_step": 4 * 2 * (p_h.numel() + a_h.numel()),
                    "d2h_bytes_per_step": 4 * out_pin.numel(), "ms_per_step": ms_e2e}}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line))


def meta_line(args):
    """`--meta`: one first-order Meta-SGD training step of PDETrainer (pde_trainer.py:122-235, 237-288) at the config's full
    size: K = 3 inner steps (nef.apply + latents-only backward + SGD update of p, a per field) from the shared latents, then the
    reconstruction loss of the adapted latents and its backward with all weight gradients.  4 forward + 4 backward passes over
    all B x C queries per step; the metric counts the B x C queries once per step."""
    import torch
    import enf_pde_b200 as E
    from enf_pde_b200 import _lib
    cfg = dict(CONFIGS[args.config])
    assert torch.cuda.is_available(), "bench.py --meta needs a CUDA device"
    dev = torch.device("cuda", 0)
    inv = E.get_ca_invariant(types.SimpleNamespace(invariant_type=cfg["invariant_type"], num_in=cfg["num_in"]))
    nef = E.EquivariantCrossAttentionNeF(cfg["d"], cfg["H"], 0, cfg["O"], cfg["L"], inv, inv, "rff", cfg["freq"], True, cfg["window"],
                                         precision=args.precision)
    B, Z, K = cfg["B"], cfg["Z"], 3
    gen = torch.Generator().manual_seed(99)
    p_h, a_h, s_h = E.init_latents(inv, B, Z, cfg["L"], polar_grid=cfg["polar_grid"])
    from enf_pde_b200.latents import make_coords
    x_d = make_coords(inv, cfg["grid"]).contiguous().to(dev)
    C = x_d.shape[0]
    img = torch.randn(B, C, cfg["O"], generator=gen).to(dev)
    variables = nef.init(0, x_d[None].cpu(), p_h.to(dev), a_h.to(dev), s_h.to(dev))
    leaves = E.params_to_leaves(variables)
    for t in leaves:
        t.requires_grad_(True)
    lrs = {"p_pos": torch.tensor([1.0]), "p_ori": torch.tensor([1.0]), "a": torch.full((cfg["L"],), 5.0), "gaussian_window": torch.tensor([0.0])}
    masks = [torch.arange(C, device=dev) for _ in range(K + 1)]       # every query at every step (the reference sub-samples to fit memory)
    p_d, a_d = p_h.to(dev), a_h.to(dev)
    s_d = s_h.to(dev) if cfg["window"] else None
    last = {}           # --dump-outputs: loss and adapted latents of the latest step

    def step():
        for t in leaves:
            t.grad = None
        loss, adapted = E.inner_loop(nef, variables, x_d, img, p_d, a_d, s_d, lrs, K, masks=masks)
        loss.backward()
        if args.dump_outputs:
            last.update({"loss": loss.detach(), **{"adapted_" + k: t.detach() for k, t in zip(("p", "a", "gaussian_window"), adapted) if t is not None}})
        return loss

    for _ in range(max(3, args.warmup)):
        step()
    torch.cuda.synchronize()
    with ClockSampler(0) as sampler:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            loss = step()
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    f_alg, _ = flops_per_pair(cfg, inv.dim)
    flop = (K + 1) * 3.0 * (f_alg * B * C * Z + flops_per_query_tail(cfg) * B * C)
    peaks = read_peaks()
    ach = flop / (ms * 1e-3) / 1e12
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {**last, **{"grad_" + n: t.grad for n, t in zip(_lib.LEAVES, leaves) if t is not None}})
    print(json.dumps({"metric": "coord-queries/sec (first-order Meta-SGD training step: 3 inner steps + outer fwd+bwd)", "value": B * C / (ms * 1e-3),
                      "unit": "queries/s", "n_gpus": 1, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms,
                      "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16 operands / f32 accumulate (tcgen05) + f32",
                      "data": "synthetic", "loss": float(loss.detach()),
                      "config": {"workload": f"{args.config}: {cfg['label']}", "B": B, "C": C, "Z": Z, "d": cfg["d"], "H": cfg["H"], "inner_steps": K,
                                 "passes": "4 forward + 3 latents-only backward + 1 full backward over all B x C queries"},
                      "roofline": {"bound": "tensor", "achieved": ach, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s", "frac": ach / peaks["bf16_sustained"],
                                   "traffic": None, "algorithmic_flop_per_step": flop,
                                   "note": "contract FLOPs of 4 forward + 4 backward passes (the latents-only backward's skipped weight-gradient products are still counted)"},
                      "clocks": sampler.summary()}))


def model_ws_mb(model, p, a):
    import ctypes
    from enf_pde_b200 import ode
    d = ode.EnfOdeDesc(**model._desc_kw(p, a))
    return ode._load().enf_ode_workspace_bytes(ctypes.byref(d)) / 1e6


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="ns64", choices=sorted(CONFIGS))
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--precision", default="bf16", choices=["fp32", "bf16"],
                    help="fp32: FMA kernels (<=1e-4 bucket); bf16: tcgen05 kernels with 16-bit operands (<=2e-3 bucket)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: the config's batch PER GPU (default, the driver's SCALE line); strong: the config's batch split over the GPUs")
    ap.add_argument("--partition", default="auto", choices=["auto", "fields", "queries"],
                    help="what is sharded over ranks; auto = fields when every rank gets one, else queries (SURVEY 8e)")
    ap.add_argument("--forward-only", action="store_true", help="forward-only roll-out line (SURVEY 8f-2)")
    ap.add_argument("--fields", type=int, default=None, help="override the number of fields per call (forward-only default: 480 = 8 x 60 frames)")
    ap.add_argument("--out-bf16", action="store_true", help="forward-only: bfloat16 decoded field (ENF_FLAG_OUT_BF16)")
    ap.add_argument("--recompute", action="store_true", help="bounded-memory training: ENF_FLAG_RECOMPUTE")
    ap.add_argument("--chunk-fields", type=int, default=0)
    ap.add_argument("--meta", action="store_true",
                    help="first-order Meta-SGD training step line (SURVEY 8f-1): K = 3 latents-only inner steps + the outer fwd+bwd")
    ap.add_argument("--ode", action="store_true",
                    help="latent ODE model line (SURVEY 8f-3): PonitaODEGen fwd + bwd at config_navier_stokes.yaml's `node:` sizes")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last device-resident step returned (output, loss, gradients) as "
                         "DIR/<name>.npy, float32 (float64 kept), at most 64 MB in all (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    if args.ode:
        return ode_line(args)
    if args.meta:
        return meta_line(args)
    cfg = dict(CONFIGS[args.config])
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    C_full = int(math.prod(cfg["grid"]))
    if args.fields is not None:
        cfg["B"] = args.fields
    elif args.forward_only:
        cfg["B"] = 480 if args.config == "ns64" else cfg["B"]          # pde_trainer.py:389-405: 8 signals x 60 roll-out frames

    if args.impl == "reference":
        if rank != 0:
            return
        kind, why = reference_probe()
        workload = {"workload": f"{args.config}: {cfg['label']}", "B_per_gpu": cfg["B"], "C": C_full, "Z": cfg["Z"], "d": cfg["d"],
                    "H": cfg["H"], "invariant": cfg["invariant_type"], "latent_dim": cfg["L"], "num_out": cfg["O"]}
        r = cpu_leg(cfg, args.steps, args.warmup, budget_s=None)
        line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
                "steps": r["steps"], "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload,
                "cpu_baseline": {**{k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}, "probe": why},
                "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    import torch
    import enf_pde_b200 as E
    from enf_pde_b200 import _lib
    from enf_pde_b200.dist import allreduce_weight_grads, allreduce_grads, field_shard, query_shard, choose_partition
    from enf_pde_b200.nef import _XAttnFunction

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback for the product path)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    lib = E.load_library()

    # ---- what this rank owns ---------------------------------------------------------------------------------------------
    B_global = cfg["B"] * (world if args.scaling == "weak" else 1)
    partition = args.partition
    if partition == "auto":
        partition = "fields" if args.scaling == "weak" else choose_partition(B_global, world)
    if partition == "fields":
        B = cfg["B"] if args.scaling == "weak" else len(range(B_global)[field_shard(B_global, rank, world)])
        q_slice = slice(0, C_full)
    else:
        B = B_global if args.scaling == "strong" else cfg["B"]
        q_slice = query_shard(C_full, rank, world)
    C = q_slice.stop - q_slice.start
    Z = cfg["Z"]
    workload = {"workload": f"{args.config}: {cfg['label']}", "B_per_gpu": B, "C": C_full, "C_per_gpu": C, "Z": Z, "d": cfg["d"],
                "H": cfg["H"], "invariant": cfg["invariant_type"], "latent_dim": cfg["L"], "num_out": cfg["O"]}

    inv = E.get_ca_invariant(types.SimpleNamespace(invariant_type=cfg["invariant_type"], num_in=cfg["num_in"]))
    nef = E.EquivariantCrossAttentionNeF(cfg["d"], cfg["H"], 0, cfg["O"], cfg["L"], inv, inv, "rff", cfg["freq"], True,
                                         cfg["window"], precision=args.precision,
                                         recompute=args.recompute, chunk_fields=args.chunk_fields, out_bf16=args.out_bf16,
                                         forward_chunk_fields=(args.chunk_fields or 96) if args.forward_only else 0)
    gen = torch.Generator().manual_seed(1234 + rank)
    p_h, a_h, s_h = E.init_latents(inv, B, Z, cfg["L"], polar_grid=cfg["polar_grid"])
    p_h = p_h + 0.02 * torch.randn(p_h.shape, generator=gen)
    a_h = a_h + 0.1 * torch.randn(a_h.shape, generator=gen)
    from enf_pde_b200.latents import make_coords
    x_h = make_coords(inv, cfg["grid"])[q_slice].contiguous()                     # (C, Dx), shared by all fields
    y_h = torch.randn(B, C, cfg["O"], generator=gen)
    variables = nef.init(0, x_h[None], p_h.to(dev), a_h.to(dev), s_h.to(dev))     # same weights on every rank
    leaves = E.params_to_leaves(variables)
    if not args.forward_only:
        for t in leaves:
            t.requires_grad_(True)
    use_sigma = cfg["window"]

    x_d, y_d = x_h.to(dev), y_h.to(dev)
    p_d, a_d, s_d = (t.to(dev).requires_grad_(not args.forward_only) for t in (p_h, a_h, s_h))
    n_out = B_global * C_full * cfg["O"] if args.scaling == "strong" else B * C * cfg["O"]
    last = {}           # --dump-outputs: decoded field (detached: its graph holds the workspace) and loss of the latest step

    def step_device(x, y, p, a, s):
        if args.forward_only:
            with torch.no_grad():
                out = nef.apply(variables, x[None].expand(B, -1, -1), p, a, s if use_sigma else None)
            if args.dump_outputs:
                last["out"] = out
            return out
        for t in leaves:
            t.grad = None
        p.grad = a.grad = None
        if s is not None:
            s.grad = None
        out = nef.apply(variables, x[None].expand(B, -1, -1), p, a, s if use_sigma else None)
        diff = out.detach() - y
        loss = (diff * diff).mean()
        if args.dump_outputs:
            last.update(out=out.detach(), loss=loss)
        out.backward(diff * (2.0 / n_out))
        if world > 1:
            if partition == "queries":      # latent gradients are sums over queries too: one packed collective for both
                wg, lg = allreduce_grads([t.grad for t in leaves], [p.grad, a.grad] + ([s.grad] if s is not None and s.grad is not None else []))
                p.grad, a.grad = lg[0], lg[1]
            else:
                allreduce_weight_grads([t.grad for t in leaves])
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing -----------------------------------------------------------------------------
    for _ in range(max(3, args.warmup)):
        step_device(x_d, y_d, p_d, a_d, s_d)
    workspace_bytes = _XAttnFunction.last_ws[2]
    chunk_used = _XAttnFunction.last_ws[0].get("chunk_fields", 0)
    lib.enf_profile_enable(1)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk:
        ev0.record()
        for _ in range(args.steps):
            step_device(x_d, y_d, p_d, a_d, s_d)
        ev1.record()
        barrier()
    ms = ev0.elapsed_time(ev1)
    if args.dump_outputs:       # what the last timed step handed its caller; the end-to-end steps below rebind, not overwrite, these
        outputs = dict(last)
        if not args.forward_only:
            outputs.update(grad_p=p_d.grad, grad_a=a_d.grad, grad_gaussian_window=s_d.grad if use_sigma else None)
            outputs.update({"grad_" + n: t.grad for n, t in zip(_lib.LEAVES, leaves) if t is not None})
    buf = (ctypes.c_float * 256)()
    n_f = lib.enf_profile_collect(0, buf, 256); fwd_ms = [buf[i] for i in range(max(n_f, 0))]
    n_b = lib.enf_profile_collect(1, buf, 256); bwd_ms = [buf[i] for i in range(max(n_b, 0))]
    lib.enf_profile_enable(0)
    launches = sum(E.last_launch_counts()) * args.steps
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())

    # ---- end to end from pinned host buffers ----------------------------------------------------------------
    pin = lambda t: t.detach().cpu().contiguous().pin_memory()
    xh, yh, ph, ah, sh = pin(x_h), pin(y_h), pin(p_h), pin(a_h), pin(s_h)
    dp_host, da_host, ds_host = (torch.empty_like(t).pin_memory() for t in (p_h, a_h, s_h))
    loss_host = torch.empty((), dtype=torch.float32).pin_memory()
    out_host = torch.empty(B, C, cfg["O"], dtype=torch.bfloat16 if args.out_bf16 else torch.float32).pin_memory() if args.forward_only else None
    if args.forward_only:
        h2d = sum(t.numel() * 4 for t in (xh, ph, ah)) + (sh.numel() * 4 if use_sigma else 0)
        d2h = out_host.numel() * out_host.element_size()
    else:
        h2d = sum(t.numel() * 4 for t in (xh, yh, ph, ah)) + (sh.numel() * 4 if use_sigma else 0)
        d2h = 4 + sum(t.numel() * 4 for t in (dp_host, da_host)) + (ds_host.numel() * 4 if use_sigma else 0)

    def step_e2e():
        x = xh.to(dev, non_blocking=True)
        p = ph.to(dev, non_blocking=True); a = ah.to(dev, non_blocking=True)
        s = sh.to(dev, non_blocking=True) if use_sigma else None
        if args.forward_only:
            out_host.copy_(step_device(x, None, p, a, s), non_blocking=True)     # the roll-out's decoded fields go back to the host
            torch.cuda.current_stream().synchronize()
            return
        y = yh.to(dev, non_blocking=True)
        p.requires_grad_(True); a.requires_grad_(True)
        if s is not None:
            s.requires_grad_(True)
        loss = step_device(x, y, p, a, s)
        loss_host.copy_(loss, non_blocking=True)
        dp_host.copy_(p.grad, non_blocking=True); da_host.copy_(a.grad, non_blocking=True)
        if use_sigma:
            ds_host.copy_(s.grad, non_blocking=True)
        torch.cuda.current_stream().synchronize()          # the caller reads the loss / latent gradients every step

    for _ in range(2):
        step_e2e()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step_e2e()
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_e2e = float(t.item())

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel, labelled from what the library actually dispatched ------------------------------
    peaks = read_peaks()
    I = inv.dim
    f_alg, f_ref = flops_per_pair(cfg, I)
    pairs = B * C * Z
    B_launch = min(B, nef.forward_chunk_fields) if (args.forward_only and nef.forward_chunk_fields > 0) else B   # fields per pair-kernel launch
    desc = _lib.EnfDesc(B=B, C=C, Z=Z, d=cfg["d"], H=cfg["H"], L=cfg["L"], O=cfg["O"], Dx=cfg["num_in"],
                        invariant_kind=_lib.INVARIANT_KINDS[cfg["invariant_type"]], use_window=int(cfg["window"]),
                        precision=nef.precision, flags=(_lib.FLAG_FORWARD_ONLY if args.forward_only else 0))
    fwd_tc, bwd_tc = _lib.dispatch(desc)
    passes = 1.0 if args.forward_only else 3.0
    clk_sum = clk.summary()
    pt = pipe_times(cfg, I, pairs, B * C, peaks, passes=passes, sm_mhz=float(clk_sum.get("sm_max_mhz") or 1965.0))
    bwd_avg = sum(bwd_ms) / len(bwd_ms) if bwd_ms else float("nan")
    fwd_avg = sum(fwd_ms) / len(fwd_ms) if fwd_ms else float("nan")
    dom_is_bwd = not args.forward_only
    dom_tc = bwd_tc if dom_is_bwd else fwd_tc
    dom_ms = bwd_avg if dom_is_bwd else fwd_avg
    dom_flop = (2.0 if dom_is_bwd else 1.0) * f_alg * (B_launch * C * Z)
    achieved = dom_flop / (dom_ms * 1e-3) / 1e12 if dom_ms == dom_ms else None
    tag = f"<{cfg['d']},{cfg['H']}>"
    if dom_is_bwd:
        kname = (f"fused pair backward = pairs_bwd_tc_a_kernel{tag} + pairs_bwd_tc_v_kernel + pairs_bwd_tc_q_kernel (tcgen05, 3 launches"
                 + (" per field chunk + the chunk's recomputed pairs_fwd_tc_kernel" if args.recompute and bwd_tc else "") + " timed as one)"
                 if bwd_tc else f"pairs_bwd_kernel<{cfg['d']}> (fused pair backward, fp32 FMA)")
    else:
        kname = f"pairs_fwd_tc_kernel{tag} (tcgen05)" if fwd_tc else f"pairs_fwd_kernel<{cfg['d']}> (fp32 FMA)"
    if dom_tc:
        bound = max(pt, key=pt.get)             # the pipe that needs the most time at 100 % (SURVEY 8d)
        peak, peak_src = peaks["bf16_sustained"], peaks["source"] + ", dense bf16 sustained"
        # achieved / peak stay in tensor TFLOP/s (the contract's unit); when another pipe binds, the fraction of THAT roof is the
        # bound's time at 100 % over the kernel's share of it
        frac = achieved / peak if achieved else None
    else:
        bound = "fp32-fma"                       # every GEMM of the fp32 kernels runs on the FMA pipe
        peak, peak_src = FP32_FMA_PEAK_TFLOPS, "nominal: 148 SM x 128 FMA lanes x 2 x 1.965 GHz (no measured fp32 peak in MEASURED_PEAKS.json)"
        frac = achieved / peak if achieved else None
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")       # dram bytes per launch from the committed ncu --set full captures
    if os.path.exists(tpath):
        with open(tpath) as f:
            tj = json.load(f).get(f"{args.config}:{args.precision}", {})
        traffic = tj.get("bwd_dram_bytes" if dom_is_bwd else "fwd_dram_bytes") if (B, C) == (CONFIGS[args.config]["B"], C_full) and not args.recompute else None
    step_flop = passes * (f_alg * pairs + flops_per_query_tail(cfg) * B * C)
    roofline = {"bound": bound, "kernel": kname, "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": frac,
                "traffic": traffic, "peak_source": peak_src,
                "pipe_time_ms_at_100pct": {k: 1e3 * v for k, v in pt.items()},
                "frac_of_bound_pipe_whole_step": (pt[max(pt, key=pt.get)] / (ms / args.steps * 1e-3)) if dom_tc else None,
                "algorithmic_flop_per_launch": dom_flop, "kernel_ms_avg": dom_ms,
                "kernel_share_of_step": dom_ms * args.steps / ms if dom_ms == dom_ms else None,
                "fwd_kernel_ms_avg": fwd_avg, "fwd_achieved": (f_alg * (B_launch * C * Z) / (fwd_avg * 1e-3) / 1e12) if fwd_ms else None,
                "whole_step_achieved": step_flop / (ms / args.steps * 1e-3) / 1e12,
                "whole_step_frac": step_flop / (ms / args.steps * 1e-3) / 1e12 / peak,
                "note": ("tcgen05 kind::f16 MMAs (fp16 operands, fp32 accumulate in TMEM)" if dom_tc else "arithmetic of this kernel is fp32 FMA")
                        + "; FLOP count is SURVEY 8d's contract figure F_pair_alg per (query, latent) pair"
                        + (", x2 for the backward (dgrad + wgrad; recompute and the 3-term split products of the relu layers are not counted)" if dom_is_bwd else "")}

    cpu = None
    if not args.no_cpu_baseline and world == 1 and not args.forward_only:
        r = cpu_leg(cfg, 40, 1, budget_s=15.0)
        cpu = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}

    q_step = (B_global * C_full) if args.scaling == "strong" else world * B * C
    q_total = q_step * args.steps
    if fwd_tc and (bwd_tc or args.forward_only):
        dtype = "f16 operands / f32 accumulate (tcgen05) + f32"
    elif fwd_tc:
        dtype = "forward: f16 operands / f32 accumulate (tcgen05); backward: f32 (FMA kernels)"
    else:
        dtype = "f32"
    metric = METRIC if not args.forward_only else "coord-queries/sec (ENF cross-attn forward only)"
    line = {"metric": metric, "value": q_total / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": dtype, "data": "synthetic",
            "config": {**workload, "precision": args.precision, "global_fields": B_global,
                       "parallelism": f"dp{world} over {partition}",
                       "dispatch": {"pair_fwd": "tcgen05" if fwd_tc else "fp32-fma", "pair_bwd": None if args.forward_only else ("tcgen05" if bwd_tc else "fp32-fma")},
                       "mode": "forward-only" if args.forward_only else ("recompute" if args.recompute else "stash"),
                       "chunk_fields": chunk_used if args.recompute else None, "forward_chunk_fields": (nef.forward_chunk_fields or None),
                       "workspace_bytes": workspace_bytes,
                       "l2": f"per-step working set ({workspace_bytes / 2**30:.2f} GiB workspace) >> 126 MB L2; no explicit flush",
                       "step": ("fwd (no_grad)" if args.forward_only else "fwd + bwd incl. all weight grads")
                               + ((" + NCCL all-reduce of weight" + (" and latent" if partition == "queries" else "") + " grads") if world > 1 and not args.forward_only else ""),
                       "step_tflop_contract": step_flop / 1e12},
            "roofline": roofline, "cpu_baseline": cpu, "clocks": clk_sum,
            "e2e": {"value": q_total / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
