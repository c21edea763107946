"""Per-element decoder outputs on one GPU (profiles/decoded_bench.md / .json), at the C5 and C2 shapes, bf16 engine (fused
tensor-core decoder), label PoE:

  1. kernel times with CUDA events over back-to-back launches in steady state (operands of one eval pass, group 0): the reducing
     forward sweep spv_dec_nb_fwd_tc, the element sweep spv_dec_nb_elems_tc with all five outputs and with `mean` only; the
     element sweep's output bytes per second against the device-to-device copy rate torch measures on the same card (1 GiB,
     read + write counted), which bounds a store-only kernel;
  2. spVIPES.get_decoded_expression(outputs=("mean",)) over every cell of both groups: cells/s with a 2 000-gene subset and
     with all genes (the latter bound by the device-to-host copy of n x G x 4 bytes per group).

    python tools/bench_decoded.py --out DIR [--iters 50] [--cells 8192]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from spvipes_b200 import _lib as L  # noqa: E402
from spvipes_b200 import synth  # noqa: E402
from spvipes_b200.engine import ELEM_OUTPUTS, HD, GroupBatch, StepEngine  # noqa: E402
from spvipes_b200.trainer import init_params  # noqa: E402

SHAPES = {"C5": (20_000, 2048), "C2": (5_000, 512)}  # genes / group, batch / group
H, S, P, NL = 128, 25, 10, 10


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = (s.strip() for s in q.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:  # the measurement stands without it, but says so
        return {"name": torch.cuda.get_device_name(), "power_limit": f"unknown ({e})", "max_sm_clock": "unknown"}


def timed(fn, iters, warm=10):
    for _ in range(warm):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1e3 / iters  # us per call


def copy_peak():
    x = torch.empty(1 << 28, dtype=torch.float32, device="cuda")
    y = torch.empty_like(x)
    us = timed(lambda: y.copy_(x), 20)
    return 2 * x.numel() * 4 / (us * 1e-6)


def kernels(shape, iters):
    G, B = SHAPES[shape]
    eng = StepEngine((G, G), H, S, P, 0.1, "label", "cuda", precision="bf16")
    init_params(eng, seed=0)
    data = synth.make_counts((4 * B, 4 * B), (G, G), NL, device="cuda", seed=1)
    batches = [GroupBatch(X=data.X[g], rows=torch.arange(B, dtype=torch.int32, device="cuda"), labels=data.labels[g]) for g in (0, 1)]
    ws = eng.forward(batches, training=False, with_grad=False)
    ctx, lib, w, d = eng._ctx, eng.lib, ws[0], eng.d
    src, xptr, ldx, rows = ctx["srcs"][0]
    dptrs = eng._dec_ptrs(0, w, xptr, rows, False)
    st = torch.cuda.current_stream().cuda_stream
    args = (L.ptr(w.amixb), w.KMp, L.ptr(w.Wstack), w.KMp, w.Gp, L.ptr(w.zcb), L.ptr(w.wzf), B, G, HD, d.Pb, d.Sb)
    fwd = lambda: L.check(lib.spv_dec_nb_fwd_tc(src, dptrs, ldx, *args, 0, d.KMIX, st), "spv_dec_nb_fwd_tc")
    outs = {k: torch.empty(B, G, device="cuda") for k in ELEM_OUTPUTS}
    all5 = L.ptr_array([outs[k] for k in ELEM_OUTPUTS])
    mean1 = L.ptr_array([outs["mean"] if k == "mean" else None for k in ELEM_OUTPUTS])
    el = lambda arr: (lambda: L.check(lib.spv_dec_nb_elems_tc(src, dptrs, ldx, *args, d.KMIX, arr, G, st), "spv_dec_nb_elems_tc"))
    res = {"B": B, "G": G, "fwd_us": timed(fwd, iters), "elems5_us": timed(el(all5), iters), "mean_us": timed(el(mean1), iters)}
    res["elems5_bytes"] = 5 * B * G * 4
    res["mean_bytes"] = B * G * 4
    # the element sweep's log-likelihood against the reducing sweep of the same pass
    rec = -outs["ll"].double().sum(1)
    fwd()
    L.check(lib.spv_dec_nb_rowreduce(L.ptr(w.part_nb), G, B, HD, L.ptr(w.rowc), L.ptr(w.rec), st), "spv_dec_nb_rowreduce")
    torch.cuda.synchronize()
    res["rec_rel_diff"] = float(((rec - w.rec.double()).abs() / w.rec.double().abs()).max())
    del eng, data
    torch.cuda.empty_cache()
    return res


def model_rate(cells, G, B, subset):
    from spvipes_b200.model import GroupedData, prepare_adatas, spVIPES
    import pandas as pd
    data = synth.make_counts((cells, cells), (G, G), NL, device="cuda", seed=2)
    ads = {}
    for gi, key in enumerate(("a", "b")):
        obs = pd.DataFrame({"cell_type": [f"t{int(v)}" for v in data.labels[gi].cpu().numpy()]})
        ads[key] = GroupedData(X=data.X[gi].cpu().numpy().astype(np.float32), obs=obs, var_names=[f"g{j}" for j in range(G)])
    del data
    adata = prepare_adatas(ads)
    spVIPES.setup_anndata(adata, groups_key="groups", label_key="cell_type")
    model = spVIPES(adata, n_hidden=H, n_dimensions_shared=S, n_dimensions_private=P, precision="bf16")
    gil = [list(ix) for ix in adata.uns["groups_obs_indices"]]
    sel = None if subset is None else [np.arange(subset), np.arange(subset)]
    model.get_decoded_expression([g[:2 * B] for g in gil], gene_indices=sel, batch_size=B)  # warm-up: device data, workspaces
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = model.get_decoded_expression(gil, gene_indices=sel, batch_size=B)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    k = G if subset is None else subset
    return {"cells": 2 * cells, "genes_out": k, "seconds": dt, "cells_per_s": 2 * cells / dt,
            "host_bytes": 2 * cells * k * 4, "host_bytes_per_s": 2 * cells * k * 4 / dt, "shape": list(out["mean"][0].shape)}


def render(r):
    c = r["card"]
    lines = ["# Per-element decoder outputs (element sweep, get_decoded_expression)", "",
             f"Measured on {c['name']}, power limit {c['power_limit']}, max SM clock {c['max_sm_clock']} "
             f"(tools/bench_decoded.py, one process).  bf16 engine, fused tensor-core decoder, label PoE, one group's operands; "
             "CUDA events over back-to-back launches after warm-up.", "",
             f"Device-to-device copy rate (torch, 1 GiB, read + write): {r['copy_peak'] / 1e12:.2f} TB/s.", "",
             "| shape | B | G | forward sweep (us) | element sweep, 5 outputs (us) | output TB/s | share of copy rate | mean only (us) | output TB/s | max rel. diff -sum ll vs rec |",
             "|---|---|---|---|---|---|---|---|---|---|"]
    for s, k in r["kernels"].items():
        b5 = k["elems5_bytes"] / (k["elems5_us"] * 1e-6)
        b1 = k["mean_bytes"] / (k["mean_us"] * 1e-6)
        lines.append(f"| {s} | {k['B']} | {k['G']} | {k['fwd_us']:.1f} | {k['elems5_us']:.1f} | {b5 / 1e12:.2f} | "
                     f"{b5 / r['copy_peak']:.0%} | {k['mean_us']:.1f} | {b1 / 1e12:.2f} | {k['rec_rel_diff']:.1e} |")
    lines += ["", "spVIPES.get_decoded_expression(outputs=(\"mean\",)), batch 2048, every cell of both groups (C5 gene count):", "",
              "| genes returned | cells | seconds | cells/s | host bytes/s |", "|---|---|---|---|---|"]
    for m in r["model"]:
        lines.append(f"| {m['genes_out']} | {m['cells']} | {m['seconds']:.3f} | {m['cells_per_s']:.0f} | {m['host_bytes_per_s'] / 1e9:.1f} GB/s |")
    return "\n".join(lines) + "\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--cells", type=int, default=8192)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_decoded needs a CUDA device")
    os.makedirs(a.out, exist_ok=True)
    r = {"card": card(), "copy_peak": copy_peak(), "kernels": {s: kernels(s, a.iters) for s in SHAPES}}
    G, B = SHAPES["C5"]
    r["model"] = [model_rate(a.cells, G, B, 2000), model_rate(a.cells, G, B, None)]
    with open(os.path.join(a.out, "decoded_bench.json"), "w") as f:
        json.dump(r, f, indent=1)
    with open(os.path.join(a.out, "decoded_bench.md"), "w") as f:
        f.write(render(r))
    print(render(r))


if __name__ == "__main__":
    main()
