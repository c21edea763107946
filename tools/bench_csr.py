"""Dense-resident against CSR-resident counts on one GPU, in one process (profiles/csr_bench.md):

  1. per shape (C5 bf16, C2 bf16, C2 fp32; label PoE): the CUDA-graph training step from a dense uint16 copy and from a CSR copy
     of the same synthetic counts, the same minibatch rows, alternated in blocks after >= 256 warm-up steps each (DESIGN.md
     section 6); spv_csr_gather alone (eager launches, CUDA events) against spv_counts_to_bf16 on the dense rows, as
     algorithmic bytes over time; the resident bytes of both formats; whether the two groups' gathers overlap in the step
     (torch.profiler on a few replays);
  2. the capability run: 2 x 4 M cells x 20 k genes CSR-resident (dense would be 320 GB), replayed steps -> cells/s, and a
     short spVIPES.train + get_latent_representation on a slice of it through the model API.

    python tools/bench_csr.py --out DIR [--steps 512] [--warmup 256] [--blocks 4] [--cap-cells 4000000]
    python tools/bench_csr.py --out DIR --render DIR/csr_bench.json     (re-write csr_bench.md from the JSON; no GPU needed)
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
from spvipes_b200.engine import CsrCounts, GroupBatch, StepEngine  # noqa: E402
from spvipes_b200.trainer import TrainLoop, init_params  # noqa: E402

SHAPES = {"C5": (1_000_000, 20_000, 2048), "C2": (50_000, 5_000, 512)}  # cells / group, genes / group, batch / group
H, S, P, NL = 128, 25, 10, 10
r8 = lambda x: (x + 7) // 8 * 8


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = (s.strip() for s in q.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:  # the measurement stands without it, but says so
        return {"name": torch.cuda.get_device_name(), "power_limit": f"unknown ({e})", "max_sm_clock": "unknown"}


def dense_to_csr(X, chunk=16384):
    """uint16 [N, G] device matrix -> CsrCounts on the device, chunk by chunk"""
    N, G = X.shape
    counts, idx, val = [torch.zeros(1, dtype=torch.int64, device=X.device)], [], []
    for r0 in range(0, N, chunk):
        c = X[r0:r0 + chunk].view(torch.int16).to(torch.int32) & 0xFFFF
        nz = c != 0
        counts.append(nz.sum(1, dtype=torch.int64))
        idx.append(nz.nonzero()[:, 1].to(torch.int32).to(torch.uint16))
        val.append(c[nz].to(torch.uint16))
    return CsrCounts(torch.cumsum(torch.cat(counts), 0), torch.cat(idx), torch.cat(val), (N, G))


class Arm:
    """one engine + captured step over a given count storage"""

    def __init__(self, X, labels, genes, B, precision):
        self.eng = StepEngine((genes, genes), H, S, P, 0.1, "label", "cuda", seed=0, precision=precision)
        init_params(self.eng, 0)
        self.loop = TrainLoop(self.eng)
        self.loop.set_epoch(1)
        self.rows = [torch.zeros(B, dtype=torch.int32, device="cuda") for _ in (0, 1)]
        self.static = [GroupBatch(X=X[g], rows=self.rows[g], labels=labels[g], labels_per_cell=True) for g in (0, 1)]
        self.graph = None

    def set_rows(self, rows, s):
        for g in (0, 1):
            self.rows[g].copy_(rows[g][s], non_blocking=True)

    def step(self, rows, s):
        self.set_rows(rows, s)
        if self.graph is None:
            self.graph = self.loop.capture(self.static)
        self.graph.replay()


def time_steps(arm, rows, s0, n):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for s in range(s0, s0 + n):
        arm.step(rows, s % rows[0].shape[0])
    ev1.record()
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1)


def kernel_times(csr, dense, B, G, rows, reps=200):
    """ms per launch of spv_csr_gather (fused bf16 mode) and of spv_counts_to_bf16 on the dense rows, eager, rows cycling through
    64 draws (their working set exceeds L2)"""
    lib = L.load()
    Gp = r8(G)
    xs = torch.zeros(B, Gp, dtype=torch.uint16, device="cuda")
    T, Tl = (torch.zeros(B, Gp, dtype=torch.bfloat16, device="cuda") for _ in range(2))
    lb = torch.zeros(B, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    nrow = rows.shape[0]

    def gather(k):
        L.check(lib.spv_csr_gather(L.SRC_U16_LOG1P, L.ptr(csr.indptr), L.ptr(csr.indices), L.ptr(csr.values), L.ptr(rows[k % nrow]),
                                   B, G, L.ptr(xs), Gp, L.ptr(T), L.ptr(Tl), Gp, L.ptr(lb), None, 0, st), "spv_csr_gather")

    def convert(k):
        L.check(lib.spv_counts_to_bf16(L.SRC_U16_LOG1P, L.ptr(dense), dense.stride(0), L.ptr(rows[k % nrow]), L.ptr(T), L.ptr(Tl), Gp,
                                       B, G, L.ptr(lb), None, 0, st), "spv_counts_to_bf16")

    out = {}
    for name, fn in (("spv_csr_gather", gather), ("spv_counts_to_bf16", convert)):
        for k in range(20):
            fn(k)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for k in range(reps):
            fn(k)
        ev1.record()
        torch.cuda.synchronize()
        out[name] = ev0.elapsed_time(ev1) / reps
    # nonzeros the gathers read: mean over the row draws
    nnz_row = (csr.indptr[1:] - csr.indptr[:-1])
    nnz = float(torch.stack([nnz_row[rows[k].long()].sum() for k in range(nrow)]).double().mean())
    return out, nnz


def copy_peak_gbs(nbytes=4 << 30, reps=20):
    a = torch.empty(nbytes // 4, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(reps):
        b.copy_(a)
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / reps
    del a, b
    return 2 * nbytes / (ms * 1e-3) / 1e9


def gather_overlap(arm, rows):
    """kernel intervals of spv_csr_gather in three replayed steps (torch.profiler): do the two groups' gathers overlap?"""
    try:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for s in range(3):
                arm.step(rows, s)
            torch.cuda.synchronize()
        ev = sorted([(e.time_range.start, e.time_range.end) for e in prof.events() if "csr_gather" in e.name])
        pairs = [(ev[i], ev[i + 1]) for i in range(0, len(ev) - 1, 2)]
        overl = [max(0.0, min(a[1], b[1]) - max(a[0], b[0])) for a, b in pairs]
        return {"gather_kernels_seen": len(ev), "pairs": len(pairs),
                "overlap_us_per_step": [round(o, 2) for o in overl],
                "gather_us": [round(e[1] - e[0], 2) for e in ev]}
    except Exception as e:
        return {"error": repr(e)}


def compare(name, precision, args, peak):
    n_cells, genes, B = SHAPES[name]
    t0 = time.time()
    data = synth.make_counts((n_cells, n_cells), (genes, genes), NL, device="cuda", seed=1234)
    csr = [dense_to_csr(data.X[g]) for g in (0, 1)]
    gen_s = time.time() - t0
    gen = torch.Generator(device="cuda").manual_seed(5)
    nrow = 64
    rows = [torch.stack([torch.randperm(n_cells, generator=gen, device="cuda")[:B] for _ in range(nrow)]).to(torch.int32)
            for _ in (0, 1)]
    arms = {"dense": Arm(data.X, data.labels, genes, B, precision), "csr": Arm(csr, data.labels, genes, B, precision)}
    for arm in arms.values():
        time_steps(arm, rows, 0, args.warmup)
    per = args.steps // args.blocks
    tot = {k: 0.0 for k in arms}
    block_ms = {k: [] for k in arms}
    for blk in range(args.blocks):
        for k in (("dense", "csr") if blk % 2 == 0 else ("csr", "dense")):
            ms = time_steps(arms[k], rows, args.warmup + blk * per, per)
            tot[k] += ms
            block_ms[k].append(round(ms / per, 4))
    step = {k: tot[k] / (per * args.blocks) for k in arms}
    # the two arms computed the same thing: their states after the same steps are equal
    same = bool(torch.equal(arms["dense"].eng.params.flat, arms["csr"].eng.params.flat))
    res = {"shape": name, "precision": precision, "cells_per_group": n_cells, "genes": genes, "batch": B,
           "steps_timed_per_arm": per * args.blocks, "warmup_per_arm": args.warmup, "blocks": args.blocks,
           "ms_per_step": {k: round(v, 4) for k, v in step.items()}, "block_ms_per_step": block_ms,
           "csr_minus_dense_ms": round(step["csr"] - step["dense"], 4),
           "csr_over_dense_pct": round(100 * (step["csr"] / step["dense"] - 1), 2),
           "params_equal_after_run": same,
           "resident_bytes": {"dense": sum(x.numel() * 2 for x in data.X), "csr": sum(c.resident_bytes() for c in csr)},
           "nnz_per_group": [int(c.indptr[-1]) for c in csr], "data_setup_s": round(gen_s, 1)}
    if precision == "bf16":
        kt, nnz = kernel_times(csr[0], data.X[0], B, genes, rows[0])
        Gp = r8(genes)
        gbytes = nnz * 4 + B * Gp * 6 + B * 8
        cbytes = B * genes * 2 + B * Gp * 4 + B * 8
        res["kernel"] = {
            "spv_csr_gather_us": round(kt["spv_csr_gather"] * 1e3, 2), "spv_csr_gather_bytes": int(gbytes),
            "spv_csr_gather_gbs": round(gbytes / (kt["spv_csr_gather"] * 1e-3) / 1e9, 1),
            "spv_csr_gather_pct_of_copy_peak": round(100 * gbytes / (kt["spv_csr_gather"] * 1e-3) / 1e9 / peak, 1),
            "spv_counts_to_bf16_us": round(kt["spv_counts_to_bf16"] * 1e3, 2), "spv_counts_to_bf16_bytes": int(cbytes),
            "spv_counts_to_bf16_gbs": round(cbytes / (kt["spv_counts_to_bf16"] * 1e-3) / 1e9, 1),
            "mean_nnz_gathered": round(nnz)}
        res["overlap"] = gather_overlap(arms["csr"], rows)
    del arms, data, csr
    torch.cuda.empty_cache()
    return res


def capability(args):
    n, genes, B = args.cap_cells, 20_000, 2048
    t0 = time.time()
    data = synth.make_counts_csr((n, n), (genes, genes), NL, device="cuda", seed=1234)
    torch.cuda.synchronize()
    gen_s = time.time() - t0
    resident = sum(c.resident_bytes() for c in data.X)
    gen = torch.Generator(device="cuda").manual_seed(5)
    rows = [torch.stack([torch.randperm(n, generator=gen, device="cuda")[:B] for _ in range(64)]).to(torch.int32) for _ in (0, 1)]
    arm = Arm(data.X, data.labels, genes, B, "bf16")
    time_steps(arm, rows, 0, args.warmup)
    ms = time_steps(arm, rows, args.warmup, args.cap_steps)
    loss = float(arm.eng.loss_out[0])
    res = {"cells_per_group": n, "genes": genes, "batch": B, "resident_bytes_csr": resident,
           "resident_bytes_dense_would_be": 2 * n * genes * 2, "nnz_per_group": [int(c.indptr[-1]) for c in data.X],
           "steps_timed": args.cap_steps, "ms_per_step": round(ms / args.cap_steps, 4),
           "cells_per_s": round(2 * B * args.cap_steps / (ms * 1e-3)), "loss_finite": bool(np.isfinite(loss)),
           "max_memory_allocated_bytes": int(torch.cuda.max_memory_allocated()), "data_setup_s": round(gen_s, 1)}
    del arm
    # the public path end to end on a slice: sparse AnnData-like objects -> prepare_adatas -> setup_anndata -> train -> latents
    import pandas as pd
    import scipy.sparse as sp
    from spvipes_b200.model import GroupedData, prepare_adatas, spVIPES
    m = args.api_cells
    ads = {}
    for g, key in enumerate(("a", "b")):
        c = data.X[g]
        end = int(c.indptr[m])
        host = sp.csr_matrix((c.values[:end].cpu().view(torch.int16).numpy().view(np.uint16).astype(np.float32),
                              c.indices[:end].cpu().view(torch.int16).numpy().view(np.uint16).astype(np.int32),
                              c.indptr[:m + 1].cpu().numpy()), shape=(m, genes))
        obs = pd.DataFrame({"cell_type": [f"t{int(v)}" for v in data.labels[g][:m].cpu().numpy()]})
        ads[key] = GroupedData(X=host, obs=obs, var_names=[f"g{j}" for j in range(genes)])
    del data
    torch.cuda.empty_cache()
    t0 = time.time()
    adata = prepare_adatas(ads)
    spVIPES.setup_anndata(adata, groups_key="groups", label_key="cell_type")
    model = spVIPES(adata, n_hidden=H, n_dimensions_shared=S, n_dimensions_private=P, precision="bf16")
    gil = [list(ix) for ix in adata.uns["groups_obs_indices"]]
    model.train(gil, max_epochs=1, batch_size=B, n_epochs_kl_warmup=None)
    lat = model.get_latent_representation(gil, batch_size=B)
    torch.cuda.synchronize()
    res["model_api"] = {"cells_per_group": m, "adata_X": type(adata.X).__name__, "device_X": type(model._device_data[0]["X"]).__name__,
                        "train_epochs": 1, "train_loss_epoch": model.history["train_loss_epoch"],
                        "latent_shapes": [list(lat["shared"][g].shape) for g in (0, 1)],
                        "latents_finite": bool(all(np.isfinite(lat["shared"][g]).all() for g in (0, 1))),
                        "wall_s": round(time.time() - t0, 1)}
    return res


def render(out) -> str:
    """profiles/csr_bench.md from the JSON this script writes"""
    c = out["card"]
    gb = lambda b: f"{b / 1e9:.1f} GB"
    lines = [f"# Dense-resident vs CSR-resident counts (`tools/bench_csr.py`)", "",
             f"One {c['name']}, power limit {c['power_limit']}, max SM clock {c['max_sm_clock']}; torch {out['torch']}. "
             f"HBM copy peak measured in the same run: {out['hbm_copy_peak_gbs']} GB/s (device-to-device copy of 4 GB).", "",
             "## CUDA-graph training step, label PoE, same synthetic counts and minibatch rows in both arms", "",
             "Arms alternated in blocks after the warm-up; ms/step is the mean over all timed steps of an arm.", "",
             "| shape | precision | dense ms/step | CSR ms/step | CSR - dense | resident dense | resident CSR | params equal after run |",
             "|---|---|---:|---:|---:|---:|---:|---|"]
    for r in out["runs"]:
        m = r["ms_per_step"]
        lines.append(f"| {r['shape']} ({r['cells_per_group']} cells x {r['genes']} genes / group, batch {r['batch']}) | {r['precision']} | "
                     f"{m['dense']:.4f} | {m['csr']:.4f} | {r['csr_minus_dense_ms']:+.4f} ms ({r['csr_over_dense_pct']:+.2f} %) | "
                     f"{gb(r['resident_bytes']['dense'])} | {gb(r['resident_bytes']['csr'])} | {r['params_equal_after_run']} |")
    lines += ["", "Per-block ms/step (block order alternates): " +
              "; ".join(f"{r['shape']} {r['precision']}: dense {r['block_ms_per_step']['dense']}, CSR {r['block_ms_per_step']['csr']}"
                        for r in out["runs"]), "",
              "## The gather kernel alone (eager launches, CUDA events, 64 row draws cycled)", "",
              "Algorithmic bytes: gather = nnz x 4 + B x Gp x 6 + B x 8 (nonzeros read; staging tile, bf16 pair written); "
              "conversion = B x G x 2 + B x Gp x 4 + B x 8.", "",
              "| shape | kernel | us / launch | bytes | GB/s | share of copy peak |", "|---|---|---:|---:|---:|---:|"]
    for r in out["runs"]:
        k = r.get("kernel")
        if not k:
            continue
        lines.append(f"| {r['shape']} | `spv_csr_gather` (fused bf16) | {k['spv_csr_gather_us']} | {k['spv_csr_gather_bytes'] / 1e6:.1f} MB | "
                     f"{k['spv_csr_gather_gbs']} | {k['spv_csr_gather_pct_of_copy_peak']} % |")
        lines.append(f"| {r['shape']} | `spv_counts_to_bf16` on dense rows (what it replaces) | {k['spv_counts_to_bf16_us']} | "
                     f"{k['spv_counts_to_bf16_bytes'] / 1e6:.1f} MB | {k['spv_counts_to_bf16_gbs']} | "
                     f"{round(100 * k['spv_counts_to_bf16_gbs'] / out['hbm_copy_peak_gbs'], 1)} % |")
    lines += ["", "Overlap of the two groups' gathers in three replayed steps (torch.profiler, separate from the timed runs):", ""]
    for r in out["runs"]:
        if "overlap" in r:
            lines.append(f"* {r['shape']}: {json.dumps(r['overlap'])}")
    cap = out.get("capability")
    if cap:
        api = cap.get("model_api", {})
        lines += ["", "## Capability: 2 x {:,} cells x {:,} genes, CSR-resident, label PoE, bf16, batch {}".format(
                      cap["cells_per_group"], cap["genes"], cap["batch"]), "",
                  f"* resident counts: {gb(cap['resident_bytes_csr'])} as CSR (dense uint16 would be "
                  f"{gb(cap['resident_bytes_dense_would_be'])}: more than the card holds); nnz per group {cap['nnz_per_group']}",
                  f"* {cap['steps_timed']} replayed steps after {out['args']['warmup']} warm-up: {cap['ms_per_step']} ms/step = "
                  f"{cap['cells_per_s']:,} cells/s (2 x {cap['batch']} cells per step); loss finite: {cap['loss_finite']}; "
                  f"peak allocated {gb(cap['max_memory_allocated_bytes'])}",
                  f"* model API on the first {api.get('cells_per_group')} cells of each group: sparse inputs -> `prepare_adatas` "
                  f"(`.X` is {api.get('adata_X')}) -> `setup_anndata` -> `spVIPES.train` (device counts: {api.get('device_X')}, "
                  f"{api.get('train_epochs')} epoch, loss {api.get('train_loss_epoch')}) -> `get_latent_representation` "
                  f"(shapes {api.get('latent_shapes')}, finite: {api.get('latents_finite')}), {api.get('wall_s')} s"]
    return "\n".join(lines) + "\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--render", default=None, help="only write csr_bench.md into --out from this csr_bench.json")
    ap.add_argument("--steps", type=int, default=512)
    ap.add_argument("--warmup", type=int, default=256)
    ap.add_argument("--blocks", type=int, default=4)
    ap.add_argument("--cap-cells", type=int, default=4_000_000)
    ap.add_argument("--cap-steps", type=int, default=300)
    ap.add_argument("--api-cells", type=int, default=20_000)
    ap.add_argument("--only", default="C5-bf16,C2-bf16,C2-fp32,cap")
    args = ap.parse_args()
    if args.render:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "csr_bench.md"), "w") as f:
            f.write(render(json.load(open(args.render))))
        return
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    # the measurement's parameters (not where its files go)
    out = {"card": card(), "torch": torch.__version__, "args": {k: v for k, v in vars(args).items() if k not in ("out", "render")}}
    out["hbm_copy_peak_gbs"] = round(copy_peak_gbs(), 1)
    print(json.dumps(out), flush=True)
    out["runs"] = []
    for tag in args.only.split(","):
        if tag == "cap":
            out["capability"] = capability(args)
            print(json.dumps(out["capability"]), flush=True)
        else:
            name, prec = tag.split("-")
            r = compare(name, prec, args, out["hbm_copy_peak_gbs"])
            print(json.dumps(r), flush=True)
            out["runs"].append(r)
    with open(os.path.join(args.out, "csr_bench.json"), "w") as f:
        json.dump(out, f, indent=1)
    with open(os.path.join(args.out, "csr_bench.md"), "w") as f:
        f.write(render(out))


if __name__ == "__main__":
    main()
