#!/usr/bin/env python
"""Benchmark of the spVIPES per-minibatch training hot path on B200 (BASELINE.json metric: training cells/sec, fwd+bwd
ELBO + optimiser, at 1/2/4/8 GPUs; NB-loglik kernel roofline).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --steps K --warmup W    # the reference algorithm on the host cores (oracle port)

A "step" is one minibatch (B cells per group, 2 groups) through inference -> generative -> loss -> backward -> Adam.

Workload: BASELINE.json's scaling config C5 (label PoE, 2 x 1M cells, 20k genes, n_hidden 128, batch 2048 / group / GPU) at
EVERY N, so that the driver's 1 -> 8 sweep compares like with like (weak scaling: the 2 x 1M cells are sharded over the ranks,
the per-GPU minibatch is fixed); 80 GB of uint16 counts fit one B200.  At N = 1 the JSON line also carries a `configs` array with
the other BASELINE configs measured the same way in the same run: C2 (configs[1]: label, 2 x 50k cells, 5k genes, batch 512),
C3 (paired OT, 2 x 100k, 10k genes, batch 1024, dense fp32 plan resident: 40 GB), C4 (cluster OT, 2 x 200k, 20k genes,
n_hidden 256, batch 2048, plan resident as bf16: 80 GB), each with value / e2e / roofline, as far as the time budget allows
(--budget seconds).  `--workload` picks another headline.

Timed region: exactly K steps (CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks),
after W untimed warm-up steps (at least MIN_WARMUP).  That one window is all that is timed, and a short one is noisy (see
DESIGN.md section 6): take K in the hundreds for a steadier number.  Prints ONE JSON line on rank 0.

    python bench.py --steps K --warmup W --dump-outputs DIR

also writes what the last timed step handed its caller to DIR/*.npy (see dump_outputs), so that two builds can be compared
output for output: with the same arguments every input is the same from run to run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (mode, cells per group, genes per group, n_hidden, batch per group, n_labels / clusters, plan dtype)
    "C1": ("label", 5_000, 2_000, 128, 512, 10, None),
    "C2": ("label", 50_000, 5_000, 128, 512, 10, None),
    "C3": ("paired", 100_000, 10_000, 128, 1024, 10, torch.float32),
    "C4": ("cluster", 200_000, 20_000, 256, 2048, 10, torch.bfloat16),
    "C5": ("label", 1_000_000, 20_000, 128, 2048, 10, None),
}
S_DIM, P_DIM, HD = 25, 10, 256
METRIC = "training cells/sec (fwd+bwd ELBO + Adam)"
T_START = time.time()
# least number of warm-up steps of the CUDA path: on a B200, C5 steps reached their steady time only after ~150 steps (the
# first 100 ran 2-3 % slower).  A count, not a time, so that what precedes the last timed step (and with it the
# --dump-outputs files) depends on the arguments alone.
MIN_WARMUP = 256
DUMP_SAMPLE = 1 << 22  # elements kept of a dumped vector longer than this (16 MB as float32)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d.get("sm_max_mhz", 1965.0)), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1965.0, "fallback (B200_PROFILING.md)"


def measured_traffic(workload, kernel):
    """dram__bytes_read + write per launch from the committed `ncu --set full` capture of this workload, if there is one
    (profiles/nb_traffic.json, written from the .ncu-rep by tools/ncu_table.py); None otherwise"""
    p = os.path.join(ROOT, "profiles", "nb_traffic.json")
    if not os.path.exists(p):
        return None
    return json.load(open(p)).get(workload, {}).get(kernel)


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region, through NVML in a background thread (pynvml, 20 ms
    period).  A resident `nvidia-smi -lms` poller was measured to stall the CUDA launch path of the benchmarked process
    (2-GPU step 0.46 ms without it, 0.60 ms with it at 20 ms, 1.28 ms at 100 ms), so it is only the fallback."""

    def __init__(self, index=0):
        self.index, self.samples, self.reason_bits, self.max_mhz = index, [], 0, None
        self.thread, self.stop_flag, self.proc, self.rows = None, False, None, []

    def start(self):
        if os.environ.get("SPV_NO_CLOCKS"):
            return
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))

            def poll():
                while not self.stop_flag:
                    try:
                        self.samples.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                        self.reason_bits |= int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(h))
                    except Exception:
                        pass
                    time.sleep(0.02)

            self._nvml = pynvml
            self.thread = threading.Thread(target=poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            t0 = time.time()
            while not self.rows and time.time() - t0 < 3.0:  # the first line arrives ~100 ms after start
                time.sleep(0.01)
            self.n_before = len(self.rows)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.thread is not None:
            self.stop_flag = True
            self.thread.join(timeout=1.0)
            nv = self._nvml
            names = [("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                     ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap)]
            return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                    "reasons": [n for n, bit in names if self.reason_bits & int(bit)], "samples": len(self.samples), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        self.rows = self.rows[getattr(self, "n_before", 0):] or self.rows[-1:]
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(len(r) > 2 + k and r[2 + k] == "Active" for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "source": "nvidia-smi"}


def workload_config(workload, n_gpus):
    mode, n_cells, genes, H, B, n_labels, plan_dtype = WORKLOADS[workload]
    plan = ""
    if plan_dtype is not None:
        plan = (f", dense transport plan {n_cells} x {n_cells} resident on the device as "
                f"{'bf16' if plan_dtype == torch.bfloat16 else 'fp32'} ({n_cells * n_cells * (2 if plan_dtype == torch.bfloat16 else 4) / 1e9:.0f} GB)")
    return {"workload": f"{workload}: {mode}-based PoE, 2 groups x {n_cells} cells, {genes} genes/group, n_hidden {H}, "
                        f"shared {S_DIM} / private {P_DIM}, batch {B}/group/GPU, {n_labels} labels{plan}",
            "cells_per_step_per_gpu": 2 * B, "parallelism": f"dp{n_gpus}",
            "l2": "inputs larger than L2: every step gathers a fresh random minibatch from the device-resident count "
                  "matrices and streams all weights/Adam state"}


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference algorithm on the host cores.  Nothing of the product package's
# engine is imported here (only the synthetic-data recipe): the oracle builds its own default-initialised state_dict.
# ------------------------------------------------------------------------------------------------
def cpu_reference_cells_per_sec(workload, steps, warmup, seed=0):
    """oracle/restatement.py (validated against the unmodified reference, tests/test_oracle.py) + autograd backward + Adam
    (scvi TrainingPlan defaults) with every host thread; bounded sample: `steps` minibatches of the workload's shape."""
    from oracle import restatement as rs
    from spvipes_b200 import synth

    mode, n_cells, genes, H, B, n_labels, plan_dtype = WORKLOADS[workload]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    n_sample = B * (steps + warmup)
    data = synth.make_counts((n_sample, n_sample), (genes, genes), n_labels, device="cpu", seed=1234)
    sd = rs.default_state_dict((genes, genes), H, S_DIM, P_DIM, seed)
    names = rs.param_names(sd)
    for k in names:
        sd[k].requires_grad_(True)
    opt = torch.optim.Adam([sd[k] for k in names], lr=1e-3, eps=0.01, weight_decay=1e-6)
    gen = torch.Generator().manual_seed(1)
    t0 = None
    for s in range(steps + warmup):
        if s == warmup:
            t0 = time.perf_counter()
        sl = slice(s * B, (s + 1) * B)
        x = [data.X[g][sl].to(torch.float32) for g in (0, 1)]
        labels = [data.labels[g][sl].numpy() for g in (0, 1)]
        sub = None
        if mode != "label":  # the reference slices the [B, B] sub-plan out of the full plan per step; only that block is needed
            sub = synth.make_plan(B, B, data.labels[0][sl], data.labels[1][sl], n_labels, device="cpu", seed=7 + s)
        eps_p = [torch.randn(B, P_DIM, generator=gen) for _ in (0, 1)]
        eps_q = [torch.randn(B, S_DIM, generator=gen) for _ in (0, 1)]
        dm = {(g, k): (torch.rand(B, H, generator=gen) < 0.9).float() / 0.9 for g in (0, 1) for k in ("private", "shared")}
        out = rs.step(sd, x, mode=mode, n_shared=S_DIM, n_private=P_DIM, eps_private=eps_p, eps_poe=eps_q,
                      labels=labels if mode in ("label", "cluster") else None, sub=sub, drop_masks=dm, kl_weight=min(1.0, s / 400.0))
        opt.zero_grad(set_to_none=True)
        out["loss"].backward()
        opt.step()
        for k, v in out["new_stats"].items():
            sd[k] = v
    dt = time.perf_counter() - t0
    return 2 * B * steps / dt, dt / steps * 1e3, cores, f"{steps} minibatches of {workload} shape (2x{B} cells, {genes} genes/group, {mode} PoE), oracle port, torch CPU"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    workload = args.workload
    steps = args.steps  # a C5-shaped minibatch costs ~1-2 s on the host
    warm = min(args.warmup, 1)
    v, ms, cores, sample = cpu_reference_cells_per_sec(workload, steps, warm)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "cells/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": workload_config(workload, args.gpus),
            "cpu_baseline": {"value": v, "unit": "cells/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "cells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
class Bench:
    """one workload on this rank's GPU: data, engine, training loop, and the measurements"""

    def __init__(self, workload, args, dev, dist, rank, world):
        from spvipes_b200 import _lib as L
        from spvipes_b200 import synth
        from spvipes_b200.engine import GroupBatch, StepEngine
        from spvipes_b200.trainer import TrainLoop, init_params
        self.L, self.GroupBatch = L, GroupBatch
        self.workload, self.args, self.dev, self.dist, self.rank, self.world = workload, args, dev, dist, rank, world
        self.mode, n_cells, self.genes, self.H, self.B, self.n_labels, plan_dtype = WORKLOADS[workload]
        self.n_cells = n_cells // world  # rank-local shard (weak scaling: the per-GPU minibatch is fixed)
        self.lib = L.load()
        self.data = synth.make_counts((self.n_cells, self.n_cells), (self.genes, self.genes), self.n_labels, device=dev,
                                      seed=1234 + 17 * rank)
        self.plan = None
        if self.mode != "label":
            self.plan = synth.make_plan(self.n_cells, self.n_cells, self.data.labels[0], self.data.labels[1], self.n_labels,
                                        device=dev, seed=7 + rank, dtype=plan_dtype)
        self.eng = StepEngine((self.genes, self.genes), self.H, S_DIM, P_DIM, 0.1, self.mode, device=dev, seed=rank,
                              plan=self.plan, precision=args.precision)
        init_params(self.eng, 0)
        self.loop = TrainLoop(self.eng)
        self.sync_kind = None
        if world > 1:
            from spvipes_b200.parallel import broadcast_params, make_grad_sync
            broadcast_params(self.eng, dist, src=0)
            self.loop.grad_sync = make_grad_sync(self.eng, dist)
            gs = self.loop.grad_sync
            self.sync_kind = f"{type(gs).__name__}: {gs.kind}" + (f" (fallback: {gs.fallback_reason})" if getattr(gs, "fallback_reason", None) else "")
        self.loop.set_epoch(1)
        self.gen = torch.Generator(device=dev).manual_seed(5 + rank)
        B = self.B
        self.rows_cur = [torch.empty(B, dtype=torch.int32, device=dev) for _ in (0, 1)]
        self.lab_cur = [torch.empty(B, dtype=torch.int32, device=dev) for _ in (0, 1)]
        self.static = self._batches(self.rows_cur, self.lab_cur)
        self.graph = None
        self.per_step_launches = None

    def _batches(self, rows, lab):
        """label mode: per-cell label arrays gathered in-kernel with the row indices; OT modes: the plan is indexed with the
        cells' positions in the resident matrix, cluster labels of the minibatch in a [B] buffer"""
        GB, d = self.GroupBatch, self.data
        if self.mode == "label":
            return [GB(X=d.X[g], rows=rows[g], labels=d.labels[g], labels_per_cell=True) for g in (0, 1)]
        return [GB(X=d.X[g], rows=rows[g], idx=rows[g], labels=lab[g] if self.mode == "cluster" else None) for g in (0, 1)]

    def draw_rows(self, n):
        return [torch.stack([torch.randperm(self.n_cells, generator=self.gen, device=self.dev)[:self.B] for _ in range(n)]).to(torch.int32)
                for _ in (0, 1)]

    def set_rows(self, rows, s):
        for g in (0, 1):
            self.rows_cur[g].copy_(rows[g][s], non_blocking=True)
            if self.mode == "cluster":
                self.lab_cur[g].copy_(self.data.labels[g][rows[g][s].long()])

    def capture(self, rows):
        self.set_rows(rows, 0)
        c0 = self.lib.spv_launch_count()
        self.graph = self.loop.capture(self.static)
        # 2 warm-up steps + 1 captured step (+ the weight re-staging launches at the end of capture())
        self.per_step_launches = (self.lib.spv_launch_count() - c0 - (4 if self.eng.bf16 else 0)) // 3

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize()

    def timed_steps(self, K, W, step_fn, profile=False):
        """W untimed warm-up steps, then exactly K timed steps; returns their ms (max over ranks) and the number of steps
        run in all.
        profile: cudaProfilerStart before the timed steps (`ncu --profile-from-start off` then sees only training steps, not
        the data generation, the index draws or the graph capture)"""
        n_steps_hint = 64
        rows = self.draw_rows(n_steps_hint)
        for s in range(W):
            step_fn(rows, s % n_steps_hint)
        self.barrier()
        if profile:
            torch.cuda.profiler.start()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for s in range(W, W + K):
            step_fn(rows, s % n_steps_hint)
        ev1.record()
        self.barrier()
        ms = ev0.elapsed_time(ev1)
        if self.dist is not None:
            t = torch.tensor([ms], device=self.dev)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, W + K

    # ---- device-resident throughput (graph replay)
    def measure_value(self, K, W):
        rows0 = self.draw_rows(1)
        use_graph = not self.args.no_graph
        if use_graph:
            self.capture(rows0)

        def step(rows, s):
            self.set_rows(rows, s)
            if use_graph:
                self.graph.replay()
            else:
                self.loop.step(self.static)

        n0 = self.lib.spv_launch_count()
        ms, n_run = self.timed_steps(K, W, step, profile=bool(os.environ.get("SPV_PROFILE_RANGE")))
        per_step = self.per_step_launches if use_graph else (self.lib.spv_launch_count() - n0) // n_run
        return {"value": self.world * 2 * self.B * K / (ms * 1e-3), "ms_per_step": ms / K, "ms": round(ms, 4),
                "launches_per_step": int(per_step), "gpu_launches": int(per_step * K)}

    # ---- the likelihood kernels alone, timed with CUDA events on the launching stream (eager passes, second group off)
    def measure_roofline(self, K):
        """the likelihood sweeps alone, each timed with CUDA events on the launching stream (eager passes, second group off):
        the forward-only sweep (evaluation passes; the kernel SURVEY 8(d)'s byte formula describes) and what a TRAINING step
        runs: one sweep that also emits the backward's operands (default), or forward + backward sweep (SPV_NB_SWEEPS=2)"""
        eng, B, G = self.eng, self.B, self.genes
        n = max(4, min(K, 20))
        rows = self.draw_rows(n)
        mk = lambda k: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(k)]
        single = bool(getattr(eng, "single_sweep", False)) and self.args.precision == "bf16"
        trn_ev, bwd_ev, fwd_ev = mk(2 * n), mk(2 * n), mk(2 * n)
        eng.parallel_groups = False  # each kernel is timed alone: no second group running beside it
        eng.nb_events, eng.nb_bwd_events = iter(trn_ev), iter(bwd_ev)
        for s in range(n):
            self.set_rows(rows, s)
            eng.forward(self.static, training=True)
            eng.backward()
        eng.nb_events, eng.nb_bwd_events = iter(fwd_ev), None
        for s in range(n):  # forward-only sweep: evaluation passes (running statistics, no gradients)
            self.set_rows(rows, s)
            eng.forward(self.static, training=False)
        torch.cuda.synchronize()
        eng.nb_events = eng.nb_bwd_events = None
        eng.parallel_groups = True
        def ms(ev):
            try:
                return float(np.mean([a.elapsed_time(b) for a, b in ev[2:]]))
            except Exception:  # events never recorded: this mode does not run that sweep as a separate kernel
                return None
        f_ms, t_ms = ms(fwd_ev), ms(trn_ev)
        b_ms = None if single else ms(bwd_ev)
        peak, sm_mhz, peak_src = peaks()
        KZ = S_DIM + P_DIM
        # SURVEY.md section 8(d): bytes of the NB-loglik forward kernel alone = counts (u16) + decoder weights read once as
        # 16-bit operands + 6 per-gene constants + per-cell decoder inputs (latents, hidden layer, library) + per-cell output
        alg_f = B * G * 2 + G * (KZ + 291) * 2 + 6 * G * 4 + B * (KZ + HD + 1) * 4 + B * 4
        # training sweep: the same reads + the backward's operands it must emit, (ep, rp, es, rs, dpi) as 16-bit values, + 2 column sums
        alg_t = alg_f + 5 * B * G * 2 + 2 * G * 4
        # separate backward sweep: the forward's reads + D3 = [dpi ; dyp ; dys] (16-bit) + 4 column sums
        alg_b = alg_f + 3 * B * G * 2 + 4 * G * 4
        elems = B * G
        # SFU (MUFU) pipe: 16 lanes per SM and clock = 4 per sub-partition; ex2 / lg2 / rcp per (cell, gene) element in nb_math.cuh
        mufu_peak = 148 * 16 * sm_mhz * 1e6
        MUFU = 8  # nb_math.cuh v5: ex2 x4, lg2 x3 (x2 in the backward-only sweep), one shared rcp (+ the rare exact variant)
        if self.args.precision == "bf16":
            kf = "nb_tc_fwd_kernel (tcgen05 decoder GEMMs + fused NB-mixture log-likelihood epilogue; forward-only sweep of evaluation passes)"
            kt = ("nb_tc_train_kernel (the training step's ONE sweep: the same + gradients w.r.t. the logits and theta, the backward GEMMs' "
                  "16-bit operands and column sums)") if single else kf.replace("forward-only sweep of evaluation passes", "forward sweep of a training step")
            kb = "nb_tc_bwd_kernel (tcgen05 recompute of the logits + likelihood gradients -> D3T, column sums)"
        else:
            kf = kt = "dec_tile_kernel<PASS_NB> (fp32 SIMT decoder GEMM + NB log-likelihood)"
            kb = "dec_tile_kernel<PASS_BWD>"
        hbm = lambda name, b, t, key: {"kernel": name, "bound": "hbm", "achieved": b / (t * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                       "frac": b / (t * 1e-3) / 1e9 / peak, "traffic": measured_traffic(self.workload, key),
                                       "algorithmic_bytes_per_launch": b, "avg_launch_ms": t}
        mufu = lambda name, t: {"kernel": name, "bound": "mufu", "achieved": MUFU * elems / (t * 1e-3) / 1e12, "peak": mufu_peak / 1e12,
                                "unit": "T SFU op/s", "frac": MUFU * elems / (t * 1e-3) / mufu_peak, "sfu_ops_per_element": MUFU,
                                "elements_per_launch": elems, "avg_launch_ms": t}
        roof = hbm(kf, alg_f, f_ms, "nb_tc_fwd_kernel")
        roof.update({"peak_source": peak_src,
                     "note": "algorithmic bytes by SURVEY 8(d) (forward-only sweep); the sweeps are bound by the SFU / issue pipes, not by HBM: "
                             "`other` carries the MUFU roofline (8 ex2/lg2/rcp per element) and the training step's sweep(s); ncu counters under profiles/",
                     "other": [mufu(kf, f_ms)]})
        if single:
            roof["other"] += [hbm(kt, alg_t, t_ms, "nb_tc_train_kernel"), mufu(kt, t_ms)]
        else:
            roof["other"] += [hbm(kt, alg_f, t_ms, "nb_tc_fwd_kernel")] + ([hbm(kb, alg_b, b_ms, "nb_tc_bwd_kernel"), mufu(kb, b_ms)] if b_ms else [])
        roof["sweeps_per_training_step"] = 1 if single else 2
        # the step's HBM-bound kernel for comparison: Adam over the whole flat parameter vector (28 bytes per parameter + staging)
        ad_ev = mk(8)
        for a, b in ad_ev:
            a.record()
            eng.adam_step(lr=0.0, eps=0.01, weight_decay=0.0)
            b.record()
        torch.cuda.synchronize()
        ad_ms = float(np.median([a.elapsed_time(b) for a, b in ad_ev[2:]]))
        ad_bytes = 28 * eng.params.numel + (2 * eng.params.numel if self.args.precision == "bf16" else 0)
        roof["other"].append({"kernel": "adam_kernel (whole parameter vector, + 16-bit operand staging)", "bound": "hbm",
                              "achieved": ad_bytes / (ad_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                              "frac": ad_bytes / (ad_ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": ad_bytes, "avg_launch_ms": ad_ms})
        return roof

    # ---- end to end through the drop-in plugin call: spVIPESmodule.forward(batch, loss_kwargs) -> loss.backward() -> torch Adam
    def measure_e2e_plugin(self, K, W, x_dtype=torch.float32, optimizer="flat"):
        """what scvi's TrainingPlan.training_step does per minibatch (reference caller: model/base/training_mixin.py:111-123),
        with pinned HOST minibatches in scvi's layout: X [B, G0 + G1] (the other group's columns zero), [B, 1] float code
        columns.  Inside the timed region every step: the host -> device copy of its inputs, the module call, loss.backward(),
        the optimiser step (Adam lr 1e-3, eps 0.01, weight_decay 1e-6: spvipes_b200.optim.FlatAdam, a torch.optim.Optimizer
        that scvi's TrainingPlan takes through optimizer_creator, or torch.optim.Adam as TrainingPlan builds it by default -
        whose multi-tensor step alone costs ~3.8 ms of host time per step), and the read-back of the loss."""
        from spvipes_b200.module import spVIPESmodule
        B, G, dev = self.B, self.genes, self.dev
        torch.manual_seed(1234 + self.rank)
        m = spVIPESmodule(groups_lengths={0: G, 1: G}, groups_obs_names=[None, None], groups_var_names={0: None, 1: None},
                          groups_obs_indices=[None, None], groups_var_indices=[np.arange(G), np.arange(G, 2 * G)],
                          transport_plan=self.plan, pair_data=self.mode == "paired", use_labels=self.mode == "label",
                          n_labels=self.n_labels, n_hidden=self.H, n_dimensions_shared=S_DIM, n_dimensions_private=P_DIM,
                          dropout_rate=0.1, device=str(dev), precision=self.args.precision)
        if self.world > 1:
            self.dist.broadcast(m.engine.params.flat, src=0)
        m.train()
        if optimizer == "flat":
            from spvipes_b200.optim import FlatAdam
            opt = FlatAdam(m, lr=1e-3, eps=0.01, weight_decay=1e-6)
        else:
            opt = torch.optim.Adam(m.parameters(), lr=1e-3, eps=0.01, weight_decay=1e-6)
        nh = 4 if B * G * 2 > 2 ** 25 else 8  # distinct pinned host minibatches, cycled (every step still copies its minibatch)
        rows = self.draw_rows(nh)
        host = []
        for s in range(nh):
            batch = []
            for g in (0, 1):
                r = rows[g][s].long()
                X = torch.zeros(B, 2 * G, dtype=x_dtype).pin_memory()
                own = self.data.X[g].view(torch.int16)[r].view(torch.uint16)
                X[:, g * G:(g + 1) * G] = (own.cpu() if x_dtype == torch.uint16 else own.to(torch.int32).to(torch.float32).cpu())
                d = {"X": X, "batch": torch.zeros(B, 1), "groups": torch.full((B, 1), float(g)),
                     "indices": r.float().reshape(-1, 1).cpu().pin_memory()}
                lab = self.data.labels[g][r].float().reshape(-1, 1).cpu().pin_memory()
                if self.mode == "label":
                    d["labels"] = lab
                elif self.mode == "cluster":
                    d["processed_transport_labels"] = lab
                batch.append(d)
            host.append(tuple(batch))
        out_host = torch.empty((), dtype=torch.float32).pin_memory()
        world, dist = self.world, self.dist

        def step(_rows, s):
            opt.zero_grad(set_to_none=True)
            _, _, lo = m(host[s % nh], loss_kwargs={"kl_weight": 0.0025})
            lo.loss.backward()
            if world > 1:  # data parallel the way a user of the module does it by hand: average the flat gradient buffer
                dist.all_reduce(m.engine.grads)
                m.engine.grads.div_(world)
            opt.step()
            out_host.copy_(lo.loss.detach(), non_blocking=True)

        ms, _ = self.timed_steps(K, max(W, 4), step)  # the first three calls run eagerly / capture the two buffer sets' graphs
        esz = 2 if x_dtype == torch.uint16 else 4
        h2d = 2 * (B * G * esz) + 2 * 2 * B * 4
        del m, opt, host
        torch.cuda.empty_cache()
        return {"value": world * 2 * B * K / (ms * 1e-3), "unit": "cells/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 4,
                "ms_per_step": ms / K,
                "api": f"spvipes_b200.module.spVIPESmodule.forward(tuple_of_group_dicts, loss_kwargs) -> loss.backward() -> "
                       f"{'spvipes_b200.optim.FlatAdam' if optimizer == 'flat' else 'torch.optim.Adam (default multi-tensor implementation)'}.step(); "
                       f"pinned host X {'uint16' if esz == 2 else 'float32'} [B, G0+G1] in scvi's layout, the group's own columns copied"}

    # ---- end to end through the training-loop API with host uint16 minibatches
    def measure_e2e_trainloop(self, K, W):
        """TrainLoop (one graph replay per step, fused Adam) fed from pinned host memory: per step the two groups' uint16 count
        minibatches [B, G] and labels are copied host -> device (double-buffered on a copy stream), the loss terms read back"""
        GB, loop, data, B, genes, dev = self.GroupBatch, self.loop, self.data, self.B, self.genes, self.dev
        if self.mode != "label":
            return None
        nh = 4 if B * genes * 2 > 2 ** 25 else 16
        rows = self.draw_rows(nh)
        host_x = [[data.X[g].view(torch.int16)[rows[g][s].long()].view(torch.uint16).cpu().pin_memory() for s in range(nh)] for g in (0, 1)]
        host_l = [[data.labels[g][rows[g][s].long()].cpu().pin_memory() for s in range(nh)] for g in (0, 1)]
        dev_x = [[torch.empty(B, genes, dtype=torch.uint16, device=dev) for _ in (0, 1)] for _ in (0, 1)]  # [buf][group]
        dev_l = [[torch.empty(B, dtype=torch.int32, device=dev) for _ in (0, 1)] for _ in (0, 1)]
        out_host = torch.empty(8, dtype=torch.float32).pin_memory()
        copy_stream = torch.cuda.Stream(device=dev)
        ready = [torch.cuda.Event() for _ in (0, 1)]
        freed = [torch.cuda.Event() for _ in (0, 1)]
        main = torch.cuda.current_stream(dev)
        bufs = [[GB(X=dev_x[b][g], labels=dev_l[b][g]) for g in (0, 1)] for b in (0, 1)]
        for b in (0, 1):
            for g in (0, 1):
                dev_x[b][g].copy_(host_x[g][0]); dev_l[b][g].copy_(host_l[g][0])
        graphs = [loop.capture(bufs[b]) for b in (0, 1)]
        for b in (0, 1):
            freed[b].record(main)
        state = {"n": 0}

        def step(_rows, s):
            i = state["n"]
            b = i % 2
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(freed[b])
                for g in (0, 1):
                    dev_x[b][g].copy_(host_x[g][i % nh], non_blocking=True)
                    dev_l[b][g].copy_(host_l[g][i % nh], non_blocking=True)
                ready[b].record(copy_stream)
            main.wait_event(ready[b])
            graphs[b].replay()
            freed[b].record(main)
            out_host.copy_(loop.engine.loss_out, non_blocking=True)
            state["n"] = i + 1

        ms, _ = self.timed_steps(K, W, step)
        h2d = sum(host_x[g][0].numel() * 2 + host_l[g][0].numel() * 4 for g in (0, 1))
        return {"value": self.world * 2 * B * K / (ms * 1e-3), "unit": "cells/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 32,
                "ms_per_step": ms / K, "api": "spvipes_b200.trainer.TrainLoop (host uint16 minibatches in pinned memory, loss terms read back)"}


def dump_outputs(eng, out_dir):
    """what the last step handed its caller, as float32 DIR/<name>.npy: the loss terms (engine.loss_terms()), the parameters
    after the optimiser step, their gradients and the BatchNorm running statistics (the engine's flat stores, in their fixed
    layout).  A vector longer than DUMP_SAMPLE is cut to the same seeded sample of positions on every run."""
    os.makedirs(out_dir, exist_ok=True)
    torch.cuda.synchronize()
    n = eng.params.numel
    keep = None
    if n > DUMP_SAMPLE:
        keep = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values.to(eng.device)
    sample = lambda t: t if keep is None else t[keep]
    arrays = {"loss_terms": eng.loss_terms(), "params": sample(eng.params.flat), "grads": sample(eng.grads),
              "running_stats": eng.buffers.flat}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def run_ours(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if os.environ.get("SPV_ALL_ON_GPU0"):
        local_rank = 0
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        backend = os.environ.get("SPV_DIST_BACKEND", "nccl")  # "gloo": debugging the multi-rank flow on a single GPU
        if backend == "nccl":
            dist.init_process_group("nccl", device_id=dev)
        else:
            dist.init_process_group(backend)
    from spvipes_b200 import _lib as L
    L.check(L.load().spv_arch_check(local_rank), "spv_arch_check (this library is sm_100a only)")
    K, W = args.steps, args.warmup
    workload = args.workload
    bench = Bench(workload, args, dev, dist, rank, world)
    clk = ClockSampler(local_rank)
    if rank == 0:
        clk.start()
    res = bench.measure_value(K, W)
    clocks = clk.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(bench.eng, args.dump_outputs)
    if hasattr(bench.loop.grad_sync, "check"):
        bench.loop.grad_sync.check()  # a handshake that timed out would have produced a number without the exchange
    sync_kind = bench.sync_kind
    loss = float(bench.eng.loss_out[0].item())
    roofline = bench.measure_roofline(K)
    e2e = e2e_u16 = e2e_tl = e2e_torch = None
    if not args.no_e2e:
        e2e = bench.measure_e2e_plugin(K, W, torch.float32)
        e2e_u16 = bench.measure_e2e_plugin(K, W, torch.uint16)
        e2e_tl = bench.measure_e2e_trainloop(K, W)
        if world == 1:
            e2e_torch = bench.measure_e2e_plugin(min(K, 10), W, torch.float32, optimizer="torch")
    line = {"metric": METRIC, "value": res["value"], "unit": "cells/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": ("f32 (tcgen05 GEMMs on split-bf16 / fp16 operands with f32 accumulation in TMEM; f32 elementwise, Adam)"
                      if args.precision == "bf16" else "f32"),
            "data": "synthetic", "config": dict(workload_config(workload, world), grad_sync=sync_kind), "clocks": clocks, "e2e": e2e,
            "e2e_uint16_input": e2e_u16, "e2e_trainloop": e2e_tl, "e2e_torch_adam": e2e_torch, "gpu_launches": res["gpu_launches"],
            "launches_per_step": res["launches_per_step"], "timing": {"timed_steps": K, "ms": res["ms"]},
            "roofline": roofline, "cpu_baseline": None, "final_loss": loss}
    # ---- the other BASELINE configs in the same run (N = 1 only), within the time budget
    configs = []
    if world == 1 and not args.no_configs:
        del bench
        torch.cuda.empty_cache()
        for wl in [w for w in ("C2", "C3", "C4") if w != workload]:
            if time.time() - T_START > args.budget:
                configs.append({"workload": wl, "skipped": f"time budget of {args.budget} s used up"})
                continue
            try:
                b2 = Bench(wl, args, dev, None, 0, 1)
                r2 = b2.measure_value(K, W)
                entry = {"config": workload_config(wl, 1), "value": r2["value"], "unit": "cells/s", "ms_per_step": r2["ms_per_step"],
                         "launches_per_step": r2["launches_per_step"],
                         "final_loss": float(b2.eng.loss_out[0].item()), "roofline": b2.measure_roofline(K)}
                if not args.no_e2e:
                    entry["e2e"] = b2.measure_e2e_plugin(K, W, torch.float32)
                configs.append(entry)
                del b2
                torch.cuda.empty_cache()
            except Exception as e:  # a config that does not fit this box is reported, not fatal
                configs.append({"workload": wl, "error": f"{type(e).__name__}: {e}"[:300]})
                torch.cuda.empty_cache()
    if rank == 0:
        line["configs"] = configs
        if world == 1 and not args.no_cpu_baseline:
            v, cms, cores, sample = cpu_reference_cells_per_sec(workload, args.cpu_steps if WORKLOADS[workload][4] <= 1024 else min(args.cpu_steps, 6), 1)
            line["cpu_baseline"] = {"value": v, "unit": "cells/s", "cores": cores, "kind": "port", "sample": sample, "ms_per_step": cms}
        line["wall_s"] = round(time.time() - T_START, 1)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=MIN_WARMUP,
                    help=f"untimed steps before the timed ones (CUDA path: at least {MIN_WARMUP})")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C5", choices=list(WORKLOADS))
    ap.add_argument("--cpu-steps", type=int, default=12)
    ap.add_argument("--budget", type=float, default=150.0, help="seconds after which no further extra config is started")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="headline workload only")
    ap.add_argument("--no-graph", action="store_true", help="issue every launch from Python instead of replaying a CUDA graph")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"],
                    help="bf16: tcgen05 tensor-core path for the large GEMMs; fp32: SIMT path")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs only: skip the host-fed measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/*.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the CUDA path's outputs (--impl ours)")
    args.warmup = max(args.warmup, MIN_WARMUP) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
