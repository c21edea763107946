"""Cost of validation during training on one GPU (profiles/validation_bench.md / .json), at the C5 and C2 minibatch shapes, bf16
engine (fused tensor-core decoder), label PoE, synthetic counts (synth.make_counts):

  1. one validation minibatch: eval forward with loss=False (encoders, PoE, decoder prologue, forward-only likelihood sweep of
     both groups) + spv_elbo_accumulate, CUDA events over back-to-back passes after warm-up;
  2. one validation epoch over a 10 % split of N cells per group (C5: N = 1,000,000 -> 100,000 cells, 49 minibatches; C2: N =
     250,000 -> 25,000 cells, 49 minibatches), run as spVIPES.train runs it: sequential minibatches whose row indices are uploaded
     from pinned host memory, the evaluation noise counter, one host read of the float64 sums at the end.  Host clock around the
     whole epoch, which ends in that read;
  3. the training step with validation off (the captured CUDA graph of TrainLoop: forward, backward, Adam), CUDA events over
     back-to-back replays, in the same process.

Only the validation cells are generated on the device (their values are synthetic; which rows of a real data set they would
be does not change the work).

    python tools/bench_validation.py [--out DIR (default profiles/)] [--iters 50] [--epochs 3]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from spvipes_b200 import synth  # noqa: E402
from spvipes_b200.engine import GroupBatch, StepEngine  # noqa: E402
from spvipes_b200.model import EVAL_NOISE_BASE  # noqa: E402
from spvipes_b200.trainer import TrainLoop, elbo_metrics, init_params  # noqa: E402
from tools.bench_decoded import H, NL, P, S, SHAPES, card, timed  # noqa: E402

N_CELLS = {"C5": 1_000_000, "C2": 250_000}
VAL_FRACTION = 0.1


def bench(shape, iters, epochs):
    G, B = SHAPES[shape]
    n_val = int(round(N_CELLS[shape] * VAL_FRACTION))
    eng = StepEngine((G, G), H, S, P, 0.1, "label", "cuda", precision="bf16")
    init_params(eng, seed=0)
    data = synth.make_counts((n_val, n_val), (G, G), NL, device="cuda", seed=1)
    # training step with validation off: the captured graph on the first B rows
    loop = TrainLoop(eng)
    loop.set_epoch(0)
    rows = [torch.arange(B, dtype=torch.int32, device="cuda") for _ in (0, 1)]
    tb = [GroupBatch(X=data.X[g], rows=rows[g], labels=data.labels[g], labels_per_cell=True, B=B) for g in (0, 1)]
    graph = loop.capture(tb)
    step_us = timed(graph.replay, iters)
    # one validation minibatch, back to back
    vb = [GroupBatch(X=data.X[g], rows=rows[g], labels=data.labels[g][:B].contiguous(), B=B) for g in (0, 1)]
    acc = torch.zeros(8, dtype=torch.float64, device="cuda")
    counter = torch.full((1,), EVAL_NOISE_BASE, dtype=torch.int32, device="cuda")

    def one_pass():
        with eng.noise_counter(counter):
            ws = eng.forward(vb, training=False, with_grad=False, loss=False)
            eng.accumulate_elbo(ws, acc)

    minibatch_us = timed(one_pass, iters)
    # a validation epoch as spVIPES._elbo_sums runs it (label mode: sequential chunks of both groups' validation rows)
    order = [np.random.RandomState(g).permutation(n_val).astype(np.int32) for g in (0, 1)]
    chunks = [[o[k:k + B] for k in range(0, n_val, B)] for o in order]

    def epoch():
        acc.zero_()
        counter.fill_(EVAL_NOISE_BASE)
        with eng.noise_counter(counter):
            for c0, c1 in zip(*chunks):
                r = [torch.from_numpy(c).pin_memory().to("cuda", non_blocking=True) for c in (c0, c1)]
                bt = [GroupBatch(X=data.X[g], rows=r[g], labels=data.labels[g][r[g].long()].contiguous(), B=len(r[g])) for g in (0, 1)]
                ws = eng.forward(bt, training=False, with_grad=False, loss=False)
                eng.accumulate_elbo(ws, acc)
        return acc.cpu()

    epoch()  # warm-up: workspaces of the ragged last minibatch, pinned buffers
    torch.cuda.synchronize()
    ep = []
    for _ in range(epochs):
        t0 = time.perf_counter()
        sums = epoch()
        ep.append((time.perf_counter() - t0) * 1e3)
    m = elbo_metrics(sums)
    res = {"B": B, "G": G, "n_val": n_val, "n_minibatches": len(chunks[0]), "train_step_us": step_us, "val_minibatch_us": minibatch_us,
           "val_epoch_ms": ep, "val_epoch_ms_min": min(ep), "elbo_validation": m["elbo_validation"]}
    res["val_epoch_per_minibatch_us"] = res["val_epoch_ms_min"] * 1e3 / res["n_minibatches"]
    del eng, data, graph
    torch.cuda.empty_cache()
    return res


def render(r):
    c = r["card"]
    lines = ["# Validation during training (eval pass + ELBO accumulation)", "",
             f"Measured on {c['name']}, power limit {c['power_limit']}, max SM clock {c['max_sm_clock']} "
             "(tools/bench_validation.py, one process).  bf16 engine, fused tensor-core decoder, label PoE, synthetic counts.  "
             "Validation minibatch: eval forward without the loss (both groups' encoders, PoE, decoder prologue and forward-only "
             "likelihood sweep) + spv_elbo_accumulate, CUDA events over back-to-back passes.  Validation epoch: a 10 % split run as "
             "spVIPES.train runs it, host clock up to the one read of the sums (best of the repeats).  Training step: the captured "
             "graph with validation off, same process.", "",
             "| shape | B | G | validation cells / group | minibatches | training step (us) | validation minibatch (us) "
             "| validation epoch (ms) | epoch / minibatch (us) |",
             "|---|---|---|---|---|---|---|---|---|"]
    for s, k in r["shapes"].items():
        lines.append(f"| {s} | {k['B']} | {k['G']} | {k['n_val']} | {k['n_minibatches']} | {k['train_step_us']:.1f} | "
                     f"{k['val_minibatch_us']:.1f} | {k['val_epoch_ms_min']:.2f} | {k['val_epoch_per_minibatch_us']:.1f} |")
    return "\n".join(lines) + "\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--epochs", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_validation needs a CUDA device")
    os.makedirs(a.out, exist_ok=True)
    r = {"card": card(), "shapes": {s: bench(s, a.iters, a.epochs) for s in SHAPES}}
    with open(os.path.join(a.out, "validation_bench.json"), "w") as f:
        json.dump(r, f, indent=1)
    with open(os.path.join(a.out, "validation_bench.md"), "w") as f:
        f.write(render(r))
    print(render(r))


if __name__ == "__main__":
    main()
