"""Count draws from the decoder's NB mixture on one GPU (profiles/sample_bench.md / .json), at the C5 and C2 minibatch shapes, bf16
engine (fused tensor-core decoder), label PoE, one group's operands of one eval pass.  CUDA events over back-to-back launches
after warm-up:

  1. the sampling sweep spv_dec_nb_sample_tc, one draw [B, G];
  2. the sampling sweep, 8 draws [8, B, G] in one launch;
  3. the element sweep spv_dec_nb_elems_tc writing `mean` only (the same prologue and MMAs, one fp32 [B, G] store);
  4. the torch route, as scvi 0.20 would run it: the element sweep writing rate_p, rate_s and pi (three fp32 [B, G]), then
     Bernoulli(sigmoid(pi)), torch.where, Gamma(theta, theta / mu).sample(), clamp, Poisson - torch's device samplers.

    python tools/bench_sample.py --out DIR [--iters 50]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from spvipes_b200 import _lib as L  # noqa: E402
from spvipes_b200 import synth  # noqa: E402
from spvipes_b200.engine import ELEM_OUTPUTS, HD, GroupBatch, StepEngine  # noqa: E402
from spvipes_b200.trainer import init_params  # noqa: E402
from tools.bench_decoded import H, NL, P, S, SHAPES, card, timed  # noqa: E402


def torch_route_sample(rate_p, rate_s, pi, theta):
    """scvi 0.20 NegativeBinomialMixture.sample (theta2 = None) on given parameters, torch's samplers"""
    mu = torch.where(torch.bernoulli(torch.sigmoid(pi)).bool(), rate_p, rate_s)
    lam = torch.distributions.Gamma(concentration=theta, rate=theta / mu).sample()
    return torch.poisson(torch.clamp(lam, max=1e8))


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
    out = torch.empty(8, B, G, device="cuda")
    samp = lambda n: (lambda: L.check(lib.spv_dec_nb_sample_tc(dptrs, *args, d.KMIX, 7, 0, 0, n, out.data_ptr(), G, B * G, st),
                                      "spv_dec_nb_sample_tc"))
    outs = {k: torch.empty(B, G, device="cuda") for k in ELEM_OUTPUTS}
    el = lambda arr: (lambda: L.check(lib.spv_dec_nb_elems_tc(src, dptrs, ldx, *args, d.KMIX, arr, G, st), "spv_dec_nb_elems_tc"))
    mean1 = L.ptr_array([outs["mean"] if k == "mean" else None for k in ELEM_OUTPUTS])
    par3 = L.ptr_array([outs[k] if k in ("rate_p", "rate_s", "pi") else None for k in ELEM_OUTPUTS])
    theta = w.genec[L.GC_THETA, :G].clone()
    elems3 = el(par3)

    def torch_route():
        elems3()
        return torch_route_sample(outs["rate_p"], outs["rate_s"], outs["pi"], theta)

    res = {"B": B, "G": G, "sample1_us": timed(samp(1), iters), "sample8_us": timed(samp(8), iters), "mean_us": timed(el(mean1), iters),
           "torch_route_us": timed(torch_route, iters)}
    res["elems3_us"] = timed(elems3, iters)
    res["sample_bytes"] = B * G * 4
    # draws of the sweep against the torch route on the same parameters: sample means over the [B, G] elements
    samp(8)()
    ref = torch.stack([torch_route() for _ in range(8)])
    el(mean1)()
    torch.cuda.synchronize()
    res["mean_count_sweep"] = float(out.double().mean())
    res["mean_count_torch"] = float(ref.double().mean())
    res["mean_of_means"] = float(outs["mean"].double().mean())
    del eng, data
    torch.cuda.empty_cache()
    return res


def render(r):
    c = r["card"]
    lines = ["# Count draws from the NB mixture (sampling sweep, torch route)", "",
             f"Measured on {c['name']}, power limit {c['power_limit']}, max SM clock {c['max_sm_clock']} "
             f"(tools/bench_sample.py, one process).  bf16 engine, fused tensor-core decoder, label PoE, one group's operands of an eval "
             "pass; CUDA events over back-to-back launches after warm-up.  The torch route is the element sweep writing rate_p, rate_s "
             "and pi, then torch's Bernoulli, Gamma and Poisson samplers, as scvi's NegativeBinomialMixture.sample runs them.", "",
             "| shape | B | G | sampling sweep, 1 draw (us) | sampling sweep, 8 draws (us) | per draw (us) | element sweep, mean only (us) "
             "| torch route, 1 draw (us) | of which element sweep, 3 outputs (us) | mean count: sweep / torch / mean |",
             "|---|---|---|---|---|---|---|---|---|---|"]
    for s, k in r["kernels"].items():
        lines.append(f"| {s} | {k['B']} | {k['G']} | {k['sample1_us']:.1f} | {k['sample8_us']:.1f} | {k['sample8_us'] / 8:.1f} | "
                     f"{k['mean_us']:.1f} | {k['torch_route_us']:.1f} | {k['elems3_us']:.1f} | "
                     f"{k['mean_count_sweep']:.4f} / {k['mean_count_torch']:.4f} / {k['mean_of_means']:.4f} |")
    return "\n".join(lines) + "\n"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--iters", type=int, default=50)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sample needs a CUDA device")
    os.makedirs(a.out, exist_ok=True)
    r = {"card": card(), "kernels": {s: kernels(s, a.iters) for s in SHAPES}}
    with open(os.path.join(a.out, "sample_bench.json"), "w") as f:
        json.dump(r, f, indent=1)
    with open(os.path.join(a.out, "sample_bench.md"), "w") as f:
        f.write(render(r))
    print(render(r))


if __name__ == "__main__":
    main()
