"""The decoder stage (factor regressors + mixing net + NB-mixture likelihood) of every decoder path against a float64
restatement of the same operation, on inputs built to take the kernels' data-dependent branches.

The end-to-end parity tests sum every element into one loss term or one max-normalised gradient, and they run on initial
weights and synthetic counts, which seldom reach the element math's edge branches.  Here the engine runs one training step
(or one eval forward) on a crafted state, and the decoder's own inputs are read back from its workspace:
zz = amix[:, HD:HD + KZ] (the [z_private_arg | z_shared_arg] ordering of quirk Q1), the library sizes and the ReLU gates of
the mixing net's hidden layer.  From those inputs, as float64 leaves, oracle.restatement.decoder + log_mixture_nb (target
log1p(counts), theta = exp(px_r)) give the reference of every output of the stage; the loss term `rec_g.mean()` is the only
one that reaches the decoder parameters and zz, so its float64 autograd is the exact reference of every decoder_g.* / px_r.g
gradient and of d zz (which the engine assembles from spv_dec_gene_bwd + spv_dec_dzz_combine, BatchNorm coupling included).

Per group, the first 64 genes are edge genes (the rest are ordinary synthetic genes, so plain full tiles exist too):
  * rate ladders: per-gene factor-regressor BatchNorm bias (private genes 0-11, shared genes 12-23), solved in float64 so that
    rho spans 1e-9 .. 1e-3 across the 1e-6 threshold of the EXACT element math, both sides inside one aligned group of 4
    genes, all with positive counts; one more rare gene alone in an otherwise ordinary tile (gene 69);
  * counts cycling through {0, 1, 15, 16, 17, 255, 256, 4095, 65535} (the table / slow-path boundary at NB_TAB = 16), plus
    {1e-3, 0.5, 2.25, 15.5, 15.999} when the source is float32;
  * px_r from -7 to 9 (genes 32-47), mixture bias +-{0, 1e-3, 5, 20, 60} (genes 48-56).
Both groups live in one [N, ld] count matrix (odd row pitch, group 1 at an odd column offset), rows gathered with scattered
indices.  The minibatch sizes pick the size-dependent forms: B = 300 (latent statistics in one 8-CTA cluster, cached
BatchNorm backward, partial row and gene tiles), 1000 (64-row statistics tiles + exact merge, 40-row last tile), 2100
(BatchNorm backward as a cluster of 3 CTAs), 8300 (uncached BatchNorm backward).

Gates.  fp32 mode: 1e-4 on reconstruction terms, latent statistics and BatchNorm running statistics, 2e-3 on gradients (the
parity gates of tests/test_gpu_shapes.py).  Tensor-core paths: each gate is at most 4x the worst error measured on a B200 over
this file's cases; TC_GATES lists them with the measurement behind each.  The reconstruction and parameter-gradient gates stay
within the north-star ceilings (1e-2, GRAD_TOL_TC).  Three weak spots found here exceed GRAD_TOL_TC and are gated on their own,
at their measured size: d px_r (and the d theta column sums) of genes with theta > e^6.5, where the d-theta form cancels;
weight gradients when the latents sit far from zero (contractions over uncentred latents, both modes); and the unfused bf16
decoder's bf16 gradient operands.  The fp16 per-element outputs of the training sweep carry their storage rounding plus the
plain element form's documented approximation (ep / es relative error 1e-8 / rho just above rho = 1e-6).
"""
import functools
import math
import os
import re

import numpy as np
import pytest
import torch

from oracle import restatement as rs
from tests.helpers import gate_consistent, grad_errors

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HD, H = 256, 128
GRAD_TOL_TC = 2e-3
RARE = 1e-6                                    # nb_math.cuh NB_X_RARE = log2(1e-6)
NEAR_RARE = 1e-4                               # above this the plain form's log(rho + 1e-8) = log(rho) is within 1e-4
COUNTS_U16 = (0, 1, 15, 16, 17, 255, 256, 4095, 65535)
COUNTS_F32 = COUNTS_U16 + (1e-3, 0.5, 2.25, 15.5, 15.999)
RATE_TARGETS = (1e-9, 1e-8, 1e-7, 3e-7, 6e-7, 9e-7, 1.2e-6, 2e-6, 5e-6, 2e-5, 1e-4, 1e-3)
RATE_P, RATE_S = range(0, 12), range(12, 24)
COUNT_GENES, THETA_GENES, PI_GENES = range(24, 32), range(32, 48), range(48, 57)
LONE_GENE, LONE_TARGET = 69, 5e-7
PI_BIAS = (0.0, 1e-3, -1e-3, 5.0, -5.0, 20.0, -20.0, 60.0, -60.0)
EDGE = 64
LADDER_GAMMA = 0.2  # BatchNorm weight of the ladder genes: rho varies by about e^(+-0.6) around the target across cells

# name: (B, (G0, G1), n_shared, n_private, count dtype, offset latents)
CASES = {
    "b300": (300, (1003, 515), 25, 10, "u16", False),
    "b300-f32": (300, (1003, 515), 25, 10, "f32", False),
    "b1000": (1000, (5001, 2048), 25, 10, "u16", False),
    "b1000-offset": (1000, (1001, 515), 25, 10, "u16", True),
    "b2100": (2100, (515, 259), 25, 10, "u16", False),
    "b8300": (8300, (259, 131), 25, 10, "u16", False),
    # latent widths around the fused decoder's limit (ZK_MAX_LATENT = 58) and at the decoder's limit (96)
    "w58": (300, (1003, 515), 40, 18, "u16", False),
    "w59": (300, (1003, 515), 40, 19, "u16", False),
    "w64": (300, (1003, 515), 40, 24, "u16", False),
    "w65": (300, (1003, 515), 40, 25, "u16", False),
    "w96": (300, (1003, 515), 48, 48, "u16", False),
}


# ------------------------------------------------------------------------------------------------------------------------
# case builder (CPU)
# ------------------------------------------------------------------------------------------------------------------------
def _ladder_counts(B, n_genes, values, seed):
    """[B, n_genes] counts cycling through `values` (a different phase per gene and per row)"""
    v = torch.tensor(values, dtype=torch.float64)
    b = torch.arange(B).unsqueeze(1)
    g = torch.arange(n_genes).unsqueeze(0)
    return v[(7 * b + 3 * g + seed) % len(values)]


def _f64_encode(sd, x, case, training=True):
    """float64 latents of the crafted state (oracle restatement): zz = [z_private_arg | z_shared_arg] and lib per group"""
    S, P = case["S"], case["P"]
    sd64 = {k: v.double() for k, v in sd.items()}
    with torch.no_grad():
        out = rs.step(sd64, x, mode="label", n_shared=S, n_private=P, eps_private=[e.double() for e in case["eps_p"]],
                      eps_poe=[e.double() for e in case["eps_q"]], labels=case["labels"],
                      drop_masks={k: v.double() for k, v in case["dm"].items()}, training=training)
    zz, lib = [], []
    for g in (0, 1):
        c = torch.cat((out["private_log_z"][g], out["poe_log_z"][g]), dim=1)
        zz.append(torch.cat((c[:, S:S + P], c[:, :S]), dim=1))
        lib.append(out["library"][g].reshape(-1))
    return zz, lib


def _branch_logits(sd, g, z, branch, training):
    """y = BatchNorm(z W^T) of one factor regressor, float64"""
    k = f"decoder_{g}.factor_regressor_{branch}.fc_layers.Layer 0"
    u = z @ sd[k + ".0.weight"].double().t()
    return rs.batch_norm(u, sd[k + ".1.weight"].double(), sd[k + ".1.bias"].double(), sd[k + ".1.running_mean"].double(),
                         sd[k + ".1.running_var"].double(), training, rs.DEC_BN_EPS, rs.DEC_BN_MOM)


@functools.lru_cache(maxsize=4)
def build_case(name):
    """inputs of one case: count matrix, row indices, labels, noise and the crafted state dict (all CPU)"""
    B, genes, S, P, src, offset = CASES[name]
    seed = sum(map(ord, name))
    gen = torch.Generator().manual_seed(seed)
    sd = rs.default_state_dict(genes, n_hidden=H, n_shared=S, n_private=P, seed=seed)
    N = B + B // 2 + 5
    # both groups in one matrix: group 1 at an odd column offset, odd row pitch
    col0 = [0, genes[0] + 1 - genes[0] % 2]
    ld = col0[1] + genes[1] + 1
    ld += 1 - ld % 2
    X = torch.zeros(N, ld, dtype=torch.float64)
    from spvipes_b200 import synth
    base = synth.make_counts((N, N), genes, 6, device="cpu", seed=seed)
    rows = [torch.randperm(N, generator=gen)[:B] for _ in (0, 1)]
    values = COUNTS_F32 if src == "f32" else COUNTS_U16
    positive = [v for v in values if v > 0]
    for g in (0, 1):
        G = genes[g]
        Xg = base.X[g].to(torch.int32).double()
        r = rows[g]
        # edge genes: ladder counts in the minibatch's rows (other rows keep their synthetic counts)
        Xg[r, :EDGE] = _ladder_counts(B, EDGE, values, g)
        rare = list(RATE_P) + list(RATE_S) + ([LONE_GENE] if G > LONE_GENE + 64 else [])
        rc = _ladder_counts(B, len(rare), positive, g + 1)
        rc[::2] = rc[::2].clamp(max=15.0)  # every other row: tabulated counts only (the quad-level plain / EXACT choice)
        Xg[r[:, None], torch.tensor(rare)] = rc
        if src == "f32":  # float32 source: some non-integer counts among the ordinary genes too
            frac = torch.rand(N, G, generator=gen) < 0.05
            frac[:, :EDGE] = False
            Xg[frac] += 0.25
        X[:, col0[g]:col0[g] + G] = Xg
    labels = [torch.randint(0, 5, (B,), generator=gen).numpy() for _ in (0, 1)]
    eps_p = [torch.randn(B, P, generator=gen) for _ in (0, 1)]
    eps_q = [torch.randn(B, S, generator=gen) for _ in (0, 1)]
    drop = [(torch.rand(B, 2 * H, generator=gen) < 0.9).float() / 0.9 for _ in (0, 1)]
    dm = {(g, k): drop[g][:, i * H:(i + 1) * H] for g in (0, 1) for i, k in enumerate(("private", "shared"))}
    case = dict(name=name, offset=offset, B=B, genes=genes, S=S, P=P, src=src, X=X, col0=col0, rows=rows, labels=labels, eps_p=eps_p,
                eps_q=eps_q, drop=drop, dm=dm)
    # crafted state
    for g in (0, 1):
        G = genes[g]
        dec = f"decoder_{g}"
        fl = "fc_layers.Layer 0"
        for br in ("factor_regressor_private", "factor_regressor_shared", "sigmoid_decoder"):
            k = f"{dec}.{br}.{fl}.1"
            n = sd[k + ".running_mean"].numel()
            sd[k + ".running_mean"] = 0.1 * torch.randn(n, generator=gen)   # eval mode: non-trivial running statistics
            sd[k + ".running_var"] = 0.5 + torch.rand(n, generator=gen)
        px = sd[f"px_r.{g}"]
        px[list(THETA_GENES)] = torch.linspace(-7.0, 9.0, len(THETA_GENES))
        bm = sd[f"{dec}.mixture.{fl}.0.bias"]
        bm[list(PI_GENES)] = torch.tensor(PI_BIAS)
        for br, ladder in (("private", RATE_P), ("shared", RATE_S)):
            idx = list(ladder) + ([LONE_GENE] if (br == "private" and G > LONE_GENE + 64) else [])
            sd[f"{dec}.factor_regressor_{br}.{fl}.1.weight"][idx] = LADDER_GAMMA
            sd[f"{dec}.factor_regressor_{br}.{fl}.1.bias"][idx] = -30.0  # out of the normaliser while it is solved
    if offset:  # latents ~ 30 + O(1): the latent statistics must centre before they square
        for g in (0, 1):
            for enc in ("private", "shared"):
                sd[f"encoder_{g}_{enc}.mu_encoder.1.bias"].fill_(30.0)
                sd[f"encoder_{g}_{enc}.lvar_encoder.1.bias"].fill_(-12.0)
    # rate ladders: solve the BatchNorm bias of each ladder gene in float64 so that its median rho over the minibatch hits the
    # target (rho = exp(lib) softmax(y); the ladder genes' own share of the normaliser is negligible)
    x = [case_counts(case, g) for g in (0, 1)]
    zz, lib = _f64_encode(sd, x, case)
    for g in (0, 1):
        G = genes[g]
        fl = "fc_layers.Layer 0"
        for br, z, ladder in (("private", zz[g][:, :P], RATE_P), ("shared", zz[g][:, P:], RATE_S)):
            idx = list(ladder) + ([LONE_GENE] if (br == "private" and G > LONE_GENE + 64) else [])
            tgt = list(RATE_TARGETS) + ([LONE_TARGET] if len(idx) > len(ladder) else [])
            y = _branch_logits(sd, g, z, br, True)
            keep = torch.ones(G, dtype=torch.bool)
            keep[idx] = False
            c = lib[g] - torch.logsumexp(y[:, keep], dim=1)
            bias = sd[f"decoder_{g}.factor_regressor_{br}.{fl}.1.bias"]
            yi = y[:, idx] - bias[idx].double()  # the gamma * xhat part of the ladder genes
            for j, (gi, t) in enumerate(zip(idx, tgt)):
                bias[gi] = float(math.log(t) - torch.median(c + yi[:, j]))
    case["sd"] = sd
    return case


def case_counts(case, g):
    """[B, G] float64 counts of group g's minibatch"""
    c0, G = case["col0"][g], case["genes"][g]
    return case["X"][case["rows"][g]][:, c0:c0 + G]


# ------------------------------------------------------------------------------------------------------------------------
# float64 reference of the decoder stage
# ------------------------------------------------------------------------------------------------------------------------
def reference(sd, g, zz, lib, xraw, P, training, gates=None, probe=None):
    """float64 decoder stage of group g from the given inputs.  Returns the per-cell reconstruction term, the gradients of
    rec.mean() w.r.t. the decoder parameters and zz, the BatchNorm running statistics, and the per-element quantities of the
    likelihood: rho, pi, ep / es = d ll / d log rho at a fixed normaliser, d ll / d pi, and the per-element contributions to
    the column sums (d loss / d y_p, d y_s, d pi, d theta with loss = rec.mean())."""
    dev = zz.device
    keys = [k for k in sd if (k.startswith(f"decoder_{g}.") or k == f"px_r.{g}")]
    sdl = {k: sd[k].to(dev, torch.float64).clone().requires_grad_("running" not in k) for k in keys}
    zzl = zz.to(torch.float64).clone().requires_grad_(training)
    lib = lib.to(torch.float64).reshape(-1, 1)
    xl = torch.log1p(xraw.to(dev, torch.float64))
    B = zz.shape[0]
    new_stats = {}
    with torch.set_grad_enabled(training):
        rate_p, rate_s, mix = rs.decoder(sdl, g, zzl[:, :P], zzl[:, P:], lib, training, new_stats, gates=gates, probe=probe)
        theta = torch.exp(sdl[f"px_r.{g}"])
        rec = -rs.log_mixture_nb(xl, rate_p, rate_s, theta, mix).sum(-1)
    out = {"rec": rec.detach(), "rho_p": rate_p.detach(), "rho_s": rate_s.detach(), "pi": mix.detach(), "new_stats": new_stats,
           "x": xraw.to(dev, torch.float64)}
    if not training:
        return out
    rec.mean().backward()
    out["grads"] = {k: v.grad for k, v in sdl.items() if v.grad is not None}
    out["grads"]["dzz"] = zzl.grad
    # per-element derivatives of ll at fixed normalisers
    lrp = torch.log(rate_p.detach()).requires_grad_()
    lrs = torch.log(rate_s.detach()).requires_grad_()
    pil = mix.detach().requires_grad_()
    th = theta.detach()
    ll = rs.log_mixture_nb(xl, torch.exp(lrp), torch.exp(lrs), th, pil)
    ep, es, dpi = torch.autograd.grad(ll.sum(), (lrp, lrs, pil))
    _, dth = torch.func.jvp(lambda t: rs.log_mixture_nb(xl, rate_p.detach(), rate_s.detach(), t, mix.detach()), (th,),
                            (torch.ones_like(th),))
    sm_p, sm_s = rate_p.detach() / torch.exp(lib), rate_s.detach() / torch.exp(lib)
    dyp = ep - sm_p * ep.sum(1, keepdim=True)  # softmax backward
    dys = es - sm_s * es.sum(1, keepdim=True)
    out.update(ep=ep, es=es, dpi=dpi, sm_p=sm_p, sm_s=sm_s,
               contrib=torch.stack([-dyp / B, -dys / B, -dpi / B, -dth / B]))  # colsum rows: dyp, dys, dpi, dtheta
    return out


def edge_classes(case, refs):
    """element / tile classes of one case from the float64 side: {class: count}, both groups together"""
    B = case["B"]
    n = {"rare_p": 0, "rare_s": 0, "rare_quad_split": 0, "rare_tabulated_quad": 0, "count_ge16": 0, "non_integer": 0, "pi_pos": 0, "pi_neg": 0,
         "pi_big_pos": 0, "pi_big_neg": 0}
    for g, r in enumerate(refs):
        x = r["x"]
        pos = x > 0
        rp, rsv = r["rho_p"] < RARE, r["rho_s"] < RARE
        n["rare_p"] += int((rp & pos).sum())
        n["rare_s"] += int((rsv & pos).sum())
        G4 = x.shape[1] // 4 * 4
        rare = ((rp | rsv) & pos)[:, :G4].reshape(B, -1, 4)
        plain = (~(rp | rsv) & pos)[:, :G4].reshape(B, -1, 4)
        n["rare_quad_split"] += int((rare.any(2) & plain.any(2)).sum())
        tab = (x < 16) & (x == torch.floor(x))
        n["rare_tabulated_quad"] += int((rare.any(2) & tab[:, :G4].reshape(B, -1, 4).all(2)).sum())
        n["count_ge16"] += int((x >= 16).sum())
        n["non_integer"] += int((x != torch.floor(x)).sum())
        n["pi_pos"] += int((r["pi"] > 0).sum())
        n["pi_neg"] += int((r["pi"] < 0).sum())
        n["pi_big_pos"] += int((r["pi"] > 15).sum())
        n["pi_big_neg"] += int((r["pi"] < -15).sum())
    n["partial_row_tile"] = int(B % 128 != 0 and B % 64 != 0)
    n["partial_gene_tile"] = sum(int(G % 64 != 0) for G in case["genes"])
    return n


def assert_classes(case, refs):
    n = edge_classes(case, refs)
    need = ["rare_p", "rare_s", "rare_quad_split", "rare_tabulated_quad", "count_ge16", "pi_pos", "pi_neg", "pi_big_pos", "pi_big_neg"]
    if case["src"] == "f32":
        need.append("non_integer")
    if case["B"] <= 1000:  # the larger minibatches test the size-dependent forms; 300 and 1000 also the ragged tiles
        need += ["partial_row_tile", "partial_gene_tile"]
    missing = [k for k in need if n[k] == 0]
    assert not missing, (case["name"], missing, n)
    return n


@pytest.mark.parametrize("name", list(CASES))
def test_case_builder_reaches_every_branch(name):
    """CPU: every case takes the branches it is built for (float64 latents of the crafted state, training-mode statistics)"""
    case = build_case(name)
    x = [case_counts(case, g) for g in (0, 1)]
    zz, lib = _f64_encode(case["sd"], x, case)
    refs = [reference(case["sd"], g, zz[g], lib[g], x[g], case["P"], True) for g in (0, 1)]
    assert_classes(case, refs)


def test_latent_limits_match_kernels():
    """the engine's latent-width limits are the kernels' (decoder_common.cuh)"""
    from spvipes_b200 import _lib as L
    src = open(os.path.join(ROOT, "spvipes_b200", "csrc", "decoder_common.cuh")).read()
    assert int(re.search(r"#define ZK_MAX_LATENT (\d+)", src).group(1)) == L.ZK_MAX_LATENT
    assert int(re.search(r"#define DEC_MAX_LATENT (\d+)", src).group(1)) == L.DEC_MAX_LATENT


@pytest.mark.parametrize("S,P,n_batch,fused", [(40, 18, 0, True), (40, 19, 0, False), (40, 24, 0, False), (25, 10, 12, False),
                                               (25, 10, 11, True), (48, 48, 0, False)])
def test_fused_decoder_only_within_its_latent_limit(S, P, n_batch, fused):
    """bf16 mode takes the fused decoder exactly when P + S (+ both covariate copies) <= ZK_MAX_LATENT"""
    from spvipes_b200.engine import StepEngine
    eng = StepEngine((70, 65), 32, S, P, 0.1, "label", "cpu", precision="bf16", n_batch=n_batch)
    assert eng.fused_nb == fused
    assert eng.single_sweep == fused


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_latent_width_beyond_decoder_limit_is_rejected(precision):
    from spvipes_b200.engine import StepEngine
    with pytest.raises(NotImplementedError):
        StepEngine((70, 65), 32, 49, 48, 0.1, "label", "cpu", precision=precision)
    with pytest.raises(NotImplementedError):
        StepEngine((70, 65), 32, 30, 20, 0.1, "label", "cpu", precision=precision, n_batch=24)


# ------------------------------------------------------------------------------------------------------------------------
# GPU: engine against the float64 reference
# ------------------------------------------------------------------------------------------------------------------------
# Tensor-core gates (relative errors as defined in _compare), measured worst over this file's cases on a B200 in brackets
TC_GATES = {
    "rec": 5e-4,                       # per cell; measured 1.61e-4 (B = 2100, single sweep)
    "stats": 1.5e-6,                   # zmean / zcov (fp32 kernels in both modes); measured 4.8e-7
    "bn_running": 8e-7,                # measured 2.0e-7
    "colsum": 1e-2,                    # per gene (_compare); measured 4.7e-3
    "colsum_large_theta": 2.4e-2,      # d theta column sums of genes with px_r > 6.5; measured 6.1e-3 (B = 1000)
    "elem_ep": 4e-2,                   # ep, es, rp', rs' of E4T (fp16), per gene; measured 1.18e-2 (offset latents)
    "elem_dpi": 2.8e-2,                # DPIT (fp16), per gene; measured 7.1e-3
    "elem_near_rare": 3.5e-2,          # elements with 1e-6 <= rho < 1e-4; measured 9.8e-3
    "grad": GRAD_TOL_TC,               # fused decoder; measured 1.3e-3 (B = 8300)
    "grad_edge": GRAD_TOL_TC,          # px_r, bm and the branch biases on the edge genes; measured 5.7e-4
    "grad_px_r_large_theta": 1.2e-2,   # d px_r of genes with px_r > 6.5; measured 3.1e-3
    "grad_offset": 1e-2,               # latents ~ 30: factor-regressor and hidden-layer weights; measured 2.5e-3
    "grad_unfused": 1e-2,              # unfused bf16 decoder (P + S > 58): hidden-layer weight; measured 2.7e-3
}
COLSUM_FLOOR = 1e-3  # column-sum errors: relative to the gene's sum of |contribution| + this fraction of the median gene's
FP32_GATES = {"rec": 1e-4, "stats": 1e-4, "bn_running": 1e-4, "colsum": 2e-3, "colsum_large_theta": 1.2e-2, "grad": 2e-3,
              "grad_edge": 2e-3, "grad_offset": 1.2e-2}  # measured: colsum_large_theta 3.3e-3, grad_offset 3.1e-3


def _run_engine(case, precision, training):
    from spvipes_b200.engine import GroupBatch, Noise, StepEngine
    B, genes, S, P = case["B"], case["genes"], case["S"], case["P"]
    eng = StepEngine(genes, H, S, P, 0.1, "label", "cuda", precision=precision)
    eng.load_state_dict(case["sd"])
    if case["src"] == "f32":
        X = case["X"].to(torch.float32).cuda()
    else:
        X = case["X"].to(torch.int32).cuda().to(torch.uint16)
    batches = [GroupBatch(X=X, rows=case["rows"][g].to(torch.int32).cuda(), col0=case["col0"][g],
                          labels=torch.from_numpy(case["labels"][g].astype(np.int32)).cuda()) for g in (0, 1)]
    noise = Noise([e.cuda() for e in case["eps_p"]], [e.cuda() for e in case["eps_q"]], [d.cuda() for d in case["drop"]])
    ws = eng.forward(batches, training=training, noise=noise)
    if training:
        eng.backward()
    torch.cuda.synchronize()
    return eng, ws


def _rel(got, want):
    got, want = got.double(), want.double()
    return float((got - want).abs().max() / (want.abs().max() + 1e-300))


def _per_gene_rel(got, want, floor_frac=1e-3):
    """max over genes (columns) of max_b |got - want| / max_b |want| (floored at floor_frac of the global max)"""
    got, want = got.double(), want.double()
    den = want.abs().amax(0).clamp(min=floor_frac * float(want.abs().max()))
    return float(((got - want).abs().amax(0) / den).max())


def _compare(eng, ws, case, training, fused, single):
    precision_fp32 = not eng.bf16
    """errors of one engine run against the float64 reference (both groups) + the element classes it covered"""
    P, KZ = case["P"], case["P"] + case["S"]
    err, where = {}, {}
    refs = []
    sd = {k: v.cuda() for k, v in case["sd"].items()}
    for g, w in enumerate(ws):
        zz = w.amix[:, HD:HD + KZ].double()
        lib = w.lib.double()
        x = case_counts(case, g).cuda()
        key = f"decoder_{g}.sigmoid_decoder"
        probe = {}  # pre-activations of the hidden layer: its ReLU gates as the engine took them where they are ambiguous
        with torch.no_grad():
            rs.decoder({k: v.double() for k, v in sd.items()}, g, zz[:, :P], zz[:, P:], lib.reshape(-1, 1), training, {},
                       probe=probe)
        gates, switched = gate_consistent({key: probe[key].cpu()}, {key: (w.amix[:, :HD] > 0).cpu()})
        ref = reference(sd, g, zz, lib, x, P, training, gates={key: gates[key].cuda()})
        refs.append(ref)
        up = lambda k, v: err.__setitem__(k, max(err.get(k, 0.0), v))
        up("rec", float(((w.rec.double() - ref["rec"]).abs() / ref["rec"].abs()).max()))
        if not training:
            continue
        up("stats", _rel(w.zmean[:KZ], zz.mean(0)))
        zc = zz - zz.mean(0)
        up("stats", _rel(w.zcov.reshape(-1)[:KZ * KZ].view(KZ, KZ), zc.t() @ zc / zz.shape[0]))
        esd = eng.state_dict()
        for k, v in ref["new_stats"].items():
            up("bn_running", _rel(esd[k], v))
        hi_theta = sd[f"px_r.{g}"] > 6.5
        # column sums, each gene normalised by its sum of |contribution|
        rows = (2, 3) if single else (0, 1, 2, 3)
        for r in rows:
            c = ref["contrib"][r]
            mag = c.abs().sum(0)
            e = (w.colsum[r].double() - c.sum(0)).abs() / (mag + COLSUM_FLOOR * mag.median())
            if r == 3:  # d theta of genes with theta > e^6.5: cancellation in the d-theta form (module docstring)
                up("colsum_large_theta", float(e[hi_theta].max()))
                e = torch.where(hi_theta, 0.0, e)
            up("colsum", float(e.max()))
            if float(e.max()) >= err["colsum"]:
                gi = int(e.argmax())
                where["colsum"] = (g, r, gi, float(w.colsum[r, gi]), float(c.sum(0)[gi]), float(mag[gi]))
        if single:  # per element: fp16 outputs of the training sweep
            B, G = zz.shape[0], x.shape[1]
            # elements just above the EXACT threshold carry the plain form's documented approximation (nb_math.cuh): compared
            # on their own (elem_near_rare), the rest against the fp16 / fast-transcendental gate
            near = (x > 0) & (((ref["rho_p"] >= RARE) & (ref["rho_p"] < NEAR_RARE)) | ((ref["rho_s"] >= RARE) & (ref["rho_s"] < NEAR_RARE)))
            e4 = w.E4T.view(w.Gp, 4 * w.Bp)[:G, :4 * B].view(G, B, 4).double().transpose(0, 1)
            dpit = w.DPIT.view(w.Gp, w.Bp)[:G, :B].double().t()
            for got_e, want_e, tag in ((e4[..., 0], ref["ep"], "elem_ep"), (e4[..., 2], ref["es"], "elem_ep"),
                                       (e4[..., 1], 4096 * ref["sm_p"], "elem_ep"), (e4[..., 3], 4096 * ref["sm_s"], "elem_ep"),
                                       (dpit, ref["dpi"], "elem_dpi")):
                up(tag, _per_gene_rel(torch.where(near, 0.0, got_e), torch.where(near, 0.0, want_e)))
                up("elem_near_rare", _per_gene_rel(torch.where(near, got_e, 0.0), torch.where(near, want_e, 0.0)))
        got = {k: v.double() for k, v in eng.grad_dict().items() if k in ref["grads"]}
        got["dzz"] = w.dzz[:, :KZ].double()
        # known weak spots, gated on their own (module docstring): d px_r of genes with theta = exp(px_r) > e^6.5 on the tensor-core
        # paths, and the hidden layer's weight gradient when the latents sit far from zero
        want = dict(ref["grads"])
        kp = f"px_r.{g}"
        if not precision_fp32:
            up("grad_px_r_large_theta", float((got[kp] - want[kp]).abs()[hi_theta].max() / want[kp].abs().max()))
            got[kp], want[kp] = torch.where(hi_theta, 0.0, got[kp]), torch.where(hi_theta, 0.0, want[kp])
        worst, wk = grad_errors(got, want)
        gk = "grad_offset" if case["offset"] else ("grad_unfused" if (not precision_fp32 and not fused) else "grad")
        up(gk, worst)
        if worst >= err[gk]:
            where[gk] = wk
        fl = "fc_layers.Layer 0"
        edge = [i for i in range(EDGE)] + ([LONE_GENE] if x.shape[1] > LONE_GENE + 64 else [])
        for k in (f"px_r.{g}", f"decoder_{g}.mixture.{fl}.0.bias", f"decoder_{g}.factor_regressor_private.{fl}.1.bias",
                  f"decoder_{g}.factor_regressor_shared.{fl}.1.bias"):
            up("grad_edge", _rel(got[k][edge], want[k][edge]))
    return err, where, refs


def _check(name, precision, training, expect_fused=None):
    case = build_case(name)
    eng, ws = _run_engine(case, precision, training)
    if expect_fused is not None:
        assert eng.fused_nb == expect_fused
    single = eng.fused_nb and training
    err, where, refs = _compare(eng, ws, case, training, eng.fused_nb, single)
    if training:
        assert_classes(case, refs)
    print(f"\n[f64] {name} {precision} {'train' if training else 'eval'} fused={eng.fused_nb}: "
          + " ".join(f"{k}={v:.2e}" for k, v in sorted(err.items())) + f" worst at {where}")
    gates = FP32_GATES if precision == "fp32" else TC_GATES
    bad = {k: v for k, v in err.items() if not v <= gates[k]}
    assert not bad, (bad, err)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["b300", "b300-f32", "b1000", "b1000-offset", "b2100", "b8300"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_training_step_against_f64(name, precision):
    """fp32 SIMT decoder and the default bf16 single-sweep decoder, one training step"""
    _check(name, precision, True, expect_fused=precision == "bf16" or None)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["b300", "b300-f32", "b1000"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_eval_forward_against_f64(name, precision):
    """eval forward: BatchNorm on the running statistics, per-cell reconstruction term"""
    _check(name, precision, False)


@pytest.mark.gpu
@pytest.mark.parametrize("name,fused", [("w58", True), ("w59", False), ("w64", False), ("w65", False), ("w96", False)])
def test_latent_width_against_f64(name, fused):
    """bf16 engines around the fused decoder's latent limit: fused up to 58 columns, the unfused bf16 decoder above"""
    _check(name, "bf16", True, expect_fused=fused)
