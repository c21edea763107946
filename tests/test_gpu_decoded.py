"""Per-element decoder outputs (StepEngine.decode_elements, px of the drop-in module, spVIPES.get_decoded_expression) against
float64: the element sweeps store what the likelihood sweeps reduce, on every decoder path.

The engine runs one forward on the crafted cases of tests/test_gpu_decoder_f64.py (rare-rate ladders across 1e-6, slow-path and
non-integer counts, px_r from -7 to 9, mixture biases of +-60, ragged tiles, odd pitches); the float64 reference is
oracle.restatement's decoder on the latents and library sizes read back from the engine's workspace.

Gates.  fp32 SIMT path: 1e-4 per gene (_per_gene_rel).  Tensor-core paths (fp16 operands, fast transcendentals): ELEM_GATES,
each at most 4x the worst error measured on a B200 over this file's cases (in brackets).
"""
import os

import numpy as np
import pandas as pd
import pytest
import torch

from oracle import restatement as rs
from tests.helpers import Golden
from tests.test_gpu_decoder_f64 import HD, H, _per_gene_rel, build_case, case_counts, reference

pytestmark = pytest.mark.gpu

NAMES = ("ll", "rate_p", "rate_s", "pi", "mean")
FP32_GATE = 1e-4
# tensor-core paths (fused bf16 decoder; unfused bf16 decoder: pi), per gene; measured worst on a B200 (1000 W) in brackets
ELEM_GATES = {"ll": 1e-2,       # 3.00e-3 (b300-f32 eval)
              "rate_p": 6.4e-3,  # 1.61e-3 (b300-f32 train)
              "rate_s": 6.9e-3,  # 1.73e-3 (b2100 train)
              "pi": 1e-2,       # 5.18e-3 (w65 train: the unfused decoder's bf16 mixture GEMM)
              "mean": 1e-2}     # 3.36e-3 (b1000-offset train)
# The fused decoder in EVAL mode on latents far from zero (b1000-offset: the encoder BatchNorm on its running statistics leaves
# latents of |z| ~ 30 and more): its fp16 operands [hm | zz] and zz (uncentred in eval mode, spv_dec_fold) round each latent to
# 2^-11 relative, and the mixing logit and the branch logits cancel over the latent columns.  The reducing sweep computes the
# same values (consistency below); test_fused_elements_equal_their_fp16_operands shows the kernel exact for those operands.
ELEM_GATES_OFFSET_EVAL = {"ll": 2.1e-2,    # 5.13e-3
                          "rate_p": 4.6e-5,  # 1.13e-5
                          "rate_s": 8.9e-2,  # 2.22e-2
                          "pi": 3.2e-1,      # 8.06e-2
                          "mean": 8.4e-2}    # 2.09e-2
# same-pass consistency; measured worst in brackets.  rec: the SIMT paths' reducing sweep sums the fp32 element form, the element
# pass evaluates ll in float64 (decoder.cu nb_ll_f64); the tensor-core sweeps share the element math.
CONSIST_GATES = {"rec_simt": 1e-4,  # 2.42e-5 (b2100 fp32 eval)
                 "rec_tc": 7.2e-7,  # 1.80e-7 (b2100 bf16 train)
                 "lib": 7.1e-5,     # 1.78e-5 (b1000-offset bf16 eval)
                 "mean": 6.7e-6}    # 1.68e-6 (b1000-offset bf16 eval)


def _engine(case, precision):
    from spvipes_b200.engine import GroupBatch, Noise, StepEngine
    eng = StepEngine(case["genes"], H, case["S"], case["P"], 0.1, "label", "cuda", precision=precision)
    eng.load_state_dict(case["sd"])
    if case["src"] == "f32":
        X = case["X"].to(torch.float32).cuda()
    else:
        X = case["X"].to(torch.int32).cuda().to(torch.uint16)
    batches = [GroupBatch(X=X, rows=case["rows"][g].to(torch.int32).cuda(), col0=case["col0"][g],
                          labels=torch.from_numpy(case["labels"][g].astype(np.int32)).cuda()) for g in (0, 1)]
    noise = Noise([e.cuda() for e in case["eps_p"]], [e.cuda() for e in case["eps_q"]], [d.cuda() for d in case["drop"]])
    return eng, batches, noise


def _alloc(eng, B, pad=0):
    """every output of both groups, [B, G + pad] (pad > 0: a row pitch that is not the gene count)"""
    return [{k: torch.full((B, G + pad), float("nan"), device="cuda")[:, :G] for k in NAMES} for G in eng.d.genes]


def _ref_elements(case, ws, g, training, sd):
    P, KZ = case["P"], case["P"] + case["S"]
    w = ws[g]
    zz = w.amix[:, HD:HD + KZ].double()
    x = case_counts(case, g).cuda()
    r = reference(sd, g, zz, w.lib.double(), x, P, training)
    theta = torch.exp(sd[f"px_r.{g}"].double())
    ll = rs.log_mixture_nb(torch.log1p(x.double()), r["rho_p"], r["rho_s"], theta, r["pi"])
    mean = torch.sigmoid(r["pi"]) * r["rho_p"] + torch.sigmoid(-r["pi"]) * r["rho_s"]
    return {"ll": ll, "rate_p": r["rho_p"], "rate_s": r["rho_s"], "pi": r["pi"], "mean": mean, "x": x}


def _elem_errors(case, precision, training):
    eng, batches, noise = _engine(case, precision)
    ws = eng.forward(batches, training=training, noise=noise, with_grad=False)
    outs = _alloc(eng, case["B"], pad=3)
    eng.decode_elements(outs)
    torch.cuda.synchronize()
    sd = {k: v.cuda() for k, v in case["sd"].items()}
    err = {k: 0.0 for k in NAMES}
    for g in (0, 1):
        ref = _ref_elements(case, ws, g, training, sd)
        for k in NAMES:
            got = outs[g][k]
            assert torch.isfinite(got).all(), (g, k)
            err[k] = max(err[k], _per_gene_rel(got, ref[k]))
    return eng, ws, outs, err


@pytest.mark.parametrize("name,precision,fused", [
    ("b300", "fp32", None), ("b300-f32", "fp32", None), ("b1000-offset", "fp32", None), ("b2100", "fp32", None),
    ("b300", "bf16", True), ("b300-f32", "bf16", True), ("b1000-offset", "bf16", True), ("b2100", "bf16", True),
    ("w65", "bf16", False)])
@pytest.mark.parametrize("training", [True, False], ids=["train", "eval"])
def test_elements_against_f64(name, precision, fused, training):
    """all five outputs on the fp32 SIMT, fused bf16 and unfused bf16 (P + S = 65) decoders, training and eval passes"""
    case = build_case(name)
    eng, ws, outs, err = _elem_errors(case, precision, training)
    if fused is not None:
        assert eng.fused_nb == fused
    print(f"\n[elem] {name} {precision} {'train' if training else 'eval'} fused={eng.fused_nb}: "
          + " ".join(f"{k}={v:.2e}" for k, v in err.items()))
    if precision == "fp32":
        gates = {k: FP32_GATE for k in NAMES}
    else:
        gates = ELEM_GATES_OFFSET_EVAL if (case["offset"] and eng.fused_nb and not training) else ELEM_GATES
    assert all(err[k] <= gates[k] for k in NAMES), err
    # same pass: -sum_g ll is the reducing sweep's reconstruction term, sum_g rate = exp(lib), mean from the returned fields
    rk = "rec_tc" if eng.fused_nb else "rec_simt"
    c = {rk: 0.0, "lib": 0.0, "mean": 0.0}
    for g in (0, 1):
        o, w = outs[g], ws[g]
        rec = -o["ll"].double().sum(1)
        c[rk] = max(c[rk], float(((rec - w.rec.double()).abs() / w.rec.double().abs()).max()))
        elib = torch.exp(w.lib.double())
        for k in ("rate_p", "rate_s"):
            c["lib"] = max(c["lib"], float(((o[k].double().sum(1) - elib).abs() / elib).max()))
        pi = o["pi"].double()
        m = torch.sigmoid(pi) * o["rate_p"].double() + torch.sigmoid(-pi) * o["rate_s"].double()
        c["mean"] = max(c["mean"], float(((o["mean"].double() - m).abs() / m.abs().clamp(min=1e-30)).max()))
    print(" consistency: " + " ".join(f"{k}={v:.2e}" for k, v in c.items()))
    assert all(c[k] <= CONSIST_GATES[k] for k in c), c


# the fused element sweep against the float64 product of its own fp16 operands (what the tensor cores multiply, fp32 accumulation):
# relative per gene, measured worst in brackets
OPERAND_GATES = {"pi": 2.5e-4,      # 6.31e-5 (b1000-offset eval)
                 "rate_p": 1.8e-5,  # 4.46e-6 (b1000-offset eval)
                 "rate_s": 3.8e-5}  # 9.59e-6 (b1000-offset eval)


@pytest.mark.parametrize("name", ["b300", "b1000-offset"])
@pytest.mark.parametrize("training", [True, False], ids=["train", "eval"])
def test_fused_elements_equal_their_fp16_operands(name, training):
    case = build_case(name)
    eng, batches, noise = _engine(case, "bf16")
    assert eng.fused_nb
    ws = eng.forward(batches, training=training, noise=noise, with_grad=False)
    outs = _alloc(eng, case["B"])
    eng.decode_elements(outs)
    torch.cuda.synchronize()
    d, err = eng.d, {k: 0.0 for k in OPERAND_GATES}
    for g, w in enumerate(ws):
        G = w.G
        pi = w.amixb[:, :d.KMIX].double() @ w.Wstack[:G, :d.KMIX].double().t() + eng.P(g, "bm").double()
        zc, wz = w.zcb.double(), w.wzf.double()
        want = {"pi": pi, "rate_p": torch.exp2(zc @ wz[:G].t()), "rate_s": torch.exp2(zc @ wz[w.Gp:w.Gp + G].t())}
        for k in OPERAND_GATES:
            err[k] = max(err[k], _per_gene_rel(outs[g][k], want[k]))
    print(f"\n[operands] {name} {'train' if training else 'eval'}: " + " ".join(f"{k}={v:.2e}" for k, v in err.items()))
    assert all(err[k] <= OPERAND_GATES[k] for k in err), err


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_target_mode(precision):
    """value given as it is: log1p(counts) reproduces the count path; zeros, non-integers and values above 20 match float64"""
    case = build_case("b300-f32")
    eng, batches, noise = _engine(case, precision)
    ws = eng.forward(batches, training=False, noise=noise, with_grad=False)
    B = case["B"]
    cnt = _alloc(eng, B)
    eng.decode_elements(cnt)
    vals, tgt = [], []
    gen = torch.Generator().manual_seed(7)
    for g, G in enumerate(eng.d.genes):
        x = case_counts(case, g)
        vals.append(torch.log1p(x).float().cuda())
        v = torch.rand(B, G, generator=gen, dtype=torch.float64) * 30.0
        v[torch.rand(B, G, generator=gen) < 0.3] = 0.0
        v[:, ::7] = torch.floor(v[:, ::7])
        tgt.append(v.float().cuda())
    o1 = [{"ll": torch.empty(B, G, device="cuda")} for G in eng.d.genes]
    eng.decode_elements(o1, vals)
    o2 = [{"ll": torch.empty(B, G, device="cuda")} for G in eng.d.genes]
    eng.decode_elements(o2, tgt)
    torch.cuda.synchronize()
    sd = {k: v.cuda() for k, v in case["sd"].items()}
    e1 = e2 = 0.0
    for g in (0, 1):
        e1 = max(e1, _per_gene_rel(o1[g]["ll"], cnt[g]["ll"]))
        ref = _ref_elements(case, ws, g, False, sd)
        theta = torch.exp(sd[f"px_r.{g}"].double())
        want = rs.log_mixture_nb(tgt[g].double(), ref["rate_p"], ref["rate_s"], theta, ref["pi"])
        e2 = max(e2, _per_gene_rel(o2[g]["ll"], want))
    print(f"\n[target] {precision}: log1p(x) vs counts {e1:.2e}, arbitrary values vs f64 {e2:.2e}")
    gate = FP32_GATE if precision == "fp32" else ELEM_GATES["ll"]
    assert e1 <= gate and e2 <= gate, (e1, e2)


def test_ragged_groups_and_state_rules():
    """B0 != B1 (no loss needed), the prologue runs once in eval mode, a training pass that did not decode refuses, and the state
    of a pass is gone after the next forward or a backward"""
    case = build_case("b300")
    eng, batches, noise = _engine(case, "bf16")
    from spvipes_b200.engine import GroupBatch, Noise
    b1 = [GroupBatch(X=b.X, rows=b.rows[:257 if g else 300].contiguous(), col0=b.col0, labels=b.labels[:257 if g else 300].contiguous())
          for g, b in enumerate(batches)]
    nz = Noise([noise.eps_private[0], noise.eps_private[1][:257].contiguous()], [noise.eps_poe[0], noise.eps_poe[1][:257].contiguous()], None)
    eng.forward(b1, training=False, noise=nz, with_grad=False, decode=False)
    outs = [{"mean": torch.empty(300, eng.d.genes[0], device="cuda")}, {"mean": torch.empty(257, eng.d.genes[1], device="cuda")}]
    eng.decode_elements(outs)
    again = [{"mean": torch.empty_like(outs[0]["mean"])}, {"mean": torch.empty_like(outs[1]["mean"])}]
    eng.decode_elements(again)
    torch.cuda.synchronize()
    assert all(torch.equal(outs[g]["mean"], again[g]["mean"]) for g in (0, 1))
    with pytest.raises(ValueError):
        eng.decode_elements([{"bogus": outs[0]["mean"]}, {}])
    eng.forward(batches, training=True, noise=noise, decode=False)
    with pytest.raises(RuntimeError, match="BatchNorm"):
        eng.decode_elements(outs)
    eng.forward(batches, training=True, noise=noise)
    eng.decode_elements([{"mean": torch.empty(300, eng.d.genes[0], device="cuda")}, {}])
    eng.backward()
    with pytest.raises(RuntimeError, match="backward or another forward"):
        eng.decode_elements([{"mean": torch.empty(300, eng.d.genes[0], device="cuda")}, {}])


# ------------------------------------------------------------------------------------------------------------------------
# module: px of generative_outputs
# ------------------------------------------------------------------------------------------------------------------------
def _module(gd):
    from tests.test_gpu_module import _module_from_golden
    return _module_from_golden(gd)


def _px_reference(m, gd, g):
    """float64 decoder of group g on the latents / library sizes in the module's last workspace (eval or training BatchNorm)"""
    w = m._last_ws[g]
    P, KZ = gd.P, gd.P + gd.S
    sd = {k: v.detach().cuda() for k, v in m.state_dict().items()}
    x = gd.x[g].double().cuda()
    r = reference(sd, g, w.amix[:, HD:HD + KZ].double(), w.lib.double(), x, P, m.training)
    theta = torch.exp(sd[f"px_r.{g}"].double())
    mean = torch.sigmoid(r["pi"]) * r["rho_p"] + torch.sigmoid(-r["pi"]) * r["rho_s"]
    return r, theta, mean, torch.log1p(x)


def _check_px(m, gd, gen):
    for g in (0, 1):
        px = gen["private_poe"][str(g)]["px"]
        r, theta, mean, xl = _px_reference(m, gd, g)
        want_ll = rs.log_mixture_nb(xl, r["rho_p"], r["rho_s"], theta, r["pi"])
        for got, want in ((px.mu1, r["rho_p"]), (px.mu2, r["rho_s"]), (px.mixture_logits, r["pi"]), (px.mean, mean),
                          (px.theta1, theta.expand_as(mean)), (px.log_prob(xl.float()), want_ll)):
            assert tuple(got.shape) == tuple(want.shape) and not got.requires_grad
            assert _per_gene_rel(got, want) <= FP32_GATE, _per_gene_rel(got, want)
        nll = -px.log_prob(xl.float()).double().sum(1)
        assert float(((nll - px.neg_log_prob_sum.double()).abs() / px.neg_log_prob_sum.double().abs()).max()) <= 1e-5


def test_module_eval_inference_then_generative():
    gd = Golden("label_tiny")
    m, batch = _module(gd)
    m.eval()
    inp = m._get_inference_input(batch)
    inf = m.inference(**inp)
    gen = m.generative(**m._get_generative_input(batch, inf))
    _check_px(m, gd, gen)


def test_module_training_plugin_call_fields_and_lifetime():
    """eager training plugin call: fields against float64 before backward; after loss.backward() an unread field raises, fields
    read before keep their values; the same after the next forward"""
    gd = Golden("label_tiny")
    m, batch = _module(gd)
    m.train()
    inf, gen, lo = m(batch, loss_kwargs={"kl_weight": gd.kl_weight})
    _check_px(m, gd, gen)
    lo.loss.backward()
    inf, gen, lo = m(batch, loss_kwargs={"kl_weight": gd.kl_weight})
    px = gen["private_poe"]["0"]["px"]
    mu1 = px.mu1.clone()  # the only member read before the backward
    lo.loss.backward()
    assert torch.equal(px.mu1, mu1)
    with pytest.raises(RuntimeError, match="next forward or backward"):
        px.mu2
    with pytest.raises(RuntimeError):
        px.log_prob(torch.zeros_like(mu1))
    inf, gen, lo = m(batch, loss_kwargs={"kl_weight": gd.kl_weight})
    px1 = gen["private_poe"]["1"]["px"]
    mean = px1.mean
    m(batch, loss_kwargs={"kl_weight": gd.kl_weight})
    with pytest.raises(RuntimeError):
        px1.mu1
    assert torch.equal(px1.mean, mean)


def test_module_captured_plugin_call_fields():
    """the captured (CUDA-graph) plugin call: px of a replayed step equals the eager step's, and expires with the replayed backward"""
    from spvipes_b200 import synth
    from spvipes_b200.module import spVIPESmodule
    B, G0, G1 = 128, 300, 260
    data = synth.make_counts((2 * B, 2 * B), (G0, G1), 5, device="cuda", seed=21)
    batch = []
    for g in (0, 1):
        X = torch.zeros(B, G0 + G1)
        X[:, (0 if g == 0 else G0):(G0 if g == 0 else G0 + G1)] = data.X[g][:B].cpu().to(torch.int32).float()
        batch.append({"X": X, "batch": torch.zeros(B, 1), "groups": torch.full((B, 1), float(g)),
                      "indices": torch.arange(B).float().reshape(-1, 1), "labels": data.labels[g][:B].cpu().float().reshape(-1, 1)})
    res = {}
    for captured in (False, True):
        torch.manual_seed(5)
        m = spVIPESmodule(groups_lengths={0: G0, 1: G1}, groups_obs_names=[None, None], groups_var_names={0: None, 1: None},
                          groups_obs_indices=[None, None], groups_var_indices=[np.arange(G0), np.arange(G0, G0 + G1)],
                          use_labels=True, n_labels=5, n_hidden=64, dropout_rate=0.0, precision="bf16")
        m.capture_steps = captured
        m.train()
        for s in range(4):  # eager warm-up, the two captures, one plain replay: every path of the captured step
            for p in m.parameters():
                p.grad = None
            inf, gen, lo = m(tuple(batch), loss_kwargs={"kl_weight": 1.0})
            px = gen["private_poe"]["1"]["px"]
            vals = {k: getattr(px, k).clone() for k in ("mu1", "mu2", "mixture_logits", "mean")}
            lo.loss.backward()
            with pytest.raises(RuntimeError):
                px.log_prob(vals["mu1"])
        res[captured] = vals
    for k in res[False]:
        assert torch.equal(res[False][k], res[True][k]), k


# ------------------------------------------------------------------------------------------------------------------------
# model: get_decoded_expression
# ------------------------------------------------------------------------------------------------------------------------
def _latent_model(name, precision, sparse=False):
    from spvipes_b200.engine import Noise
    from spvipes_b200.model import GroupedData, prepare_adatas, spVIPES
    import scipy.sparse as sp
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden_latent", name + ".npz"))
    mode = str(z["meta_mode"])
    n0, n1, G0, G1, Hh, S, P, nl, bs = (int(v) for v in z["meta_dims"])
    ads = {}
    for gi, key in enumerate(("a_first", "b_second")):
        obs = pd.DataFrame({"cell_type": [f"t{int(v)}" for v in z[f"labels{gi}"]]})
        if mode == "cluster":
            obs["processed_transport_labels"] = z[f"labels{gi}"]
        X = z[f"x{gi}"].astype(np.float32)
        ads[key] = GroupedData(X=sp.csr_matrix(X) if sparse else X, obs=obs, var_names=[f"g{j}" for j in range((G0, G1)[gi])])
    adata = prepare_adatas(ads)
    if mode != "label":
        adata.uns["transport_plan"] = z["plan"]
    spVIPES.setup_anndata(adata, groups_key="groups", label_key="cell_type" if mode == "label" else None,
                          transport_plan_key="transport_plan" if mode != "label" else None, match_clusters=mode == "cluster")
    model = spVIPES(adata, n_hidden=Hh, n_dimensions_shared=S, n_dimensions_private=P, dropout_rate=0.1, precision=precision)
    model.module.load_state_dict({k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd/")}, strict=True)

    def noise(k, B0, B1):  # the generator of oracle/make_golden_latent.batch_noise
        g = torch.Generator().manual_seed(1000 + k)
        ep = [torch.randn(B, P, generator=g) for B in (B0, B1)]
        eq = [torch.randn(B, S, generator=g) for B in (B0, B1)]
        return Noise([e.cuda() for e in ep], [e.cuda() for e in eq], None)

    gil = [list(ix) for ix in adata.uns["groups_obs_indices"]]
    return model, adata, gil, bs, noise, (S, P)


OUTS = ("mean", "px_rate_private", "px_rate_shared", "px_mixing", "log_prob")


@pytest.mark.parametrize("name", ["latent_label_ragged", "latent_paired_cycling"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_decoded_expression_against_f64(name, precision):
    """decoded outputs == the float64 eval-mode decoder applied to the latents get_latent_representation returns (same
    minibatches, cycling, truncation and injected noise); a gene subset is the same columns, bitwise"""
    model, adata, gil, bs, noise, (S, P) = _latent_model(name, precision)
    lat = model.get_latent_representation(gil, batch_size=bs, _noise_fn=noise)
    dec = model.get_decoded_expression(gil, outputs=OUTS, batch_size=bs, _noise_fn=noise)
    sd = {k: v.detach().cuda() for k, v in model.module.state_dict().items()}
    uns = adata.uns
    X = np.asarray(adata.X.todense() if hasattr(adata.X, "todense") else adata.X)
    worst = {}
    for g in (0, 1):
        x = torch.from_numpy(X[np.asarray(uns["groups_obs_indices"][g])][:, np.asarray(uns["groups_var_indices"][g])]).double().cuda()
        c = torch.cat((torch.from_numpy(lat["private"][g]), torch.from_numpy(lat["shared"][g])), 1).double().cuda()
        zz = torch.cat((c[:, S:S + P], c[:, :S]), 1)  # [z_private_arg | z_shared_arg], quirk Q1
        lib = torch.log(torch.log1p(x).sum(1))
        r = reference(sd, g, zz, lib, x, P, False)
        theta = torch.exp(sd[f"px_r.{g}"].double())
        want = {"px_rate_private": r["rho_p"], "px_rate_shared": r["rho_s"], "px_mixing": r["pi"],
                "mean": torch.sigmoid(r["pi"]) * r["rho_p"] + torch.sigmoid(-r["pi"]) * r["rho_s"],
                "log_prob": rs.log_mixture_nb(torch.log1p(x), r["rho_p"], r["rho_s"], theta, r["pi"])}
        for k in OUTS:
            got = dec[k][g]
            assert got.shape == tuple(want[k].shape) and got.dtype == np.float32, (k, got.shape)
            worst[k] = max(worst.get(k, 0.0), _per_gene_rel(torch.from_numpy(got), want[k].cpu()))
    print(f"\n[decoded] {name} {precision}: " + " ".join(f"{k}={v:.2e}" for k, v in worst.items()))
    gate = FP32_GATE if precision == "fp32" else max(ELEM_GATES.values())
    assert all(v <= gate for v in worst.values()), worst
    sub = [[3, 0, 5], None]
    part = model.get_decoded_expression(gil, outputs=("mean", "log_prob"), gene_indices=sub, batch_size=bs, _noise_fn=noise)
    for k in ("mean", "log_prob"):
        assert np.array_equal(part[k][0], dec[k][0][:, sub[0]])
        assert np.array_equal(part[k][1], dec[k][1])
    with pytest.raises(ValueError):
        model.get_decoded_expression(gil, outputs=("rate",))


def test_decoded_expression_csr_equals_dense():
    """bitwise, on gene counts whose dense rows are 16-byte aligned: the condition under which spv_csr_gather reproduces the dense
    conversion bit for bit, library size included (the library size reaches every rate)"""
    from spvipes_b200 import synth
    from spvipes_b200.engine import Noise
    from spvipes_b200.model import GroupedData, prepare_adatas, spVIPES
    import scipy.sparse as sp
    n, G, S, P = (300, 260), (64, 72), 12, 6
    data = synth.make_counts(n, G, n_labels=3, device="cuda", seed=17)

    def noise(k, B0, B1):
        g = torch.Generator().manual_seed(2000 + k)
        return Noise([torch.randn(B, P, generator=g).cuda() for B in (B0, B1)],
                     [torch.randn(B, S, generator=g).cuda() for B in (B0, B1)], None)

    outs = {}
    for sparse in (False, True):
        ads = {}
        for gi, key in enumerate(("mouse", "human")):
            obs = pd.DataFrame({"cell_type": [f"t{int(v)}" for v in data.labels[gi].cpu().numpy()]})
            X = data.X[gi].cpu().numpy().astype(np.float32)
            ads[key] = GroupedData(X=sp.csr_matrix(X) if sparse else X, obs=obs, var_names=[f"g{j}" for j in range(G[gi])])
        adata = prepare_adatas(ads)
        spVIPES.setup_anndata(adata, groups_key="groups", label_key="cell_type")
        torch.manual_seed(0)
        model = spVIPES(adata, n_hidden=64, n_dimensions_shared=S, n_dimensions_private=P, dropout_rate=0.1, precision="bf16")
        gil = [list(ix) for ix in adata.uns["groups_obs_indices"]]
        outs[sparse] = model.get_decoded_expression(gil, outputs=OUTS, batch_size=128, _noise_fn=noise)
    for k in OUTS:
        for g in (0, 1):
            assert np.array_equal(outs[False][k][g], outs[True][k][g]), k


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_decoded_expression_with_batch_covariate(precision):
    """a batch-covariate model (ragged last batch of group 0): sum_g rate = exp(library) per cell, finite log-probabilities"""
    from spvipes_b200 import synth
    from spvipes_b200.model import GroupedData, prepare_adatas, spVIPES
    n, G = (300, 260), (64, 72)
    data = synth.make_counts(n, G, n_labels=3, device="cuda", seed=15)
    ads = {}
    rng = np.random.RandomState(0)
    for gi, key in enumerate(("mouse", "human")):
        obs = pd.DataFrame({"cell_type": [f"t{int(v)}" for v in data.labels[gi].cpu().numpy()], "lab": rng.choice(["b0", "b1"], n[gi])})
        ads[key] = GroupedData(X=data.X[gi].cpu().numpy().astype(np.float32), obs=obs, var_names=[f"g{j}" for j in range(G[gi])])
    adata = prepare_adatas(ads)
    spVIPES.setup_anndata(adata, groups_key="groups", label_key="cell_type", batch_key="lab")
    model = spVIPES(adata, n_hidden=64, n_dimensions_shared=12, n_dimensions_private=6, dropout_rate=0.1, precision=precision)
    gil = [list(ix) for ix in adata.uns["groups_obs_indices"]]
    dec = model.get_decoded_expression(gil, outputs=("log_prob", "px_rate_private", "px_rate_shared"), batch_size=n[1])
    x1 = torch.from_numpy(np.asarray(adata.X)[np.asarray(gil[1])][:, np.asarray(adata.uns["groups_var_indices"][1])]).double()
    lib1 = torch.log(torch.log1p(x1).sum(1))
    for k in ("px_rate_private", "px_rate_shared"):
        s = dec[k][1].astype(np.float64).sum(1)
        assert np.abs(s / np.exp(lib1.numpy()) - 1).max() < (1e-5 if precision == "fp32" else 1e-3)
    assert np.isfinite(dec["log_prob"][0]).all() and np.isfinite(dec["log_prob"][1]).all()
