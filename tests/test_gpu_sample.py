"""Count draws from the decoder's NB mixture: the SIMT sampler against the exact mixture distribution, the tensor-core sampling
sweep against the SIMT sampler on the sweep's own rates (bitwise), the keying of the draws, px.sample and
spVIPES.posterior_predictive_sample.  Every seed is fixed, so the statistical gates are deterministic."""
import numpy as np
import pytest
import torch
from scipy import stats

from tests.test_gpu_decoded import _engine, _latent_model
from tests.test_gpu_decoder_f64 import build_case

pytestmark = pytest.mark.gpu

GC_THETA = 8


def _lib():
    from spvipes_b200 import _lib as L
    return L, L.load()


def _simt_sample(mu1, mu2, pi, theta, n_draws, seed, group=0, draw0=0):
    """spv_nb_mixture_sample on [B, G] parameters (unit gene stride, any row pitch) -> [n_draws, B, G]"""
    L, lib = _lib()
    B, G = mu1.shape
    out = torch.full((n_draws, B, G), float("nan"), device="cuda")
    L.check(lib.spv_nb_mixture_sample(mu1.data_ptr(), mu2.data_ptr(), pi.data_ptr(), mu1.stride(0), theta.data_ptr(), B, G, n_draws,
                                      out.data_ptr(), G, B * G, seed, group, draw0, torch.cuda.current_stream().cuda_stream),
            "spv_nb_mixture_sample")
    return out


# ------------------------------------------------------------------------------------------------------------------------
# 1. exact distribution of the SIMT sampler
# ------------------------------------------------------------------------------------------------------------------------
THETAS = np.exp([-6.0, -2.0, 0.0, 2.0, 8.0])
MUS = [0.0, 1e-4, 0.3, 3.0, 9.99, 10.0, 40.0, 2e3, 1e5]
PIS = [-30.0, -2.0, 0.0, 2.0, 30.0]
ROWS, DRAWS = 4096, 16            # 65 536 draws per column
BIN = 50                          # least expected count of a chi-square bin
# integer grid of bin edges: every count up to 2000, then geometric (steps of 0.06 %) up to the 1e8 clamp and beyond
GRID = np.unique(np.concatenate([np.arange(0, 2000), np.round(np.geomspace(2000, 4e8, 20000))]).astype(np.int64))


def _component_cdf(theta, mu):
    if mu == 0.0:
        return np.ones(GRID.size)
    return stats.nbinom.cdf(GRID, theta, theta / (theta + mu))


def _moments(theta, mu):
    """raw moments E X, E X^2, E X^3, E X^4 of NB(theta, mu) (0 for mu = 0)"""
    if mu == 0.0:
        return np.zeros(4)
    m, v, s, k = (float(x) for x in stats.nbinom.stats(theta, theta / (theta + mu), moments="mvsk"))
    c3, c4 = s * v ** 1.5, (k + 3.0) * v * v
    return np.array([m, v + m * m, c3 + 3 * m * v + m ** 3, c4 + 4 * m * c3 + 6 * m * m * v + m ** 4])


def test_simt_sampler_exact_distribution():
    cols = [(t, a, b, p) for t in THETAS for a in MUS for b in MUS for p in PIS]
    C = len(cols)
    th = torch.tensor([c[0] for c in cols], dtype=torch.float32, device="cuda")
    rows = lambda k: torch.tensor([c[k] for c in cols], dtype=torch.float32, device="cuda").expand(ROWS, C).contiguous()
    out = _simt_sample(rows(1), rows(2), rows(3), th, DRAWS, seed=20261022, group=1)
    x = out.permute(2, 0, 1).reshape(C, -1).cpu().numpy().astype(np.float64)  # [column, 65 536 draws]
    N = x.shape[1]
    assert np.isfinite(x).all() and (x >= 0).all() and (x == np.round(x)).all()
    cdf = {(t, m): _component_cdf(t, m) for t in THETAS for m in MUS}
    mom = {(t, m): _moments(t, m) for t in THETAS for m in MUS}
    pmin, worst_z, n_chi, n_mom = 1.0, 0.0, 0, 0
    for j, (t, a, b, p) in enumerate(cols):
        xs = x[j]
        if a == 0.0 and b == 0.0:
            assert (xs == 0).all(), (t, a, b, p)
            continue
        w = 1.0 / (1.0 + np.exp(-p))
        # lam = Gamma(theta, theta / mu) is clamped at 1e8: leave out the columns where that changes the distribution
        clamp = w * stats.gamma.sf(1e8, t, scale=a / t) if a else 0.0
        clamp += (1 - w) * stats.gamma.sf(1e8, t, scale=b / t) if b else 0.0
        F = w * cdf[(t, a)] + (1 - w) * cdf[(t, b)]
        # bins (u_{i-1}, u_i] with >= BIN expected draws each; the tail beyond the last edge merged into the last bin
        cum = N * F
        cut = np.unique(np.searchsorted(cum, np.arange(BIN, N * F[-1] - BIN, BIN)))
        edges = GRID[cut]
        if edges.size >= 2:
            exp_ = np.diff(np.concatenate([[0.0], cum[cut], [N]]))
            obs = np.bincount(np.searchsorted(edges, xs, side="left"), minlength=edges.size + 1).astype(np.float64)
            exp_[-2] += exp_[-1]
            obs[-2] += obs[-1]
            exp_, obs = exp_[:-1], obs[:-1]
            chi = float(((obs - exp_) ** 2 / exp_).sum())
            pv = float(stats.chi2.sf(chi, exp_.size - 1))
            pmin = min(pmin, pv)
            n_chi += 1
            assert pv * C >= 1e-3, (t, a, b, p, chi, exp_.size, pv)
        if clamp > 1e-7:
            continue
        r = w * mom[(t, a)] + (1 - w) * mom[(t, b)]
        mean, var = r[0], r[1] - r[0] ** 2
        mu4 = r[3] - 4 * mean * r[2] + 6 * mean * mean * r[1] - 3 * mean ** 4
        if var <= 0:
            continue
        z_m = (xs.mean() - mean) / np.sqrt(var / N)
        z_v = (xs.var(ddof=1) - var) / np.sqrt(max(mu4 - var * var, 0.0) / N + 1e-300)
        worst_z = max(worst_z, abs(z_m), abs(z_v))
        n_mom += 1
        assert abs(z_m) <= 5 and abs(z_v) <= 5, (t, a, b, p, z_m, z_v)
    print(f"\n[sample] {C} columns, {n_chi} chi-square (min p {pmin:.2e}), {n_mom} moment checks (worst z {worst_z:.2f})")


# ------------------------------------------------------------------------------------------------------------------------
# 2. fused sampling sweep == SIMT sampler on the sweep's own rates
# ------------------------------------------------------------------------------------------------------------------------
def _c2_engine():
    from spvipes_b200 import synth
    from spvipes_b200.engine import GroupBatch, StepEngine
    from spvipes_b200.trainer import init_params
    G, B = 5_000, 512
    eng = StepEngine((G, G), 128, 25, 10, 0.1, "label", "cuda", precision="bf16")
    init_params(eng, seed=0)
    data = synth.make_counts((4 * B, 4 * B), (G, G), 10, device="cuda", seed=1)
    batches = [GroupBatch(X=data.X[g], rows=torch.arange(7, 7 + B, dtype=torch.int32, device="cuda"), labels=data.labels[g][7:7 + B].contiguous())
               for g in (0, 1)]
    return eng, batches, None


def _pass(name, training, precision="bf16"):
    if name == "C2":
        eng, batches, noise = _c2_engine()
    else:
        eng, batches, noise = _engine(build_case(name), precision)
    ws = eng.forward(batches, training=training, noise=noise, with_grad=False)
    return eng, ws


def _elements(eng, ws):
    outs = [{k: torch.empty(ws[g].B, eng.d.genes[g], device="cuda") for k in ("rate_p", "rate_s", "pi")} for g in (0, 1)]
    eng.decode_elements(outs)
    return outs


@pytest.mark.parametrize("name", ["b300", "b300-f32", "b1000-offset", "b2100", "C2"])
@pytest.mark.parametrize("training", [True, False], ids=["train", "eval"])
def test_fused_sweep_equals_simt_sampler(name, training):
    eng, ws = _pass(name, training)
    assert eng.fused_nb
    el = _elements(eng, ws)
    pad = 5
    outs = [torch.full((3, ws[g].B, eng.d.genes[g] + pad), float("nan"), device="cuda")[:, :, :eng.d.genes[g]] for g in (0, 1)]
    eng.decode_sample(outs, seed=99, draw0=4)
    for g in (0, 1):
        want = _simt_sample(el[g]["rate_p"], el[g]["rate_s"], el[g]["pi"], ws[g].genec[GC_THETA, :eng.d.genes[g]].contiguous(), 3,
                            seed=99, group=g, draw0=4)
        assert torch.isfinite(outs[g]).all()
        assert torch.equal(outs[g], want), (g, int((outs[g] != want).sum()))
    assert float(outs[0].sum()) > 0


# ------------------------------------------------------------------------------------------------------------------------
# 3. keying
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_draw_keying(precision):
    eng, ws = _pass("b300", False, precision)
    Bs, Gs = [w.B for w in ws], eng.d.genes
    new = lambda n, g: torch.empty(n, Bs[g], Gs[g], device="cuda")
    a = [new(8, 0), new(8, 1)]
    eng.decode_sample(a, seed=5)
    b = [new(8, 0), new(8, 1)]
    eng.decode_sample(b, seed=5)
    assert all(torch.equal(a[g], b[g]) for g in (0, 1))
    other = [new(8, 0), new(8, 1)]
    eng.decode_sample(other, seed=6)
    for g in (0, 1):
        assert float((other[g] != a[g]).float().mean()) > 0.05
        assert float((a[g][0] != a[g][1]).float().mean()) > 0.05  # another draw index
    assert float((a[0][:, :, :Gs[1]] != a[1][:, :, :Gs[1]]).float().mean()) > 0.05  # another group
    alone = new(8, 1)
    eng.decode_sample([None, alone], seed=5)
    assert torch.equal(alone, a[1])
    part = [new(2, 0), None]
    eng.decode_sample(part, seed=5, draw0=3)
    assert torch.equal(part[0], a[0][3:5])
    with pytest.raises(ValueError):
        eng.decode_sample([torch.empty(2, Bs[0], Gs[0] - 1, device="cuda"), None], seed=5)
    with pytest.raises(ValueError):
        eng.decode_sample([torch.empty(2, Bs[0], Gs[0], device="cuda", dtype=torch.float64), None], seed=5)
    with pytest.raises(ValueError):
        eng.decode_sample([new(2, 0), None], seed=-1)
    with pytest.raises(ValueError):
        eng.decode_sample([new(2, 0), None], seed=5, draw0=2 ** 32 - 1)
    # a training pass that did not decode: running the decoder here would update its BatchNorm statistics a second time
    eng.forward(eng._ctx["batches"], training=True, with_grad=False, decode=False)
    with pytest.raises(RuntimeError, match="BatchNorm"):
        eng.decode_sample([new(1, 0), None], seed=5)


# ------------------------------------------------------------------------------------------------------------------------
# 4. px.sample
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,precision,fused", [("b300", "fp32", False), ("b300", "bf16", True), ("w65", "bf16", False)])
def test_px_sample(name, precision, fused):
    from spvipes_b200.module import _NBMixtureHandle
    eng, ws = _pass(name, False, precision)
    assert eng.fused_nb == fused
    tested = 0
    for g in (0, 1):
        px = _NBMixtureHandle(ws[g].rec, eng, g, ws[g])
        B, G = ws[g].B, eng.d.genes[g]
        one = px.sample()
        assert one.shape == (B, G) and one.dtype == torch.float32
        assert not torch.equal(px.sample(), px.sample())  # seed=None: a new seed per call
        assert torch.equal(px.sample(seed=3), px.sample(seed=3))
        k = 256
        s = px.sample((k,), seed=11)
        assert s.shape == (k, B, G)
        assert px.sample((2, 3), seed=1).shape == (2, 3, B, G)
        mu1, mu2, pi, th = px.mu1.double(), px.mu2.double(), px.mixture_logits.double(), px.theta1.double()
        w = torch.sigmoid(pi)
        m = w * mu1 + (1 - w) * mu2
        ex2 = w * (mu1 + mu1 ** 2 / th + mu1 ** 2) + (1 - w) * (mu2 + mu2 ** 2 / th + mu2 ** 2)
        var = ex2 - m * m
        # elements where the mean of 256 draws is close to normal: theta >= 1 and at least 30 expected counts over the draws
        ok = (th >= 1.0) & (k * m >= 30)
        z = (s.double().mean(0) - px.mean.double()) / torch.sqrt(var / k)
        tested += int(ok.sum())
        assert float(z[ok].abs().max()) <= 6.0, float(z[ok].abs().max())
    assert tested > 1000
    eng.forward(eng._ctx["batches"], training=False, with_grad=False)
    with pytest.raises(RuntimeError):
        px.sample()


# ------------------------------------------------------------------------------------------------------------------------
# 5. posterior_predictive_sample
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["latent_label_ragged", "latent_paired_cycling"])
def test_posterior_predictive_sample(name):
    model, adata, gil, bs, noise, _ = _latent_model(name, "bf16")
    n = [len(g) for g in gil]
    genes = model.module.engine.d.genes
    one = model.posterior_predictive_sample(gil, batch_size=bs, seed=4, _noise_fn=noise)
    three = model.posterior_predictive_sample(gil, n_samples=3, batch_size=bs, seed=4, _noise_fn=noise)
    dec = model.get_decoded_expression(gil, outputs=("px_rate_private", "px_rate_shared", "px_mixing"), batch_size=bs, _noise_fn=noise)
    for g in (0, 1):
        assert one[g].shape == (n[g], genes[g]) and one[g].dtype == np.float32
        assert three[g].shape == (n[g], genes[g], 3)
        assert np.array_equal(three[g][:, :, 0], one[g])  # the first sample pass is the n_samples = 1 pass
        # row order: each cell's total count against the decoded mixture of the same cell (same latents: same noise)
        th = np.exp(model.module.state_dict()[f"px_r.{g}"].double().cpu().numpy())
        m1, m2 = dec["px_rate_private"][g].astype(np.float64), dec["px_rate_shared"][g].astype(np.float64)
        w = 1.0 / (1.0 + np.exp(-dec["px_mixing"][g].astype(np.float64)))
        m = w * m1 + (1 - w) * m2
        var = w * (m1 + m1 ** 2 / th + m1 ** 2) + (1 - w) * (m2 + m2 ** 2 / th + m2 ** 2) - m * m
        z = (one[g].sum(1) - m.sum(1)) / np.sqrt(var.sum(1))
        assert np.abs(z).max() <= 6.0, np.abs(z).max()
        assert np.abs(np.corrcoef(one[g].sum(1), m.sum(1))[0, 1]) > 0.5 or m.sum(1).std() < 1e-3 * m.sum(1).mean()
    sub = [[3, 0, 5], None]
    part = model.posterior_predictive_sample(gil, n_samples=3, gene_indices=sub, batch_size=bs, seed=4, _noise_fn=noise)
    assert np.array_equal(part[0], three[0][:, sub[0]])
    assert np.array_equal(part[1], three[1])
    for bad in (dict(n_samples=0), dict(gene_indices=[[0]]), dict(gene_indices=[[genes[0]], None]), dict(seed=-1)):
        with pytest.raises(ValueError):
            model.posterior_predictive_sample(gil, batch_size=bs, _noise_fn=noise, **bad)


def test_posterior_predictive_sample_csr_equals_dense():
    """the setting of test_gpu_decoded.test_decoded_expression_csr_equals_dense, where the rates are bitwise equal"""
    from spvipes_b200 import synth
    from spvipes_b200.engine import Noise
    from spvipes_b200.model import GroupedData, prepare_adatas, spVIPES
    import pandas as pd
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
        outs[sparse] = model.posterior_predictive_sample(gil, n_samples=2, batch_size=128, seed=8, _noise_fn=noise)
    for g in (0, 1):
        assert outs[False][g].shape == (n[g], G[g], 2)
        assert np.array_equal(outs[False][g], outs[True][g])
