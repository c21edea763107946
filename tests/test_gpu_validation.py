"""Validation during spVIPES.train, early stopping and get_elbo on the GPU.

The validation metrics are checked against the CPU oracle (oracle.restatement.step in eval mode, float64) recomputed minibatch by
minibatch on the trained model's state_dict, with the same injected noise.  rs.step sums the two groups' per-cell terms into the
reference's loss, which is not defined for B_0 != B_1 (a ragged final minibatch); the per-cell terms are therefore captured where
rs.step computes them (log_mixture_nb, kl_std_normal), and rs.step is handed shape-[1] stand-ins so that it completes."""
import itertools
from unittest import mock

import numpy as np
import pandas as pd
import pytest
import torch

from oracle import restatement as rs

pytestmark = pytest.mark.gpu

GATES = {"fp32": 1e-4, "bf16": 1e-2}
N_CELLS, GENES, S, P, BS = (350, 300), (64, 72), 12, 6, 32  # validation splits of 70 / 60 cells: ragged, unequal
KEYS = ("elbo_validation", "reconstruction_loss_validation", "kl_local_validation", "validation_loss")


def _model(mode="label", precision="bf16", n_batch=0, sparse=False, seed=17):
    import scipy.sparse as sp
    from spvipes_b200 import synth
    from spvipes_b200.model import GroupedData, prepare_adatas, spVIPES
    data = synth.make_counts(N_CELLS, GENES, n_labels=3, device="cuda", seed=seed)
    rng = np.random.RandomState(3)
    ads = {}
    for gi, key in enumerate(("mouse", "human")):
        obs = pd.DataFrame({"cell_type": [f"t{int(v)}" for v in data.labels[gi].cpu().numpy()]})
        if n_batch:
            obs["lab"] = rng.choice([f"b{k}" for k in range(n_batch)], N_CELLS[gi])
        X = data.X[gi].cpu().numpy().astype(np.float32)
        ads[key] = GroupedData(X=sp.csr_matrix(X) if sparse else X, obs=obs, var_names=[f"g{j}" for j in range(GENES[gi])])
    adata = prepare_adatas(ads)
    if mode == "paired":
        adata.uns["transport_plan"] = synth.make_plan(N_CELLS[0], N_CELLS[1], data.labels[0], data.labels[1], 3).cpu().numpy()
        spVIPES.setup_anndata(adata, groups_key="groups", transport_plan_key="transport_plan")
    else:
        spVIPES.setup_anndata(adata, groups_key="groups", label_key="cell_type", batch_key="lab" if n_batch else None)
    torch.manual_seed(0)
    model = spVIPES(adata, n_hidden=64, n_dimensions_shared=S, n_dimensions_private=P, dropout_rate=0.1, precision=precision)
    assert model.module.engine.mode == mode
    gil = [list(ix) for ix in adata.uns["groups_obs_indices"]]
    return model, adata, gil


def _noise(k, B0, B1):
    from spvipes_b200.engine import Noise
    g = torch.Generator().manual_seed(5000 + k)
    ep = [torch.randn(B, P, generator=g) for B in (B0, B1)]
    eq = [torch.randn(B, S, generator=g) for B in (B0, B1)]
    return Noise([e.cuda() for e in ep], [e.cuda() for e in eq], None)


def _minibatches(idx, bs, cycling):
    """the minibatches of get_latent_representation: sequential chunks, zip(largest, cycle(other)); the paired mode's cycling path"""
    def process(lists):
        chunks = [[np.asarray(l)[k:k + bs] for k in range(0, len(l), bs)] for l in lists]
        largest = int(np.argmax([len(c) for c in chunks]))
        return list(zip(*[iter(c) if g == largest else itertools.cycle(c) for g, c in enumerate(chunks)]))
    if not cycling:
        return process(idx)
    n = [len(v) for v in idx]
    out = []
    for start in range(0, max(n), min(n)):
        out += process([[idx[g][(start + i) % n[g]] for i in range(min(n))] for g in (0, 1)])
    return out


def _oracle_terms(sd, x, **kw):
    """per-cell (rec, klp, klq) of both groups from rs.step(training=False), for any two minibatch sizes"""
    cap = {"ll": [], "kl": []}
    lmnb, kl = rs.log_mixture_nb, rs.kl_std_normal

    def lmnb_cap(*a, **k):
        v = lmnb(*a, **k)
        cap["ll"].append(v)
        return torch.zeros(1, v.shape[1], dtype=v.dtype)

    def kl_cap(loc, scale):
        v = kl(loc, scale)
        cap["kl"].append(v)
        return torch.zeros(1, dtype=v.dtype)

    with mock.patch.object(rs, "log_mixture_nb", lmnb_cap), mock.patch.object(rs, "kl_std_normal", kl_cap):
        rs.step(sd, x, training=False, **kw)
    return [(-cap["ll"][g].sum(-1), cap["kl"][2 * g], cap["kl"][2 * g + 1]) for g in (0, 1)]


def _oracle_metrics(model, adata, mode, n_batch, kl_weight):
    sd = {k: v.detach().double().cpu() for k, v in model.module.state_dict().items()}
    uns = adata.uns
    X = np.asarray(adata.X.todense() if hasattr(adata.X, "todense") else adata.X, dtype=np.float64)
    cell_type = pd.Categorical(adata.obs["cell_type"]).codes
    within = np.asarray(adata.obs["indices"])
    bcodes = pd.Categorical(adata.obs["lab"]).codes if n_batch else None
    plan = torch.from_numpy(np.asarray(uns["transport_plan"], dtype=np.float64)) if mode == "paired" else None
    rec = kl_sum = n_obs = 0.0
    for k, st in enumerate(_minibatches(model.val_idx, BS, mode == "paired")):
        x = [torch.from_numpy(X[np.asarray(st[g])][:, np.asarray(uns["groups_var_indices"][g])]) for g in (0, 1)]
        nz = _noise(k, len(st[0]), len(st[1]))
        kw = dict(mode=mode, n_shared=S, n_private=P, eps_private=[e.double().cpu() for e in nz.eps_private],
                  eps_poe=[e.double().cpu() for e in nz.eps_poe])
        if mode == "paired":
            kw["sub"] = rs.sub_plan(plan, within[np.asarray(st[0])], within[np.asarray(st[1])])
        else:
            kw["labels"] = [cell_type[np.asarray(st[g])] for g in (0, 1)]
        if n_batch:
            kw["batch_index"] = [torch.from_numpy(bcodes[np.asarray(st[g])].astype(np.int64)) for g in (0, 1)]
            kw["n_batch"] = n_batch
        terms = _oracle_terms(sd, x, **kw)
        rec += sum(float(t[0].sum()) for t in terms)
        kl_sum += sum(float(t[1].sum() + t[2].sum()) for t in terms)
        n_obs += len(st[0])
    return {"reconstruction_loss_validation": rec / n_obs, "kl_local_validation": kl_sum / n_obs,
            "elbo_validation": (rec + kl_sum) / n_obs, "validation_loss": (rec + kl_weight * kl_sum) / n_obs}


@pytest.mark.parametrize("mode,n_batch", [("label", 0), ("paired", 0), ("label", 3)], ids=["label", "paired", "label-nbatch3"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_validation_metrics_against_oracle(mode, n_batch, precision):
    model, adata, gil = _model(mode, precision, n_batch)
    model.train(gil, max_epochs=2, batch_size=BS, train_size=0.8, check_val_every_n_epoch=1, n_epochs_kl_warmup=4, _noise_fn=_noise)
    assert [len(v) for v in model.val_idx] == [70, 60]
    h = model.history
    for k in KEYS + ("elbo_train", "reconstruction_loss_train", "kl_local_train", "train_loss_epoch"):
        assert len(h[k]) == 2 and all(np.isfinite(h[k])), k
    assert model.early_stopped_epoch_ is None and model.is_trained_
    want = _oracle_metrics(model, adata, mode, n_batch, kl_weight=1 / 4)  # weight of the last epoch (index 1)
    err = {k: abs(h[k][-1] - want[k]) / abs(want[k]) for k in KEYS}
    print(f"\n[validation] {mode} n_batch={n_batch} {precision}: " + " ".join(f"{k}={v:.2e}" for k, v in err.items()))
    assert all(v <= GATES[precision] for v in err.values()), (err, want, {k: h[k][-1] for k in KEYS})
    # the ELBO of get_elbo on the validation split is the last validation run's, for injected and for in-kernel noise
    assert model.get_elbo(model.val_idx, batch_size=BS, _noise_fn=_noise) == -h["elbo_validation"][-1]


def test_get_elbo_philox_noise_matches_last_validation():
    model, adata, gil = _model("label", "bf16")
    model.train(gil, max_epochs=2, batch_size=BS, train_size=0.8, check_val_every_n_epoch=2)
    assert len(model.history["elbo_validation"]) == 1
    elbo = model.get_elbo(model.val_idx, batch_size=BS)
    assert elbo == -model.history["elbo_validation"][-1]
    assert model.get_elbo(model.val_idx, batch_size=BS) == elbo  # the evaluation noise stream restarts on every call
    with pytest.raises(ValueError):
        model.get_elbo([[], gil[1]], batch_size=BS)


@pytest.mark.parametrize("mode,precision", [("label", "fp32"), ("label", "bf16"), ("paired", "bf16")])
def test_training_is_independent_of_validation(mode, precision):
    """the captured (label) and eager (paired) training steps: parameters, buffers and train_loss_epoch bitwise equal with and
    without a validation run after every epoch"""
    res = {}
    for every in (None, 1):
        model, adata, gil = _model(mode, precision)
        torch.manual_seed(1)
        model.train(gil, max_epochs=3, batch_size=BS, train_size=0.8, check_val_every_n_epoch=every)
        res[every] = ({k: v.detach().clone() for k, v in model.module.state_dict().items()}, list(model.history["train_loss_epoch"]),
                      model.history)
    assert "elbo_validation" not in res[None][2] and len(res[1][2]["elbo_validation"]) == 3
    assert res[None][1] == res[1][1]
    for k, v in res[None][0].items():
        assert torch.equal(v, res[1][0][k]), k


def test_early_stopping_fires_where_the_rule_says():
    model, adata, gil = _model("label", "bf16")
    model.train(gil, max_epochs=10, batch_size=BS, train_size=0.8, early_stopping=True, early_stopping_patience=2,
                early_stopping_min_delta=1e9)
    assert model.is_trained_ and model.early_stopped_epoch_ == 2
    assert len(model.history["train_loss_epoch"]) == 3 and len(model.history["elbo_validation"]) == 3
    with pytest.raises(ValueError, match="validation split"):
        model.train(gil, max_epochs=1, batch_size=BS, train_size=1.0, early_stopping=True)


def test_csr_validation_history_equals_dense():
    hist = {}
    for sparse in (False, True):
        model, adata, gil = _model("label", "bf16", sparse=sparse)
        torch.manual_seed(1)
        model.train(gil, max_epochs=2, batch_size=BS, train_size=0.8, check_val_every_n_epoch=1)
        hist[sparse] = model.history
    for k in KEYS:
        assert hist[False][k] == hist[True][k], k


def test_ragged_eval_pass_without_loss():
    from spvipes_b200 import synth
    from spvipes_b200.engine import GroupBatch, StepEngine
    data = synth.make_counts((300, 260), GENES, n_labels=3, device="cuda", seed=4)
    eng = StepEngine(GENES, 64, S, P, 0.1, "label", "cuda", precision="bf16")
    Bs = (100, 77)
    batches = [GroupBatch(X=data.X[g], rows=torch.arange(Bs[g], dtype=torch.int32, device="cuda"), labels=data.labels[g],
                          labels_per_cell=True) for g in (0, 1)]
    before = eng.loss_out.clone()
    ws = eng.forward(batches, training=False, with_grad=False, loss=False)
    acc = torch.zeros(8, dtype=torch.float64, device="cuda")
    eng.set_kl_weight(0.5)
    eng.accumulate_elbo(ws, acc)
    eng.accumulate_elbo(ws, acc)
    torch.cuda.synchronize()
    assert torch.equal(eng.loss_out, before)
    sums = [ws[0].rec, ws[1].rec, ws[0].klp, ws[0].klq, ws[1].klp, ws[1].klq]
    assert all(bool(torch.isfinite(t).all()) for t in sums)
    want = torch.tensor([float(t.double().sum()) for t in sums], dtype=torch.float64)
    got = acc.cpu()
    assert torch.allclose(got[:6], 2 * want, rtol=1e-5)
    assert float(got[6]) == 2 * Bs[0]
    assert abs(float(got[7]) - 2 * float(want[:2].sum() + 0.5 * want[2:].sum())) <= 1e-5 * abs(float(got[7]))
    with pytest.raises(ValueError, match="equally sized"):
        eng.forward(batches, training=False, with_grad=False)
    with pytest.raises(ValueError):
        eng.accumulate_elbo(ws, torch.zeros(8, dtype=torch.float32, device="cuda"))
