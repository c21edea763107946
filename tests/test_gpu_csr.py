"""-m gpu: a minibatch gathered from a device-resident CSR count matrix gives BITWISE the same results as the same minibatch
gathered from a dense matrix holding the same counts.  The dense reference keeps a 16-byte aligned row pitch (a [N, Gp]
buffer viewed as [:, :G]), so that its count consumers take the same vectorised path as the staging tile.
  * kernel: spv_csr_gather against spv_counts_to_bf16 + the gathered dense rows (xs, T, T_lo, library size);
  * engine: a training step (forward, backward, Adam) and an eval forward in every mode / precision / path switch;
  * graph: four replays of a captured CSR step equal four replays of the dense one;
  * model: spVIPES on scipy-sparse data trains and extracts latents exactly as on the same data dense."""
import numpy as np
import pandas as pd
import pytest
import scipy.sparse as sp
import torch

pytestmark = pytest.mark.gpu

r8 = lambda x: (x + 7) // 8 * 8


def _bits(t):
    return t.view(torch.int16) if t.element_size() == 2 else t.view(torch.int32)


def _same(a, b):
    return a.shape == b.shape and torch.equal(_bits(a), _bits(b))


def _matrix(N, G, kind, seed):
    """[N, G] counts with an empty row (0), a fully dense row (1), counts >= 256 (the slow log1p) and, for "f32", non-integers"""
    rng = np.random.default_rng(seed)
    X = rng.poisson(0.4, (N, G)) * (rng.random((N, G)) < 0.3)
    X[1] = rng.integers(1, 9, G)
    big = rng.random((N, G)) < 0.01
    X[big] = rng.integers(256, 65536, int(big.sum()))
    X[0] = 0
    X = X.astype(np.float32)
    if kind == "f32":
        X[2:] += np.where(X[2:] > 0, rng.random((N - 2, G)).astype(np.float32) * 0.75, 0)
        X[3, : min(G, 4)] = 0.25
    return X


def _dense_aligned(X, dtype):
    N, G = X.shape
    buf = torch.zeros(N, r8(G), dtype=dtype, device="cuda")
    src = torch.from_numpy(X.astype(np.int32) if dtype == torch.uint16 else X).cuda()
    buf[:, :G] = src.to(dtype)
    return buf


KERNEL_CASES = [  # (kind, B, G, n_cov)
    ("u16", 1, 7, 0), ("u16", 300, 5000, 3), ("u16", 2048, 20000, 0), ("u16", 300, 65536, 2), ("u16", 2048, 7, 2),
    ("f32", 300, 7, 0), ("f32", 2048, 5000, 2), ("f32", 1, 20000, 0), ("f32", 300, None, 0), ("f32", 2, None, 3),
]


@pytest.mark.parametrize("kind,B,G,n_cov", KERNEL_CASES)
def test_gather_kernel_matches_dense_conversion(kind, B, G, n_cov):
    from spvipes_b200 import _lib as L
    from spvipes_b200.engine import CsrCounts
    lib = L.load()
    src = L.SRC_U16_LOG1P if kind == "u16" else L.SRC_F32_LOG1P
    G = G or int(lib.spv_csr_max_genes(src))  # None: the largest float32 row
    N = 37
    X = _matrix(N, G, kind, seed=G + B)
    csr = CsrCounts.from_scipy(sp.csr_matrix(X), "cuda")
    dt = torch.uint16 if kind == "u16" else torch.float32
    assert csr.values.dtype == dt
    Xd = _dense_aligned(X, dt)
    gen = torch.Generator(device="cuda").manual_seed(B)
    rows = torch.randint(0, N, (B,), generator=gen, device="cuda", dtype=torch.int32)  # repeated and scattered
    rows[:min(B, 2)] = torch.tensor([0, 1][:min(B, 2)], dtype=torch.int32, device="cuda")  # the empty and the dense row
    cov = torch.randint(0, max(n_cov, 1), (B,), generator=gen, device="cuda", dtype=torch.int32) if n_cov else None
    Gp, Gpe = r8(G), r8(G + n_cov)
    bf = lambda: torch.full((B, Gpe), 7.0, dtype=torch.bfloat16, device="cuda")
    T, Tl, lib_ref = bf(), bf(), torch.zeros(B, device="cuda")
    L.check(lib.spv_counts_to_bf16(src, L.ptr(Xd), Gp, L.ptr(rows), L.ptr(T), L.ptr(Tl), Gpe, B, G, L.ptr(lib_ref), L.ptr(cov),
                                   n_cov, None), "spv_counts_to_bf16")
    T2, Tl2, lib2 = bf(), bf(), torch.zeros(B, device="cuda")
    xs = torch.full((B, Gp), 3, dtype=dt, device="cuda") if dt == torch.float32 else \
        torch.full((B, Gp), 3, dtype=torch.int16, device="cuda").view(torch.uint16)
    L.check(lib.spv_csr_gather(src, L.ptr(csr.indptr), L.ptr(csr.indices), L.ptr(csr.values), L.ptr(rows), B, G, L.ptr(xs), Gp,
                               L.ptr(T2), L.ptr(Tl2), Gpe, L.ptr(lib2), L.ptr(cov), n_cov, None), "spv_csr_gather")
    xs_only = torch.zeros_like(xs)
    L.check(lib.spv_csr_gather(src, L.ptr(csr.indptr), L.ptr(csr.indices), L.ptr(csr.values), L.ptr(rows), B, G, L.ptr(xs_only),
                               Gp, None, None, 0, None, None, 0, None), "spv_csr_gather")
    torch.cuda.synchronize()
    ref_rows = Xd.view(torch.int16 if dt == torch.uint16 else torch.int32)[rows.long()]
    assert torch.equal(_bits(xs), ref_rows) and torch.equal(_bits(xs_only), ref_rows)
    assert _same(T2, T) and _same(Tl2, Tl) and _same(lib2, lib_ref)
    assert torch.isinf(lib2[rows == 0]).all()  # the empty row: log(0)


# ------------------------------------------------------------------------------------------------ engine level
N0, N1, GE, BE, H, S, P, NL = 600, 520, (1000, 517), 256, 128, 25, 10, 5


def _engine_data(counts="u16", seed=4):
    from spvipes_b200 import synth
    data = synth.make_counts((N0, N1), GE, NL, device="cuda", seed=seed)
    dense, csr = [], []
    from spvipes_b200.engine import CsrCounts
    for g in (0, 1):
        X = data.X[g].cpu().numpy().astype(np.float32)
        if counts == "f32":
            X = X * 0.5
        dt = torch.uint16 if counts == "u16" else torch.float32
        dense.append(_dense_aligned(X, dt)[:, :GE[g]])
        csr.append(CsrCounts.from_scipy(sp.csr_matrix(X), "cuda"))
        assert csr[g].values.dtype == dt
    return data, dense, csr


def _engine(mode, precision, n_batch=0, plan=None):
    from spvipes_b200.engine import StepEngine
    from spvipes_b200.trainer import init_params
    eng = StepEngine(GE, H, S, P, 0.1, mode, "cuda", seed=21, plan=plan, precision=precision, n_batch=n_batch)
    init_params(eng, 5)
    return eng


def _batches(X, data, rows, mode, bcodes):
    from spvipes_b200.engine import GroupBatch
    out = []
    for g in (0, 1):
        r = rows[g].long()
        lab = data.labels[g][r].contiguous() if mode != "paired" else None
        out.append(GroupBatch(X=X[g], rows=rows[g], labels=lab, idx=rows[g], batch=bcodes[g] if bcodes else None))
    return out


def _noise(seed=8):
    from spvipes_b200.engine import Noise
    gen = torch.Generator().manual_seed(seed)
    return Noise([torch.randn(BE, P, generator=gen).cuda() for _ in (0, 1)], [torch.randn(BE, S, generator=gen).cuda() for _ in (0, 1)],
                 [((torch.rand(BE, 2 * H, generator=gen) < 0.9).float() / 0.9).cuda() for _ in (0, 1)])


ENGINE_CASES = [  # (id, mode, precision, env, n_batch, counts, training)
    ("label-bf16", "label", "bf16", {}, 0, "u16", True),
    ("label-fp32", "label", "fp32", {}, 0, "u16", True),
    ("paired-bf16", "paired", "bf16", {}, 0, "u16", True),
    ("cluster-bf16", "cluster", "bf16", {}, 0, "u16", True),
    ("paired-fp32", "paired", "fp32", {}, 0, "u16", True),
    ("label-bf16-covariates", "label", "bf16", {}, 3, "u16", True),
    ("label-fp32-covariates", "label", "fp32", {}, 3, "u16", True),
    ("label-bf16-two-sweeps", "label", "bf16", {"SPV_NB_SWEEPS": "2"}, 0, "u16", True),
    ("label-bf16-fused-fc1", "label", "bf16", {"SPV_FUSED_FC1": "1"}, 0, "u16", True),
    ("label-bf16-float-counts", "label", "bf16", {}, 0, "f32", True),
    ("label-fp32-float-counts", "label", "fp32", {}, 0, "f32", True),
    ("label-bf16-eval", "label", "bf16", {}, 0, "u16", False),
    ("label-fp32-eval", "label", "fp32", {}, 0, "u16", False),
]


@pytest.mark.parametrize("case", ENGINE_CASES, ids=[c[0] for c in ENGINE_CASES])
def test_engine_step_csr_equals_dense(case, monkeypatch):
    from spvipes_b200 import synth
    from spvipes_b200.trainer import TrainLoop
    _, mode, precision, env, n_batch, counts, training = case
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    data, dense, csr = _engine_data(counts)
    gen = torch.Generator(device="cuda").manual_seed(77)
    rows = [torch.randint(0, n, (BE,), generator=gen, device="cuda", dtype=torch.int32) for n in (N0, N1)]
    bcodes = [torch.randint(0, n_batch, (BE,), generator=gen, device="cuda", dtype=torch.int32) for _ in (0, 1)] if n_batch else None
    plan = synth.make_plan(N0, N1, data.labels[0], data.labels[1], NL, device="cuda") if mode != "label" else None
    res = []
    for X in (dense, csr):
        eng = _engine(mode, precision, n_batch, plan)
        noise = _noise()
        if training:
            loop = TrainLoop(eng)
            loop.set_epoch(3)
            for _ in range(2):
                loop.step(_batches(X, data, rows, mode, bcodes), noise)
        else:
            ws = eng.forward(_batches(X, data, rows, mode, bcodes), training=False, noise=noise, with_grad=False)
        torch.cuda.synchronize()
        out = [eng.loss_out.clone(), eng.grads.clone(), eng.params.flat.clone(), eng.buffers.flat.clone()]
        if not training:
            out += [w.zpoe.clone() for w in ws] + [w.rec.clone() for w in ws] + [w.lib.clone() for w in ws]
        res.append(out)
    for a, b in zip(*res):
        assert torch.equal(a, b)


def test_graph_replay_csr_equals_dense():
    from spvipes_b200.engine import GroupBatch
    from spvipes_b200.trainer import TrainLoop
    data, dense, csr = _engine_data()
    res = []
    for X in (dense, csr):
        eng = _engine("label", "bf16")
        loop = TrainLoop(eng)
        loop.set_epoch(10)
        rows_cur = [torch.zeros(BE, dtype=torch.int32, device="cuda") for _ in (0, 1)]
        static = [GroupBatch(X=X[g], rows=rows_cur[g], labels=data.labels[g], labels_per_cell=True) for g in (0, 1)]
        gen = torch.Generator(device="cuda").manual_seed(100)
        step_rows = [[torch.randperm(n, generator=gen, device="cuda")[:BE].to(torch.int32) for n in (N0, N1)] for _ in range(5)]
        for g in (0, 1):
            rows_cur[g].copy_(step_rows[0][g])
        graph = loop.capture(static)
        for s in range(1, 5):
            for g in (0, 1):
                rows_cur[g].copy_(step_rows[s][g])
            graph.replay()
        torch.cuda.synchronize()
        res.append((eng.loss_out.clone(), eng.params.flat.clone(), eng.adam_m.clone(), eng.buffers.flat.clone(), int(eng.step_dev)))
    for a, b in zip(*res):
        assert torch.equal(a, b) if torch.is_tensor(a) else a == b


# ------------------------------------------------------------------------------------------------ model level
def _adata(sparse, mode, n=(450, 330), G=(96, 64), seed=12):
    from spvipes_b200 import synth
    from spvipes_b200.model import GroupedData, prepare_adatas
    data = synth.make_counts(n, G, n_labels=4, device="cpu", seed=seed)
    ads = {}
    for gi, key in enumerate(("mouse", "human")):
        X = data.X[gi].numpy().astype(np.float32)
        obs = pd.DataFrame({"cell_type": [f"t{int(v)}" for v in data.labels[gi].numpy()]})
        ads[key] = GroupedData(X=sp.csr_matrix(X) if sparse else X, obs=obs, var_names=[f"g{j}" for j in range(G[gi])])
    adata = prepare_adatas(ads)
    assert sp.issparse(adata.X) == sparse
    if mode == "paired":
        adata.uns["transport_plan"] = synth.make_plan(n[0], n[1], data.labels[0], data.labels[1], 4, device="cpu").numpy()
    return adata


@pytest.mark.parametrize("mode,precision", [("label", "bf16"), ("paired", "fp32"), ("paired", "bf16")])
def test_model_sparse_equals_dense(mode, precision):
    from spvipes_b200.engine import CsrCounts
    from spvipes_b200.model import spVIPES
    out, init = [], None
    for sparse in (False, True):
        adata = _adata(sparse, mode)
        spVIPES.setup_anndata(adata, groups_key="groups", label_key="cell_type" if mode == "label" else None,
                              transport_plan_key="transport_plan" if mode == "paired" else None)
        torch.manual_seed(0)
        model = spVIPES(adata, n_hidden=64, n_dimensions_shared=12, n_dimensions_private=6, dropout_rate=0.1, precision=precision)
        if init is None:
            init = {k: v.detach().clone() for k, v in model.module.state_dict().items()}
        else:
            model.module.load_state_dict(init, strict=True)
        gil = [list(ix) for ix in adata.uns["groups_obs_indices"]]
        torch.manual_seed(1)
        model.train(gil, max_epochs=2, batch_size=128, n_epochs_kl_warmup=None)
        assert isinstance(model._device_data[0]["X"], CsrCounts) == sparse
        # batch 100 leaves ragged last batches (450 = 4 x 100 + 50, 330 = 3 x 100 + 30); the paired mode cycles over chunks
        lat = model.get_latent_representation(gil, batch_size=100)
        torch.cuda.synchronize()
        out.append((list(model.history["train_loss_epoch"]), model.module.engine.params.flat.clone(),
                    model.module.engine.buffers.flat.clone(), lat))
    (h0, p0, b0, l0), (h1, p1, b1, l1) = out
    assert h0 == h1 and len(h0) == 2
    assert torch.equal(p0, p1) and torch.equal(b0, b1)
    for key in ("shared", "private", "shared_reordered", "private_reordered"):
        for g in (0, 1):
            assert np.array_equal(l0[key][g], l1[key][g]), (key, g)
