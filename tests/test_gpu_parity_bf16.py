"""-m gpu: the tensor-core path (tcgen05 GEMMs: encoder fc1 on split-bf16 operands, decoder mixture / branch logits in bf16,
fused NB-likelihood epilogue) against the golden vectors from the unmodified reference and against the oracle.

Tolerances (BASELINE.json north_star, "bf16 tensor-core path"): indices bit-exact; per-batch ELBO and each of the
2 reconstruction + 4 KL terms <= 1e-2 relative; latent means / log-variances / scales <= 1e-3 (the encoders' K = genes
contraction runs as hi.hi + hi.lo + lo.hi on bf16 pairs, so the latents are fp32-grade in this mode too).
Gradients: per parameter, max |error| / max |gradient| <= GRAD_TOL (the decoder-side gradient GEMMs read bf16 operands:
dpi / dy rounded to 2^-9 relative, averaged over the minibatch rows).  The exact BASELINE minibatch shapes are in
tests/test_gpu_shapes.py."""
import numpy as np
import pytest
import torch

from tests.helpers import Golden, golden_names, grad_errors, relerr, run_oracle
from tests.gpu_helpers import engine_from_golden, engine_outputs, gate_consistent_grads

pytestmark = pytest.mark.gpu

TERMS = ("rec", "kl_private", "kl_poe")
LATENTS = ("private_loc", "private_logvar", "shared_loc", "shared_logvar", "poe_loc", "poe_logvar", "poe_scale")
GRAD_TOL = 2e-3


@pytest.mark.parametrize("name", golden_names())
def test_bf16_forward_matches_golden(name):
    gd = Golden(name)
    eng, batches, noise = engine_from_golden(gd, precision="bf16")
    ws = eng.forward(batches, training=gd.training, noise=noise)
    torch.cuda.synchronize()
    out = engine_outputs(eng, ws)
    assert relerr(out["loss"], gd.out["loss"]) < 1e-2
    for k in TERMS:
        for g in (0, 1):
            assert relerr(out[k][g].reshape(-1), gd.out[f"{k}{g}"].reshape(-1)) < 1e-2, (k, g)
    for g in (0, 1):
        assert relerr(out["library"][g].reshape(-1), gd.out[f"library{g}"].reshape(-1)) < 1e-5  # library stays fp32
    for k in LATENTS:
        for g in (0, 1):
            assert relerr(out[k][g], gd.out[f"{k}{g}"]) < 1e-3, (k, g, relerr(out[k][g], gd.out[f"{k}{g}"]))
    if gd.mode in ("label", "paired"):
        for g in (0, 1):
            assert np.array_equal(out["partners"][g], gd.out[f"partner{g}"]), g


@pytest.mark.parametrize("name", golden_names(training=True))
def test_bf16_backward_matches_golden(name):
    gd = Golden(name)
    eng, batches, noise = engine_from_golden(gd, precision="bf16")
    ws = eng.forward(batches, training=True, noise=noise)
    eng.backward()
    torch.cuda.synchronize()
    got = {k: v.cpu() for k, v in eng.grad_dict().items()}
    probe = {}
    run_oracle(gd, backward=False, probe=probe)
    want, switched = gate_consistent_grads(eng, ws, probe, gd.grads, lambda gates: run_oracle(gd, gates=gates)[1], gd.drop_masks())
    worst, where = grad_errors(got, want)
    assert worst < GRAD_TOL, (worst, where, switched)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_c1_shape_against_oracle(precision):
    """BASELINE.json configs[0] minibatch shape (2 x 512 cells, 2000 genes, H 128, 10 labels, label PoE): the CUDA path
    against the fp32 oracle on the same seeded inputs, explicit noise and dropout masks."""
    from oracle import restatement as rs
    from spvipes_b200 import synth
    from spvipes_b200.engine import GroupBatch, Noise, StepEngine
    from spvipes_b200.trainer import init_params

    B, G, H, S, P = 512, 2000, 128, 25, 10
    data = synth.make_counts((B, B), (G, G), 10, device="cuda", seed=4321)
    eng = StepEngine((G, G), H, S, P, 0.1, "label", "cuda", precision=precision)
    sd0 = init_params(eng, 3)
    eng.set_kl_weight(0.25)
    gen = torch.Generator().manual_seed(11)
    eps_p = [torch.randn(B, P, generator=gen) for _ in (0, 1)]
    eps_q = [torch.randn(B, S, generator=gen) for _ in (0, 1)]
    drop = [(torch.rand(B, 2 * H, generator=gen) < 0.9).float() / 0.9 for _ in (0, 1)]
    noise = Noise([e.cuda() for e in eps_p], [e.cuda() for e in eps_q], [d.cuda() for d in drop])
    batches = [GroupBatch(X=data.X[g], labels=data.labels[g]) for g in (0, 1)]
    ws = eng.forward(batches, training=True, noise=noise)
    eng.backward()
    torch.cuda.synchronize()
    out = engine_outputs(eng, ws)
    # oracle
    dm = {(g, k): drop[g][:, i * H:(i + 1) * H] for g in (0, 1) for i, k in enumerate(("private", "shared"))}

    def oracle(gates=None, probe=None):
        sd = {k: v.clone().requires_grad_("running" not in k) for k, v in sd0.items()}
        o = rs.step(sd, [data.X[g].cpu().to(torch.float32) for g in (0, 1)], mode="label", n_shared=S, n_private=P,
                    eps_private=eps_p, eps_poe=eps_q, labels=[data.labels[g].cpu().numpy() for g in (0, 1)], drop_masks=dm,
                    kl_weight=0.25, gates=gates, probe=probe)
        o["loss"].backward()
        return o, {k: sd[k].grad for k in rs.param_names(sd)}

    probe = {}
    want, grads = oracle(probe=probe)
    tol = 1e-4 if precision == "fp32" else 1e-2
    assert relerr(out["loss"], want["loss"].detach()) < tol
    for k in TERMS:
        for g in (0, 1):
            assert relerr(out[k][g], want[k][g].detach()) < tol, (k, g)
    for g in (0, 1):
        assert np.array_equal(out["partners"][g], want["partners"][g])
    for k in LATENTS:
        for g in (0, 1):
            assert relerr(out[k][g], want[k][g].detach()) < 1e-3, (k, g)
    grads, switched = gate_consistent_grads(eng, ws, probe, grads, lambda gates: oracle(gates=gates)[1], dm)
    worst, where = grad_errors({k: v.cpu() for k, v in eng.grad_dict().items()}, grads)
    assert worst < (2e-3 if precision == "fp32" else GRAD_TOL), (worst, where, switched)


def test_stats_tc_matches_simt_statistics():
    """softmax normalisers from the tensor-core statistics kernel (bf16 logits) vs the fp32 SIMT phase on the same state"""
    import torch
    from spvipes_b200 import _lib as L
    gd = Golden("label_tiny")
    eng, batches, noise = engine_from_golden(gd, precision="bf16")
    assert eng.fused_nb
    ws = eng.forward(batches, training=True, noise=noise)
    torch.cuda.synchronize()
    d = eng.d
    for g, w in enumerate(ws):
        got = w.rowc[:, :2].clone()
        bt = batches[g]
        src, esz = eng._src_of(bt.X)
        ptrs = eng._dec_ptrs(g, w, bt.X.data_ptr(), bt.rows, True)
        L.check(eng.lib.spv_dec_nb_fwd(src, ptrs, bt.X.stride(0), d.KMIX, w.B, w.G, 256, d.n_private, d.n_shared, 1, None, 0, 0,
                                       torch.cuda.current_stream().cuda_stream), "spv_dec_nb_fwd")
        torch.cuda.synchronize()
        want = w.rowc[:, :2]
        assert float((got - want).abs().max()) < 2e-2, g


def test_early_adam_is_the_same_update():
    """optimiser step interleaved with the backward (per parameter range) == backward followed by one Adam launch"""
    import torch
    from spvipes_b200.trainer import TrainLoop
    gd = Golden("label_tiny")
    out = []
    for early in (True, False):
        eng, batches, noise = engine_from_golden(gd, precision="bf16")
        loop = TrainLoop(eng)  # (also for the reference: it sets the engine's stage_in_adam)
        loop.set_epoch(1)
        for _ in range(3):
            if early:
                loop.step(batches, noise)
            else:
                eng.forward(batches, training=True, noise=noise)
                eng.backward()
                eng.adam_step(lr=loop.lr, eps=loop.eps, weight_decay=loop.weight_decay)
        torch.cuda.synchronize()
        out.append((eng.params.flat.clone(), eng.adam_m.clone(), eng.adam_v.clone(), int(eng.step_dev), eng.wb[0][0].clone(),
                    eng.wb[0][1][:eng.d.genes[0]].clone()))
    for a, b in zip(*out):
        assert torch.equal(a, b) if torch.is_tensor(a) else a == b
    off, shape = eng.params.offsets[0]["W1"]
    W1 = out[0][0][off:off + shape[0] * shape[1]].view(shape)
    assert torch.equal(out[0][4][:, :shape[1]], W1.bfloat16())  # the bf16 operand copy tracks the fp32 master
    lo = eng.wb[0][2][:, :shape[1]]                               # and its residual plane: hi + lo ~ W1 to 2^-17
    assert torch.equal(lo, (W1 - W1.bfloat16().float()).bfloat16())


def test_philox_noise_is_the_same_in_forward_and_backward():
    """TrainLoop.step with in-kernel Philox noise (noise=None): the backward must regenerate the eps of ITS forward.  The
    optimiser's step counter advances on an auxiliary stream during the backward; the Philox streams read their own counter.
    Recover eps from the forward's outputs, replay the step on a second engine with that eps given explicitly, compare the
    gradients."""
    from spvipes_b200.engine import Noise
    from spvipes_b200.trainer import TrainLoop
    for name in ("label_tiny", "paired_tiny"):
        gd = Golden(name)
        engA, batches, _ = engine_from_golden(gd, precision="fp32")
        engA.dropout_rate = 0.0
        p0, b0 = engA.params.flat.clone(), engA.buffers.flat.clone()
        loop = TrainLoop(engA)
        loop.set_epoch(200)
        for _ in range(3):  # several steps: the counters move apart
            p0.copy_(engA.params.flat); b0.copy_(engA.buffers.flat)
            loop.step(batches)
        torch.cuda.synchronize()
        ws = engA._ctx["ws"]
        P_ = gd.P
        eps_p = [((w.zpriv - w.stats[:, :P_]) / torch.exp(0.5 * w.stats[:, P_:2 * P_])).clone() for w in ws]
        sc = [w.poe_scale if gd.mode == "label" else w.poe_scale.clamp(min=1e-6) for w in ws]
        eps_q = [((w.zpoe - w.poe_loc) / s).clone() for w, s in zip(ws, sc)]
        gA = engA.grads.clone()
        engB, batchesB, _ = engine_from_golden(gd, precision="fp32")
        engB.dropout_rate = 0.0
        engB.params.flat.copy_(p0); engB.buffers.flat.copy_(b0)
        engB.set_kl_weight(0.5)
        engB.forward(batchesB, training=True, noise=Noise(eps_p, eps_q, None))
        engB.backward()
        torch.cuda.synchronize()
        err = float((gA - engB.grads).abs().max() / engB.grads.abs().max())
        assert err < 1e-4, (name, err)
        assert int(engA.step_dev) == 3 and int(engA.noise_dev) == 3


@pytest.mark.parametrize("mode,precision", [("paired", "fp32"), ("cluster", "fp32"), ("paired", "bf16"), ("cluster", "bf16")])
def test_ot_modes_hidden256_against_oracle(mode, precision):
    """BASELINE.json configs[2] / [3] flavour at a size the oracle finishes in seconds: OT-paired and OT-cluster PoE with
    n_hidden 256 (fc2 at the K = 256 limit of the whole-K GEMM), gene counts that are not multiples of the tile sizes,
    different gene counts per group.  Indices bit-exact, loss terms within the north-star tolerances."""
    from oracle import restatement as rs
    from spvipes_b200 import synth
    from spvipes_b200.engine import GroupBatch, Noise, StepEngine
    from spvipes_b200.trainer import init_params

    B, G0, G1, H, S, P, NL = 256, 1003, 1210, 256, 25, 10, 6
    data = synth.make_counts((B, B), (G0, G1), NL, device="cuda", seed=77)
    plan = synth.make_plan(B, B, data.labels[0], data.labels[1], NL, device="cuda", seed=7)
    eng = StepEngine((G0, G1), H, S, P, 0.1, mode, "cuda", plan=plan, precision=precision)
    sd0 = init_params(eng, 5)
    eng.set_kl_weight(0.5)
    gen = torch.Generator().manual_seed(13)
    eps_p = [torch.randn(B, P, generator=gen) for _ in (0, 1)]
    eps_q = [torch.randn(B, S, generator=gen) for _ in (0, 1)]
    drop = [(torch.rand(B, 2 * H, generator=gen) < 0.9).float() / 0.9 for _ in (0, 1)]
    noise = Noise([e.cuda() for e in eps_p], [e.cuda() for e in eps_q], [d.cuda() for d in drop])
    idx = [torch.arange(B, dtype=torch.int32, device="cuda") for _ in (0, 1)]
    labels = [data.labels[g] if mode == "cluster" else None for g in (0, 1)]
    batches = [GroupBatch(X=data.X[g], labels=labels[g], idx=idx[g]) for g in (0, 1)]
    ws = eng.forward(batches, training=True, noise=noise)
    eng.backward()
    torch.cuda.synchronize()
    out = engine_outputs(eng, ws)
    dm = {(g, k): drop[g][:, i * H:(i + 1) * H] for g in (0, 1) for i, k in enumerate(("private", "shared"))}

    def oracle(gates=None, probe=None):
        sd = {k: v.clone().requires_grad_("running" not in k) for k, v in sd0.items()}
        o = rs.step(sd, [data.X[g].cpu().to(torch.float32) for g in (0, 1)], mode=mode, n_shared=S, n_private=P,
                    eps_private=eps_p, eps_poe=eps_q, sub=plan.cpu(),
                    labels=[data.labels[g].cpu().numpy() for g in (0, 1)] if mode == "cluster" else None, drop_masks=dm,
                    kl_weight=0.5, gates=gates, probe=probe)
        o["loss"].backward()
        return o, {k: sd[k].grad for k in rs.param_names(sd)}

    probe = {}
    want, grads = oracle(probe=probe)
    tol = 1e-4 if precision == "fp32" else 1e-2
    assert relerr(out["loss"], want["loss"].detach()) < tol
    for k in TERMS:
        for g in (0, 1):
            assert relerr(out[k][g], want[k][g].detach()) < tol, (k, g)
    if mode == "paired":
        for g in (0, 1):
            assert np.array_equal(out["partners"][g], want["partners"][g])
    for k in LATENTS:
        for g in (0, 1):
            assert relerr(out[k][g], want[k][g].detach()) < 1e-3, (k, g)
    grads, switched = gate_consistent_grads(eng, ws, probe, grads, lambda gates: oracle(gates=gates)[1], dm)
    worst, where = grad_errors({k: v.cpu() for k, v in eng.grad_dict().items()}, grads)
    assert worst < (2e-3 if precision == "fp32" else GRAD_TOL), (worst, where, switched)


def test_exploding_latent_stays_finite():
    """the model does not clamp its log-variances, so an outlier cell can sample a latent far beyond fp16's range (seen in
    C5-shaped training: KL spikes of 1e8).  The fp16 decoder operands saturate instead of overflowing: every loss term and
    gradient stays finite, as in the fp32 mode."""
    gd = Golden("label_tiny")
    for precision in ("fp32", "bf16"):
        eng, batches, noise = engine_from_golden(gd, precision=precision)
        eng.state_dict()["encoder_0_private.lvar_encoder.1.bias"].fill_(26.0)  # scale = e^13 ~ 4e5: |z| beyond 65504
        ws = eng.forward(batches, training=True, noise=noise)
        eng.backward()
        torch.cuda.synchronize()
        assert float(ws[0].zpriv.abs().max()) > 65504.0
        assert bool(torch.isfinite(eng.loss_out[:7]).all()), (precision, eng.loss_out)
        assert bool(torch.isfinite(eng.grads).all()), precision
