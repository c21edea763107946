"""Drop-in replacement of the reference's `spVIPESmodule` (reference src/spVIPES/module/spVIPESmodule.py:18-899) whose
per-minibatch arithmetic runs in the sm_100a kernels of libspvipes_b200.so.

Same constructor signature (reference :74-95), same parameter / buffer names (state_dict of a reference model loads 1:1),
same five methods and output-dict layouts (key ORDER included: model/spvipes.py:539-551 unpacks them positionally):

    _get_inference_input(tensors_by_group)                        reference :381-405
    inference(x, batch_index, groups, global_indices, **kw)       reference :425-472
    _get_generative_input(tensors_by_group, inference_outputs)    reference :407-423
    generative(private_stats, shared_stats, poe_stats, library, groups, batch_index)   reference :720-771
    loss(tensors_by_group, inference_outputs, generative_outputs, kl_weight)           reference :809-899
    forward(tensors, ..., loss_kwargs={"kl_weight": w}) -> (inference_outputs, generative_outputs, LossOutput)
                                                                  scvi BaseModuleClass.forward
    get_loadings(dataset, type_latent)                            reference :773-807

`forward` returns a loss tensor that carries an autograd node: `loss.backward()` runs the hand-written backward kernels and
deposits `.grad` on the nn.Parameters, so scvi's TrainingPlan (or any torch optimiser) drives it unchanged.  There is no CPU
fallback: constructing the module without a CUDA device / without the built library raises.

Differences that are deliberate: reparameterisation noise and dropout masks come from an in-kernel Philox generator seeded
from torch.initial_seed() (the reference consumes the global torch RNG, including draws it discards: quirk Q9).
"""
from __future__ import annotations

from collections import OrderedDict
from dataclasses import dataclass, field
from typing import Dict, Iterable, Optional

import numpy as np
import torch
from torch import nn
from torch.distributions import Normal

from ._lib import GC_THETA
from .engine import GroupBatch, Noise, StepEngine

X_KEY, BATCH_KEY, LABELS_KEY = "X", "batch", "labels"  # scvi.REGISTRY_KEYS


@dataclass
class LossOutput:
    """scvi.module.base.LossOutput (0.20.0), the fields the training plan reads"""
    loss: torch.Tensor
    reconstruction_loss: Optional[Dict[str, torch.Tensor]] = None
    kl_local: Optional[Dict[str, torch.Tensor]] = None
    kl_global: Optional[torch.Tensor] = None
    extra_metrics: Dict[str, torch.Tensor] = field(default_factory=dict)
    n_obs_minibatch: Optional[int] = None

    def __post_init__(self):
        if self.n_obs_minibatch is None and self.reconstruction_loss:
            self.n_obs_minibatch = int(next(iter(self.reconstruction_loss.values())).shape[0])

    @property
    def reconstruction_loss_sum(self):
        return sum(v.sum() for v in self.reconstruction_loss.values())

    @property
    def kl_local_sum(self):
        return sum(v.sum() for v in self.kl_local.values())


class _NBMixtureHandle:
    """stands where the reference puts scvi's NegativeBinomialMixture (`px`) of one group (module/spVIPESmodule.py:759).
    neg_log_prob_sum = -log_prob(log1p(x)).sum(-1), evaluated by the likelihood sweep of the pass.  The per-gene members are
    device tensors [B, G] without autograd, each computed on first access by one element launch (StepEngine.decode_elements) from
    the decoder state of the pass that built this handle, and cached: mu1 = px_rate_private, mu2 = px_rate_shared,
    mixture_logits = px_mixing, theta1 = exp(px_r) (an expanded view), mean = sigmoid(pi) mu1 + (1 - sigmoid(pi)) mu2 and
    log_prob(value) (eps 1e-8); sample(sample_shape, seed) draws counts (not cached).  Once the engine has run another forward or backward that state is gone: a member not read by
    then raises RuntimeError; members already read are independent tensors and keep their values."""

    def __init__(self, rec: torch.Tensor, engine=None, group: int = 0, ws=None):
        self.neg_log_prob_sum = rec
        self._eng, self._g, self._ws = engine, group, ws
        self._gen = engine.generation if engine is not None else None
        self._cache = {}

    def _check(self, what):
        if self._eng is None:
            raise RuntimeError(f"px.{what}: this handle carries the reconstruction term only")
        if self._eng.generation != self._gen:
            raise RuntimeError(f"px.{what} was not read before the engine's next forward or backward pass, which replaced the decoder "
                               f"state it is computed from; read the px fields of a pass before running the next one")

    def _elements(self, what, key, value=None):
        self._check(what)
        w, eng = self._ws, self._eng
        out = torch.empty(w.B, w.G, dtype=torch.float32, device=eng.device)
        outs, vals = [{}, {}], None
        outs[self._g] = {key: out}
        if value is not None:
            vals = [None, None]
            vals[self._g] = value
        eng.decode_elements(outs, vals)
        return out

    def _field(self, name, key):
        if name not in self._cache:
            self._cache[name] = self._elements(name, key)
        return self._cache[name]

    @property
    def mu1(self):
        return self._field("mu1", "rate_p")

    @property
    def mu2(self):
        return self._field("mu2", "rate_s")

    @property
    def mixture_logits(self):
        return self._field("mixture_logits", "pi")

    @property
    def mean(self):
        return self._field("mean", "mean")

    @property
    def theta1(self):
        if "theta1" not in self._cache:
            self._check("theta1")
            w = self._ws
            self._cache["theta1"] = w.genec[GC_THETA, :w.G].clone().unsqueeze(0).expand(w.B, w.G)
        return self._cache["theta1"]

    @property
    def theta2(self):  # scvi: theta2 = None means theta1 for both components (the reference's shared dispersion)
        return None

    def sample(self, sample_shape=torch.Size(), seed=None):
        """count draws [*sample_shape, B, G] float32 on the device (scvi NegativeBinomialMixture.sample, theta2 = None): per draw
        and element, mu1 with probability sigmoid(mixture_logits), else mu2; then Poisson(min(Gamma(theta1, theta1 / mu), 1e8)).
        seed: an int gives reproducible draws (a function of seed, group, draw index, cell and gene); None takes the engine's
        seed plus a counter the engine advances on every such call, so that repeated calls differ.  Not cached."""
        self._check("sample")
        shape = torch.Size(sample_shape)
        w, eng = self._ws, self._eng
        if seed is None:
            seed = (eng.seed + eng.sample_calls) % 2 ** 64
            eng.sample_calls += 1
        out = torch.empty(shape.numel(), w.B, w.G, dtype=torch.float32, device=eng.device)
        if out.numel():
            outs = [None, None]
            outs[self._g] = out
            eng.decode_sample(outs, seed)
        return out.view(*shape, w.B, w.G)

    def log_prob(self, value):
        """log_mixture_nb(value; mu1, mu2, theta1, mixture_logits), eps 1e-8, per element [B, G]; value: a [B, G] float tensor,
        evaluated as given (the reference passes log1p(x): quirk Q3)"""
        w = self._ws
        if self._eng is None:
            self._check("log_prob")
        v = torch.as_tensor(value, device=self._eng.device)
        if v.dim() != 2 or tuple(v.shape) != (w.B, w.G):
            raise ValueError(f"px.log_prob: value must be [{w.B}, {w.G}], got {tuple(v.shape)}")
        v = v.to(torch.float32).contiguous()
        return self._elements("log_prob", "ll", v)


class _LazyDict(OrderedDict):
    """ordered dict whose values may be zero-argument callables, evaluated on first access.  The reference's callers unpack
    the stats dicts positionally (model/spvipes.py:539-551), so key order is the contract; scvi's TrainingPlan never reads
    them, so building Normal / softmax objects per training step would be wasted launches."""

    def _force(self, k):
        v = OrderedDict.__getitem__(self, k)
        if callable(v) and not isinstance(v, (torch.Tensor, torch.distributions.Distribution)):
            v = v()
            OrderedDict.__setitem__(self, k, v)
        return v

    def __getitem__(self, k):
        return self._force(k)

    def get(self, k, default=None):
        return self._force(k) if k in self else default

    def values(self):
        return [self._force(k) for k in self.keys()]

    def items(self):
        return [(k, self._force(k)) for k in self.keys()]


class _CapturedStep:
    """the plugin call `module(batch, loss_kwargs)` -> `loss.backward()` for one minibatch signature, as two CUDA graphs
    (forward; backward) over static input buffers.  Two buffer sets alternate, so the host -> device copy of step s + 1 (copy
    stream) overlaps the kernels of step s; of the scvi minibatch matrix X [B, G0 + G1] only the group's own gene columns are
    moved (one strided cudaMemcpy2DAsync per group)."""

    def __init__(self, module, sig):
        self.module, self.sig = module, sig
        eng = module.engine
        dev = eng.device
        self.B = sig["B"]
        self.bufs = []
        for _ in (0, 1):
            X = [torch.zeros(self.B, G, dtype=dt, device=dev) for G, dt in zip(eng.d.genes, sig["x_dtypes"])]
            lab = [torch.zeros(self.B, dtype=torch.int32, device=dev) for _ in (0, 1)] if sig["labels"] else [None, None]
            idx = [torch.zeros(self.B, dtype=torch.int32, device=dev) for _ in (0, 1)]
            tmp = [[torch.zeros(self.B, dtype=torch.float32, device=dev) for _ in (0, 1)] for _ in (0, 1)]  # [labels | idx][group]
            batches = [GroupBatch(X=X[g], labels=lab[g], idx=idx[g], B=self.B) for g in (0, 1)]
            self.bufs.append({"X": X, "lab": lab, "idx": idx, "tmp": tmp, "batches": batches, "fwd": None, "bwd": None,
                              "ready": torch.cuda.Event(), "free": torch.cuda.Event()})
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.turn = 0
        self.warm = False
        main = torch.cuda.current_stream(dev)
        for b in self.bufs:
            b["free"].record(main)

    def stage(self, x, global_indices, labels):
        """copy this call's minibatch into the next buffer set (asynchronous for pinned host tensors / device tensors)"""
        from . import _lib as L
        m, eng = self.module, self.module.engine
        b = self.bufs[self.turn]
        lib = eng.lib
        cs = self.copy_stream
        cs.wait_event(b["free"])  # the previous step that used this buffer set has finished reading it
        with torch.cuda.stream(cs):
            for g in (0, 1):
                X = x[g]
                G = eng.d.genes[g]
                col0 = m._col0[g] if X.shape[1] != G else 0
                if col0 is None:  # scattered gene subset: gather (data movement only)
                    b["X"][g].copy_(X.to(eng.device, non_blocking=True).index_select(1, m._var_idx_dev[g]), non_blocking=True)
                elif X.device.type == "cpu":
                    esz = X.element_size()
                    L.check(lib.spv_copy2d_h2d(b["X"][g].data_ptr(), G * esz, X.data_ptr() + col0 * esz, X.stride(0) * esz, G * esz,
                                               self.B, cs.cuda_stream), "spv_copy2d_h2d")
                else:
                    b["X"][g].copy_(X[:, col0:col0 + G], non_blocking=True)
                for which, src, dst in ((0, labels[g] if labels is not None else None, b["lab"][g]), (1, global_indices[g], b["idx"][g])):
                    if src is None or dst is None:
                        continue
                    t = b["tmp"][which][g]
                    t.copy_(src.reshape(-1), non_blocking=True)   # float codes as scvi delivers them
                    dst.copy_(t)                                   # -> int32 on the device
            b["ready"].record(cs)
        return b

    def forward(self, b):
        eng = self.module.engine
        main = torch.cuda.current_stream(eng.device)
        main.wait_event(b["ready"])
        if not self.warm:  # first use: lazily configured kernels, workspaces (not capturable)
            eng.forward(b["batches"], training=True, noise=None)
            self.warm = True
        elif b["fwd"] is None:
            side = torch.cuda.Stream(device=eng.device)
            side.wait_stream(main)
            torch.cuda.synchronize(eng.device)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                eng.forward(b["batches"], training=True, noise=None)
            b["fwd"] = g
            b["ctx"] = eng._ctx  # the pass state (count pointers of this buffer set) that decode_elements reads after a replay
            g.replay()
            eng.note_replay(forward=True)
        else:
            if eng.bf16 and eng.stage_in_adam and eng._staged_version != eng.params.flat._version:
                eng.stage_weights()  # the parameters were written through torch since the 16-bit operand copies were made
            eng._ctx = b["ctx"]
            b["fwd"].replay()
            eng.note_replay(forward=True)
        return eng._ctx["ws"] if eng._ctx is not None else eng.workspace(self.B, self.B, True)

    def backward(self, b):
        eng = self.module.engine
        if b["fwd"] is None:  # the eager first step
            eng._ctx["batches"] = b["batches"]
            eng.backward(grad_scale=1.0)
        elif b["bwd"] is None:
            torch.cuda.synchronize(eng.device)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                eng.backward(grad_scale=1.0)
            b["bwd"] = g
            g.replay()
            eng.note_replay(forward=False)
        else:
            b["bwd"].replay()
            eng.note_replay(forward=False)
        b["free"].record(torch.cuda.current_stream(eng.device))


class _GraphStepFunction(torch.autograd.Function):
    """autograd node of the captured plugin step: forward = one graph replay, backward = one graph replay.  Its only autograd
    input is a scalar anchor leaf: the backward kernels write every parameter gradient into the engine's flat gradient buffer and
    `.grad` of each nn.Parameter is (re)bound to its view of that buffer - 66 AccumulateGrad nodes, gradient copies and scaling
    launches per step would cost more host time than the whole step takes on the GPU (tools/profile_plugin.py).  Consequence:
    gradients do not accumulate over several backward calls (each backward overwrites), as documented in INTEGRATION.md."""

    @staticmethod
    def forward(ctx, module, plan, buf, anchor):
        ws = plan.forward(buf)
        ctx.module, ctx.plan, ctx.buf = module, plan, buf
        module._last_ws = ws
        return module.engine.loss_out[0].clone()

    @staticmethod
    def backward(ctx, grad_loss):
        module, eng = ctx.module, ctx.module.engine
        ctx.plan.backward(ctx.buf)
        if module.scale_grads_by_upstream:
            eng.grads.mul_(grad_loss)  # one launch over the flat buffer (d total / d loss; 1.0 for a plain loss.backward())
        for p, gv in module._param_grad_pairs:
            if p.grad is None:
                p.grad = gv
        return None, None, None, None


class _StepFunction(torch.autograd.Function):
    """loss = fused CUDA forward; backward = hand-written CUDA backward, gradients for every parameter"""

    @staticmethod
    def forward(ctx, module, batches, training, *params):
        eng = module.engine
        ws = eng.forward(batches, training=training, noise=module._noise)
        ctx.module = module
        ctx.n_params = len(params)
        module._last_ws = ws
        return eng.loss_out[0].clone()

    @staticmethod
    def backward(ctx, grad_loss):
        module = ctx.module
        eng = module.engine
        eng.backward(grad_scale=1.0)
        grads = []
        for name in module._param_names:
            g = eng.params.view(name, eng.grads)
            grads.append(g * grad_loss)
        return (None, None, None, *grads)


class spVIPESmodule(nn.Module):
    def __init__(self, groups_lengths, groups_obs_names, groups_var_names, groups_obs_indices, groups_var_indices,
                 transport_plan: Optional[torch.Tensor] = None, pair_data: bool = False, use_labels: bool = False,
                 n_labels: Optional[int] = None, n_batch: int = 0, n_hidden: int = 128, n_dimensions_shared: int = 25,
                 n_dimensions_private: int = 10, dropout_rate: float = 0.1, use_batch_norm: bool = True,
                 use_layer_norm: bool = False, log_variational_inference: bool = True, log_variational_generative: bool = True,
                 dispersion: str = "gene", device: Optional[str] = None, precision: str = "fp32"):
        super().__init__()
        if not (log_variational_inference and log_variational_generative) or use_layer_norm or not use_batch_norm:
            raise NotImplementedError("only the reference's default normalisation switches are implemented")
        if len(groups_lengths) != 2:
            raise ValueError("the only supported number of groups is 2")  # reference :723-726
        self.n_dimensions_shared, self.n_dimensions_private, self.n_batch = n_dimensions_shared, n_dimensions_private, n_batch
        self.input_dims = groups_lengths
        self.groups_barcodes, self.groups_genes = groups_obs_names, groups_var_names
        self.groups_obs_indices, self.groups_var_indices = groups_obs_indices, groups_var_indices
        self.use_batch_norm, self.use_layer_norm, self.dispersion = use_batch_norm, use_layer_norm, dispersion
        self.log_variational_inference, self.log_variational_generative = log_variational_inference, log_variational_generative
        self.use_transport_plan = transport_plan is not None
        self.transport_plan = transport_plan
        self.use_labels, self.n_labels, self.pair_data = use_labels, n_labels, pair_data
        mode = "label" if use_labels else ("paired" if pair_data else "cluster")  # dispatcher priority, reference :484-509
        if not use_labels and transport_plan is None:
            raise ValueError("either labels or a transport plan is needed for the supervised PoE")
        dev = torch.device(device or "cuda")
        if dev.type != "cuda":
            raise RuntimeError("spvipes_b200.spVIPESmodule needs a CUDA (sm_100a) device: there is no CPU fallback")
        genes = tuple(int(v) for v in groups_lengths.values())
        plan = None
        if transport_plan is not None and not use_labels:
            # resident on the device in fp32 (paired mode: the argmax over the sub-plan is a bit-exact contract); a plan handed
            # over as bf16 is kept as bf16 (cluster mode at sizes where fp32 does not fit: 200k x 200k = 160 GB)
            keep = transport_plan.dtype == torch.bfloat16 and not pair_data
            plan = transport_plan.to(dev, torch.bfloat16 if keep else torch.float32).contiguous()
        self.engine = StepEngine(genes, n_hidden, n_dimensions_shared, n_dimensions_private, dropout_rate, mode, dev,
                                 seed=int(torch.initial_seed() % (2 ** 62)), plan=plan, precision=precision, n_batch=n_batch)
        # parameters / buffers are VIEWS of the engine's flat stores under the reference's names
        self._param_names = self.engine.params.names()
        self._torch_params = OrderedDict()
        for name in self._param_names:
            p = nn.Parameter(self.engine.params.view(name))
            self._torch_params[name] = p
            self._register(name, p, is_param=True)
        for name in self.engine.buffers.names():
            self._register(name, self.engine.buffers.view(name), is_param=False)
            if name.endswith("running_mean"):  # nn.BatchNorm1d carries this counter in its state_dict
                self._register(name[:-len("running_mean")] + "num_batches_tracked",
                               torch.zeros((), dtype=torch.long, device=dev), is_param=False)
        self._init_like_reference()
        self._grad_views = {n: self.engine.params.view(n, self.engine.grads) for n in self._param_names}
        self._param_grad_pairs = [(self._torch_params[n], self._grad_views[n]) for n in self._param_names]
        self._anchor = torch.zeros((), device=dev, requires_grad=True)  # the captured step's only autograd input
        # loss.backward() hands the node d total / d loss = 1; callers that scale the loss before backward() (gradient
        # accumulation, loss scaling) set this so that the flat gradient buffer is multiplied by the upstream gradient
        self.scale_grads_by_upstream = False
        # where a group's genes sit in the combined var axis of the scvi minibatch matrix: a column offset when they form a
        # contiguous ascending block (what prepare_adatas produces), else None (gathered)
        self._col0, self._var_idx_dev = [], []
        for g in (0, 1):
            vi = np.asarray(groups_var_indices[g])
            contiguous = vi.size > 0 and np.array_equal(vi, np.arange(vi[0], vi[0] + vi.size))
            self._col0.append(int(vi[0]) if contiguous else None)
            self._var_idx_dev.append(None if contiguous else torch.as_tensor(vi, device=dev))
        self._plans: Dict[tuple, _CapturedStep] = {}
        self.capture_steps = True  # training-mode forward(): replay captured CUDA graphs per minibatch signature
        self._noise = None      # tests may set a Noise(...) with explicit eps / dropout multipliers
        self._last_ws = None
        self._last_batches = None

    # ------------------------------------------------------------------ parameter plumbing
    def _register(self, dotted: str, tensor, is_param: bool):
        parts = dotted.split(".")
        mod = self
        for p in parts[:-1]:
            if p not in mod._modules:
                mod.add_module(p, nn.Module())
            mod = mod._modules[p]
        if is_param:
            mod.register_parameter(parts[-1], tensor)
        else:
            mod.register_buffer(parts[-1], tensor)

    def _init_like_reference(self):
        from .trainer import init_params
        init_params(self.engine, seed=int(torch.initial_seed() % (2 ** 31)))

    @property
    def device(self):
        return self.engine.device

    # ------------------------------------------------------------------ reference API
    def _get_inference_input(self, tensors_by_group):
        x = {i: group[X_KEY] for i, group in enumerate(tensors_by_group)}
        input_dict = {"x": x, "batch_index": [g[BATCH_KEY] for g in tensors_by_group],
                      "groups": [g["groups"] for g in tensors_by_group],
                      "global_indices": [g["indices"] for g in tensors_by_group]}
        if self.use_transport_plan and not self.pair_data:
            if "processed_transport_labels" not in tensors_by_group[0]:
                raise ValueError("processed_transport_labels are required when using transport plan.")
            input_dict["processed_labels"] = [g["processed_transport_labels"] for g in tensors_by_group]
        if self.use_labels:
            if "labels" not in tensors_by_group[0]:
                raise ValueError("Labels are required when using label-based POE.")
            input_dict["labels"] = [g["labels"].flatten() for g in tensors_by_group]
        return input_dict

    def _get_generative_input(self, tensors_by_group, inference_outputs):
        return {"private_stats": inference_outputs["private_stats"], "shared_stats": inference_outputs["shared_stats"],
                "poe_stats": inference_outputs["poe_stats"], "library": inference_outputs["library"],
                "groups": [g["groups"] for g in tensors_by_group], "batch_index": [g[BATCH_KEY] for g in tensors_by_group]}

    def _batches(self, x, global_indices, labels=None, processed_labels=None, batch_index=None):
        dev = self.engine.device
        out = []
        nb = self.engine.d.nb
        if nb and batch_index is None:
            raise ValueError("batch_index is required: the module was built with n_batch > 1")
        for g in (0, 1):
            X = x[g].to(dev)
            vi = np.asarray(self.groups_var_indices[g])
            G = int(vi.shape[0])
            if X.shape[1] == G:      # already this group's own genes
                col0 = 0
            elif np.array_equal(vi, np.arange(vi[0], vi[0] + G)):  # contiguous, ascending block of the combined var axis: zero-copy column offset
                col0 = int(vi[0])
            else:                    # arbitrary gene subset: gather once (data movement only)
                X, col0 = X.index_select(1, torch.as_tensor(vi, device=dev)).contiguous(), 0
            if X.dtype not in (torch.float32, torch.uint16):
                X = X.to(torch.float32)
            lab = None
            if labels is not None:
                lab = labels[g].to(dev).flatten().to(torch.int32)
            elif processed_labels is not None:
                lab = processed_labels[g].to(dev).flatten().to(torch.int32)
            idx = global_indices[g].to(dev).flatten().to(torch.int32) if global_indices is not None else None
            bc = batch_index[g].to(dev).flatten().to(torch.int32) if nb else None
            out.append(GroupBatch(X=X.contiguous() if X.stride(1) != 1 else X, col0=col0, labels=lab, idx=idx, B=int(X.shape[0]), batch=bc))
        return out

    def _stats_dicts(self, ws):
        """the reference's output dicts (key order = the contract, model/spvipes.py:539-551); derived entries (scales, softmax,
        Normal objects) are built on access"""
        P, S = self.n_dimensions_private, self.n_dimensions_shared
        private_stats, shared_stats, poe_stats, library = {}, {}, {}, {}
        for g, w in enumerate(ws):
            st = w.stats
            loc, lv = st[:, :P], st[:, P:2 * P]
            sloc, slv = st[:, 2 * P:2 * P + S], st[:, 2 * P + S:]
            clamp = not self.use_labels
            private_stats[g] = _LazyDict(logtheta_loc=loc, logtheta_logvar=lv,
                                         logtheta_scale=lambda lv=lv: torch.exp(0.5 * lv), log_z=w.zpriv,
                                         theta=lambda w=w: torch.softmax(w.zpriv, -1),
                                         qz=lambda loc=loc, lv=lv: Normal(loc, torch.exp(0.5 * lv)))
            shared_stats[g] = _LazyDict(logtheta_loc=sloc, logtheta_logvar=slv,
                                        logtheta_scale=lambda slv=slv: torch.exp(0.5 * slv), log_z=None, theta=None,
                                        qz=lambda sloc=sloc, slv=slv: Normal(sloc, torch.exp(0.5 * slv)))
            poe_stats[g] = _LazyDict(logtheta_loc=w.poe_loc, logtheta_logvar=w.poe_lv, logtheta_scale=w.poe_scale,
                                     logtheta_qz=lambda w=w, clamp=clamp: Normal(w.poe_loc, w.poe_scale.clamp(min=1e-6) if clamp else w.poe_scale),
                                     logtheta_log_z=w.zpoe, logtheta_theta=lambda w=w: torch.softmax(w.zpoe, -1))
            library[g] = w.lib.unsqueeze(1)
        return {"private_stats": private_stats, "shared_stats": shared_stats, "poe_stats": poe_stats, "library": library}

    @torch.no_grad()
    def inference(self, x, batch_index, groups, global_indices, **kwargs):
        """encoders + PoE only (used by get_latent_representation, reference model/spvipes.py:537-538)"""
        batches = self._batches(x, global_indices, kwargs.get("labels"), kwargs.get("processed_labels"), batch_index)
        ws = self.engine.forward(batches, training=self.training, noise=self._noise, with_grad=False, decode=False)
        self._last_ws, self._last_batches = ws, batches
        return self._stats_dicts(ws)

    @torch.no_grad()
    def generative(self, private_stats, shared_stats, poe_stats, library, groups, batch_index):
        if len(private_stats) > 2 or len(shared_stats) > 2:
            raise ValueError("the only supported number of groups is 2, make sure you passed only 2 groups to `prepare_adatas`")
        if self._last_batches is None:
            raise RuntimeError("generative() follows inference() on the same minibatch")
        ws = self.engine.decode()  # decoders + likelihood on the latents inference() left in the workspace (its arguments are views of it)
        self._last_ws = ws
        return self._generative_dict(ws)

    def _generative_dict(self, ws):
        return {"private_shared": {}, "private_poe": {str(g): {"px": _NBMixtureHandle(w.rec, self.engine, g, w)} for g, w in enumerate(ws)}}

    def _loss_output(self, loss, ws):
        out = self.engine.loss_out
        rec = {"reconst_loss_groups_1_poe": ws[0].rec, "reconst_loss_groups_2_poe": ws[1].rec}
        kl = OrderedDict(kl_divergence_groups_1_private=ws[0].klp, kl_divergence_groups_1_poe=ws[0].klq,
                         kl_divergence_groups_2_private=ws[1].klp, kl_divergence_groups_2_poe=ws[1].klq)
        extra = {"kl_divergence_private_groups_1": out[1], "kl_divergence_poe_groups_1": out[2],
                 "kl_divergence_private_groups_2": out[3], "kl_divergence_poe_groups_2": out[4]}
        return LossOutput(loss=loss, reconstruction_loss=rec, kl_local=kl, extra_metrics=extra)

    @torch.no_grad()
    def loss(self, tensors_by_group, inference_outputs, generative_outputs, kl_weight: float = 1.0):
        self.engine.set_kl_weight(kl_weight)
        ws = self._last_ws
        rec = [generative_outputs["private_poe"][str(g)]["px"].neg_log_prob_sum for g in (0, 1)]
        loss = torch.mean(rec[0] + rec[1] + kl_weight * (ws[0].klp + ws[0].klq + ws[1].klp + ws[1].klq))
        return self._loss_output(loss, ws)

    def forward(self, tensors, get_inference_input_kwargs=None, get_generative_input_kwargs=None, inference_kwargs=None,
                generative_kwargs=None, loss_kwargs=None, compute_loss=True):
        """scvi BaseModuleClass.forward: inference -> generative -> loss, here as ONE fused CUDA step"""
        inp = self._get_inference_input(tensors)
        kl_weight = float((loss_kwargs or {}).get("kl_weight", 1.0))
        self.engine.set_kl_weight(kl_weight)
        plan = self._plan_for(inp) if (self.training and torch.is_grad_enabled() and self.capture_steps and self._noise is None) else None
        if plan is not None:  # captured step: stage the inputs, replay the forward graph; loss.backward() replays the backward graph
            labels = inp.get("labels") if self.use_labels else inp.get("processed_labels")
            buf = plan.stage(inp["x"], inp["global_indices"], labels)
            plan.turn ^= 1
            self._last_batches = buf["batches"]
            loss = _GraphStepFunction.apply(self, plan, buf, self._anchor)
            ws = self._last_ws
            inference_outputs = self._stats_dicts(ws)
            generative_outputs = self._generative_dict(ws)
            if not compute_loss:
                return inference_outputs, generative_outputs
            return inference_outputs, generative_outputs, self._loss_output(loss, ws)
        batches = self._batches(inp["x"], inp["global_indices"], inp.get("labels"), inp.get("processed_labels"), inp["batch_index"])
        self._last_batches = batches
        if self.training and torch.is_grad_enabled():
            loss = _StepFunction.apply(self, batches, True, *[self._torch_params[n] for n in self._param_names])
            ws = self._last_ws
        else:
            with torch.no_grad():
                ws = self.engine.forward(batches, training=self.training, noise=self._noise, with_grad=False)
                self._last_ws = ws
                loss = self.engine.loss_out[0].clone()
        inference_outputs = self._stats_dicts(ws)
        generative_outputs = self._generative_dict(ws)
        if not compute_loss:
            return inference_outputs, generative_outputs
        return inference_outputs, generative_outputs, self._loss_output(loss, ws)

    def _plan_for(self, inp):
        """captured-step plan for this minibatch signature, or None when the step has to run eagerly (unequal group sizes,
        unsupported dtypes)"""
        x = inp["x"]
        B0, B1 = int(x[0].shape[0]), int(x[1].shape[0])
        if B0 != B1 or any(x[g].dtype not in (torch.float32, torch.uint16) for g in (0, 1)) or self.engine.d.nb:
            return None  # (batch covariates: the eager path stages the batch codes)
        has_labels = self.use_labels or (self.use_transport_plan and not self.pair_data)
        key = (B0, x[0].dtype, x[1].dtype, int(x[0].shape[1]), int(x[1].shape[1]), has_labels)
        plan = self._plans.get(key)
        if plan is None:
            plan = _CapturedStep(self, {"B": B0, "x_dtypes": (x[0].dtype, x[1].dtype), "labels": has_labels})
            self._plans[key] = plan
        return plan

    @torch.inference_mode()
    def get_loadings(self, dataset: int, type_latent: str) -> np.ndarray:
        """per-gene weights B W of the linear decoder, B = diag(gamma / sqrt(running_var + eps))  (reference :773-807)"""
        if type_latent not in ["shared", "private"]:
            raise ValueError(f"Invalid value for type_latent: {type_latent}. It can only be 'shared' or 'private'")
        tag = "p" if type_latent == "private" else "s"
        e = self.engine
        w = e.P(dataset, "W" + tag)
        if e.d.nb:
            w = w[:, :-e.d.nb]  # the covariate columns are not loadings (reference :804-805)
        sigma = torch.sqrt(e.Bf(dataset, "rv_" + tag) + 1e-3)
        loadings = (e.P(dataset, "g" + tag) / sigma).unsqueeze(1) * w
        return loadings.detach().cpu().numpy()
