"""Model-level API of spVIPES on top of the B200 hot path: `prepare_adatas`, `spVIPES.setup_anndata`,
`spVIPES(adata, n_dimensions_shared, n_dimensions_private, n_hidden, dropout_rate)`, `.train`, `.get_latent_representation`,
`.get_loadings` with the reference's signatures and semantics (reference model/spvipes.py:216-677,
model/base/training_mixin.py:19-123, data/prepare_adatas.py:7-134).

anndata / scvi-tools / lightning are not dependencies of this package: any object with `.X` (scipy sparse or ndarray),
`.obs` (pandas DataFrame), `.var_names`, `.obs_names` and `.uns` (dict) works, a real AnnData included; `GroupedData` is the
minimal stand-in.  What differs from the reference is WHERE things run: the count matrices live on the GPU as uint16 (or as
CSR when `.X` is scipy-sparse), a minibatch is a list of row indices gathered on the device (no per-step host-side
densification / host->device copy), the step
is one CUDA-graph replay, and the optimiser is the fused Adam kernel with the scvi TrainingPlan defaults
(lr 1e-3, eps 0.01, weight_decay 1e-6, KL warm-up over n_epochs_kl_warmup epochs).
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from itertools import cycle
from typing import Dict, List, Optional, Sequence

import numpy as np
import pandas as pd
import torch

from .engine import CsrCounts, GroupBatch
from .module import spVIPESmodule
from .trainer import (VALIDATION_METRICS, EarlyStopping, TrainLoop, elbo_metrics, epoch_batches, is_validation_epoch,
                      split_indices, validation_interval)

TRAIN_METRICS = ("elbo_train", "reconstruction_loss_train", "kl_local_train")
# Philox counter of the evaluation passes of a validation run or get_elbo (reset to this value at the start of each run): the top
# bit of the counter word, so it stays disjoint from the training passes, which count up from 0
EVAL_NOISE_BASE = -2 ** 31  # int32 bit pattern 0x80000000


@dataclass
class GroupedData:
    """minimal AnnData stand-in"""
    X: object
    obs: pd.DataFrame
    var_names: Sequence[str]
    obs_names: Optional[Sequence[str]] = None
    uns: Dict = field(default_factory=dict)

    def __post_init__(self):
        if self.obs_names is None:
            self.obs_names = [str(i) for i in range(self.X.shape[0])]

    @property
    def n_obs(self):
        return self.X.shape[0]

    @property
    def shape(self):
        return self.X.shape


def _dense(X):
    return np.asarray(X.todense()) if hasattr(X, "todense") else np.asarray(X)


def _is_sparse(X):
    return hasattr(X, "tocsr")


def prepare_adatas(adatas: Dict[str, object], layers: Optional[Sequence[Optional[str]]] = None) -> GroupedData:
    """concatenate two groups on the obs axis with an OUTER join on genes prefixed by their group key, and record the
    per-group obs / var index lists in `.uns` (reference data/prepare_adatas.py:94-132).

    The joined `.X` is a dense float32 array when every input `.X` is dense.  When any input `.X` is scipy-sparse it is a
    float32 scipy CSR matrix (the group blocks stacked with empty blocks for the other group's genes, as the reference's
    anndata concat keeps it): the dense join of two 1 M-cell x 20 k-gene groups would take 320 GB of host memory.
    `spVIPES` then keeps each group's counts as CSR on the GPU as well."""
    if len(adatas) != 2:
        raise ValueError("spVIPES currently supports exactly 2 groups")
    keys = list(adatas.keys())
    sparse = any(_is_sparse(a.X) for a in adatas.values())
    blocks, obs_frames, var_names, lengths = [], [], [], {}
    groups_obs_names, groups_var_names, groups_obs_indices, groups_var_indices = [], {}, [], []
    col0 = row0 = 0
    total_genes = sum(a.X.shape[1] for a in adatas.values())
    for gi, k in enumerate(keys):
        a = adatas[k]
        n, G = a.X.shape
        vn = [f"{k}_{v}" for v in a.var_names]
        var_names += vn
        if sparse:
            import scipy.sparse as sp
            own = sp.csr_matrix(a.X, dtype=np.float32)
            parts = [sp.csr_matrix((n, col0), dtype=np.float32), own, sp.csr_matrix((n, total_genes - col0 - G), dtype=np.float32)]
            blocks.append(sp.hstack(parts, format="csr"))
        else:
            full = np.zeros((n, total_genes), dtype=np.float32)  # the other group's genes are absent: zero fill of the outer join
            full[:, col0:col0 + G] = _dense(a.X)
            blocks.append(full)
        obs = a.obs.copy()
        obs["groups"] = k
        obs["indices"] = np.arange(n)  # within-group position (reference :94-97)
        obs_frames.append(obs)
        lengths[gi] = G
        groups_obs_names.append(list(getattr(a, "obs_names", range(n))))
        groups_var_names[k] = vn  # keyed by group name, as the reference (data/prepare_adatas.py:111)
        groups_obs_indices.append(np.arange(row0, row0 + n))
        groups_var_indices.append(np.arange(col0, col0 + G))
        col0 += G
        row0 += n
    obs = pd.concat(obs_frames, ignore_index=True)
    uns = {"groups_lengths": lengths, "groups_obs_names": groups_obs_names, "groups_var_names": groups_var_names,
           "groups_obs_indices": groups_obs_indices, "groups_var_indices": groups_var_indices, "groups_mapping": dict(enumerate(keys))}
    if sparse:
        import scipy.sparse as sp
        X = sp.vstack(blocks, format="csr")
    else:
        X = np.concatenate(blocks, 0)
    return GroupedData(X=X, obs=obs, var_names=var_names, uns=uns)


class spVIPES:
    """reference model/spvipes.py:165-677"""

    _setup: Dict[int, Dict] = {}

    @classmethod
    def setup_anndata(cls, adata, groups_key: str, match_clusters: bool = False, transport_plan_key: Optional[str] = None,
                      label_key: Optional[str] = None, batch_key: Optional[str] = None, layer: Optional[str] = None, **kwargs):
        """register which obs columns / uns entries drive the PoE (reference :285-422): labels take priority, then a
        transport plan (cluster-based when match_clusters, i.e. when `processed_transport_labels` exists, else paired)."""
        if groups_key not in adata.obs.columns:
            raise KeyError(f"{groups_key} not in adata.obs")
        if transport_plan_key is not None and transport_plan_key not in adata.uns:
            raise ValueError(f"Transport plan not found in adata.uns['{transport_plan_key}']")
        if match_clusters and transport_plan_key is not None and "processed_transport_labels" not in adata.obs.columns:
            # reference :362-370: derive the shared cluster labels from the plan (transport.process_transport_plan; the
            # clustering step is scanpy's Leiden when scanpy is installed, kNN + Louvain otherwise, or `cluster_fn=` in kwargs)
            from .transport import process_transport_plan
            labels = process_transport_plan(adata.uns[transport_plan_key], adata, groups_key, cluster_fn=kwargs.pop("cluster_fn", None))
            adata.obs["processed_transport_labels"] = pd.Categorical(labels)
        if match_clusters and "processed_transport_labels" not in adata.obs.columns:
            raise ValueError("match_clusters=True needs a transport plan (transport_plan_key) or adata.obs['processed_transport_labels']")
        if batch_key is not None and batch_key not in adata.obs.columns:
            raise KeyError(f"{batch_key} not in adata.obs")
        cls._setup[id(adata)] = {"groups_key": groups_key, "match_clusters": match_clusters, "transport_plan_key": transport_plan_key,
                                 "label_key": label_key, "batch_key": batch_key, "layer": layer}

    def __init__(self, adata, n_hidden: int = 128, n_dimensions_shared: int = 25, n_dimensions_private: int = 10,
                 dropout_rate: float = 0.1, **model_kwargs):
        if id(adata) not in self._setup:
            raise ValueError("Please run `spVIPES.setup_anndata` on this object first")
        self.adata = adata
        self.setup_args = self._setup[id(adata)]
        self.n_dimensions_private, self.n_dimensions_shared = n_dimensions_private, n_dimensions_shared
        uns = adata.uns
        tp_key = self.setup_args["transport_plan_key"]
        transport_plan = torch.tensor(np.asarray(uns[tp_key]), dtype=torch.float32) if tp_key else None
        pair_data = "processed_transport_labels" not in adata.obs.columns  # reference :249 (quirk Q10)
        label_key = self.setup_args["label_key"]
        use_labels = label_key is not None
        self._label_codes = None
        n_labels = None
        if use_labels:
            cat = pd.Categorical(adata.obs[label_key])  # categories sorted, as scvi's CategoricalObsField
            self._label_codes = np.asarray(cat.codes, dtype=np.int32)
            n_labels = len(cat.categories)
        elif not pair_data:
            self._label_codes = np.asarray(pd.Categorical(adata.obs["processed_transport_labels"]).codes, dtype=np.int32)
        # batch covariate: categorical codes (scvi CategoricalObsField: sorted categories); n_batch = number of categories, the
        # one-hot code is injected when n_batch > 1 (reference model/spvipes.py:230, 252; nn/networks.py:60-68)
        batch_key = self.setup_args["batch_key"]
        self._batch_codes, n_batch = None, 0
        if batch_key is not None:
            bcat = pd.Categorical(adata.obs[batch_key])
            self._batch_codes, n_batch = np.asarray(bcat.codes, dtype=np.int32), len(bcat.categories)
        self.module = spVIPESmodule(groups_lengths=uns["groups_lengths"], groups_obs_names=uns["groups_obs_names"],
                                    groups_var_names=uns["groups_var_names"], groups_var_indices=uns["groups_var_indices"],
                                    groups_obs_indices=uns["groups_obs_indices"], transport_plan=transport_plan, pair_data=pair_data,
                                    use_labels=use_labels, n_labels=n_labels, n_batch=n_batch, n_hidden=n_hidden,
                                    n_dimensions_shared=n_dimensions_shared, n_dimensions_private=n_dimensions_private,
                                    dropout_rate=dropout_rate, **model_kwargs)
        self.is_trained_ = False
        self.history: Dict[str, List[float]] = {"train_loss_epoch": []}
        self.early_stopped_epoch_: Optional[int] = None
        self._device_data = None

    # ------------------------------------------------------------------ device-resident data
    def _to_device(self):
        """per group: uint16 [N_g, G_g] counts of the group's own genes (float32 if the data are not small integers); a
        scipy-sparse `adata.X` stays sparse: each group becomes a CSR matrix on the GPU (engine.CsrCounts)"""
        if self._device_data is not None:
            return self._device_data
        dev = self.module.device
        uns = self.adata.uns
        X = self.adata.X
        Xcsr = X.tocsr() if _is_sparse(X) else None
        data = []
        for g in (0, 1):
            rows, cols = np.asarray(uns["groups_obs_indices"][g]), np.asarray(uns["groups_var_indices"][g])
            if Xcsr is not None:
                # the group's rows and its column range (contiguous as prepare_adatas lays it out: a sparse slice)
                contiguous = len(cols) > 0 and np.array_equal(cols, np.arange(cols[0], cols[0] + len(cols)))
                sel = slice(int(cols[0]), int(cols[0]) + len(cols)) if contiguous else cols
                t = CsrCounts.from_scipy(Xcsr[rows][:, sel], dev)
            else:
                blk = _dense(X[rows][:, cols])
                integral = np.all(blk == np.round(blk)) and blk.min() >= 0 and blk.max() <= 65535
                # (numpy's column selection hands back a Fortran-ordered block: make it row-major, the kernels read rows)
                t = torch.from_numpy(np.ascontiguousarray(blk.astype(np.uint16 if integral else np.float32))).to(dev)
            labels = None
            if self._label_codes is not None:
                labels = torch.from_numpy(self._label_codes[rows].astype(np.int32)).to(dev)
            idx = torch.from_numpy(np.asarray(self.adata.obs["indices"])[rows].astype(np.int32)).to(dev)
            batch = None
            if self.module.engine.d.nb:
                batch = torch.from_numpy(self._batch_codes[rows].astype(np.int32)).to(dev)
            data.append({"X": t, "labels": labels, "idx": idx, "row0": int(rows[0]), "rows": rows, "batch": batch})
        self._device_data = data
        return data

    def _local_rows(self, g, global_rows):
        """global obs row ids -> positions inside group g's device matrix"""
        rows = self._device_data[g]["rows"]
        if np.array_equal(rows, np.arange(rows[0], rows[0] + len(rows))):
            return np.asarray(global_rows) - rows[0]
        lut = {int(r): i for i, r in enumerate(rows)}
        return np.array([lut[int(r)] for r in global_rows])

    def _static_batches(self, B):
        dev = self.module.device
        data = self._to_device()
        bufs = [torch.zeros(B, dtype=torch.int32, device=dev) for _ in (0, 1)]
        # batch codes of the minibatch: a static buffer refreshed from the per-cell codes before every step
        self._batch_bufs = [torch.zeros(B, dtype=torch.int32, device=dev) if data[g]["batch"] is not None else None for g in (0, 1)]
        batches = []
        for g in (0, 1):
            d = data[g]
            batches.append(GroupBatch(X=d["X"], rows=bufs[g], labels=d["labels"], idx=d["idx"], labels_per_cell=True, B=B,
                                      batch=self._batch_bufs[g]))
        return bufs, batches

    # ------------------------------------------------------------------ training
    def train(self, group_indices_list: Sequence[Sequence[int]], max_epochs: Optional[int] = None, use_gpu=None,
              train_size: float = 0.9, validation_size: Optional[float] = None, batch_size: int = 128,
              early_stopping: bool = False, n_steps_kl_warmup: Optional[int] = None, n_epochs_kl_warmup: Optional[int] = 400,
              plan_kwargs: Optional[dict] = None, seed: int = 0, use_cuda_graph: bool = True,
              check_val_every_n_epoch: Optional[int] = None, early_stopping_monitor: str = "elbo_validation",
              early_stopping_patience: int = 45, early_stopping_min_delta: float = 0.0, early_stopping_mode: str = "min",
              _noise_fn=None, **kwargs):
        """reference model/base/training_mixin.py:19-123 + scvi TrainingPlan / TrainRunner / Trainer semantics.

        Validation (scvi 0.20 Trainer arguments): after epoch e when (e + 1) % check_val_every_n_epoch == 0; None means every epoch
        with early_stopping and never without.  A validation run takes the minibatches get_latent_representation takes on
        self.val_idx (batch_size, drop_last=False) through eval-mode passes and appends elbo_validation,
        reconstruction_loss_validation, kl_local_validation and validation_loss to history (trainer.elbo_metrics).  Its latent
        noise comes from a Philox counter of its own and eval mode updates no BatchNorm statistics, so validation leaves the
        training itself unchanged.  early_stopping: Lightning's EarlyStopping rule (trainer.EarlyStopping) on
        early_stopping_monitor after each validation run; a stop ends training after that epoch (early_stopped_epoch_) with the
        last epoch's parameters.  Every epoch also appends elbo_train, reconstruction_loss_train and kl_local_train.
        _noise_fn (tests): as in get_latent_representation, for the validation passes."""
        n_obs = self.adata.X.shape[0]
        if max_epochs is None:
            max_epochs = int(min(round((20000 / n_obs) * 400), 400))  # reference :89-91
        plan_kwargs = dict(plan_kwargs or {})
        lr, eps, wd = plan_kwargs.get("lr", 1e-3), plan_kwargs.get("eps", 0.01), plan_kwargs.get("weight_decay", 1e-6)
        every = validation_interval(check_val_every_n_epoch, early_stopping)
        stopper = EarlyStopping(early_stopping_monitor, early_stopping_patience, early_stopping_min_delta, early_stopping_mode)
        train_idx, self.val_idx, self.test_idx = split_indices(group_indices_list, train_size, validation_size, seed)
        self.train_idx = train_idx
        if every is not None and min(len(v) for v in self.val_idx) == 0:
            raise ValueError("validation (early_stopping or check_val_every_n_epoch) needs a non-empty validation split in both "
                             f"groups, got {[len(v) for v in self.val_idx]} cells: lower train_size or set validation_size")
        self._to_device()
        for k in TRAIN_METRICS + (VALIDATION_METRICS if every is not None else ()):
            self.history.setdefault(k, [])
        self.early_stopped_epoch_ = None
        eng = self.module.engine
        if eng.mode != "label":
            # the OT modes index the plan / cluster labels with per-minibatch arrays: gather them on the host per step
            use_cuda_graph = False
        loop = TrainLoop(eng, lr=lr, eps=eps, weight_decay=wd, n_epochs_kl_warmup=n_epochs_kl_warmup)
        global_step = 0
        self.module.train()
        bufs, batches = self._static_batches(batch_size)
        graph = None
        for epoch in range(max_epochs):
            loop.set_epoch(epoch)
            steps = epoch_batches(train_idx, batch_size, shuffle=True, drop_last=True)
            if not steps:
                raise ValueError("batch_size is larger than the training split of a group")
            local = [[torch.from_numpy(self._local_rows(g, st[g]).astype(np.int32)) for g in (0, 1)] for st in steps]
            dev_rows = [torch.stack([l[g] for l in local]).to(eng.device) for g in (0, 1)]
            tot = torch.zeros(7, device=eng.device)  # per-step loss_out[:7] summed over the epoch
            for s in range(len(steps)):
                if n_steps_kl_warmup:  # scvi TrainingPlan: the step-based warm-up takes precedence over the epoch-based one
                    eng.set_kl_weight(min(1.0, global_step / n_steps_kl_warmup))
                global_step += 1
                for g in (0, 1):
                    bufs[g].copy_(dev_rows[g][s], non_blocking=True)
                    if self._batch_bufs[g] is not None:
                        self._batch_bufs[g].copy_(self._device_data[g]["batch"][dev_rows[g][s].long()])
                if eng.mode != "label":
                    step_batches = self._ot_batches(bufs, batch_size)
                    loop.step(step_batches)
                elif use_cuda_graph:
                    if graph is None:
                        graph = loop.capture(batches)
                    graph.replay()
                    eng.note_replay(forward=True)   # one training step: a forward and a backward pass
                    eng.note_replay(forward=False)
                else:
                    loop.step(batches)
                tot += eng.loss_out[:7]
            t = [float(v) for v in tot.cpu()]
            self.history["train_loss_epoch"].append(t[0] / len(steps))
            # every training minibatch holds batch_size cells in both groups: the mean over steps of the per-step means is the sum
            # over the epoch divided by the epoch's n_obs
            rec, kl = (t[5] + t[6]) / len(steps), (t[1] + t[2] + t[3] + t[4]) / len(steps)
            for k, v in zip(TRAIN_METRICS, (rec + kl, rec, kl)):
                self.history[k].append(v)
            if is_validation_epoch(epoch, every):
                if n_steps_kl_warmup:  # the weight after the epoch's last step (the next step sets its own before it runs)
                    eng.set_kl_weight(min(1.0, global_step / n_steps_kl_warmup))
                metrics = elbo_metrics(self._elbo_sums(self.val_idx, batch_size, False, _noise_fn))
                self.module.train()
                for k, v in metrics.items():
                    self.history[k].append(v)
                if early_stopping and stopper.update(metrics[early_stopping_monitor]):
                    self.early_stopped_epoch_ = epoch
                    break
        self.module.eval()
        self.is_trained_ = True
        return self

    def _ot_batches(self, bufs, B):
        data = self._device_data
        out = []
        for g in (0, 1):
            d = data[g]
            r = bufs[g].long()
            lab = d["labels"][r].contiguous() if d["labels"] is not None else None
            out.append(GroupBatch(X=d["X"], rows=bufs[g], labels=lab, idx=d["idx"][r].contiguous(), B=B, batch=self._batch_bufs[g]))
        return out

    # ------------------------------------------------------------------ latent extraction
    @torch.no_grad()
    def get_latent_representation(self, group_indices_list: Sequence[Sequence[int]], adata=None, indices=None,
                                  normalized: bool = False, give_mean: bool = True, mc_samples: int = 5000,
                                  batch_size: Optional[int] = None, drop_last: Optional[bool] = None, _noise_fn=None) -> dict:
        """reference model/spvipes.py:424-650: sequential minibatches, the shorter group cycled (zip(largest, cycle(other))),
        module in eval mode; returns the SAMPLED log_z of the PoE / private posteriors, truncated to the group sizes and
        re-ordered by within-group index.

        normalized=True cannot complete in the reference either: _process_batches appends nothing to the shared lists in that
        branch (spvipes.py:542-544, 552) and _format_results then calls torch.cat on the empty lists (:634-635), which raises
        RuntimeError; with give_mean=False it fails earlier on an unbound local (:556-563).  The same error type is raised here
        instead of inventing a result the reference never produced.

        _noise_fn (tests): callable(batch number, B0, B1) -> engine.Noise with the eps of that minibatch; None = in-kernel Philox."""
        if normalized:
            raise RuntimeError("normalized=True: the reference collects no shared latents in this branch and fails in "
                               "torch.cat on an empty list (model/spvipes.py:542-544, 634); use normalized=False")
        n = [len(g) for g in group_indices_list]
        res = {"shared": [[], []], "private": [[], []], "idx": [[], []]}
        for batches, ws in self._eval_passes(group_indices_list, batch_size, drop_last, _noise_fn):
            for g in (0, 1):
                res["shared"][g].append(ws[g].zpoe.cpu().clone())
                res["private"][g].append(ws[g].zpriv.cpu().clone())
                res["idx"][g].append(batches[g].idx.cpu().clone())
        # reference _format_results (:628-650): truncate to the group sizes; group 2 re-ordered by its within-group index
        shared = {g: torch.cat(res["shared"][g]).numpy()[:n[g]] for g in (0, 1)}
        private = {g: torch.cat(res["private"][g]).numpy()[:n[g]] for g in (0, 1)}
        idx2 = torch.cat(res["idx"][1]).numpy().flatten()[:n[1]]
        order = np.argsort(idx2)
        return {"shared": shared, "private": private,
                "shared_reordered": {0: shared[0], 1: shared[1][order]},
                "private_reordered": {0: private[0], 1: private[1][order]}}

    def _eval_passes(self, group_indices_list, batch_size, drop_last, _noise_fn, decode=False):
        """the minibatches of the reference's latent extraction, each through an eval-mode encoder pass
        (engine.forward(..., decode=False); decode=True: the whole pass without the loss, engine.forward(..., loss=False)): yields
        (batches, workspaces) per minibatch.  Sequential chunks of batch_size cells per
        group; reference :478-515: drop_last defaults to False in every mode; the paired OT mode (no labels) then goes through the
        cycling path, every other mode through one ConcatDataLoader over the two index lists"""
        self._to_device()
        eng = self.module.engine
        batch_size = batch_size or 128  # scvi.settings.batch_size
        n = [len(g) for g in group_indices_list]
        self.module.eval()
        drop_last = False if drop_last is None else bool(drop_last)
        use_cycling = eng.mode == "paired" and not drop_last
        counter = [0]

        def process(index_lists):
            """reference _process_batches (:537-576) over ConcatDataLoader(shuffle=False): sequential chunks per group, the
            loader with the most batches drives and the other one is cycled (dataloaders/_concat_dataloader.py:101-110)"""
            chunks = [[np.asarray(gi)[k:k + batch_size] for k in range(0, len(gi), batch_size)] for gi in index_lists]
            if drop_last:
                chunks = [[c for c in ch if len(c) == batch_size] for ch in chunks]
            largest = int(np.argmax([len(c) for c in chunks]))
            its = [iter(c) if g == largest else cycle(c) for g, c in enumerate(chunks)]
            for st in zip(*its):
                # (pinned host memory: the upload does not wait for the previous minibatch's kernels)
                rows = [torch.from_numpy(self._local_rows(g, st[g]).astype(np.int32)).pin_memory().to(eng.device, non_blocking=True)
                        for g in (0, 1)]
                batches = []
                for g in (0, 1):
                    d = self._device_data[g]
                    r = rows[g].long()
                    lab = d["labels"][r].contiguous() if d["labels"] is not None else None
                    bc = d["batch"][r].contiguous() if d["batch"] is not None else None
                    batches.append(GroupBatch(X=d["X"], rows=rows[g], labels=lab, idx=d["idx"][r].contiguous(), B=len(st[g]), batch=bc))
                noise = _noise_fn(counter[0], len(st[0]), len(st[1])) if _noise_fn is not None else None
                counter[0] += 1
                yield batches, eng.forward(batches, training=False, noise=noise, with_grad=False, decode=decode, loss=False)

        if use_cycling:
            # reference _process_all_cells_with_cycling (:578-626): chunks of min(n) cells, the indices of BOTH groups taken
            # modulo their group's length, each chunk through its own loader
            lo, hi = min(n), max(n)
            if lo == 0:
                raise ValueError("One of the groups is empty")
            for start in range(0, hi, lo):
                yield from process([[group_indices_list[g][(start + i) % n[g]] for i in range(lo)] for g in (0, 1)])
        else:
            yield from process(group_indices_list)

    def _elbo_sums(self, group_indices_list, batch_size, drop_last, _noise_fn):
        """float64 [8] host tensor of StepEngine.accumulate_elbo summed over the eval passes of _eval_passes (one host read).  The
        latent noise is drawn on a counter that starts at EVAL_NOISE_BASE for every run: the training noise stream is not
        advanced, and the same weights give the same value on every call."""
        eng = self.module.engine
        self._to_device()
        acc = torch.zeros(8, dtype=torch.float64, device=eng.device)
        counter = torch.full((1,), EVAL_NOISE_BASE, dtype=torch.int32, device=eng.device)
        with eng.noise_counter(counter):
            for _, ws in self._eval_passes(group_indices_list, batch_size, drop_last, _noise_fn, decode=True):
                eng.accumulate_elbo(ws, acc)
        # the passes overwrote the engine's per-pass decoder state: decode_elements / decode_sample need a forward of their own
        eng._ctx = None
        acc = acc.cpu()
        if acc[6] <= 0:
            raise ValueError("no minibatch to evaluate: a group's index list is empty (or drop_last removed every minibatch)")
        return acc

    @torch.no_grad()
    def get_elbo(self, group_indices_list: Sequence[Sequence[int]], batch_size: Optional[int] = None,
                 drop_last: Optional[bool] = None, _noise_fn=None) -> float:
        """the evidence lower bound of the eval-mode model on the given cells (scvi VAEMixin.get_elbo sign convention: the ELBO,
        i.e. minus the elbo metric (reconstruction loss + local KL per observation) that history["elbo_validation"] records).
        Same minibatches as get_latent_representation (batch_size, drop_last, cycling); n_obs of a minibatch is the size of
        group 0's part.  get_elbo(model.val_idx, batch_size) reproduces -history["elbo_validation"][-1] for the current weights.
        _noise_fn (tests): as in get_latent_representation."""
        return -elbo_metrics(self._elbo_sums(group_indices_list, batch_size, drop_last, _noise_fn))["elbo_validation"]

    # decoded outputs of get_decoded_expression -> StepEngine.decode_elements names
    DECODED_OUTPUTS = {"mean": "mean", "px_rate_private": "rate_p", "px_rate_shared": "rate_s", "px_mixing": "pi", "log_prob": "ll"}

    @torch.no_grad()
    def get_decoded_expression(self, group_indices_list: Sequence[Sequence[int]], outputs: Sequence[str] = ("mean",),
                               gene_indices=None, batch_size: Optional[int] = None, drop_last: Optional[bool] = None,
                               _noise_fn=None) -> dict:
        """per-cell, per-gene decoder outputs of the eval-mode model (module/spVIPESmodule.py:751-759) on the latents that
        get_latent_representation samples with the same arguments (same minibatches, cycling, truncation and noise):
          mean             sigmoid(px_mixing) px_rate_private + (1 - sigmoid(px_mixing)) px_rate_shared (NegativeBinomialMixture.mean)
          px_rate_private  exp(library) softmax over the genes of the private factor regressor's output
          px_rate_shared   the same from the shared latents
          px_mixing        the mixing logit: how much of a gene's expression the private branch explains (sigmoid of it)
          log_prob         per-gene log-likelihood of the cell's own counts at log1p(x) (quirk Q3); minus its row sum is the
                           reconstruction loss
        gene_indices: None (all of each group's own genes) or one sequence per group of positions within that group's genes
        (None entries: all); the gene selection is made on the GPU before the copy to the host.
        Returns {output: {0: ndarray [n0, k0], 1: ndarray [n1, k1]}} float32, rows in the order of group_indices_list[g]; each
        output takes n * k * 4 bytes of host memory per group (n cells, k genes), and the whole [batch, genes] block of a
        minibatch passes through GPU memory before the gene selection.
        _noise_fn (tests): as in get_latent_representation."""
        outputs = (outputs,) if isinstance(outputs, str) else tuple(outputs)
        bad = [o for o in outputs if o not in self.DECODED_OUTPUTS]
        if bad or not outputs:
            raise ValueError(f"unknown decoded output(s) {bad or outputs}; choose from {sorted(self.DECODED_OUTPUTS)}")
        eng = self.module.engine
        genes = eng.d.genes
        sel = self._gene_selection(gene_indices)
        n = [len(g) for g in group_indices_list]
        res = {o: [[], []] for o in outputs}
        for _, ws in self._eval_passes(group_indices_list, batch_size, drop_last, _noise_fn):
            outs = [{self.DECODED_OUTPUTS[o]: torch.empty(ws[g].B, genes[g], dtype=torch.float32, device=eng.device) for o in outputs}
                    for g in (0, 1)]
            eng.decode_elements(outs)
            for g in (0, 1):
                for o in outputs:
                    t = outs[g][self.DECODED_OUTPUTS[o]]
                    res[o][g].append((t if sel[g] is None else t.index_select(1, sel[g])).cpu())
        return {o: {g: torch.cat(res[o][g]).numpy()[:n[g]] for g in (0, 1)} for o in outputs}

    def _gene_selection(self, gene_indices):
        """gene_indices (None, or one sequence or None per group) -> per group None or a device index tensor, checked"""
        eng = self.module.engine
        genes = eng.d.genes
        sel = [None, None]
        if gene_indices is not None:
            if len(gene_indices) != 2:
                raise ValueError("gene_indices: one sequence (or None) per group")
            for g in (0, 1):
                if gene_indices[g] is None:
                    continue
                gi = np.asarray(gene_indices[g], dtype=np.int64).reshape(-1)
                if gi.size and (gi.min() < 0 or gi.max() >= genes[g]):
                    raise ValueError(f"gene_indices[{g}]: positions must lie in [0, {genes[g]})")
                sel[g] = torch.from_numpy(gi).to(eng.device)
        return sel

    @torch.no_grad()
    def posterior_predictive_sample(self, group_indices_list: Sequence[Sequence[int]], n_samples: int = 1, gene_indices=None,
                                    batch_size: Optional[int] = None, drop_last: Optional[bool] = None, seed: Optional[int] = None,
                                    _noise_fn=None) -> dict:
        """counts drawn from the eval-mode model's NB mixture (scvi 0.20 posterior_predictive_sample / VAE.sample): each of the
        n_samples draws takes its own latent sample (its own eval pass over the minibatches of get_decoded_expression, with the
        same cycling, truncation and row order) and one count draw per cell and gene from it (px.sample).
        gene_indices: as in get_decoded_expression (selected on the GPU before the copy to the host).
        seed: an int gives reproducible count draws for given latents; None takes the engine's seed plus its sample-call counter.
        Every eval pass draws under its own draw index (its position among all passes), so no two minibatches share counters.  The latent noise comes from the engine's Philox streams (or _noise_fn).
        Returns {0: ndarray, 1: ndarray} float32: [n_g, k_g] when n_samples == 1, else [n_g, k_g, n_samples]."""
        n_samples = int(n_samples)
        if n_samples < 1:
            raise ValueError(f"n_samples must be >= 1, got {n_samples}")
        eng = self.module.engine
        if seed is None:
            seed = (eng.seed + eng.sample_calls) % 2 ** 64
            eng.sample_calls += 1
        elif not 0 <= int(seed) < 2 ** 64:
            raise ValueError(f"seed must lie in [0, 2**64), got {seed}")
        seed = int(seed)
        genes = eng.d.genes
        sel = self._gene_selection(gene_indices)
        n = [len(g) for g in group_indices_list]
        res = [[[] for _ in range(n_samples)] for _ in (0, 1)]
        passes = 0

        def noise_fn(_, b0, b1):  # the test hook numbers the passes across all samples
            return _noise_fn(passes, b0, b1)

        for s in range(n_samples):
            for _, ws in self._eval_passes(group_indices_list, batch_size, drop_last, noise_fn if _noise_fn is not None else None):
                outs = [torch.empty(1, ws[g].B, genes[g], dtype=torch.float32, device=eng.device) for g in (0, 1)]
                eng.decode_sample(outs, seed, draw0=passes)
                passes += 1
                for g in (0, 1):
                    t = outs[g][0]
                    res[g][s].append((t if sel[g] is None else t.index_select(1, sel[g])).cpu())
        out = {}
        for g in (0, 1):
            draws = [torch.cat(res[g][s]).numpy()[:n[g]] for s in range(n_samples)]
            out[g] = draws[0] if n_samples == 1 else np.stack(draws, axis=-1)
        return out

    def get_loadings(self) -> dict:
        """reference model/spvipes.py:652-677"""
        out = {}
        for g in (0, 1):
            names = list(self.adata.uns["groups_var_names"].values())[g]
            for kind, dim in (("shared", self.n_dimensions_shared), ("private", self.n_dimensions_private)):
                w = self.module.get_loadings(g, kind)
                out[(g, kind)] = pd.DataFrame(w, index=names, columns=[f"Z_{kind}_{i}" for i in range(w.shape[1])])
        return out
