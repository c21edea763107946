"""Training loop around StepEngine: minibatch index schedule with the reference's semantics, device-resident or
host-fed minibatches, KL warm-up and the optimiser step.

Index semantics restated from the reference (bit-exact contract, SURVEY.md section 8a row a1):
  * split: np.random.RandomState(seed).permutation per group, in group order; val first, then train
    (data/_multi_datasplitter.py:65-85; n_train = ceil(train_size * n), scvi validate_data_split)
  * per epoch and group: a BatchSampler(RandomSampler) over the train subset, batch_size B, drop_last=True
    (dataloaders/_ann_dataloader.py:85-92); RandomSampler draws its seed from the global torch CPU RNG and then
    torch.randperm(n, generator=...)
  * the group with fewer batches is replayed with itertools.cycle, i.e. its FIRST pass is cached and repeated
    (dataloaders/_concat_dataloader.py:108-110)
  * kl_weight = min(1, epoch / n_epochs_kl_warmup) (scvi TrainingPlan, model/base/training_mixin.py:93-101)
"""
from __future__ import annotations

import math
import os
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from .engine import GroupBatch, Noise, StepEngine


def validate_data_split(n: int, train_size: float, validation_size: Optional[float] = None) -> Tuple[int, int]:
    """scvi.dataloaders._data_splitting.validate_data_split (0.20.0)"""
    n_train = math.ceil(train_size * n)
    n_val = n - n_train if validation_size is None else math.floor(n * validation_size)
    return n_train, n_val


def split_indices(group_indices_list: Sequence[np.ndarray], train_size=0.9, validation_size=None, seed=0):
    """reference data/_multi_datasplitter.py:65-79 -> (train, val, test) index lists per group"""
    rs = np.random.RandomState(seed=seed)
    train, val, test = [], [], []
    for gi in group_indices_list:
        gi = np.asarray(gi)
        n_train, n_val = validate_data_split(len(gi), train_size, validation_size)
        perm = rs.permutation(gi)
        val.append(perm[:n_val])
        train.append(perm[n_val:n_val + n_train])
        test.append(perm[n_val + n_train:])
    return train, val, test


def _random_sampler_perm(n: int) -> torch.Tensor:
    """torch.utils.data.RandomSampler.__iter__ (replacement=False, generator=None): seed from the global CPU RNG"""
    seed = int(torch.empty((), dtype=torch.int64).random_().item())
    gen = torch.Generator()
    gen.manual_seed(seed)
    return torch.randperm(n, generator=gen)


def epoch_batches(train_idx: Sequence[np.ndarray], batch_size: int, shuffle=True, drop_last=True) -> List[List[np.ndarray]]:
    """one epoch of ConcatDataLoader: list over steps of [rows_group0, rows_group1] (global row ids).
    The global torch CPU RNG is consumed exactly as the reference's loader stack consumes it
    (dataloaders/_concat_dataloader.py:108-110 on top of torch.utils.data): creating each DataLoader iterator draws one
    int64 (its base seed) — the cycled loaders when `cycle(dl)` is built, the largest when zip() starts — and only then, at
    the first batch, each RandomSampler draws its own seed in list order and builds torch.randperm from it.
    tests/test_index_semantics.py checks this against the real torch DataLoader / BatchSampler / RandomSampler classes."""
    per_group = []
    if shuffle is not None:  # one base-seed draw per DataLoader iterator (shuffled or not)
        for _ in train_idx:
            torch.empty((), dtype=torch.int64).random_()
    for idx in train_idx:
        n = len(idx)
        order = _random_sampler_perm(n).numpy() if shuffle else np.arange(n)
        nb = n // batch_size if drop_last else math.ceil(n / batch_size)
        per_group.append([np.asarray(idx)[order[k * batch_size:(k + 1) * batch_size]] for k in range(nb)])
    lens = [len(p) for p in per_group]
    largest = int(np.argmax(lens))
    steps = lens[largest]
    out = []
    for s in range(steps):
        out.append([per_group[g][s] if g == largest else per_group[g][s % lens[g]] for g in range(len(per_group))])
    return out


class TrainLoop:
    """fwd + bwd + Adam per minibatch on one GPU (one process per GPU; see parallel.py for the data-parallel wrapper)."""

    def __init__(self, engine: StepEngine, lr=1e-3, eps=0.01, weight_decay=1e-6, n_epochs_kl_warmup=400):
        self.engine = engine
        self.lr, self.eps, self.weight_decay = lr, eps, weight_decay
        self.n_epochs_kl_warmup = n_epochs_kl_warmup
        self.epoch = 0
        self.grad_sync = None  # optional callable(engine) run between backward and the optimiser step (data parallel)
        self._dp_stream = None
        # this loop owns the optimiser step: Adam also refreshes the bf16 tensor-core copies of the large weights
        # (largest staged block must stay below 2^24 elements, the range of the kernel's index arithmetic)
        if engine.bf16 and max(engine.d.genes) * max(engine.d.KMIX, 2 * engine.d.n_hidden) < (1 << 24):
            engine.stage_in_adam = True

    def set_epoch(self, epoch: int):
        self.epoch = epoch
        w = 1.0 if not self.n_epochs_kl_warmup else min(1.0, epoch / self.n_epochs_kl_warmup)
        self.engine.set_kl_weight(w)

    def step(self, batches: Sequence[GroupBatch], noise: Optional[Noise] = None):
        e = self.engine
        e.forward(batches, training=True, noise=noise)
        if self.grad_sync is None:  # single GPU: the optimiser step is interleaved with the backward
            e.backward(adam={"lr": self.lr, "eps": self.eps, "weight_decay": self.weight_decay})
        elif getattr(self.grad_sync, "in_graph", False):
            self._step_nvlink(e)
        else:  # data parallel: the decoder range is all-reduced while the encoder backward runs
            from .engine import PHASE_DEC, PHASE_ENC
            e.backward(stage="decoder", tick=True)
            self.grad_sync.start(e, PHASE_DEC)
            e.backward(stage="encoder")
            self.grad_sync.start(e, PHASE_ENC)
            gs = self.grad_sync.finish()
            for ph in (PHASE_DEC, PHASE_ENC):
                e.adam_range_step(ph, lr=self.lr, eps=self.eps, weight_decay=self.weight_decay, grad_scale=gs)
        return e.loss_terms()

    def _step_nvlink(self, e):
        """backward + gradient all-reduce + Adam of the data-parallel step, every launch on CUDA streams (capturable as one
        graph): decoder / PoE backward -> on a side stream [all-reduce of the decoder range (csrc/xgpu.cu) -> Adam on it] beside
        the encoder backward -> per group, as soon as its encoder backward ends, [all-reduce of the group's encoder range -> Adam
        on it] on the group's stream (the first group's exchange and update run beside the other group's first-layer weight
        gradient).  Adam folds the 1 / world factor.  Channels: 0 decoder range, 1 / 2 the groups' encoder ranges; every rank
        replays the same graph, so the launch order per channel is the same everywhere."""
        from .engine import PHASE_DEC, PHASE_ENC
        gs, dev = self.grad_sync, e.device
        kw = {"lr": self.lr, "eps": self.eps, "weight_decay": self.weight_decay, "grad_scale": 1.0 / gs.world}
        e.backward(stage="decoder", tick=True)
        main = torch.cuda.current_stream(dev)
        if self._dp_stream is None:
            self._dp_stream = torch.cuda.Stream(device=dev)
        fork, done = torch.cuda.Event(), torch.cuda.Event()
        fork.record(main)
        self._dp_stream.wait_event(fork)
        with torch.cuda.stream(self._dp_stream):
            gs.allreduce(PHASE_DEC, 0, blocks=int(os.environ.get("SPV_DP_BLOCKS_DEC", "8")))
            e.adam_range_step(PHASE_DEC, **kw)
            done.record(self._dp_stream)
        nb_enc = int(os.environ.get("SPV_DP_BLOCKS_ENC", "16"))
        if os.environ.get("SPV_DP_ENC_SPLIT", "1") == "1":
            enc = e.params.group_ranges[PHASE_ENC]
            e.backward(stage="encoder", adam=dict(kw, enc_only=True, sync=lambda g: gs.allreduce_range(enc[g][0], enc[g][1], 1 + g, blocks=nb_enc)))
        else:  # A/B: the whole encoder range in one exchange after both groups' backward
            e.backward(stage="encoder")
            gs.allreduce(PHASE_ENC, 1, blocks=nb_enc)
            e.adam_range_step(PHASE_ENC, **kw)
        main.wait_event(done)

    def capture(self, batches: Sequence[GroupBatch], noise: Optional[Noise] = None) -> "torch.cuda.CUDAGraph":
        """record one step (every kernel launch of forward, backward, gradient sync and Adam) into a CUDA graph.
        `batches` must reference STATIC device buffers (count matrix, row-index buffer, labels): the caller refreshes their
        contents before each replay.  Steps are launch-latency bound at the BASELINE shapes (~100 kernels of 2-100 us),
        so replaying a graph instead of issuing the launches from Python is what keeps the GPU busy.
        Engine state (parameters, Adam moments, BatchNorm running statistics, step counter) is restored after the
        warm-up launches that precede the capture, so capturing does not advance training."""
        e = self.engine
        keep = [e.params.flat.clone(), e.buffers.flat.clone(), (e.step_dev.clone(), e.noise_dev.clone()),
                None if e.adam_m is None else e.adam_m.clone(), None if e.adam_v is None else e.adam_v.clone()]
        cur = torch.cuda.current_stream(e.device)
        side = torch.cuda.Stream(device=e.device)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for _ in range(2):
                self.step(batches, noise)
        cur.wait_stream(side)
        torch.cuda.synchronize(e.device)
        if self.grad_sync is None or getattr(self.grad_sync, "in_graph", False):
            # (data parallel over NVLink: the all-reduce kernels are part of the graph - every rank replays the same launch order)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                self.step(batches, noise)
        else:
            # data parallel: forward + decoder/PoE backward, encoder backward and the two halves of the optimiser step are four
            # graphs; the two gradient all-reduces are issued eagerly between the replays (collectives stay out of capture)
            from .engine import PHASE_DEC, PHASE_ENC
            g1, g2, g3, g4 = (torch.cuda.CUDAGraph() for _ in range(4))
            scale = 1.0 / self.grad_sync.world
            with torch.cuda.graph(g1):
                e.forward(batches, training=True, noise=noise)
                e.backward(stage="decoder", tick=True)
            with torch.cuda.graph(g2):
                e.backward(stage="encoder")
            with torch.cuda.graph(g3):
                e.adam_range_step(PHASE_DEC, lr=self.lr, eps=self.eps, weight_decay=self.weight_decay, grad_scale=scale)
            with torch.cuda.graph(g4):
                e.adam_range_step(PHASE_ENC, lr=self.lr, eps=self.eps, weight_decay=self.weight_decay, grad_scale=scale)
            graph = _SyncedGraphs(g1, g2, g3, g4, self.grad_sync, e)
        torch.cuda.synchronize(e.device)
        e.params.flat.copy_(keep[0]); e.buffers.flat.copy_(keep[1]); e.step_dev.copy_(keep[2][0]); e.noise_dev.copy_(keep[2][1])
        if keep[3] is None:
            e.adam_m.zero_(); e.adam_v.zero_()
        else:
            e.adam_m.copy_(keep[3]); e.adam_v.copy_(keep[4])
        e.stage_weights()  # the restore above went through torch: bring the bf16 operand copies back in line
        return graph


class _SyncedGraphs:
    """replay(): [forward + decoder/PoE backward] -> all-reduce(decoder range, async) -> [encoder backward] on the main
    stream while a side stream waits for that all-reduce and runs [Adam, decoder range] -> all-reduce(encoder range) ->
    [Adam, encoder range]"""

    def __init__(self, g_dec, g_enc, g_opt_dec, g_opt_enc, grad_sync, engine):
        self.g_dec, self.g_enc, self.g_opt_dec, self.g_opt_enc = g_dec, g_enc, g_opt_dec, g_opt_enc
        self.grad_sync, self.engine = grad_sync, engine
        self.side = torch.cuda.Stream(device=engine.device)

    def replay(self):
        from .engine import PHASE_DEC, PHASE_ENC
        main = torch.cuda.current_stream(self.engine.device)
        self.g_dec.replay()
        self.grad_sync.start(self.engine, PHASE_DEC)
        with torch.cuda.stream(self.side):  # decoder half of the optimiser step beside the encoder backward
            self.grad_sync.finish()
            self.g_opt_dec.replay()
        self.g_enc.replay()
        self.grad_sync.start(self.engine, PHASE_ENC)
        self.grad_sync.finish()
        main.wait_stream(self.side)
        self.g_opt_enc.replay()
        self.engine.note_replay(forward=True)
        self.engine.note_replay(forward=False)
        self.side.wait_stream(main)  # the next replay's decoder-range Adam must not start before this step is done


def init_params(engine: StepEngine, seed: int = 0):
    """reference default initialisation, restated: nn.Linear -> U(+-1/sqrt(fan_in)) for weight and bias
    (kaiming_uniform(a=sqrt(5))), BatchNorm weight 1 / bias 0, px_r ~ N(0, 1) (module/spVIPESmodule.py:115-117)."""
    gen = torch.Generator().manual_seed(seed)
    sd = {}
    for name in engine.params.names():
        v = engine.params.view(name)
        shape = tuple(v.shape)
        if name.startswith("px_r"):
            t = torch.randn(shape, generator=gen)
        elif ".1.weight" in name:  # BatchNorm affine
            t = torch.ones(shape)
        elif ".1.bias" in name:
            t = torch.zeros(shape)
        elif name.endswith("weight"):
            bound = 1.0 / math.sqrt(shape[1])
            t = (torch.rand(shape, generator=gen) * 2 - 1) * bound
        else:  # Linear bias: fan_in of the matching weight
            wname = name[:-4] + "weight"
            fan_in = engine.params.view(wname).shape[1]
            t = (torch.rand(shape, generator=gen) * 2 - 1) / math.sqrt(fan_in)
        sd[name] = t
    for name in engine.buffers.names():
        v = engine.buffers.view(name)
        sd[name] = torch.ones(v.shape) if name.endswith("running_var") else torch.zeros(v.shape)
    engine.load_state_dict(sd)
    return sd
