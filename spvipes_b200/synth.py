"""Synthetic NB-sampled count matrices of the BASELINE.json shapes (SURVEY.md section 8d recipe).

Per group g: per-label gene-mean profiles softmax(N(0, 1.5^2)), library sizes LogNormal(log 3000, 0.5), inverse
dispersions LogNormal(0, 0.5); counts ~ Gamma-Poisson; stored as uint16 (clipped).  Labels: uniform over n_labels
(seed 99 + g).  Generated on the given device in row chunks so that the 2 x 1M x 20k case never holds an f32 copy.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Tuple

import torch


@dataclass
class SynthData:
    X: List[torch.Tensor]        # per group uint16 [N_g, G_g] (make_counts_csr: engine.CsrCounts)
    labels: List[torch.Tensor]   # per group int32 [N_g]
    n_labels: int


def _group_chunks(g, N, G, n_labels, device, seed, chunk):
    """(labels, iterator over (r0, r1, int32 counts [r1 - r0, G])) of group g, in the order that fixes the random streams"""
    gen = torch.Generator(device=device).manual_seed(seed + g)
    prof = torch.softmax(1.5 * torch.randn(n_labels, G, generator=gen, device=device), dim=1)
    theta = torch.exp(0.5 * torch.randn(G, generator=gen, device=device))
    lgen = torch.Generator(device=device).manual_seed(99 + g)
    labels = torch.randint(0, n_labels, (N,), generator=lgen, device=device, dtype=torch.int32)

    def chunks():
        for r0 in range(0, N, chunk):
            r1 = min(N, r0 + chunk)
            lib = torch.exp(torch.log(torch.tensor(3000.0, device=device)) + 0.5 * torch.randn(r1 - r0, 1, generator=gen, device=device))
            mean = prof[labels[r0:r1].long()] * lib
            # Gamma-Poisson: rate ~ Gamma(shape theta, scale mean / theta)
            gam = torch._standard_gamma(theta.expand(r1 - r0, G).contiguous(), generator=gen)
            rate = gam * (mean / theta)
            cnt = torch.poisson(rate, generator=gen).clamp_(max=65535.0)
            yield r0, r1, cnt.to(torch.int32)
    return labels, chunks()


def make_counts(n_cells: Tuple[int, int], genes: Tuple[int, int], n_labels: int = 10, device="cuda", seed: int = 1234,
                chunk: int = 8192) -> SynthData:
    Xs, Ls = [], []
    for g in (0, 1):
        N, G = int(n_cells[g]), int(genes[g])
        labels, chunks = _group_chunks(g, N, G, n_labels, device, seed, chunk)
        X = torch.empty(N, G, dtype=torch.uint16, device=device)
        for r0, r1, cnt in chunks:
            X[r0:r1] = cnt.to(torch.uint16)
        Xs.append(X)
        Ls.append(labels)
    return SynthData(Xs, Ls, n_labels)


def make_counts_csr(n_cells: Tuple[int, int], genes: Tuple[int, int], n_labels: int = 10, device="cuda", seed: int = 1234,
                    chunk: int = 8192) -> SynthData:
    """make_counts with the same recipe, seeds and chunk order, each group stored as an engine.CsrCounts: every chunk is
    converted to CSR where it was sampled, so no more than one dense chunk exists at a time (2 x 4 M cells x 20 k genes
    fit in 66 GB of HBM instead of 320 GB).  Densified, X equals make_counts' X exactly."""
    from .engine import CsrCounts
    Xs, Ls = [], []
    for g in (0, 1):
        N, G = int(n_cells[g]), int(genes[g])
        if G > 65536:
            raise ValueError(f"uint16 column indices hold at most 65536 genes, got {G}")
        labels, chunks = _group_chunks(g, N, G, n_labels, device, seed, chunk)
        counts, idx, val = [torch.zeros(1, dtype=torch.int64, device=device)], [], []
        for r0, r1, cnt in chunks:
            nz = cnt != 0
            counts.append(nz.sum(1, dtype=torch.int64))
            idx.append(nz.nonzero()[:, 1].to(torch.int32).to(torch.uint16))  # row-major order: sorted columns per row
            val.append(cnt[nz].to(torch.uint16))
            del nz, cnt
        indptr = torch.cumsum(torch.cat(counts), 0)
        Xs.append(CsrCounts(indptr, torch.cat(idx), torch.cat(val), (N, G)))
        del idx, val
        Ls.append(labels)
    return SynthData(Xs, Ls, n_labels)


def make_plan(n0: int, n1: int, labels0: torch.Tensor, labels1: torch.Tensor, n_labels: int, device="cuda", seed: int = 7,
              tau: float = 4.0, dtype=torch.float32) -> torch.Tensor:
    """dense OT-like plan T[i, j] = exp(-|u_i - v_j|^2 / tau) from 8-dim label-centred Gaussian embeddings; dtype bfloat16
    halves its residency (200k x 200k: 80 GB instead of 160 GB)"""
    gen = torch.Generator(device=device).manual_seed(seed)
    centres = 3.0 * torch.randn(n_labels, 8, generator=gen, device=device)
    u = centres[labels0.long()] + torch.randn(n0, 8, generator=gen, device=device)
    v = centres[labels1.long()] + torch.randn(n1, 8, generator=gen, device=device)
    T = torch.empty(n0, n1, dtype=dtype, device=device)
    for r0 in range(0, n0, 4096):
        r1 = min(n0, r0 + 4096)
        T[r0:r1] = torch.exp(-torch.cdist(u[r0:r1], v) ** 2 / tau).to(dtype)
    return T
