"""Host-side orchestration of one spVIPES training step on a B200: flat parameter layout, workspaces and the
sequence of C-ABI kernel launches for inference -> generative -> loss, their backward and Adam.

Mirrors reference module/spVIPESmodule.py:425-472 (inference), :720-771 (generative), :809-899 (loss) and
nn/networks.py (Encoder, LinearDecoderSPVIPE); the optimiser restates scvi TrainingPlan's defaults
(model/base/training_mixin.py:93-111: Adam lr 1e-3, eps 0.01, weight_decay 1e-6).

torch is used for device memory and streams only; every arithmetic step is a launch into libspvipes_b200.so.
"""
from __future__ import annotations

import contextlib
import math
from collections import OrderedDict
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _lib as L

HD = 256  # decoder hidden width is fixed (reference nn/networks.py:194, quirk Q8)
ENC_BN_EPS, ENC_BN_MOM = 1e-5, 0.1
DEC_BN_EPS, DEC_BN_MOM = 1e-3, 0.01
# grid cap of the decoder-range Adam update that overlaps the encoder backward (measured optimum on B200 at C5, DESIGN.md section 5)
ADAM_OVERLAP_BLOCKS = 296


# ------------------------------------------------------------------------------------------------
# flat parameter layout (names follow the reference state_dict so checkpoints load 1:1)
# ------------------------------------------------------------------------------------------------
@dataclass
class Dims:
    genes: Tuple[int, int]
    n_hidden: int = 128
    n_shared: int = 25
    n_private: int = 10
    n_batch: int = 0   # batch covariate: its one-hot code (n_batch columns) is appended to the input of the encoders' first layer
                       # and of the four decoder nets when n_batch > 1 (reference nn/networks.py:60-68, scvi FCLayers)

    @property
    def nb(self):
        return self.n_batch if self.n_batch > 1 else 0

    @property
    def KZ(self):   # latent columns [z_private_arg | z_shared_arg]
        return self.n_shared + self.n_private

    @property
    def KMIX(self):  # input width of the mixture layer and row width of amix = [hm | zz | covariates]
        return HD + self.KZ + self.nb

    @property
    def Pb(self):   # input width of the private factor regressor
        return self.n_private + self.nb

    @property
    def Sb(self):
        return self.n_shared + self.nb

    @property
    def KZb(self):  # [z_private_arg | covariates | z_shared_arg | covariates]: the two regressors' inputs side by side
        return self.KZ + 2 * self.nb

    @property
    def NST(self):
        return 2 * self.n_shared + 2 * self.n_private


PHASE_ENC, PHASE_DEC = 0, 1
# per-element decoder outputs of decode_elements, in the order of the kernels' output array (include/spvipes_b200.h)
ELEM_OUTPUTS = ("ll", "rate_p", "rate_s", "pi", "mean")
_ENCODER_BLOCKS = ("W1", "b1", "W2", "b2", "Whp", "Whs", "bhd", "ghd", "bthd")


def _group_param_entries(g: int, G: int, d: Dims):
    """[(fused name, shape, [(state_dict name, row slice / index)])] in flat order for group g."""
    H, S, P, KZ, KMIX, NST = d.n_hidden, d.n_shared, d.n_private, d.KZ, d.KMIX, d.NST
    ep, es, dec = f"encoder_{g}_private", f"encoder_{g}_shared", f"decoder_{g}"
    fl = "fc_layers.Layer 0"
    Gc = G + d.nb  # the covariate columns sit behind the genes / the latents in every first-layer weight
    return [
        ("W1", (2 * H, Gc), [(f"{ep}.fc1.weight", (0, H)), (f"{es}.fc1.weight", (H, 2 * H))]),
        ("b1", (2 * H,), [(f"{ep}.fc1.bias", (0, H)), (f"{es}.fc1.bias", (H, 2 * H))]),
        ("W2", (2 * H, H), [(f"{ep}.fc2.weight", (0, H)), (f"{es}.fc2.weight", (H, 2 * H))]),
        ("b2", (2 * H,), [(f"{ep}.fc2.bias", (0, H)), (f"{es}.fc2.bias", (H, 2 * H))]),
        ("Whp", (2 * P, H), [(f"{ep}.mu_encoder.0.weight", (0, P)), (f"{ep}.lvar_encoder.0.weight", (P, 2 * P))]),
        ("Whs", (2 * S, H), [(f"{es}.mu_encoder.0.weight", (0, S)), (f"{es}.lvar_encoder.0.weight", (S, 2 * S))]),
        ("bhd", (NST,), [(f"{ep}.mu_encoder.0.bias", (0, P)), (f"{ep}.lvar_encoder.0.bias", (P, 2 * P)),
                         (f"{es}.mu_encoder.0.bias", (2 * P, 2 * P + S)), (f"{es}.lvar_encoder.0.bias", (2 * P + S, NST))]),
        ("ghd", (NST,), [(f"{ep}.mu_encoder.1.weight", (0, P)), (f"{ep}.lvar_encoder.1.weight", (P, 2 * P)),
                         (f"{es}.mu_encoder.1.weight", (2 * P, 2 * P + S)), (f"{es}.lvar_encoder.1.weight", (2 * P + S, NST))]),
        ("bthd", (NST,), [(f"{ep}.mu_encoder.1.bias", (0, P)), (f"{ep}.lvar_encoder.1.bias", (P, 2 * P)),
                          (f"{es}.mu_encoder.1.bias", (2 * P, 2 * P + S)), (f"{es}.lvar_encoder.1.bias", (2 * P + S, NST))]),
        ("Wp", (G, d.Pb), [(f"{dec}.factor_regressor_private.{fl}.0.weight", None)]),
        ("gp", (G,), [(f"{dec}.factor_regressor_private.{fl}.1.weight", None)]),
        ("bp", (G,), [(f"{dec}.factor_regressor_private.{fl}.1.bias", None)]),
        ("Ws", (G, d.Sb), [(f"{dec}.factor_regressor_shared.{fl}.0.weight", None)]),
        ("gs", (G,), [(f"{dec}.factor_regressor_shared.{fl}.1.weight", None)]),
        ("bs", (G,), [(f"{dec}.factor_regressor_shared.{fl}.1.bias", None)]),
        ("Wh", (HD, KZ + d.nb), [(f"{dec}.sigmoid_decoder.{fl}.0.weight", None)]),
        ("bh", (HD,), [(f"{dec}.sigmoid_decoder.{fl}.0.bias", None)]),
        ("gh", (HD,), [(f"{dec}.sigmoid_decoder.{fl}.1.weight", None)]),
        ("bth", (HD,), [(f"{dec}.sigmoid_decoder.{fl}.1.bias", None)]),
        ("Wm", (G, KMIX), [(f"{dec}.mixture.{fl}.0.weight", None)]),
        ("bm", (G,), [(f"{dec}.mixture.{fl}.0.bias", None)]),
        ("px_r", (G,), [(f"px_r.{g}", None)]),
    ]


def _group_buffer_entries(g: int, G: int, d: Dims):
    S, P, NST = d.n_shared, d.n_private, d.NST
    ep, es, dec = f"encoder_{g}_private", f"encoder_{g}_shared", f"decoder_{g}"
    fl = "fc_layers.Layer 0"
    out = []
    for kind in ("running_mean", "running_var"):
        tag = "rm" if kind == "running_mean" else "rv"
        out += [
            (f"{tag}_hd", (NST,), [(f"{ep}.mu_encoder.1.{kind}", (0, P)), (f"{ep}.lvar_encoder.1.{kind}", (P, 2 * P)),
                                   (f"{es}.mu_encoder.1.{kind}", (2 * P, 2 * P + S)), (f"{es}.lvar_encoder.1.{kind}", (2 * P + S, NST))]),
            (f"{tag}_p", (G,), [(f"{dec}.factor_regressor_private.{fl}.1.{kind}", None)]),
            (f"{tag}_s", (G,), [(f"{dec}.factor_regressor_shared.{fl}.1.{kind}", None)]),
            (f"{tag}_h", (HD,), [(f"{dec}.sigmoid_decoder.{fl}.1.{kind}", None)]),
        ]
    return out


class FlatStore:
    """one flat fp32 tensor + named views (fused blocks per group, and reference state_dict names)"""

    def __init__(self, entries_per_group, device, phase_of=None):
        """phase_of(name) -> int: blocks are laid out phase by phase (all groups' phase-0 blocks, then phase 1, ...), so that
        e.g. every encoder parameter and every decoder parameter form one contiguous range each (`self.ranges[phase]`,
        per group `self.group_ranges[phase][g]`): the data-parallel step all-reduces a whole phase with one call."""
        self.offsets: List[Dict[str, Tuple[int, Tuple[int, ...]]]] = [dict() for _ in entries_per_group]
        self.sd_index: "OrderedDict[str, Tuple[int, str, Optional[Tuple[int, int]]]]" = OrderedDict()
        phases = sorted({(phase_of(n) if phase_of else 0) for entries in entries_per_group for n, _, _ in entries})
        self.ranges: Dict[int, Tuple[int, int]] = {}
        self.group_ranges: Dict[int, List[Tuple[int, int]]] = {}
        off = 0
        for ph in phases:
            lo_ph = off
            self.group_ranges[ph] = []
            for g, entries in enumerate(entries_per_group):
                lo_g = off
                for name, shape, subs in entries:
                    if (phase_of(name) if phase_of else 0) != ph:
                        continue
                    self.offsets[g][name] = (off, shape)
                    off += (int(math.prod(shape)) + 3) // 4 * 4  # keep every block 16-byte aligned
                self.group_ranges[ph].append((lo_g, off))
            self.ranges[ph] = (lo_ph, off)
        for g, entries in enumerate(entries_per_group):  # state_dict key order: group by group, as the reference registers them
            for name, shape, subs in entries:
                for sd_name, sl in subs:
                    self.sd_index[sd_name] = (g, name, sl)
        self.numel = off
        self.flat = torch.zeros(off, dtype=torch.float32, device=device)

    def block(self, g: int, name: str, flat: Optional[torch.Tensor] = None) -> torch.Tensor:
        off, shape = self.offsets[g][name]
        base = self.flat if flat is None else flat
        return base[off:off + int(math.prod(shape))].view(shape)

    def view(self, sd_name: str, flat: Optional[torch.Tensor] = None) -> torch.Tensor:
        g, name, sl = self.sd_index[sd_name]
        blk = self.block(g, name, flat)
        return blk if sl is None else blk[sl[0]:sl[1]]

    def names(self):
        return list(self.sd_index.keys())


# ------------------------------------------------------------------------------------------------
def _count_dtype(values) -> "np.dtype":
    """uint16 when every value is an integer in [0, 65535], float32 otherwise (the rule of the dense model path)"""
    import numpy as np
    v = np.asarray(values)
    if v.size == 0:
        return np.dtype(np.uint16)
    if v.dtype.kind in "ui":
        return np.dtype(np.uint16) if v.min() >= 0 and v.max() <= 65535 else np.dtype(np.float32)
    return np.dtype(np.uint16) if np.all(v == np.round(v)) and v.min() >= 0 and v.max() <= 65535 else np.dtype(np.float32)


@dataclass
class CsrCounts:
    """one group's count matrix [N, G] as device-resident CSR: a minibatch is gathered into a dense staging tile by
    spv_csr_gather, so the matrix itself takes 4 bytes per nonzero (uint16 values) instead of 2 G bytes per row.
    Canonical: every row's columns sorted and distinct, no stored zeros."""
    indptr: torch.Tensor    # int64 [N + 1]
    indices: torch.Tensor   # uint16 [nnz] column indices
    values: torch.Tensor    # uint16 or float32 [nnz]
    shape: Tuple[int, int]

    @property
    def dtype(self):
        return self.values.dtype

    @staticmethod
    def canonical_arrays(mat):
        """host side of from_scipy: (indptr int64, indices uint16, values uint16 | float32, shape) of a scipy sparse matrix, with
        duplicate entries summed (scipy's meaning of them), explicit zeros dropped and the columns of every row sorted"""
        import numpy as np
        import scipy.sparse as sp
        m = sp.csr_matrix(mat, copy=True)
        m.sum_duplicates()  # also sorts the indices
        m.eliminate_zeros()
        N, G = (int(x) for x in m.shape)
        data = m.data
        if data.dtype.kind == "f" and data.dtype != np.float32:
            data = data.astype(np.float32)  # the dtype rule looks at the values the kernels will see
        dt = _count_dtype(data)
        limit = int(L.load().spv_csr_max_genes(L.SRC_U16_LOG1P if dt == np.uint16 else L.SRC_F32_LOG1P))
        if G > limit:
            raise ValueError(f"a CSR count matrix with {dt.name} values holds at most {limit} genes (a row is assembled in "
                             f"shared memory), got {G}")
        return (m.indptr.astype(np.int64), m.indices.astype(np.uint16), data.astype(dt), (N, G))

    @classmethod
    def from_scipy(cls, mat, device="cuda") -> "CsrCounts":
        indptr, indices, values, shape = cls.canonical_arrays(mat)
        up = lambda a: torch.from_numpy(a).to(device)
        return cls(up(indptr), up(indices), up(values), shape)

    def resident_bytes(self) -> int:
        return sum(t.numel() * t.element_size() for t in (self.indptr, self.indices, self.values))


@dataclass
class GroupBatch:
    """one group's minibatch: a device-resident count matrix plus optional row-gather indices"""
    X: object                             # [N, ld] uint16 or float32 counts (device tensor); columns col0 .. col0+G are this group's
                                          # genes; or a CsrCounts of the group's own genes (col0 = 0)
    rows: Optional[torch.Tensor] = None   # int32 [B] row indices into X, or None for X[:B]
    col0: int = 0
    labels: Optional[torch.Tensor] = None  # int32 [B] cell-type labels (label mode) or cluster labels (cluster mode)
    idx: Optional[torch.Tensor] = None     # int32 [B] within-group indices into the transport plan
    B: Optional[int] = None
    labels_per_cell: bool = False          # labels (and idx) are indexed by X's row, i.e. gathered with `rows`
    batch: Optional[torch.Tensor] = None   # int32 [B] batch codes of the minibatch (n_batch > 1 only)

    def batch_size(self):
        if self.B is not None:
            return self.B
        return int(self.rows.shape[0]) if self.rows is not None else int(self.X.shape[0])  # (a CsrCounts has .shape too)


@dataclass
class Noise:
    """explicit reparameterisation noise / dropout multipliers (parity tests); None -> in-kernel Philox"""
    eps_private: Optional[Sequence[torch.Tensor]] = None   # per group [B, P]
    eps_poe: Optional[Sequence[torch.Tensor]] = None       # per group [B, S]
    drop: Optional[Sequence[torch.Tensor]] = None          # per group [B, 2H] multipliers (private | shared)


class _GroupWS:
    def __init__(self, B, G, d: Dims, dev, with_grad: bool, bf16: bool = False, wb=None, fused=False):
        H, S, P, KZ, KMIX, NST = d.n_hidden, d.n_shared, d.n_private, d.KZ, d.KMIX, d.NST
        f = lambda *s: torch.empty(*s, dtype=torch.float32, device=dev)
        self.B, self.G = B, G
        self.xs = None
        self.nTG, self.nTB = (G + 63) // 64, (B + 63) // 64
        self.lib = f(B)
        self.h1, self.h2 = f(B, 2 * H), f(B, 2 * H)
        self.r, self.stats = f(B, NST), f(B, NST)
        self.bn_hd_mean, self.bn_hd_istd = f(NST), f(NST)
        self.zpriv, self.zpoe = f(B, P), f(B, S)
        self.poe_loc, self.poe_lv, self.poe_scale = f(B, S), f(B, S), f(B, S)
        self.klp, self.klq, self.rec = f(B), f(B), f(B)
        self.partner = torch.empty(B, dtype=torch.int32, device=dev)
        nb, KZb = d.nb, d.KZb
        self.amix = torch.zeros(B, KMIX, dtype=torch.float32, device=dev)
        self.zzb = f(B, KZb) if nb else None      # [z_private_arg | oh | z_shared_arg | oh] (batch covariates)
        self.oh = f(B, nb) if nb and not bf16 else None  # one-hot batch codes (fp32 path of the encoders' first layer)
        self.zsum, self.zmean, self.zcov = f(KZb), f(KZb), f(KZb, KZb)
        # scratch of the latent statistics (spv_dec_fold, minibatches > 512 rows): per 64-row tile, column sums + centred second moments
        self.cov_part = torch.zeros(self.nTB, KZb + KZb * KZb, dtype=torch.float32, device=dev)
        self.wfold, self.genec = f(G, KZb), f(L.GENEC_ROWS, G)
        self.ah = f(B, HD)
        self.bn_h_mean, self.bn_h_istd = f(HD), f(HD)
        self.part_stats = f(2 * self.nTG, B, 4)
        self.part_nb = f(max(2 * self.nTG * B * 3, int(L.load().spv_dec_nb_part_floats(B, G))))
        self.rowc = f(B, 4)
        self.pi = f(B, G)
        self.expert = f(B, 2 * S)  # cluster mode: plan-weighted expert statistics
        # split-K workspace: the largest user is fc1 forward (B x 2H) and d Amix (B x KMIX)
        self.splits_fc1 = max(1, min(16, G // 512))
        self.splits_g = max(1, min(32, G // 256))       # reductions over the gene axis with a small output
        self.splits_b = max(1, min(8, B // 64))         # reductions over the minibatch with a small output
        big = max(2 * H, KMIX)
        self.ws = f(max(32 * B * big, self.splits_b * G * KZb, 2 * self.splits_b * big * big, 1))
        self.ws2 = f(max(2 * self.splits_b * big * big, 1))  # split-K scratch of the auxiliary (weight-gradient) streams
        self.ws3 = f(max(2 * self.splits_b * big * big, 1))
        r8 = lambda x: (x + 7) // 8 * 8
        # Gp: gene pitch of the decoder operands; Gpe: pitch of the encoder operands (genes + covariate columns);
        # KMp: row pitch of the 16-bit [hm | zz | covariates] operand and of Wstack (whose folded-weight rows use columns
        # HD .. HD + KZb)
        self.Gp, self.Gpe, self.KMp = r8(G), r8(G + nb), r8(max(KMIX, HD + KZb))
        if bf16:
            h = lambda *s: torch.zeros(*s, dtype=torch.bfloat16, device=dev)
            hd = lambda *s: torch.zeros(*s, dtype=torch.float16 if fused else torch.bfloat16, device=dev)  # decoder operands
            self.amixb = hd(B, self.KMp)
            self.Tb, self.Tb_lo = h(B, self.Gpe), h(B, self.Gpe)  # log1p(counts) as a bf16 pair: the first layer's input
            # fp16 operands of the branch-logit MMAs (spv_dec_fold writes them): centred latents and folded weights
            self.zcb = torch.zeros(B, 64, dtype=torch.float16, device=dev)
            self.wzf = torch.zeros(2 * self.Gp, 64, dtype=torch.float16, device=dev)
            # count tables of the likelihood sweeps (spv_dec_theta_tables): [G, 16] float2 lgamma terms, [G, 16] digamma terms
            self.tgf = f(G, 16, 2)
            self.tb1 = f(G, 16) if (with_grad and fused) else None
            # bf16 weight operands are per engine (shared by every workspace): W1b [2H, Gp] and the stacked operand
            # Wstack [3 Gp, KMp]: rows [0, G) mixture weight, [Gp, Gp+G) / [2Gp, 2Gp+G) the folded private / shared
            # factor-regressor weights of the current minibatch in the latent columns (zero elsewhere)
            self.W1b, self.Wstack, self.W1b_lo = wb
            self.Wmb = self.Wstack[:G]
            if with_grad:
                self.dh1b, self.dh1b_lo = h(B, 2 * H), h(B, 2 * H)
                if fused:
                    # outputs of the training sweep (csrc/nb_tc_train.cu), gene-major fp16: E4T [Gp, 4 Bp] = (ep, rp', es, rs') per
                    # cell, DPIT [Gp, Bp] = d ll / d pi; and the small operands / results of the backward GEMMs
                    self.Bp = r8(B)
                    self.E4T, self.DPIT = hd(self.Gp * 4 * self.Bp), hd(self.Gp * self.Bp)
                    self.ldq4 = r8(KZb + 2)
                    self.ZQ4 = hd(4 * self.Bp, self.ldq4)
                    self.CQ = f(self.Gp, KZb + 2)        # [Qp | colsum dyp | Qs | colsum dys]
                    self.T4 = f(4 * self.Bp, KZb)
                    self.Wcomb = hd(self.Gp, r8(KZb))    # [W'p | W's] (fp16 copy of wfold)
                    self.tc_splits_dz4 = max(1, min(148 // ((4 * B + 127) // 128), (self.Gp + 63) // 64 // 2))
                else:
                    self.dpib = hd(B, self.Gp)  # d ll / d pi of spv_dec_nb_bwd (bf16): operand of the two mixture-weight GEMMs
            # split-K factors of the tensor-core GEMMs (128-wide tiles): fill the 148 SMs
            tiles = ((B + 127) // 128) * ((2 * H + 127) // 128)
            self.tc_splits_fc1 = max(1, min(148 // tiles, (G + 63) // 64 // 2))
            tiles = ((B + 127) // 128) * ((KMIX + 127) // 128)
            self.tc_splits_damix = max(1, min(148 // tiles, (G + 63) // 64 // 2))
        if with_grad:
            self.dyp, self.dys, self.dpi = f(B, G), f(B, G), f(B, G)
            self.colpart, self.colsum = f(self.nTB, 4, G), f(4, G)
            self.Qp, self.Qs = f(G, d.Pb), f(G, d.Sb)
            self.damix, self.dzraw, self.dzz = f(B, KMIX), f(B, KZb), f(B, KZ)
            self.dzzb = f(B, KZb) if nb else self.dzz
            self.dzraw_sum = f(KZb)
            self.nGB = L.load().spv_dec_gene_bwd_parts(G)
            self.vpart, self.mpart = f(self.nGB, KZb), f(self.nGB, KZb * KZb)  # per-CTA partials of spv_dec_gene_bwd
            self.dah = f(B, HD)
            self.dstats, self.dr = f(B, NST), f(B, NST)
            self.g_own, self.g_contrib, self.dexpert = f(B, 2 * S), f(B, 2 * S), f(B, 2 * S)
            self.dh2, self.dh1 = f(B, 2 * H), f(B, 2 * H)

    def need_xs(self, dtype, dev):
        """dense staging tile [B, Gp] of a CSR minibatch (spv_csr_gather): what every count consumer reads with rows = NULL"""
        if self.xs is None or self.xs.dtype != dtype:
            self.xs = torch.zeros(self.B, self.Gp, dtype=dtype, device=dev)
        return self.xs


class StepEngine:
    """fwd / bwd / Adam of the spVIPES step for two groups on one GPU."""

    def __init__(self, genes: Tuple[int, int], n_hidden=128, n_shared=25, n_private=10, dropout_rate=0.1, mode="label",
                 device="cuda", seed: int = 0, plan: Optional[torch.Tensor] = None, precision: str = "fp32", n_batch: int = 0):
        """precision: "fp32" = fp32 SIMT GEMMs everywhere (parity gate 1e-4); "bf16" = the large contractions (encoder fc1
        forward / weight gradient, decoder mixture GEMM forward / weight gradient / input gradient) run on the tcgen05
        tensor-core path with bf16 operands and fp32 accumulation (parity gate 1e-2, BASELINE.json north_star)."""
        if precision not in ("fp32", "bf16"):
            raise ValueError("precision must be 'fp32' or 'bf16'")
        self.precision = precision
        self.bf16 = precision == "bf16"
        # fused tcgen05 decoder-GEMMs + NB-likelihood kernel (bf16 mode); the latent columns must fit the 64-wide branch k-block
        # below its six additive columns (decoder_common.cuh ZK_MAX_LATENT); wider latents take the unfused bf16 decoder
        nb_cols = int(n_batch) if int(n_batch) > 1 else 0
        kz_dec = int(n_shared) + int(n_private) + 2 * nb_cols
        if kz_dec > L.DEC_MAX_LATENT:
            raise NotImplementedError(f"n_dimensions_shared + n_dimensions_private (+ 2 n_batch) = {kz_dec} is not implemented (the "
                                      f"decoder kernels take at most {L.DEC_MAX_LATENT} latent columns)")
        self.fused_nb = self.bf16 and kz_dec <= L.ZK_MAX_LATENT
        # one sweep over [B, G] per training step on the fused path: the forward sweep also emits what the backward needs
        # (csrc/nb_tc_train.cu)
        self.single_sweep = self.fused_nb
        # operands of the decoder GEMMs: fp16 on the fused path (2^-12 rounding, three bits more than bf16; every operand's range
        # is bounded: activations after BatchNorm, weights, gradients stored in natural units), bf16 on the unfused fallback
        self.dec_dtype = torch.float16 if self.fused_nb else torch.bfloat16
        self.dec_fmt = 3 if self.fused_nb else 0
        self.lib = L.load()
        self.d = Dims(tuple(int(x) for x in genes), int(n_hidden), int(n_shared), int(n_private), int(n_batch))
        if self.d.n_private > self.d.n_shared:
            # the reference's slicing of [private | poe] (c[:, :S], c[:, S:S+P]) is defined for P > S as well; this implementation's
            # zz column mapping covers P <= S (every BASELINE config and the reference's defaults, 10 / 25) - see INTEGRATION.md
            raise NotImplementedError("n_dimensions_private > n_dimensions_shared is not implemented (the kernels' latent column "
                                      "mapping covers n_dimensions_private <= n_dimensions_shared)")
        self.mode = mode
        self.mode_id = L.POE_MODES[mode]
        self.dropout_rate = float(dropout_rate)
        self.device = torch.device(device)
        self.seed = int(seed)
        # parameter layout: [encoders of group 0 | encoders of group 1 | decoders of group 0 | decoders of group 1]
        self.params = FlatStore([_group_param_entries(g, G, self.d) for g, G in enumerate(self.d.genes)], self.device,
                                phase_of=lambda n: PHASE_ENC if n in _ENCODER_BLOCKS else PHASE_DEC)
        self.buffers = FlatStore([_group_buffer_entries(g, G, self.d) for g, G in enumerate(self.d.genes)], self.device)
        for n in self.buffers.names():
            if n.endswith("running_var"):
                self.buffers.view(n).fill_(1.0)
        self.grads = torch.zeros_like(self.params.flat)
        self.adam_m: Optional[torch.Tensor] = None
        self.adam_v: Optional[torch.Tensor] = None
        self.step_dev = torch.zeros(1, dtype=torch.int32, device=self.device)   # Adam's t: only the optimiser kernels write it
        # counter of the Philox streams (reparameterisation noise, dropout masks): advanced once at the start of every
        # forward and left alone until the matching backward has regenerated its noise from it
        self.noise_dev = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._noise_events = []
        self.kl_weight = torch.ones(1, dtype=torch.float32, device=self.device)
        self.loss_out = torch.zeros(8, dtype=torch.float32, device=self.device)
        self.plan = plan
        self._ws: Dict[Tuple[int, int, bool], List[_GroupWS]] = {}
        self._ctx = None
        self._side = None
        self._aux = None
        self._pending = {}
        self.parallel_groups = True
        r8 = lambda x: (x + 7) // 8 * 8
        self.wb = None
        if self.bf16:
            kmp = r8(max(self.d.KMIX, HD + self.d.KZb))
            self.wb = [(torch.zeros(2 * self.d.n_hidden, r8(G + self.d.nb), dtype=torch.bfloat16, device=self.device),
                        torch.zeros(3 * r8(G), kmp, dtype=self.dec_dtype, device=self.device),
                        torch.zeros(2 * self.d.n_hidden, r8(G + self.d.nb), dtype=torch.bfloat16, device=self.device))
                       for G in self.d.genes]
        # bf16 copies of W1 / Wm: refreshed by conversion kernels at the start of every forward, or (stage_in_adam, set by
        # the owner of the optimiser step: TrainLoop) written by the Adam kernel itself; _staged_version detects parameter
        # writes made through torch (load_state_dict, .copy_, a torch optimiser) since the last staging
        self.stage_in_adam = False
        self._staged_version = -1
        self.adam_ticket = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.nb_events = None  # bench hook: iterator of (start, end) CUDA events bracketing the NB-loglik sweep
        # advanced by every forward and every backward pass, eager or replayed from a CUDA graph (note_replay): a pass's decoder
        # state in the workspaces (what decode_elements reads) is current while the generation is the one it was made in
        self.generation = 0

    # -------------------------------------------------------------------------------- helpers
    def P(self, g, name):
        return self.params.block(g, name)

    def Gd(self, g, name):
        return self.params.block(g, name, self.grads)

    def Bf(self, g, name):
        return self.buffers.block(g, name)

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _gemm(self, A, B, C, M, N, K, *, lda, ldb, ldc, ta=0, tb=0, srcA=L.SRC_F32, srcB=L.SRC_F32, rowsA=None, rowsB=None,
              batch=1, sA=0, sB=0, sC=0, bias=None, sBias=0, relu=0, acc=0, splits=1, ws=None, gate=None, drop=None, c_bf16=None):
        """gate = (y ptr, ld, mask ptr or None, ld, scale); drop = (p, mask ptr or None, stream id, ld); c_bf16 = (ptr, lo ptr or None, ld):
        fused epilogue stages of spv_gemm_fused (whole-K kernel only: see self._can_fuse)"""
        if gate is None and drop is None and c_bf16 is None:
            L.check(self.lib.spv_gemm(srcA, ta, srcB, tb, A, lda, L.ptr(rowsA), B, ldb, L.ptr(rowsB), C, ldc, M, N, K, batch,
                                      sA, sB, sC, bias, sBias, relu, acc, splits, L.ptr(ws), self._stream()), "spv_gemm")
            return
        gy, gld, gm, gmld, gs = gate if gate is not None else (None, 0, None, 0, 1.0)
        dp, dm, dsid, dld = drop if drop is not None else (0.0, None, 0, 0)
        cb, cblo, cbld = c_bf16 if c_bf16 is not None else (None, None, 0)
        L.check(self.lib.spv_gemm_fused(srcA, ta, srcB, tb, A, lda, L.ptr(rowsA), B, ldb, L.ptr(rowsB), C, ldc, M, N, K, batch,
                                        sA, sB, sC, bias, sBias, relu, acc, splits, L.ptr(ws), gy, gld, gm, gmld, gs, dp, dm,
                                        self.seed, dsid, L.ptr(self.noise_dev), dld, cb, cblo, cbld, self._stream()), "spv_gemm_fused")

    def _can_fuse(self, K):
        return K <= 256

    def _tc_gemm(self, A, B, C, M, N, K, *, lda, ldb, ldc, a_mn=0, b_mn=0, bias=None, relu=0, acc=0, splits=1, ws=None, fmt=0,
                 alpha=1.0):
        L.check(self.lib.spv_tc_gemm_ex(fmt, alpha, a_mn, b_mn, A, lda, B, ldb, C, ldc, M, N, K, bias, relu, acc, splits, L.ptr(ws),
                                        self._stream()), "spv_tc_gemm_ex")

    def _to_dec(self, src, ld_src, dst, ld_dst, R, C):
        """fp32 -> the decoder's 16-bit operand format"""
        fn, name = (self.lib.spv_to_f16, "spv_to_f16") if self.fused_nb else (self.lib.spv_to_bf16, "spv_to_bf16")
        L.check(fn(src, ld_src, dst, ld_dst, R, C, self._stream()), name)

    def _tc_gemm_split(self, A, Alo, B, Blo, C, M, N, K, *, lda, ldb, ldc, a_mn=0, b_mn=0, bias=None, relu=0, acc=0, splits=1, ws=None):
        """split-bf16 operands (hi + lo planes): three MMAs per k-step, fp32-grade products (spv_tc_gemm_split)"""
        L.check(self.lib.spv_tc_gemm_split(a_mn, b_mn, A, Alo, lda, B, Blo, ldb, C, ldc, M, N, K, bias, relu, acc, splits,
                                           L.ptr(ws), self._stream()), "spv_tc_gemm_split")

    def _fork_groups(self):
        """iterate over the two groups, issuing each group's launches on its own stream (forked from the current stream and
        joined back after the loop).  The two groups' encoder / decoder chains are independent and most of their kernels
        fill only part of the 148 SMs, so they overlap; inside a CUDA graph the fork/join becomes two parallel branches."""
        if not self.parallel_groups or self.device.type != "cuda":
            for g in (0, 1):
                yield g
            return
        if self._side is None:
            # (stream priorities were tried in r2 - main chains high, weight-gradient / optimiser lanes low: no effect on the replayed
            # graph's step time at C5 or C2)
            self._side = [torch.cuda.Stream(device=self.device) for _ in (0, 1)]
        cur = torch.cuda.current_stream(self.device)
        fork = torch.cuda.Event()
        fork.record(cur)
        joins = []
        for g in (0, 1):
            s = self._side[g]
            s.wait_event(fork)
            with torch.cuda.stream(s):
                yield g
            ev = torch.cuda.Event()
            ev.record(s)
            joins.append(ev)
        for ev in joins:
            cur.wait_event(ev)

    @contextlib.contextmanager
    def _branch(self, g, tag, lane=0):
        """run the enclosed launches on one of group g's two auxiliary streams (`lane`), forked from the current stream;
        `_join(g, tag)` makes the current stream wait for them.  Used for work that is off the critical path of the step
        (weight-gradient GEMMs, bias column sums, operand staging that does not depend on the minibatch)."""
        if not self.parallel_groups or self.device.type != "cuda":
            yield
            return
        if self._aux is None:
            self._aux = [[torch.cuda.Stream(device=self.device) for _ in (0, 1)] for _ in (0, 1)]
        cur = torch.cuda.current_stream(self.device)
        fork = torch.cuda.Event()
        fork.record(cur)
        aux = self._aux[g][lane]
        aux.wait_event(fork)
        with torch.cuda.stream(aux):
            yield
        done = torch.cuda.Event()
        done.record(aux)
        self._pending.setdefault((g, tag), []).append(done)

    def _join(self, g, tag=None):
        cur = torch.cuda.current_stream(self.device)
        for key in [k for k in self._pending if k[0] == g and (tag is None or k[1] == tag)]:
            for ev in self._pending.pop(key):
                cur.wait_event(ev)

    def _gene_bwd(self, g, w, Qp, Qs, ldq, B, G, colsum_in_q=0):
        gb = L.ptr_array([self.P(g, "Wp"), self.P(g, "Ws"), Qp, Qs, w.genec, w.colsum, w.zmean, w.zcov,
                          self.Gd(g, "Wp"), self.Gd(g, "Ws"), self.Gd(g, "gp"), self.Gd(g, "bp"), self.Gd(g, "gs"),
                          self.Gd(g, "bs"), self.Gd(g, "px_r"), self.Gd(g, "bm"), w.vpart, w.mpart])
        L.check(self.lib.spv_dec_gene_bwd(gb, ldq, B, G, self.d.Pb, self.d.Sb, colsum_in_q, self._stream()), "spv_dec_gene_bwd")

    def _hidden_mix(self, g, w, B, tr, zzp):
        """hm = relu(BatchNorm(zz Wh^T + bh)) into the first HD columns of amix   (reference nn/networks.py:322-323)"""
        d = self.d
        # input [zz | covariates]: the latent and covariate columns are contiguous in amix
        self._gemm(zzp, L.ptr(self.P(g, "Wh")), L.ptr(w.ah), B, HD, d.KZ + d.nb, lda=d.KMIX, ldb=d.KZ + d.nb, ldc=HD, tb=1,
                   bias=L.ptr(self.P(g, "bh")))
        L.check(self.lib.spv_bn_fwd(L.ptr(w.ah), HD, L.ptr(w.amix), d.KMIX, B, HD, L.ptr(self.P(g, "gh")),
                                    L.ptr(self.P(g, "bth")), DEC_BN_EPS, DEC_BN_MOM, L.ptr(self.Bf(g, "rm_h")),
                                    L.ptr(self.Bf(g, "rv_h")), L.ptr(w.bn_h_mean), L.ptr(w.bn_h_istd), tr, 1, self._stream()),
                 "spv_bn_fwd")

    def workspace(self, B0, B1, with_grad=True):
        key = (B0, B1, with_grad)
        if key not in self._ws:
            self._ws[key] = [_GroupWS(B, G, self.d, self.device, with_grad, self.bf16, self.wb[g] if self.bf16 else None,
                                      self.fused_nb) for g, (B, G) in enumerate(zip((B0, B1), self.d.genes))]
        return self._ws[key]

    @staticmethod
    def _src_of(X):
        if X.dtype == torch.uint16:
            return L.SRC_U16_LOG1P, 2
        if X.dtype == torch.float32:
            return L.SRC_F32_LOG1P, 4
        raise TypeError(f"counts must be uint16 or float32, got {X.dtype}")

    # -------------------------------------------------------------------------------- forward
    def forward(self, batches: Sequence[GroupBatch], training: bool = True, noise: Optional[Noise] = None,
                with_grad: Optional[bool] = None, decode: bool = True):
        """inference -> generative -> loss.  Returns the workspaces (device tensors) holding every output."""
        with_grad = training if with_grad is None else with_grad
        self.generation += 1
        ctx = self._encode(batches, training, noise, with_grad, stage_wm=decode)
        if not decode:
            for g in (0, 1):
                self._join(g)
            return ctx["ws"]
        return self._decode(ctx)

    def decode(self):
        """generative + loss on the latents of the preceding forward(decode=False) (same minibatch, same noise, BatchNorm
        running statistics of the encoders not updated a second time): reference module/spVIPESmodule.py:720-771, 809-899"""
        if self._ctx is None:
            raise RuntimeError("decode() follows forward(..., decode=False)")
        return self._decode(self._ctx)

    def _encode(self, batches, training, noise, with_grad, stage_wm=True):
        d, st, lib = self.d, self._stream(), self.lib
        H, S, P, KZ, KMIX, NST = d.n_hidden, d.n_shared, d.n_private, d.KZ, d.KMIX, d.NST
        Bs = [b.batch_size() for b in batches]
        ws = self.workspace(Bs[0], Bs[1], with_grad)
        noise = noise or Noise()
        tr = 1 if training else 0
        srcs = []
        decode = stage_wm
        # new Philox counter value for this pass (off the critical path; the first consumers wait for it below)
        with self._branch(0, "ntick", lane=1):
            L.check(lib.spv_adam_tick(L.ptr(self.noise_dev), self._stream()), "spv_adam_tick")
        self._noise_events = self._pending.pop((0, "ntick"), [])
        if self.mode == "label":  # integer pairing needs only the labels: off the critical path, beside the encoders
            if batches[0].labels is None or batches[1].labels is None:
                raise ValueError("Labels are required when using label-based POE.")  # reference :401-402
            with self._branch(0, "pair", lane=1):
                self._pair_label(batches, ws, Bs)
        convert = self.bf16 and not (self.stage_in_adam and self._staged_version == self.params.flat._version)
        # ---------------- encoders (reference nn/networks.py:119-125, module :428-448)
        for g in self._fork_groups():
            bt, w, st = batches[g], ws[g], self._stream()
            G, B = d.genes[g], Bs[g]
            src, esz = self._src_of(bt.X)
            nb, Gc = d.nb, G + d.nb
            if nb and bt.batch is None:
                raise ValueError("batch codes are required when the model was built with n_batch > 1")
            # (src, xptr, ldx, count_rows): where every consumer of the counts reads this minibatch
            if isinstance(bt.X, CsrCounts):
                if bt.col0 != 0 or bt.X.shape[1] != G:
                    raise ValueError(f"a CSR count matrix holds exactly the group's own {G} genes (col0 = 0), got shape "
                                     f"{bt.X.shape} and col0 = {bt.col0}")
                # gather the minibatch into the dense staging tile; in the default bf16 mode the same launch writes the encoder's
                # split-bf16 input and the library size (what spv_counts_to_bf16 does on dense rows)
                xs = w.need_xs(bt.X.dtype, self.device)
                conv = self.bf16
                L.check(lib.spv_csr_gather(src, L.ptr(bt.X.indptr), L.ptr(bt.X.indices), L.ptr(bt.X.values), L.ptr(bt.rows), B, G,
                                           L.ptr(xs), w.Gp, L.ptr(w.Tb) if conv else None, L.ptr(w.Tb_lo) if conv else None, w.Gpe,
                                           L.ptr(w.lib) if conv else None, L.ptr(bt.batch) if (conv and nb) else None,
                                           nb if conv else 0, st), "spv_csr_gather")
                xptr, ldx, count_rows = L.ptr(xs), w.Gp, None
            else:
                if bt.X.dim() != 2 or bt.X.stride(1) != 1:
                    raise ValueError("the count matrix must be row-major (unit stride along the genes)")
                conv = False
                xptr, ldx, count_rows = bt.X.data_ptr() + bt.col0 * esz, bt.X.stride(0), bt.rows
            srcs.append((src, xptr, ldx, count_rows))
            if convert:  # bf16 copies of the two big weights do not depend on the minibatch: off the critical path
                with self._branch(g, "w1"):
                    L.check(lib.spv_to_bf16_split(L.ptr(self.P(g, "W1")), Gc, L.ptr(w.W1b), L.ptr(w.W1b_lo), w.Gpe, 2 * H, Gc,
                                                  self._stream()), "spv_to_bf16_split")
                if decode or self.stage_in_adam:
                    with self._branch(g, "wm"):
                        self._to_dec(L.ptr(self.P(g, "Wm")), KMIX, L.ptr(w.Wmb), w.KMp, G, KMIX)
            if self.bf16:  # encoder input and library size from one pass over the gathered rows
                # (with batch covariates: their one-hot columns behind the genes, so that fc1 stays one GEMM over K = G + nb)
                if not conv:  # (a CSR minibatch was converted by its gather)
                    L.check(lib.spv_counts_to_bf16(src, xptr, ldx, L.ptr(count_rows), L.ptr(w.Tb), L.ptr(w.Tb_lo), w.Gpe, B, G,
                                                   L.ptr(w.lib), L.ptr(bt.batch) if nb else None, nb, st), "spv_counts_to_bf16")
                self._join(g, "w1")
                self._tc_gemm_split(L.ptr(w.Tb), L.ptr(w.Tb_lo), L.ptr(w.W1b), L.ptr(w.W1b_lo), L.ptr(w.h1), B, 2 * H, Gc, lda=w.Gpe,
                                    ldb=w.Gpe, ldc=2 * H, bias=L.ptr(self.P(g, "b1")), relu=1, splits=w.tc_splits_fc1, ws=w.ws)
            else:
                with self._branch(g, "lib"):
                    L.check(lib.spv_library_size(src, xptr, ldx, L.ptr(count_rows), B, G, L.ptr(w.lib), self._stream()),
                            "spv_library_size")
                if nb:  # covariate term + bias first (pre-activation), then the count GEMM adds to it and applies the ReLU
                    L.check(lib.spv_one_hot(L.ptr(bt.batch), L.ptr(w.oh), nb, B, nb, st), "spv_one_hot")
                    self._gemm(L.ptr(w.oh), self.P(g, "W1").data_ptr() + 4 * G, L.ptr(w.h1), B, 2 * H, nb, lda=nb, ldb=Gc, ldc=2 * H,
                               tb=1, bias=L.ptr(self.P(g, "b1")))
                self._gemm(xptr, L.ptr(self.P(g, "W1")), L.ptr(w.h1), B, 2 * H, G, lda=ldx, ldb=Gc, ldc=2 * H, tb=1, srcA=src,
                           rowsA=count_rows, bias=None if nb else L.ptr(self.P(g, "b1")), relu=1, acc=2 if nb else 0,
                           splits=w.splits_fc1, ws=w.ws)
            mask = noise.drop[g] if (training and noise.drop is not None) else None
            dropping = training and (mask is not None or self.dropout_rate > 0)
            for ev in self._noise_events:
                torch.cuda.current_stream(self.device).wait_event(ev)
            fuse_drop = dropping and self._can_fuse(H)  # dropout in the fc2 epilogue (same keep mask as spv_dropout)
            self._gemm(L.ptr(w.h1), L.ptr(self.P(g, "W2")), L.ptr(w.h2), B, H, H, lda=2 * H, ldb=H, ldc=2 * H, tb=1, batch=2,
                       sA=H, sB=H * H, sC=H, bias=L.ptr(self.P(g, "b2")), sBias=H, relu=1,
                       drop=(0.0 if mask is not None else self.dropout_rate, L.ptr(mask), 8 + g, 2 * H) if fuse_drop else None)
            if dropping and not fuse_drop:
                L.check(lib.spv_dropout(L.ptr(w.h2), 2 * H, B, 2 * H, L.ptr(mask), 2 * H, self.dropout_rate, self.seed,
                                        8 + g, L.ptr(self.noise_dev), st), "spv_dropout")
            bhd = self.P(g, "bhd")
            with self._branch(g, "headp"):  # the private and the shared heads are independent
                self._gemm(L.ptr(w.h2), L.ptr(self.P(g, "Whp")), L.ptr(w.r), B, 2 * P, H, lda=2 * H, ldb=H, ldc=NST, tb=1,
                           bias=L.ptr(bhd))
            self._gemm(w.h2.data_ptr() + 4 * H, L.ptr(self.P(g, "Whs")), w.r.data_ptr() + 4 * 2 * P, B, 2 * S, H, lda=2 * H,
                       ldb=H, ldc=NST, tb=1, bias=bhd.data_ptr() + 4 * 2 * P)
            self._join(g, "headp")
            L.check(lib.spv_bn_fwd(L.ptr(w.r), NST, L.ptr(w.stats), NST, B, NST, L.ptr(self.P(g, "ghd")),
                                   L.ptr(self.P(g, "bthd")), ENC_BN_EPS, ENC_BN_MOM, L.ptr(self.Bf(g, "rm_hd")),
                                   L.ptr(self.Bf(g, "rv_hd")), L.ptr(w.bn_hd_mean), L.ptr(w.bn_hd_istd), tr, 0, st), "spv_bn_fwd")
        if convert and self.stage_in_adam:
            self._staged_version = self.params.flat._version
        # ---------------- pairing (integer work) and PoE (reference :484-718)
        aux = self._pairing(batches, ws, Bs)
        self._poe_fwd(ws, Bs, noise, aux)
        ctx = {"batches": batches, "ws": ws, "Bs": Bs, "noise": noise, "srcs": srcs, "aux": aux, "training": training,
               "with_grad": with_grad, "wm_staged": (not convert) or decode or self.stage_in_adam, "gen": self.generation}
        self._ctx = ctx
        return ctx

    def note_replay(self, forward: bool):
        """a CUDA graph replayed a forward (forward=True; with its decoder, whose state is then current) or a backward pass of this
        engine: advance the generation as forward() / backward() do"""
        self.generation += 1
        if forward and self._ctx is not None:
            self._ctx["dec_gen"] = self.generation

    def _decode(self, ctx):
        # ---------------- decoders + NB likelihood (reference nn/networks.py:314-325, module :751-759, :817-824)
        Bs, ws = ctx["Bs"], ctx["ws"]
        for g in self._fork_groups():
            self._dec_prologue(ctx, g)
            self._dec_sweep(ctx, g)
        ctx["dec_gen"] = self.generation
        if Bs[0] != Bs[1]:
            raise ValueError("the loss needs equally sized minibatches in both groups (reference :886-893)")
        L.check(self.lib.spv_loss(L.ptr(ws[0].rec), L.ptr(ws[1].rec), L.ptr(ws[0].klp), L.ptr(ws[0].klq), L.ptr(ws[1].klp),
                                  L.ptr(ws[1].klq), Bs[0], L.ptr(self.kl_weight), L.ptr(self.loss_out), self._stream()), "spv_loss")
        return ws

    def _dec_prologue(self, ctx, g):
        """group g's decoder up to the likelihood sweep: mixture-weight staging, covariate expansion, count tables, hidden layer,
        BatchNorm fold and softmax normalisers (on the current stream of _fork_groups)"""
        d, lib = self.d, self.lib
        H, S, P, KZ, KMIX, NST = d.n_hidden, d.n_shared, d.n_private, d.KZ, d.KMIX, d.NST
        batches, ws, Bs, srcs, training, with_grad = ctx["batches"], ctx["ws"], ctx["Bs"], ctx["srcs"], ctx["training"], ctx["with_grad"]
        tr = 1 if training else 0
        bt, w, st = batches[g], ws[g], self._stream()
        G, B = d.genes[g], Bs[g]
        src, xptr, ldx, count_rows = srcs[g]
        if self.bf16 and not ctx["wm_staged"]:  # decode() after an encoder-only pass: the mixture weight's bf16 copy
            self._to_dec(L.ptr(self.P(g, "Wm")), KMIX, L.ptr(w.Wmb), w.KMp, G, KMIX)
        zzp = w.amix.data_ptr() + 4 * HD
        nb, Pb, Sb, KZb = d.nb, d.Pb, d.Sb, d.KZb
        # zb / ld_zb: the two factor regressors' inputs side by side.  Without covariates these are the latent columns of
        # amix; with them each regressor's input carries its own copy of the one-hot columns (spv_cov_expand, which also
        # fills the covariate columns behind [hm | zz] in amix)
        zb, ld_zb = zzp, KMIX
        if nb:
            L.check(lib.spv_cov_expand(zzp, KMIX, L.ptr(bt.batch), L.ptr(w.zzb), KZb, zzp + 4 * KZ, KMIX, B, P, S, nb, st),
                    "spv_cov_expand")
            zb, ld_zb = L.ptr(w.zzb), KZb
        fold = L.ptr_array([self.P(g, "Wp"), self.P(g, "Ws"), self.P(g, "gp"), self.P(g, "bp"), self.P(g, "gs"),
                            self.P(g, "bs"), self.P(g, "px_r"), self.Bf(g, "rm_p"), self.Bf(g, "rv_p"),
                            self.Bf(g, "rm_s"), self.Bf(g, "rv_s"), zb, w.zsum, w.cov_part, w.wfold, w.genec, w.zmean,
                            w.zcov])
        wz = w.Wstack.data_ptr() + 2 * w.Gp * w.KMp if self.fused_nb else None
        if self.fused_nb:
            # count tables of the likelihood sweeps: a function of px_r only, on the second auxiliary stream
            with self._branch(g, "tg", lane=1):
                L.check(lib.spv_dec_theta_tables(L.ptr(self.P(g, "px_r")), G, L.ptr(w.tgf), L.ptr(w.tb1), self._stream()),
                        "spv_dec_theta_tables")
            # hidden layer of the mixing net (needs only zz) on the auxiliary stream, beside latent stats / fold / normalisers;
            # the bf16 operand [hm | zz] of the mixture GEMM in one conversion pass after it
            with self._branch(g, "hm"):
                self._hidden_mix(g, w, B, tr, zzp)
                self._to_dec(L.ptr(w.amix), KMIX, L.ptr(w.amixb), w.KMp, B, KMIX)
        L.check(lib.spv_dec_fold(fold, ld_zb, B, G, Pb, Sb, tr, DEC_BN_EPS, DEC_BN_MOM, wz, w.KMp if self.fused_nb else 0,
                                 w.Gp, HD, L.ptr(w.wzf) if self.fused_nb else None, L.ptr(w.zcb) if self.fused_nb else None, st),
                "spv_dec_fold")
        if self.fused_nb:  # softmax normalisers on the tensor cores (main stream: latent stats -> fold -> normalisers)
            self._join(g, "lib")
            L.check(lib.spv_dec_stats_tc(L.ptr(w.zcb), L.ptr(w.wzf), w.Gp, L.ptr(w.genec), L.ptr(w.lib),
                                         L.ptr(w.part_stats), L.ptr(w.rowc), B, G, Pb, Sb, st), "spv_dec_stats_tc")
            self._join(g, "hm")
        else:
            self._hidden_mix(g, w, B, tr, zzp)
        dptrs = self._dec_ptrs(g, w, xptr, count_rows, with_grad)
        self._join(g, "lib")
        if not self.fused_nb:
            L.check(lib.spv_dec_nb_fwd(src, dptrs, ldx, KMIX, B, G, HD, Pb, Sb, 1, L.ptr(w.zzb) if nb else None, KZb, KMIX, st), "spv_dec_nb_fwd")

    def _dec_sweep(self, ctx, g):
        """group g's reducing likelihood sweep (per-cell reconstruction term; training: also what the backward needs)"""
        d, lib = self.d, self.lib
        KMIX = d.KMIX
        ws, Bs, srcs, training, with_grad = ctx["ws"], ctx["Bs"], ctx["srcs"], ctx["training"], ctx["with_grad"]
        w, st = ws[g], self._stream()
        G, B = d.genes[g], Bs[g]
        src, xptr, ldx, count_rows = srcs[g]
        nb, Pb, Sb, KZb = d.nb, d.Pb, d.Sb, d.KZb
        dptrs = self._dec_ptrs(g, w, xptr, count_rows, with_grad)
        evs = next(self.nb_events) if self.nb_events is not None else None
        if self.fused_nb:
            self._join(g, "wm")
            self._join(g, "tg")
        elif self.bf16:  # mixture logits on the tensor cores, consumed by the NB sweep
            self._to_dec(L.ptr(w.amix), KMIX, L.ptr(w.amixb), w.KMp, B, KMIX)
            self._join(g, "wm")
        if evs is not None:
            evs[0].record()
        if self.bf16:
            if self.fused_nb:
                if training and with_grad:  # one sweep: likelihood + everything the backward needs
                    L.check(lib.spv_dec_nb_train_tc(src, dptrs, ldx, L.ptr(w.amixb), w.KMp, L.ptr(w.Wstack), w.KMp, w.Gp,
                                                    L.ptr(w.zcb), L.ptr(w.wzf), L.ptr(w.E4T), 4 * w.Bp, L.ptr(w.DPIT), w.Bp, B, G, HD,
                                                    Pb, Sb, KMIX, st), "spv_dec_nb_train_tc")
                else:
                    L.check(lib.spv_dec_nb_fwd_tc(src, dptrs, ldx, L.ptr(w.amixb), w.KMp, L.ptr(w.Wstack), w.KMp, w.Gp, L.ptr(w.zcb),
                                                  L.ptr(w.wzf), B, G, HD, Pb, Sb, 0, KMIX, st), "spv_dec_nb_fwd_tc")  # backward recomputes pi
                if evs is not None:
                    evs[1].record()
                    evs = None
                L.check(lib.spv_dec_nb_rowreduce(L.ptr(w.part_nb), G, B, HD, L.ptr(w.rowc), L.ptr(w.rec), st), "spv_dec_nb_rowreduce")
            else:  # unfused: tensor-core GEMM writes pi, the SIMT sweep consumes it
                self._tc_gemm(L.ptr(w.amixb), L.ptr(w.Wmb), L.ptr(w.pi), B, G, KMIX, lda=w.KMp, ldb=w.KMp, ldc=G,
                              bias=L.ptr(self.P(g, "bm")))
                L.check(lib.spv_dec_nb_fwd(src, dptrs, ldx, KMIX, B, G, HD, Pb, Sb, 2 | 4, L.ptr(w.zzb) if nb else None, KZb, KMIX, st), "spv_dec_nb_fwd")
        else:
            L.check(lib.spv_dec_nb_fwd(src, dptrs, ldx, KMIX, B, G, HD, Pb, Sb, 2, L.ptr(w.zzb) if nb else None, KZb, KMIX, st), "spv_dec_nb_fwd")
        if evs is not None:
            evs[1].record()

    def _on_device(self, t):
        dev = self.device
        return t.device.type == dev.type and (dev.index is None or t.device.index == dev.index)

    def decode_elements(self, outs, value=None):
        """per-element decoder outputs of the current pass: outs[g] maps names of ELEM_OUTPUTS to float32 device tensors [B_g, ld]
        (unit stride along the genes, one row pitch per group, ld >= the group's genes; a group may be omitted or map to {}):
          ll      log_mixture_nb per element (eps 1e-8) of t = log1p(counts of the minibatch), or of value[g] (float32 [B_g, >= G_g],
                  unit stride) as given when `value` is a sequence of two such tensors (None entries: that group's counts)
          rate_p  px_rate_private = exp(lib) softmax(BN_p(z_private_arg Wp^T)),  rate_s  px_rate_shared
          pi      px_mixing (the mixing logit, bias included),  mean  sigmoid(pi) rate_p + (1 - sigmoid(pi)) rate_s
        The state is the one the pass left in the workspaces: after forward(..., decode=False) in eval mode the decoder's prologue
        runs here (not the likelihood sweep: no loss, so the groups may differ in size).  No spv_loss, no gradient state."""
        ctx = self._ctx
        if ctx is None:
            raise RuntimeError("decode_elements() follows a forward pass")
        if ctx.get("dec_gen") != self.generation:
            if "dec_gen" in ctx or self.generation != ctx["gen"]:
                raise RuntimeError("the decoder state of the last forward is gone: a backward or another forward ran since")
            if ctx["training"]:
                raise RuntimeError("decode_elements() after a training-mode forward(..., decode=False): running the decoder here would "
                                   "update its BatchNorm running statistics a second time; decode the training pass instead")
        d, lib = self.d, self.lib
        idx = {k: i for i, k in enumerate(ELEM_OUTPUTS)}
        for g in (0, 1):
            for k in (outs[g] or {}):
                if k not in idx:
                    raise ValueError(f"unknown decoder output {k!r}; choose from {ELEM_OUTPUTS}")
        run_prologue = ctx.get("dec_gen") != self.generation
        for g in self._fork_groups():
            if run_prologue:
                self._dec_prologue(ctx, g)
            self._join(g)
            og = outs[g] or {}
            if not og:
                continue
            w, B, G, st = ctx["ws"][g], ctx["Bs"][g], d.genes[g], self._stream()
            ld = None
            for k, t in og.items():
                if t.dtype != torch.float32 or not self._on_device(t) or t.dim() != 2 or t.shape[0] != B or t.shape[1] < G or \
                        t.stride(1) != 1 or (ld is not None and t.stride(0) != ld):
                    raise ValueError(f"decoder output {k!r} of group {g}: a float32 {self.device} tensor [{B}, >= {G}] with unit stride "
                                     f"along the genes and the row pitch of the group's other outputs is needed, got "
                                     f"{tuple(t.shape)} {t.dtype} strides {t.stride()}")
                ld = t.stride(0)
            arr = L.ptr_array([og.get(k) for k in ELEM_OUTPUTS])
            src, xptr, ldx, rows = ctx["srcs"][g]
            v = value[g] if value is not None else None
            if v is not None:
                if v.dtype != torch.float32 or not self._on_device(v) or v.dim() != 2 or v.shape[0] != B or v.shape[1] < G or v.stride(1) != 1:
                    raise ValueError(f"value of group {g}: a float32 {self.device} tensor [{B}, >= {G}] with unit stride along the genes is "
                                     f"needed, got {tuple(v.shape)} {v.dtype}")
                src, xptr, ldx, rows = L.SRC_F32, v.data_ptr(), v.stride(0), None
            dptrs = self._dec_ptrs(g, w, xptr, rows, False)
            nb, Pb, Sb, KZb, KMIX = d.nb, d.Pb, d.Sb, d.KZb, d.KMIX
            if self.fused_nb:
                L.check(lib.spv_dec_nb_elems_tc(src, dptrs, ldx, L.ptr(w.amixb), w.KMp, L.ptr(w.Wstack), w.KMp, w.Gp, L.ptr(w.zcb),
                                                L.ptr(w.wzf), B, G, HD, Pb, Sb, KMIX, arr, ld, st), "spv_dec_nb_elems_tc")
                continue
            if self.bf16:  # the unfused bf16 decoder's mixture logits: the tensor-core GEMM of its sweep
                self._to_dec(L.ptr(w.amix), KMIX, L.ptr(w.amixb), w.KMp, B, KMIX)
                self._tc_gemm(L.ptr(w.amixb), L.ptr(w.Wmb), L.ptr(w.pi), B, G, KMIX, lda=w.KMp, ldb=w.KMp, ldc=G, bias=L.ptr(self.P(g, "bm")))
            L.check(lib.spv_dec_nb_elems(src, dptrs, ldx, KMIX, B, G, HD, Pb, Sb, 1 if self.bf16 else 0, L.ptr(w.zzb) if nb else None,
                                         KZb, KMIX, arr, ld, st), "spv_dec_nb_elems")
        if run_prologue:
            ctx["dec_gen"] = self.generation

    def _dec_ptrs(self, g, w, xptr, rows, with_grad):
        wg = with_grad
        return L.ptr_array([xptr, rows, w.amix, w.wfold, self.P(g, "Wm"), self.P(g, "bm"), w.genec, w.lib, w.part_stats,
                            w.rowc, w.pi, w.part_nb, w.dyp if wg else None, w.dys if wg else None, w.dpi if wg else None,
                            w.colpart if wg else None, w.rec, getattr(w, "tgf", None), getattr(w, "tb1", None)])

    def _pairing(self, batches, ws, Bs):
        lib, st, d = self.lib, self._stream(), self.d
        aux = {}
        if self.mode == "label":  # launched at the start of forward
            self._join(0, "pair")
            return aux
        if self.plan is None:
            raise ValueError("a transport plan is required for the OT PoE modes")
        if Bs[0] != Bs[1]:
            raise ValueError("OT PoE needs equally sized minibatches (reference :521-523)")
        key = ("sub", Bs[0], Bs[1])
        if key not in self._ws:
            self._ws[key] = {"sub": torch.empty(Bs[0], Bs[1], dtype=torch.float32, device=self.device),
                             "P1": torch.empty(Bs[0], Bs[1], dtype=torch.float32, device=self.device),
                             "P2": torch.empty(Bs[1], Bs[0], dtype=torch.float32, device=self.device)}
        aux = self._ws[key]
        gather = lib.spv_plan_gather_bf16 if self.plan.dtype == torch.bfloat16 else lib.spv_plan_gather
        L.check(gather(L.ptr(self.plan), self.plan.stride(0), L.ptr(batches[0].idx), L.ptr(batches[1].idx),
                       Bs[0], Bs[1], L.ptr(aux["sub"]), st), "spv_plan_gather")
        if self.mode == "paired":
            L.check(lib.spv_plan_argmax(L.ptr(aux["sub"]), Bs[0], Bs[1], L.ptr(ws[0].partner), L.ptr(ws[1].partner), st),
                    "spv_plan_argmax")
            return aux
        # cluster mode (reference :184-280)
        if batches[0].labels is None or batches[1].labels is None:
            raise ValueError("processed_transport_labels are required when using transport plan.")  # reference :394-397
        self._pair_label(batches, ws, Bs)
        L.check(lib.spv_plan_cluster_norm(L.ptr(aux["sub"]), Bs[0], Bs[1], L.ptr(batches[0].labels), L.ptr(batches[1].labels),
                                          L.ptr(aux["P1"]), L.ptr(aux["P2"]), st), "spv_plan_cluster_norm")
        S, P, NST = d.n_shared, d.n_private, d.NST
        # expert A = P1 @ stats_0[:, shared], expert B = P2 @ stats_1[:, shared]  (cross-indexing quirk Q5, :222, :228)
        # (K = the other group's minibatch: split-K so that more than B / 64 CTAs share a 2048-deep reduction; nothing else uses
        # the groups' split-K scratch at this point of the step)
        sk = lambda K: max(1, min(8, K // 256))
        self._gemm(L.ptr(aux["P1"]), ws[0].stats.data_ptr() + 4 * 2 * P, L.ptr(ws[0].expert), Bs[0], 2 * S, Bs[1], lda=Bs[1],
                   ldb=NST, ldc=2 * S, splits=sk(Bs[1]), ws=ws[0].ws)
        self._gemm(L.ptr(aux["P2"]), ws[1].stats.data_ptr() + 4 * 2 * P, L.ptr(ws[1].expert), Bs[1], 2 * S, Bs[0], lda=Bs[0],
                   ldb=NST, ldc=2 * S, splits=sk(Bs[0]), ws=ws[1].ws)
        return aux

    def _pair_label(self, batches, ws, Bs):
        """labels are either per-minibatch [B] arrays, or per-cell arrays gathered with the batch's row indices"""
        lr = [bt.rows if (bt.labels_per_cell and bt.rows is not None) else None for bt in batches]
        L.check(self.lib.spv_pair_label(L.ptr(batches[0].labels), L.ptr(batches[1].labels), L.ptr(lr[0]), L.ptr(lr[1]), Bs[0],
                                        Bs[1], L.ptr(ws[0].partner), L.ptr(ws[1].partner), self._stream()), "spv_pair_label")

    def _poe_sides(self, ws):
        d = self.d
        S, P, NST = d.n_shared, d.n_private, d.NST
        if self.mode == "cluster":
            own = [(w.expert.data_ptr(), w.expert.data_ptr() + 4 * S, 2 * S) for w in ws]
        else:
            own = [(w.stats.data_ptr() + 4 * 2 * P, w.stats.data_ptr() + 4 * (2 * P + S), NST) for w in ws]
        return own

    def _poe_fwd(self, ws, Bs, noise, aux):
        d = self.d
        S, P, NST, KMIX = d.n_shared, d.n_private, d.NST, d.KMIX
        own = self._poe_sides(ws)
        arrs = []
        for g in (0, 1):
            o, t, w = own[g], own[1 - g], ws[g]
            ep = noise.eps_private[g] if noise.eps_private is not None else None
            eq = noise.eps_poe[g] if noise.eps_poe is not None else None
            ptrs = L.ptr_array([o[0], o[1], t[0], t[1], w.stats, w.partner, ep, eq, w.zpriv, w.poe_loc, w.poe_lv, w.poe_scale,
                                w.zpoe, w.klp, w.klq, w.amix.data_ptr() + 4 * HD])
            lds = L.ll_array([o[2], t[2], NST, KMIX])
            arrs.append((ptrs, lds))
        L.check(self.lib.spv_poe_fwd(self.mode_id, S, P, Bs[0], Bs[1], arrs[0][0], arrs[0][1], arrs[1][0], arrs[1][1], self.seed,
                                     L.ptr(self.noise_dev), self._stream()), "spv_poe_fwd")

    # -------------------------------------------------------------------------------- backward
    def backward(self, grad_scale: float = 1.0, adam: Optional[dict] = None, stage: str = "all", tick: bool = False):
        """gradients of loss * grad_scale w.r.t. every parameter, written into self.grads.
        adam (keys lr, betas, eps, weight_decay[, grad_scale]; data parallel: enc_only = True and sync = callable(g), which enqueues the
        all-reduce of group g's encoder range on the current stream before its update): also apply the optimiser step, per parameter range
        as soon as its gradients are complete: the decoder ranges (55 % of the parameters) update on an auxiliary stream
        while the encoder backward, a chain of small latency-bound kernels that leaves HBM idle, is still running.
        stage: "all", or "decoder" (decoders + PoE: every decoder-range gradient final) followed by "encoder" - the
        data-parallel step all-reduces the decoder range while the encoder stage runs.  tick: advance the optimiser step
        counter now (off the critical path), for callers that apply Adam per range afterwards (`adam_range_step`)."""
        ctx = self._ctx
        if ctx is None or not ctx["training"]:
            raise RuntimeError("backward needs a preceding training-mode forward")
        self.generation += 1
        if stage not in ("all", "decoder", "encoder") or (adam is not None and stage == "decoder") or \
                (adam is not None and stage == "encoder" and not adam.get("enc_only")):
            raise ValueError("stage must be 'all', 'decoder' or 'encoder' (the interleaved optimiser step needs 'all', or 'encoder' "
                             "with adam['enc_only'])")
        tick_events = []
        if (adam is not None and not adam.get("enc_only")) or (tick and stage != "encoder"):  # (enc_only: the decoder stage ticked)
            if self.adam_m is None:
                self.adam_m = torch.zeros_like(self.params.flat)
                self.adam_v = torch.zeros_like(self.params.flat)
            with self._branch(0, "tick", lane=1):  # the step count of this update, off the critical path
                L.check(self.lib.spv_adam_tick(L.ptr(self.step_dev), self._stream()), "spv_adam_tick")
            tick_events = self._pending.pop((0, "tick"), [])
        if stage != "encoder":
            self._backward_decoders(ctx, grad_scale)
        if stage == "decoder":
            for g in (0, 1):  # every auxiliary branch back on the calling stream (a graph capture may end here)
                self._join(g)
            for ev in tick_events:
                torch.cuda.current_stream(self.device).wait_event(ev)
            return
        self._backward_encoders(ctx, grad_scale, adam, tick_events)

    def _backward_decoders(self, ctx, grad_scale):
        d, st, lib = self.d, self._stream(), self.lib
        H, S, P, KZ, KMIX, NST = d.n_hidden, d.n_shared, d.n_private, d.KZ, d.KMIX, d.NST
        batches, ws, Bs, noise, srcs, aux = ctx["batches"], ctx["ws"], ctx["Bs"], ctx["noise"], ctx["srcs"], ctx["aux"]
        # ---------------- decoders
        for g in self._fork_groups():
            bt, w, st = batches[g], ws[g], self._stream()
            G, B = d.genes[g], Bs[g]
            src, xptr, ldx, count_rows = srcs[g]
            zzp = w.amix.data_ptr() + 4 * HD
            nb, Pb, Sb, KZb = d.nb, d.Pb, d.Sb, d.KZb
            zb, ld_zb = (L.ptr(w.zzb), KZb) if nb else (zzp, KMIX)
            if self.fused_nb:
                # the training sweep of the forward left E4T = (ep, rp', es, rs') and DPIT = d ll / d pi (fp16, gene-major): the
                # backward of the likelihood is four GEMMs; the softmax coupling rides in their small operands (csrc/nb_tc_train.cu)
                f3, al = self.dec_fmt, -float(grad_scale) / B
                Bp, ldq = w.Bp, KZb + 2
                L.check(lib.spv_dec_nb_train_colsum(L.ptr(w.colpart), B, G, al, w.colsum.data_ptr() + 4 * 2 * G, st), "spv_dec_nb_train_colsum")
                with self._branch(g, "dzg"):  # d zz through the two softmax branches: T = E4T^T [W'p | W's], then the row combination
                    self._to_dec(L.ptr(w.wfold), KZb, L.ptr(w.Wcomb), w.Wcomb.stride(0), G, KZb)
                    self._tc_gemm(L.ptr(w.E4T), L.ptr(w.Wcomb), L.ptr(w.T4), 4 * B, KZb, w.Gp, lda=4 * Bp, ldb=w.Wcomb.stride(0), ldc=KZb,
                                  a_mn=1, b_mn=1, splits=w.tc_splits_dz4, ws=w.ws2, fmt=f3, alpha=al)
                    L.check(lib.spv_dec_dz4_combine(L.ptr(w.T4), KZb, L.ptr(w.rowc), L.ptr(w.dzraw), KZb, B, Pb, Sb, self._stream()),
                            "spv_dec_dz4_combine")
                with self._branch(g, "wgrad"):  # d Wm = dpi^T [hm | zz]
                    self._tc_gemm(L.ptr(w.DPIT), L.ptr(w.amixb), L.ptr(self.Gd(g, "Wm")), G, KMIX, B, lda=Bp, ldb=w.KMp, ldc=KMIX,
                                  a_mn=0, b_mn=1, fmt=f3, alpha=al)
                with self._branch(g, "gene", lane=1):
                    # [Qp | sum dyp | Qs | sum dys] = E4T . ZQ4 (K = 4 B: the coupling -D' [z 1] rides in ZQ4's odd rows); unsplit:
                    # measured faster in the step than a split that fills the SMs evenly (DESIGN.md section 8)
                    L.check(lib.spv_dec_zq4(zb, ld_zb, L.ptr(w.rowc), L.ptr(w.ZQ4), w.ldq4, B, Pb, Sb, self._stream()), "spv_dec_zq4")
                    self._tc_gemm(L.ptr(w.E4T), L.ptr(w.ZQ4), L.ptr(w.CQ), G, ldq, 4 * B, lda=4 * Bp, ldb=w.ldq4, ldc=ldq,
                                  a_mn=0, b_mn=1, fmt=f3, alpha=al)
                    self._gene_bwd(g, w, w.CQ.data_ptr(), w.CQ.data_ptr() + 4 * (Pb + 1), ldq, B, G, colsum_in_q=1)
                dzraw = None
                # d [hm | zz] (mixture part) = dpi Wm
                self._tc_gemm(L.ptr(w.DPIT), L.ptr(w.Wstack), L.ptr(w.damix), B, KMIX, G, lda=Bp, ldb=w.KMp, ldc=KMIX, a_mn=1, b_mn=1,
                              splits=w.tc_splits_damix, ws=w.ws, fmt=f3, alpha=al)
            else:
                L.check(lib.spv_dec_nb_bwd(src, self._dec_ptrs(g, w, xptr, count_rows, True), ldx, KMIX, B, G, HD, Pb, Sb,
                                           -float(grad_scale) / B, L.ptr(w.colsum), L.ptr(w.dpib) if self.bf16 else None,
                                           w.Gp if self.bf16 else 0, L.ptr(w.zzb) if nb else None, KZb, KMIX, st),
                        "spv_dec_nb_bwd")
                # d Wm = dpi^T [hm | zz];   d [hm | zz] = dpi Wm
                if self.bf16:
                    self._tc_gemm(L.ptr(w.dpib), L.ptr(w.amixb), L.ptr(self.Gd(g, "Wm")), G, KMIX, B, lda=w.Gp, ldb=w.KMp,
                                  ldc=KMIX, a_mn=1, b_mn=1)
                    self._tc_gemm(L.ptr(w.dpib), L.ptr(w.Wmb), L.ptr(w.damix), B, KMIX, G, lda=w.Gp, ldb=w.KMp, ldc=KMIX,
                                  b_mn=1, splits=w.tc_splits_damix, ws=w.ws)
                else:
                    self._gemm(L.ptr(w.dpi), L.ptr(w.amix), L.ptr(self.Gd(g, "Wm")), G, KMIX, B, lda=G, ldb=KMIX, ldc=KMIX, ta=1)
                    self._gemm(L.ptr(w.dpi), L.ptr(self.P(g, "Wm")), L.ptr(w.damix), B, KMIX, G, lda=G, ldb=KMIX, ldc=KMIX,
                               splits=w.splits_g, ws=w.ws)
                # Q = dy^T z ;  dz (softmax branches) = dy W'
                self._gemm(L.ptr(w.dyp), zb, L.ptr(w.Qp), G, Pb, B, lda=G, ldb=ld_zb, ldc=Pb, ta=1, splits=w.splits_b, ws=w.ws)
                self._gemm(L.ptr(w.dys), zb + 4 * Pb, L.ptr(w.Qs), G, Sb, B, lda=G, ldb=ld_zb, ldc=Sb, ta=1, splits=w.splits_b, ws=w.ws)
                self._gemm(L.ptr(w.dyp), L.ptr(w.wfold), L.ptr(w.dzraw), B, Pb, G, lda=G, ldb=KZb, ldc=KZb, splits=w.splits_g, ws=w.ws)
                self._gemm(L.ptr(w.dys), w.wfold.data_ptr() + 4 * Pb, w.dzraw.data_ptr() + 4 * Pb, B, Sb, G, lda=G, ldb=KZb, ldc=KZb,
                           splits=w.splits_g, ws=w.ws)
                Qp, Qs, ldq, dzraw = L.ptr(w.Qp), L.ptr(w.Qs), 0, L.ptr(w.dzraw)
            # hidden layer of the mixing net: ReLU + BatchNorm backward (needs only d [hm | zz]); its Linear's input and
            # weight gradients run on the auxiliary stream next to the per-gene BatchNorm backward
            L.check(lib.spv_bn_bwd(L.ptr(w.damix), KMIX, L.ptr(w.ah), HD, L.ptr(w.amix), KMIX, L.ptr(w.dah), HD, B, HD,
                                   L.ptr(self.P(g, "gh")), L.ptr(w.bn_h_mean), L.ptr(w.bn_h_istd), L.ptr(self.Gd(g, "gh")),
                                   L.ptr(self.Gd(g, "bth")), st), "spv_bn_bwd")
            def hidden_input_grad(dst):
                """dzraw += dah Wh (the latent columns; the covariate columns of Wh carry no input gradient)"""
                wh, kh = self.P(g, "Wh").data_ptr(), KZ + nb
                if not nb:
                    self._gemm(L.ptr(w.dah), wh, dst, B, KZ, HD, lda=HD, ldb=kh, ldc=KZb, acc=1)
                else:  # dzraw is laid out [z_private_arg | oh | z_shared_arg | oh], Wh's columns [z_private_arg | z_shared_arg | oh]
                    self._gemm(L.ptr(w.dah), wh, dst, B, P, HD, lda=HD, ldb=kh, ldc=KZb, acc=1)
                    self._gemm(L.ptr(w.dah), wh + 4 * P, dst + 4 * Pb, B, S, HD, lda=HD, ldb=kh, ldc=KZb, acc=1)

            if dzraw is None:  # fused path: dzraw already holds the softmax-branch part (branch "dzg", same auxiliary stream)
                dzraw = L.ptr(w.dzraw)
                with self._branch(g, "hid"):
                    hidden_input_grad(dzraw)
            else:
                hidden_input_grad(dzraw)
            with self._branch(g, "wgrad"):
                self._gemm(L.ptr(w.dah), zzp, L.ptr(self.Gd(g, "Wh")), HD, KZ + nb, B, lda=HD, ldb=KMIX, ldc=KZ + nb, ta=1,
                           splits=w.splits_b, ws=w.ws2)
            with self._branch(g, "wgrad1", lane=1):
                L.check(lib.spv_colsum(L.ptr(w.dah), HD, B, HD, L.ptr(self.Gd(g, "bh")), self._stream()), "spv_colsum")
            if not self.fused_nb:
                self._gene_bwd(g, w, Qp, Qs, ldq, B, G)
            self._join(g, "hid")
            if self.fused_nb:  # column sums of the branch / hidden-layer input gradient (the consistent mean-coupling term)
                L.check(lib.spv_colsum(dzraw, KZb, B, KZb, L.ptr(w.dzraw_sum), st), "spv_colsum")
            self._join(g, "gene")
            # without covariates the mixture layer's input gradient (latent columns of damix) has the regressors' layout and is
            # added here; with them it is added by the compaction below
            L.check(lib.spv_dec_dzz_combine(None if nb else w.damix.data_ptr() + 4 * HD, KMIX, dzraw, L.ptr(w.vpart), L.ptr(w.mpart),
                                            w.nGB, zb, ld_zb, L.ptr(w.zmean), L.ptr(w.dzzb), B, Pb, Sb,
                                            L.ptr(w.dzraw_sum) if self.fused_nb else None, st), "spv_dec_dzz_combine")
            if nb:
                L.check(lib.spv_cov_compact(L.ptr(w.dzzb), KZb, L.ptr(w.dzz), KZ, B, P, S, nb, w.damix.data_ptr() + 4 * HD, KMIX, st),
                        "spv_cov_compact")
        # ---------------- PoE
        own = self._poe_sides(ws)
        arrs = []
        for g in (0, 1):
            o, t, w = own[g], own[1 - g], ws[g]
            ep = noise.eps_private[g] if noise.eps_private is not None else None
            eq = noise.eps_poe[g] if noise.eps_poe is not None else None
            if self.mode == "cluster":
                out, ld_out = w.dexpert.data_ptr(), 2 * S
            else:
                out, ld_out = w.dstats.data_ptr() + 4 * 2 * P, NST
            ptrs = L.ptr_array([o[0], o[1], t[0], t[1], w.stats, w.partner, ep, eq, w.dzz, w.dstats, w.g_own, w.g_contrib, out])
            lds = L.ll_array([o[2], t[2], NST, KZ, NST, ld_out])
            arrs.append((ptrs, lds))
        L.check(lib.spv_poe_bwd(self.mode_id, S, P, Bs[0], Bs[1], arrs[0][0], arrs[0][1], arrs[1][0], arrs[1][1], self.seed,
                                L.ptr(self.noise_dev), L.ptr(self.kl_weight), float(grad_scale) / Bs[0], self._stream()),
                "spv_poe_bwd")
        if self.mode == "cluster":
            # d stats_0[:, shared] += P1^T d expertA ;  d stats_1[:, shared] += P2^T d expertB   (quirk Q5)
            sk = lambda K: max(1, min(8, K // 256))
            self._gemm(L.ptr(aux["P1"]), L.ptr(ws[0].dexpert), ws[0].dstats.data_ptr() + 4 * 2 * P, Bs[1], 2 * S, Bs[0],
                       lda=Bs[1], ldb=2 * S, ldc=NST, ta=1, acc=1, splits=sk(Bs[0]), ws=ws[0].ws)
            self._gemm(L.ptr(aux["P2"]), L.ptr(ws[1].dexpert), ws[1].dstats.data_ptr() + 4 * 2 * P, Bs[0], 2 * S, Bs[1],
                       lda=Bs[0], ldb=2 * S, ldc=NST, ta=1, acc=1, splits=sk(Bs[1]), ws=ws[1].ws)
    def _backward_encoders(self, ctx, grad_scale, adam, tick_events):
        d, st, lib = self.d, self._stream(), self.lib
        H, S, P, KZ, KMIX, NST = d.n_hidden, d.n_shared, d.n_private, d.KZ, d.KMIX, d.NST
        batches, ws, Bs, noise, srcs, aux = ctx["batches"], ctx["ws"], ctx["Bs"], ctx["noise"], ctx["srcs"], ctx["aux"]
        # ---------------- encoders
        for g in self._fork_groups():
            bt, w, st = batches[g], ws[g], self._stream()
            G, B = d.genes[g], Bs[g]
            src, xptr, ldx, count_rows = srcs[g]
            L.check(lib.spv_bn_bwd(L.ptr(w.dstats), NST, L.ptr(w.r), NST, None, 0, L.ptr(w.dr), NST, B, NST,
                                   L.ptr(self.P(g, "ghd")), L.ptr(w.bn_hd_mean), L.ptr(w.bn_hd_istd), L.ptr(self.Gd(g, "ghd")),
                                   L.ptr(self.Gd(g, "bthd")), st), "spv_bn_bwd")
            drs = w.dr.data_ptr() + 4 * 2 * P
            mask = noise.drop[g] if noise.drop is not None else None
            scale = 1.0 / (1.0 - self.dropout_rate) if self.dropout_rate > 0 else 1.0
            fuse2 = self._can_fuse(2 * S)  # ReLU + dropout backward in the epilogue of the two head input-gradient GEMMs
            gate_p = (L.ptr(w.h2), 2 * H, L.ptr(mask), 2 * H, scale) if fuse2 else None
            gate_s = (w.h2.data_ptr() + 4 * H, 2 * H, mask.data_ptr() + 4 * H if mask is not None else None, 2 * H, scale) if fuse2 else None
            with self._branch(g, "dh2p"):  # first on its auxiliary stream: this one is on the critical path
                self._gemm(L.ptr(w.dr), L.ptr(self.P(g, "Whp")), L.ptr(w.dh2), B, H, 2 * P, lda=NST, ldb=H, ldc=2 * H, gate=gate_p)
            if adam is not None and not adam.get("enc_only"):  # every decoder gradient of this group is final: update that range now
                self._join(g, "wgrad")
                self._join(g, "wgrad1")
                with self._branch(g, "adam", lane=1):
                    for ev in tick_events:
                        torch.cuda.current_stream(self.device).wait_event(ev)
                    lo, hi = self.params.group_ranges[PHASE_DEC][g]
                    self._adam_range(lo, hi, adam, max_blocks=ADAM_OVERLAP_BLOCKS)
            with self._branch(g, "wgrad1", lane=1):
                L.check(lib.spv_colsum(L.ptr(w.dr), NST, B, NST, L.ptr(self.Gd(g, "bhd")), self._stream()), "spv_colsum")
            with self._branch(g, "wgrad"):
                self._gemm(L.ptr(w.dr), L.ptr(w.h2), L.ptr(self.Gd(g, "Whp")), 2 * P, H, B, lda=NST, ldb=2 * H, ldc=H, ta=1,
                           splits=w.splits_b, ws=w.ws2)
                self._gemm(drs, w.h2.data_ptr() + 4 * H, L.ptr(self.Gd(g, "Whs")), 2 * S, H, B, lda=NST, ldb=2 * H, ldc=H, ta=1,
                           splits=w.splits_b, ws=w.ws2)
            self._gemm(drs, L.ptr(self.P(g, "Whs")), w.dh2.data_ptr() + 4 * H, B, H, 2 * S, lda=NST, ldb=H, ldc=2 * H, gate=gate_s)
            self._join(g, "dh2p")
            if not fuse2:
                L.check(lib.spv_relu_bwd(L.ptr(w.dh2), 2 * H, L.ptr(w.h2), 2 * H, B, 2 * H, L.ptr(mask), 2 * H, scale, st),
                        "spv_relu_bwd")
            with self._branch(g, "wgrad1", lane=1):
                self._gemm(L.ptr(w.dh2), L.ptr(w.h1), L.ptr(self.Gd(g, "W2")), H, H, B, lda=2 * H, ldb=2 * H, ldc=H, ta=1,
                           batch=2, sA=H, sB=H, sC=H * H, splits=w.splits_b, ws=w.ws3)
                L.check(lib.spv_colsum(L.ptr(w.dh2), 2 * H, B, 2 * H, L.ptr(self.Gd(g, "b2")), self._stream()), "spv_colsum")
            fuse1 = self._can_fuse(H)  # ReLU backward + bf16 copy in the fc2 input-gradient GEMM's epilogue
            self._gemm(L.ptr(w.dh2), L.ptr(self.P(g, "W2")), L.ptr(w.dh1), B, H, H, lda=2 * H, ldb=H, ldc=2 * H, batch=2,
                       sA=H, sB=H * H, sC=H, gate=(L.ptr(w.h1), 2 * H, None, 0, 1.0) if fuse1 else None,
                       c_bf16=(L.ptr(w.dh1b), L.ptr(w.dh1b_lo), 2 * H) if (fuse1 and self.bf16) else None)
            if not fuse1:
                L.check(lib.spv_relu_bwd(L.ptr(w.dh1), 2 * H, L.ptr(w.h1), 2 * H, B, 2 * H, None, 0, 1.0, st), "spv_relu_bwd")
            if self.bf16:
                if not fuse1:
                    L.check(lib.spv_to_bf16_split(L.ptr(w.dh1), 2 * H, L.ptr(w.dh1b), L.ptr(w.dh1b_lo), 2 * H, B, 2 * H, st),
                            "spv_to_bf16_split")
                self._tc_gemm_split(L.ptr(w.dh1b), L.ptr(w.dh1b_lo), L.ptr(w.Tb), L.ptr(w.Tb_lo), L.ptr(self.Gd(g, "W1")), 2 * H,
                                    G + d.nb, B, lda=2 * H, ldb=w.Gpe, ldc=G + d.nb, a_mn=1, b_mn=1)
            else:
                self._gemm(L.ptr(w.dh1), xptr, L.ptr(self.Gd(g, "W1")), 2 * H, G, B, lda=2 * H, ldb=ldx, ldc=G + d.nb, ta=1, srcB=src,
                           rowsB=count_rows)
                if d.nb:  # covariate columns of the first layer's weight: dh1^T one_hot
                    self._gemm(L.ptr(w.dh1), L.ptr(w.oh), self.Gd(g, "W1").data_ptr() + 4 * G, 2 * H, d.nb, B, lda=2 * H, ldb=d.nb,
                               ldc=G + d.nb, ta=1)
            # last bias gradient on the main stream: queued behind the auxiliary lanes' weight-gradient GEMMs it would finish later
            L.check(lib.spv_colsum(L.ptr(w.dh1), 2 * H, B, 2 * H, L.ptr(self.Gd(g, "b1")), st), "spv_colsum")
            self._join(g)
            if adam is not None:  # encoder range of this group
                for ev in tick_events:
                    torch.cuda.current_stream(self.device).wait_event(ev)
                if adam.get("sync") is not None:  # data parallel: sum this group's encoder gradients over the ranks first
                    adam["sync"](g)
                self._adam_range(*self.params.group_ranges[PHASE_ENC][g], adam)

    # -------------------------------------------------------------------------------- optimiser
    def adam_step(self, lr=1e-3, betas=(0.9, 0.999), eps=0.01, weight_decay=1e-6, grad_scale=1.0):
        if self.adam_m is None:
            self.adam_m = torch.zeros_like(self.params.flat)
            self.adam_v = torch.zeros_like(self.params.flat)
        st = self._stream()
        segs = self._stage_segments() if (self.bf16 and self.stage_in_adam) else []
        L.check(self.lib.spv_adam(L.ptr(self.params.flat), L.ptr(self.grads), L.ptr(self.adam_m), L.ptr(self.adam_v),
                                  self.params.numel, lr, betas[0], betas[1], eps, weight_decay, grad_scale,
                                  L.ptr(self.step_dev), L.ptr(self.adam_ticket), len(segs),
                                  L.ll_array([s[0] for s in segs]), L.int_array([s[1] for s in segs]),
                                  L.int_array([s[2] for s in segs]), L.ptr_array([s[3] for s in segs]),
                                  L.ptr_array([s[5] for s in segs]), L.int_array([s[6] for s in segs]),
                                  L.ll_array([s[4] for s in segs]), 0, st), "spv_adam")

    def adam_range_step(self, phase, lr=1e-3, betas=(0.9, 0.999), eps=0.01, weight_decay=1e-6, grad_scale=1.0):
        """Adam on one phase of the flat layout (PHASE_ENC / PHASE_DEC); the step counter must have been advanced already
        (backward(..., tick=True))"""
        self._adam_range(*self.params.ranges[phase], {"lr": lr, "betas": betas, "eps": eps, "weight_decay": weight_decay,
                                                      "grad_scale": grad_scale})

    def _adam_range(self, lo, hi, cfg, max_blocks=0):
        """Adam on the flat parameter range [lo, hi); *step already holds this update's index (spv_adam_tick)"""
        segs = ([s for s in self._stage_segments() if s[0] < hi and lo < s[0] + s[1] * s[2]]  # any overlap with the range
                if (self.bf16 and self.stage_in_adam) else [])
        betas = cfg.get("betas", (0.9, 0.999))
        off = 4 * lo
        L.check(self.lib.spv_adam(self.params.flat.data_ptr() + off, self.grads.data_ptr() + off, self.adam_m.data_ptr() + off,
                                  self.adam_v.data_ptr() + off, hi - lo, cfg["lr"], betas[0], betas[1], cfg["eps"],
                                  cfg["weight_decay"], cfg.get("grad_scale", 1.0), L.ptr(self.step_dev), None, len(segs),
                                  L.ll_array([s[0] - lo for s in segs]), L.int_array([s[1] for s in segs]),
                                  L.int_array([s[2] for s in segs]), L.ptr_array([s[3] for s in segs]),
                                  L.ptr_array([s[5] for s in segs]), L.int_array([s[6] for s in segs]),
                                  L.ll_array([s[4] for s in segs]), max_blocks, self._stream()), "spv_adam")

    def _stage_segments(self):
        """(flat offset, rows, cols, 16-bit destination, destination row pitch, residual plane or None, destination is fp16) of the
        weights the tensor-core path reads"""
        out = []
        for g, G in enumerate(self.d.genes):
            W1b, Wstack, W1b_lo = self.wb[g]
            out.append((self.params.offsets[g]["W1"][0], 2 * self.d.n_hidden, G + self.d.nb, W1b, W1b.stride(0), W1b_lo, 0))
            out.append((self.params.offsets[g]["Wm"][0], G, self.d.KMIX, Wstack, Wstack.stride(0), None, 1 if self.fused_nb else 0))
        return out

    def stage_weights(self):
        """refresh the bf16 operand copies of W1 / Wm from the fp32 parameters (bf16 mode; a no-op otherwise)"""
        if not self.bf16:
            return
        for off, rows, cols, dst, ld, dst_lo, f16 in self._stage_segments():
            src = self.params.flat[off:off + rows * cols]
            if dst_lo is None:
                self._to_dec(L.ptr(src), cols, L.ptr(dst), ld, rows, cols)
            else:
                L.check(self.lib.spv_to_bf16_split(L.ptr(src), cols, L.ptr(dst), L.ptr(dst_lo), ld, rows, cols, self._stream()),
                        "spv_to_bf16_split")
        self._staged_version = self.params.flat._version

    # -------------------------------------------------------------------------------- state
    def load_state_dict(self, sd: Dict[str, torch.Tensor]):
        """copy a reference-format state_dict (torch CPU/GPU tensors) into the flat stores"""
        missing = []
        for store in (self.params, self.buffers):
            for n in store.names():
                if n not in sd:
                    missing.append(n)
                    continue
                store.view(n).copy_(sd[n].to(self.device, torch.float32).reshape(store.view(n).shape))
        if missing:
            raise KeyError(f"state_dict is missing {missing[:4]}... ({len(missing)} keys)")

    def state_dict(self) -> "OrderedDict[str, torch.Tensor]":
        out = OrderedDict()
        for store in (self.params, self.buffers):
            for n in store.names():
                out[n] = store.view(n)
        return out

    def grad_dict(self) -> "OrderedDict[str, torch.Tensor]":
        return OrderedDict((n, self.params.view(n, self.grads)) for n in self.params.names())

    def set_kl_weight(self, w: float):
        self.kl_weight.fill_(float(w))

    def loss_terms(self):
        """(loss, kl_private0, kl_poe0, kl_private1, kl_poe1 means, rec0 mean, rec1 mean) as a device tensor"""
        return self.loss_out[:7]
