"""-m "not gpu": the flat parameter layout carries exactly the reference's state_dict names and shapes."""
import torch

from tests.helpers import Golden


def test_state_dict_roundtrip_matches_reference_names():
    from spvipes_b200.engine import StepEngine
    gd = Golden("label_tiny")
    eng = StepEngine((gd.G0, gd.G1), gd.H, gd.S, gd.P, gd.dropout, gd.mode, device="cpu")
    eng.load_state_dict(gd.sd)
    sd = eng.state_dict()
    ref_names = [k for k in gd.sd if not k.endswith("num_batches_tracked")]
    assert sorted(sd.keys()) == sorted(ref_names)
    for k in ref_names:
        assert tuple(sd[k].shape) == tuple(gd.sd[k].shape), k
        assert torch.equal(sd[k], gd.sd[k].float()), k
    # fused blocks are contiguous concatenations of the per-encoder tensors
    H = gd.H
    W1 = eng.P(0, "W1")
    assert torch.equal(W1[:H], gd.sd["encoder_0_private.fc1.weight"]) and torch.equal(W1[H:], gd.sd["encoder_0_shared.fc1.weight"])
    assert set(eng.grad_dict().keys()) == set(gd.grads.keys())


def test_flat_ranges_are_float4_aligned():
    """every phase / group range of the flat parameter layout starts and ends on a multiple of 4 floats: the gradient exchange
    kernel (csrc/xgpu.cu) and Adam work on float4"""
    from spvipes_b200.engine import StepEngine
    for genes in ((5000, 4999), (37, 41)):
        e = StepEngine(genes, 32, 7, 3, 0.1, "label", "cpu", precision="fp32")
        for ph, (lo, hi) in e.params.ranges.items():
            assert lo % 4 == 0 and hi % 4 == 0
            for glo, ghi in e.params.group_ranges[ph]:
                assert glo % 4 == 0 and ghi % 4 == 0 and lo <= glo <= ghi <= hi
