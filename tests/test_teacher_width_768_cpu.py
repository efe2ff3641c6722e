"""CPU: the host-side pieces of the DeiT-Base (768-wide) teacher support: the model stand-in, the synthetic features
and the per-entry-point table of supported (student, teacher) widths."""
import torch

from deltakd_b200 import deit, synth
from deltakd_b200 import functional as Fn
from deltakd_b200.features import FrozenTeacher, forward_with_features


def test_deit_base_stand_in():
    for name, distilled in (("deit_base_patch16_224", False), ("deit_base_distilled_patch16_224", True)):
        m = deit.create_model(name, num_classes=10)
        assert m.embed_dim == 768 and len(m.blocks) == 12 and m.distilled == distilled
        assert all(b.attn.num_heads == 12 for b in m.blocks)
    ft = FrozenTeacher(m, dtype=None)
    out, feats = forward_with_features(ft, torch.randn(1, 3, 224, 224), layers=(0, 11))
    assert out.shape == (1, 10) and ft.embed_dim == 768
    assert feats[0].shape == (1, 198, 768) and feats[11].shape == (1, 198, 768) and feats[1] is None


def test_make_features_teacher_width():
    s, t = synth.make_features(2, 5, layers=[0, 3])
    s2, t2 = synth.make_features(2, 5, layers=[0, 3], teacher_dim=768)
    assert t[0].shape == (2, 198, 384) and t2[3].shape == (2, 198, 768)
    assert torch.equal(s[0], s2[0]) and torch.equal(s[3], s2[3])   # the student draws do not depend on the teacher width


def test_supported_pairs_table():
    both = ((192, 384), (192, 768))
    assert Fn.SUPPORTED_PAIRS["dkd_align_mse"] == both and Fn.SUPPORTED_PAIRS["dkd_wass_l1"] == both
    for op in ("dkd_align_nmse", "dkd_wass_sinkhorn", "masked generation", "LRKD"):
        assert Fn.SUPPORTED_PAIRS[op] == ((192, 384),), op
