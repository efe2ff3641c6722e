"""CPU: the host-side pieces of 384-px inputs (a 24 x 24 patch grid, 576 patch tokens): the model stand-in's `img_size`,
the synthetic features at 576 tokens and the per-entry-point table of supported patch-token counts."""
import pytest
import torch

from deltakd_b200 import deit, synth
from deltakd_b200 import functional as Fn
from deltakd_b200.features import FrozenTeacher, forward_with_features


def test_create_model_img_size():
    s = deit.create_model("deit_tiny_patch16_224", num_classes=10, img_size=384)
    t = deit.create_model("deit_small_distilled_patch16_224", num_classes=10, img_size=384)
    assert s.pos_embed.shape == (1, 577, 192) and t.pos_embed.shape == (1, 578, 384)
    assert deit.create_model("deit_tiny_patch16_224", num_classes=10).pos_embed.shape == (1, 197, 192)
    ft = FrozenTeacher(t, dtype=None)
    out, feats = forward_with_features(ft, torch.randn(1, 3, 384, 384), layers=(11,))
    assert out.shape == (1, 10) and feats[11].shape == (1, 578, 384)


def test_make_features_576_tokens():
    s, t = synth.make_features(2, 5, layers=[0, 11])
    s2, t2 = synth.make_features(2, 5, layers=[0, 11], n_tok=196)
    for a, b in zip(s + t, s2 + t2):          # the default is the 196-token draw, unchanged
        assert (a is None and b is None) or torch.equal(a, b)
    s3, t3 = synth.make_features(2, 5, layers=[0, 11], n_tok=576)
    assert s[0].shape == (2, 197, 192) and t[0].shape == (2, 198, 384)
    assert s3[11].shape == (2, 577, 192) and t3[11].shape == (2, 578, 384)
    s4, t4 = synth.make_features(2, 5, layers=[0], n_tok=576, teacher_dim=768)
    assert t4[0].shape == (2, 578, 768) and torch.equal(s4[0], s3[0])


def test_supported_grid_tokens_table():
    assert Fn.SUPPORTED_GRID_TOKENS == {"masked generation": (196, 576), "dkd_wass_sinkhorn": (196,)}


@pytest.mark.parametrize("n_tok", [225, 200])
def test_grid_check_names_the_supported_grids(monkeypatch, n_tok):
    """Masked generation names both grids, Sinkhorn its one grid; hidden-state matching takes any token count.  (The
    check follows the CUDA-tensor check, which is stubbed out here to exercise it on CPU tensors.)"""
    monkeypatch.setattr(Fn, "_require_cuda", lambda *a: None)
    s, t = torch.zeros(1, 1 + n_tok, 192), torch.zeros(1, 2 + n_tok, 384)
    with pytest.raises(ValueError, match=r"built for 196 patch tokens .* or 576 patch tokens .*got %d" % n_tok):
        Fn._check_feature_pair(s, t, 1, 2, op="masked generation")
    with pytest.raises(ValueError, match=r"built for 196 patch tokens .*got %d" % n_tok):
        Fn._check_feature_pair(s, t, 1, 2, op="dkd_wass_sinkhorn")
    Fn._check_feature_pair(s, t, 1, 2, op="dkd_align_mse")
    Fn._check_feature_pair(torch.zeros(1, 577, 192), torch.zeros(1, 578, 384), 1, 2, op="masked generation")
