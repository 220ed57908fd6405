"""Host-side pieces of fine-tuning above 224 px: the entry point's ``--img-size`` and the 384 px model names."""
import importlib.util
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _vit_cp():
    import sys
    sys.path.insert(0, os.path.join(ROOT, "image_classification"))
    spec = importlib.util.spec_from_file_location("vit_cp_img_size", os.path.join(ROOT, "image_classification", "vit_cp.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_img_size_defaults_and_accepts_patch_multiples():
    m = _vit_cp()
    assert m._parse_args([]).img_size == 224
    assert m._parse_args(["--img-size=384"]).img_size == 384
    assert m._parse_args(["--model=vit_base_patch16_384"]).img_size == 384
    assert m._parse_args(["--model=vit_huge_patch14_224_in21k", "--img-size=518"]).img_size == 518


@pytest.mark.parametrize("argv", [["--img-size=100"], ["--img-size=0"], ["--img-size=-16"],
                                  ["--model=vit_huge_patch14_224_in21k", "--img-size=384"]])
def test_img_size_rejects_non_multiples_of_the_patch(argv, capsys):
    m = _vit_cp()
    with pytest.raises(SystemExit) as e:
        m._parse_args(argv)
    assert e.value.code == 2
    assert "not a positive multiple of the patch size" in capsys.readouterr().err


@pytest.mark.parametrize("name,width", [("vit_base_patch16_384", 768), ("vit_large_patch16_384", 1024)])
def test_384_models_have_577_tokens(name, width):
    from cara_b200.vit import create_model
    vit = create_model(name, depth=1)
    assert vit.pos_embed.shape == (1, 577, width)
    assert vit.head.out_features == 1000


def test_synthetic_data_follows_img_size():
    import sys
    sys.path.insert(0, os.path.join(ROOT, "image_classification"))
    import vtab
    tr, va = vtab.get_data("svhn", batch_size=4, synthetic=True, train_len=8, val_len=4, img_size=384)
    x, _ = next(iter(tr))
    assert x.shape == (4, 3, 384, 384)
