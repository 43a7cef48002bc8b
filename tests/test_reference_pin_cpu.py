"""Pins the oracle (and the engine's host-side API) to the REFERENCE ITSELF.

TensorFlow cannot be installed here, so ``oracle/ref_runner.py`` executes the unmodified reference sources
(``tfimm/architectures/{vit,swin,convnext,efficientnet,resnet}.py`` + ``tfimm/layers`` +
``tfimm/models/{factory,registry}.py`` + ``tfimm/utils/timm.py`` of the reference) on a torch-CPU restatement of the
TF/Keras calls they make (``oracle/tf_shim``).  ``tools/make_reference_pin_golden.py`` ran that code on the seeded
inputs below and stored what it computed under ``tests/golden/reference_pin``; every test here compares with those
stored results, so the suite needs no copy of the reference.

Tensors too large to store whole are stored as a digest (``digest``): max|t|, a fixed-weight projection of every
element and a seeded sample of elements.  ``assert_close`` checks the elementwise bound on the sampled elements and
the two conditions it implies for all the others.
"""
import dataclasses
import hashlib
import importlib
import json
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent
for p in (str(ROOT), str(ROOT / "tensorflow-image-models_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

from oracle import params  # noqa: E402

GOLDEN = Path(__file__).resolve().parent / "golden" / "reference_pin"
IGNORE = ("attn_mask", "relative_position_index", "blur_kernel")

# (family, registered name, create_model overrides) -- the small configurations of the reference's own test-suite
# (tests/models/architectures.py: *_test_model) expressed as overrides of registered models, plus real registrations.
CASES = [
    ("vit", "vit_tiny_patch16_224", {"input_size": (32, 32), "patch_size": 8, "embed_dim": 4, "nb_blocks": 2, "nb_heads": 2, "nb_classes": 12}),
    ("vit", "deit_tiny_distilled_patch16_224", {"input_size": (32, 32), "patch_size": 8, "embed_dim": 4, "nb_blocks": 2, "nb_heads": 2, "nb_classes": 12}),
    ("vit", "vit_base_patch32_224_in21k", {"input_size": (64, 64), "embed_dim": 24, "nb_blocks": 2, "nb_heads": 3, "representation_size": 16, "nb_classes": 7}),
    ("vit", "vit_tiny_patch16_224", {"input_size": (96, 64), "nb_blocks": 3}),
    ("swin", "swin_tiny_patch4_window7_224", {"input_size": (32, 32), "patch_size": 2, "embed_dim": 4, "nb_blocks": (2, 2), "nb_heads": (1, 2), "window_size": 4, "nb_classes": 12}),
    ("swin", "swin_tiny_patch4_window7_224", {"input_size": (112, 112), "nb_blocks": (2, 2, 2), "nb_heads": (3, 6, 12)}),
    ("convnext", "convnext_tiny", {"input_size": (32, 32), "embed_dim": (3, 4, 5, 6), "nb_blocks": (1, 1, 1, 1), "nb_classes": 12}),
    ("convnext", "convnext_tiny", {"input_size": (64, 96), "nb_blocks": (1, 1, 2, 1)}),
    ("convnext", "convnext_tiny_in22k", {"input_size": (64, 64), "nb_blocks": (1, 1, 1, 1), "conv_mlp_block": True}),
    ("efficientnet", "efficientnet_b0", {"input_size": (64, 64)}),
    ("efficientnet", "efficientnet_b4", {"input_size": (76, 76)}),
    ("efficientnet", "pt_efficientnet_b0", {"input_size": (64, 80)}),
    ("efficientnet", "mobilenet_v2_100", {"input_size": (64, 64)}),
    ("efficientnet", "efficientnet_es", {"input_size": (64, 64)}),
    ("efficientnet", "efficientnet_lite0", {"input_size": (64, 64)}),
    ("efficientnet", "efficientnet_v2_b0", {"input_size": (64, 64)}),
    ("resnet", "resnet18", {"input_size": (64, 64)}),
    ("resnet", "resnet50", {"input_size": (64, 64)}),
    ("resnet", "resnet50d", {"input_size": (64, 64)}),
    ("resnet", "resnext50_32x4d", {"input_size": (64, 64)}),
    ("resnet", "seresnext26d_32x4d", {"input_size": (64, 64)}),
    ("resnet", "ecaresnet26t", {"input_size": (64, 64)}),
    ("resnet", "resnetblur50", {"input_size": (64, 64)}),
    ("resnet", "resnet50_gn", {"input_size": (64, 64)}),
    ("resnet", "resnetrs50", {"input_size": (64, 64)}),
]
INITIAL_VALUE_CASES = [("convnext_tiny", {"input_size": (32, 32), "nb_blocks": (1, 1, 1, 1)}),
                       ("vit_tiny_patch16_224", {"input_size": (32, 32), "nb_blocks": 1}),
                       ("resnet18", {"input_size": (32, 32)}), ("resnet50_gn", {"input_size": (32, 32)})]
REGISTRY_CONFIGS = ("vit_base_patch16_224", "swin_base_patch4_window7_224", "convnext_base", "efficientnet_b4",
                    "resnet50")
PREPROCESSING_MODELS = ["vit_base_patch16_224", "convnext_base", "efficientnet_b4", "resnet50"]
TRANSFER_MODELS = [("resnet18", {"input_size": (32, 32)}),
                   ("vit_tiny_patch16_224", {"input_size": (32, 32), "nb_blocks": 1}),
                   ("convnext_tiny", {"input_size": (32, 32), "nb_blocks": (1, 1, 1, 1)})]
TRANSFER_CHANGES = [{"in_channels": 1}, {"in_channels": 5}, {"nb_classes": 7}]
CONVERSION_ARCHS = ["resnet50", "vit_b_16"]

LOGIT_SAMPLES = 256
FEATURE_SAMPLES = 16


# ------------------------------------------------------------------------------------------ digests of stored tensors
def _sample_index(n, k):
    return np.arange(n) if n <= k else np.sort(np.random.default_rng(n).choice(n, k, replace=False))


def _projection_weights(n):
    return (np.arange(n) * 0.6180339887498949) % 1.0 - 0.5  # fixed weights in [-0.5, 0.5), no RNG


def digest(t, k):
    """[max|t|, sum_i w_i t_i, t at k seeded positions] in float64 (every element when t has at most k)."""
    a = np.asarray(t, dtype=np.float64).ravel()
    return np.concatenate([[np.abs(a).max(), a @ _projection_weights(a.size)], a[_sample_index(a.size, k)]])


def digest_len(shape, k):
    return 2 + min(int(np.prod(shape)), k)


def assert_close(t, dig, k, tol, relative=True, what=""):
    """|t - ref| < tol * scale elementwise, scale = max|ref| + 1e-6 (the reference's own metric, tests/test_timm.py:71)
    or 1 (relative=False), for the tensor ``ref`` that ``dig`` digests: asserted on the sampled elements; max|t| and
    the projection must then lie within tol * scale and tol * scale * sum|w| of the stored ones."""
    a = np.asarray(t, dtype=np.float64).ravel()
    bound = tol * ((dig[0] + 1e-6) if relative else 1.0)
    err = np.abs(a[_sample_index(a.size, k)] - dig[2:]).max()
    assert err < bound, (what, "sampled elements", err / bound * tol)
    assert abs(np.abs(a).max() - dig[0]) <= bound, (what, "max|t|", np.abs(a).max(), dig[0])
    w = _projection_weights(a.size)
    assert abs(a @ w - dig[1]) <= bound * np.abs(w).sum(), (what, "projection", a @ w, dig[1])


def _load(name):
    return np.load(GOLDEN / f"{name}.npz")


def _meta(data, key="meta"):
    return json.loads(str(data[key]))


def _nerr(a, b):
    a, b = a.double(), b.double()
    return (a - b).abs().max().item() / (b.abs().max().item() + 1e-6)


def _engine_cfg(name, overrides):
    import tfimm

    base = tfimm.models.model_config(name)
    return type(base)(**{**base.__dict__, **overrides})


def _plain(v):
    """Config values as JSON stores them (tuples become lists)."""
    return json.loads(json.dumps(v))


def array_hash(a):
    """Exact identity of a float32 array: its shape and bytes."""
    a = np.ascontiguousarray(np.asarray(a, dtype=np.float32))
    return hashlib.blake2b(repr(a.shape).encode() + a.tobytes(), digest_size=16).hexdigest()


def conversion_case(arch):
    """(engine model name, overrides, seeded timm-named state_dict) for a torchvision architecture."""
    import torchvision

    if arch == "resnet50":
        tv = torchvision.models.resnet50(weights=None)
        name, ov = "resnet50", {"input_size": (32, 32)}
        sd = {k: v for k, v in tv.state_dict().items()}
    else:
        tv = torchvision.models.VisionTransformer(image_size=32, patch_size=8, num_layers=2, num_heads=2, hidden_dim=16,
                                                  mlp_dim=64, num_classes=10)
        name, ov = "vit_tiny_patch16_224", {"input_size": (32, 32), "patch_size": 8, "embed_dim": 16, "nb_blocks": 2,
                                             "nb_heads": 2, "nb_classes": 10}
        # torchvision -> timm key names (the reference converts timm checkpoints)
        sd = {}
        for k, v in tv.state_dict().items():
            k = (k.replace("encoder.layers.encoder_layer_", "blocks.").replace("ln_1", "norm1").replace("ln_2", "norm2")
                 .replace("self_attention.in_proj_", "attn.qkv.").replace("self_attention.out_proj", "attn.proj")
                 .replace("mlp.0", "mlp.fc1").replace("mlp.3", "mlp.fc2").replace("encoder.ln", "norm")
                 .replace("conv_proj", "patch_embed.proj").replace("heads.head", "head")
                 .replace("class_token", "cls_token").replace("encoder.pos_embedding", "pos_embed"))
            sd[k] = v
    g = torch.Generator().manual_seed(0)
    sd = {k: (torch.randn(v.shape, generator=g) if v.is_floating_point() else v) for k, v in sd.items()}
    return name, ov, sd


# ------------------------------------------------------------------------------------------ the tests
@pytest.mark.parametrize("family,name,overrides", CASES, ids=[f"{c[1]}-{i}" for i, c in enumerate(CASES)])
def test_oracle_equals_reference_code_run_on_the_shim(family, name, overrides):
    """Same variables (names + shapes) and, in float64, the same logits to 1e-12: the oracle restates the
    reference's graph exactly.  (float32 run of the same comparison: ~3e-7, see tools/make_golden.py.)"""
    i = [c[1:] for c in CASES].index((name, overrides))
    data = _load("shim_float64")
    meta = _meta(data, f"c{i}_meta")
    assert (meta["model"], _plain(meta["overrides"])) == (name, _plain(overrides))
    omod = importlib.import_module(f"oracle.{family}")
    cfg = _engine_cfg(name, overrides)
    shapes = omod.param_shapes(cfg)
    loadable = {k: tuple(v) for k, v in meta["weight_shapes"].items() if not any(p in k for p in IGNORE)}
    assert set(loadable) == set(shapes), (sorted(set(loadable) ^ set(shapes))[:6])
    for k, shp in shapes.items():
        assert tuple(shp) == loadable[k], (k, shp, loadable[k])
    w = params.random_params(shapes, seed=31, dtype=torch.float64)
    x = params.test_images(2, *cfg.input_size, cfg.in_channels).double()
    with torch.no_grad():
        y_or, f_or = omod.forward(cfg, w, x, return_features=True)
    assert y_or.dtype == torch.float64 and list(y_or.shape) == meta["logits_shape"]
    assert_close(y_or, data[f"c{i}_logits"], LOGIT_SAMPLES, 1e-12, what="logits")
    # intermediate features: same keys in the same order, same values (tests/models/test_factory.py:205-222)
    assert list(f_or.keys()) == [k for k, _ in meta["features"]]
    digests, at = data[f"c{i}_features"], 0
    for k, shape in meta["features"]:
        assert list(f_or[k].shape) == shape, k
        n = digest_len(shape, FEATURE_SAMPLES)
        assert_close(f_or[k], digests[at:at + n], FEATURE_SAMPLES, 1e-11, what=k)
        at += n
    assert at == digests.size


def test_oracle_equals_reference_in_float32_at_full_size():
    """The reference's default dtype and a real registration at its native 224 px."""
    from oracle import vit as ovit

    cfg = _engine_cfg("vit_tiny_patch16_224", {})
    w = params.random_params(ovit.param_shapes(cfg), seed=3)
    x = params.test_images(1, 224, 224)
    want = torch.from_numpy(_load("vit_logits")["float32_224"])
    assert want.dtype == torch.float32
    assert _nerr(ovit.forward(cfg, w, x), want) < 2e-6


def test_vit_interpolate_input_equals_reference():
    """interpolate_input=True resamples pos_embed with tf.image.resize(bicubic) (layers/transformers.py:13-47)."""
    from oracle import vit as ovit

    ov = {"input_size": (64, 64), "nb_blocks": 1, "interpolate_input": True}
    cfg = _engine_cfg("vit_tiny_patch16_224", ov)
    w = params.random_params(ovit.param_shapes(cfg), seed=4, dtype=torch.float64)
    x = params.test_images(1, 96, 128).double()
    want = torch.from_numpy(_load("vit_logits")["interpolate_input_float64"])
    # tf.image.resize returns float32, so agreement is at float32 rounding of the position table
    assert _nerr(ovit.forward(cfg, w, x), want) < 1e-6


def test_reference_initial_values_match_engine_initialisers():
    """Variables created by build(): the engine's ParamSpec initialisers name the same constants
    (zeros cls/pos tokens vit.py:378-400, ConvNeXt layer scale 1e-6 convnext.py:211-217, zero-init last BN gamma
    with moving_variance = zeros only where the reference passes it, resnet.py:147-155).
    Stored: [min, max] of every reference variable right after build()."""
    import tfimm

    ranges = _meta(_load("initial_values"))
    for name, ov in INITIAL_VALUE_CASES:
        ref = ranges[name]
        eng = tfimm.create_model(name, device="cpu", **ov)
        for key, spec in eng.param_specs().items():
            kind, _, arg = spec.init.partition(":")
            if kind in ("zeros", "ones", "const"):
                want = {"zeros": 0.0, "ones": 1.0}.get(kind, float(arg) if arg else 0.0)
                assert np.allclose(ref[key], want), (name, key, spec.init, ref[key])


def test_list_models_and_configs_equal_the_reference_registry():
    import tfimm

    ref = _meta(_load("registry"))
    assert sorted(ref["list_models"]) == sorted(("vit", "swin", "convnext", "efficientnet", "resnet"))
    for fam, ref_names in ref["list_models"].items():
        assert tfimm.list_models(module=fam) == ref_names
    assert sorted(ref["configs"]) == sorted(REGISTRY_CONFIGS)
    for n, rc in ref["configs"].items():
        ec = dataclasses.asdict(tfimm.models.model_config(n))
        for k, v in rc.items():
            assert _plain(ec[k]) == v, (n, k, ec[k], v)


@pytest.mark.parametrize("name", PREPROCESSING_MODELS)
def test_create_preprocessing_equals_reference(name):
    import tfimm

    img = np.random.default_rng(0).integers(0, 256, (2, 16, 16, 3)).astype(np.uint8)
    data = _load("preprocessing")
    a = data[name]
    b = np.asarray(tfimm.create_preprocessing(name, dtype="float32")(img))
    assert a.shape == b.shape
    assert np.abs(a - b).max() < 1e-6
    assert _meta(data)["unknown_model_raises"] == "ValueError"
    with pytest.raises(ValueError):
        tfimm.create_preprocessing("not_a_model")


@pytest.mark.parametrize("name,ov", TRANSFER_MODELS)
@pytest.mark.parametrize("change", TRANSFER_CHANGES)
def test_transfer_weights_equals_reference(name, ov, change):
    """in_channels / nb_classes adaptation (tfimm/models/factory.py:174-305; tests/models/test_factory.py:37-90):
    the engine's transfer_weights writes the same values into the same variables as the reference's.
    Stored per reference variable: "unchanged" (the reference left its initial value), "source" (it copied the
    source model's value) or a digest of what it wrote."""
    import tfimm

    fam = {"resnet18": "resnet", "vit_tiny_patch16_224": "vit", "convnext_tiny": "convnext"}[name]
    omod = importlib.import_module(f"oracle.{fam}")
    cfg = _engine_cfg(name, ov)
    w = params.random_params(omod.param_shapes(cfg), seed=17)
    data = _load("transfer_weights")
    case = f"{name}_{TRANSFER_CHANGES.index(change)}"
    meta = _meta(data, f"{case}_meta")
    digests, at = data[f"{case}_digests"], 0

    src = tfimm.create_model(name, device="cpu", **ov)
    src.load_weights_dict(w)
    dst = tfimm.create_model(name, device="cpu", **ov, **change)
    init = dst.weights_dict()
    tfimm.models.transfer_weights(src, dst)
    got = dst.weights_dict()
    for k, how in meta:
        if how == "unchanged":
            if not np.array_equal(got[k], init[k]):
                raise AssertionError(f"{k}: the reference left it at its initial value, the engine overwrote it")
        elif how == "source":
            assert np.abs(got[k] - w[k].numpy()).max() < 1e-6, k
        else:
            assert list(got[k].shape) == how, k
            n = digest_len(how, FEATURE_SAMPLES)
            assert_close(got[k], digests[at:at + n], FEATURE_SAMPLES, 1e-6, relative=False, what=k)
            at += n
    assert at == digests.size


@pytest.mark.parametrize("arch", CONVERSION_ARCHS)
def test_pytorch_state_dict_conversion_equals_reference(arch):
    """N1: tfimm.utils.timm.convert_state_dict produces exactly what the reference's
    load_pytorch_weights_in_tf2_model (tfimm/utils/timm.py:109-229) writes into its variables.
    Stored: ``array_hash`` of every variable the reference loads."""
    import tfimm
    from tfimm.utils import timm as etimm

    name, ov, sd = conversion_case(arch)
    want = _meta(_load("state_dict_conversion"), arch)
    eng = tfimm.create_model(name, device="cpu", **ov)
    got, missing, unexpected = etimm.convert_state_dict(eng, sd)
    assert not missing
    for k, v in got.items():
        assert array_hash(v) == want[k], k
    assert set(got) == set(want)
