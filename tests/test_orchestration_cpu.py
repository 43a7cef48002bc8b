"""The engine's HOST side, on CPU: weight layout transforms, BatchNorm folding, Swin row maps / bias tables / region
masks, the pruned last ViT block, squeeze-excite gate routing, the fused-MLP and gated-GEMM call sites -- everything in
``tfimm/architectures/*.py`` that decides WHAT is launched -- executed with every ``tfimm.backend.ops`` launcher
replaced by its exact float64 torch restatement (``oracle/emulate_bf16.py``, test infrastructure) and compared with the
reference-pinned oracle.  No kernel runs here: the product path still refuses a CPU device (checked below); the test
lifts that guard for itself only.

fp32 models (no bf16 storage anywhere) must reproduce the oracle to 1e-5; bf16 models exercise the bf16-only branches
(fused MLP, gate inside the projection GEMM, tensor-core window attention tables) and must land within the bf16 error
budget measured on B200 (DESIGN.md section 5).
"""
import importlib

import pytest
import torch


def _nerr(out, ref):
    out, ref = out.float().cpu(), ref.float().cpu()
    return (out - ref).abs().max().item() / (ref.abs().max().item() + 1e-6)


@pytest.fixture
def cpu_engine():
    from oracle.launch_census import host_plan_on_cpu

    with host_plan_on_cpu():
        yield


CASES = [
    ("vit", "vit_tiny_patch16_224", {"nb_blocks": 2, "input_size": (64, 64)}, 2),
    ("vit", "deit_tiny_distilled_patch16_224", {"nb_blocks": 2, "input_size": (64, 64)}, 2),
    ("swin", "swin_tiny_patch4_window7_224", {"input_size": (112, 112), "nb_blocks": (2, 2), "nb_heads": (3, 6)}, 1),
    ("convnext", "convnext_tiny", {"input_size": (64, 96), "nb_blocks": (1, 1, 1, 1)}, 1),
    ("efficientnet", "efficientnet_b0", {"input_size": (96, 96)}, 1),
    ("efficientnet", "efficientnet_v2_b0", {"input_size": (64, 64)}, 1),
    ("resnet", "resnet18", {"input_size": (64, 64)}, 2),
    ("resnet", "seresnext26d_32x4d", {"input_size": (64, 64)}, 1),
]


def _build(family, name, overrides, precision):
    import tfimm
    from oracle import params

    omod = importlib.import_module(f"oracle.{family}")
    model = tfimm.create_model(name, precision=precision, device="cpu", **overrides)
    w = params.random_params(omod.param_shapes(model.cfg), seed=7)
    model.load_weights_dict(w)
    return model, omod, w


def test_product_path_refuses_cpu():
    import tfimm
    from tfimm.backend.lib import KernelLibraryError

    model = tfimm.create_model("vit_tiny_patch16_224", precision="fp32", device="cpu", nb_blocks=1)
    with pytest.raises(KernelLibraryError, match="no CPU fallback"):
        model(torch.zeros(1, 224, 224, 3))


@pytest.mark.parametrize("family,name,overrides,batch", CASES, ids=[c[1] for c in CASES])
def test_fp32_orchestration_reproduces_the_oracle(cpu_engine, family, name, overrides, batch):
    from oracle import emulate_bf16, params

    model, omod, w = _build(family, name, overrides, "fp32")
    x = params.test_images(batch, *model.cfg.input_size, model.cfg.in_channels)
    with emulate_bf16.emulated_ops():
        y = model(x)
        feats = model(x, return_features=True)[1]
    with torch.no_grad():
        ref = omod.forward(model.cfg, w, x)
    assert y.shape == ref.shape
    assert _nerr(y, ref) < 1e-5
    assert _nerr(feats["logits"], ref) < 1e-5       # the return_features route computes every block in full


@pytest.mark.parametrize("family,name,overrides,batch", CASES, ids=[c[1] for c in CASES])
def test_bf16_orchestration_stays_inside_the_bf16_budget(cpu_engine, family, name, overrides, batch):
    from oracle import emulate_bf16, params
    from tfimm.backend import ops

    model, omod, w = _build(family, name, overrides, "bf16")
    x = params.test_images(batch, *model.cfg.input_size, model.cfg.in_channels)
    called = set()
    with emulate_bf16.emulated_ops():
        for n in ("mlp_fused", "gemm_gated", "window_attention_tc", "attention_cls", "conv_gemm"):
            f = getattr(ops, n)
            setattr(ops, n, (lambda f, n: lambda *a, **k: (called.add(n), f(*a, **k))[1])(f, n))
        y = model(x)
    with torch.no_grad():
        ref = omod.forward(model.cfg, w, x)
    assert _nerr(y, ref) < 1.2e-2
    expect = {"vit": {"attention_cls"}, "swin": {"window_attention_tc", "mlp_fused"}, "convnext": {"mlp_fused"},
              "efficientnet": set(), "resnet": {"conv_gemm"} if name == "resnet18" else set()}[family]
    assert expect <= called, (expect, called)


def test_efficientnet_gate_routing(cpu_engine):
    """>= 256 pixels per image: the squeeze-excite gate rides in the projection GEMM; smaller maps keep scale_channels_."""
    from oracle import emulate_bf16, params
    from tfimm.backend import ops

    model, omod, w = _build("efficientnet", "efficientnet_b0", {"input_size": (128, 128)}, "bf16")
    x = params.test_images(1, 128, 128, 3)
    gated_hw, scaled_hw = [], []
    with emulate_bf16.emulated_ops():
        g0, s0 = ops.gemm_gated, ops.scale_channels_
        ops.gemm_gated = lambda a, gate, hw, *r, **k: (gated_hw.append(hw), g0(a, gate, hw, *r, **k))[1]
        ops.scale_channels_ = lambda t, gate: (scaled_hw.append(t.shape[1] * t.shape[2]), s0(t, gate))[1]
        y = model(x)
    ref = omod.forward(model.cfg, w, x)
    assert _nerr(y, ref) < 1.2e-2
    assert gated_hw and min(gated_hw) >= 256
    assert scaled_hw and max(scaled_hw) < 256
