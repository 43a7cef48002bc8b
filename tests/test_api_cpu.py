"""CPU tests of the drop-in boundary: registry, factory, preprocessing, weight transfer, cache, C ABI exports.

They mirror the reference's tests/models/test_factory.py, tests/utils/test_cache.py and tests/utils/test_etc.py
for everything that does not need a forward pass (forward parity lives in the -m gpu tests).
"""
import json
import logging
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest
import torch

import tfimm
from tfimm.models import registry
from tfimm.models.factory import transfer_weights

ROOT = Path(__file__).resolve().parent.parent
ZOO = ROOT / "tensorflow-image-models_b200" / "tfimm" / "architectures" / "zoo"


def test_every_reference_registration_is_present():
    """list_models() == the names dumped from the reference's own registry (tools/extract_zoo.py)."""
    expected = set()
    for fam in ("vit", "swin", "convnext", "efficientnet", "resnet"):
        table = json.loads((ZOO / f"{fam}.json").read_text())
        expected |= set(table)
        assert set(tfimm.list_models(module=fam)) == set(table)
    assert set(tfimm.list_models()) == expected
    assert len(expected) == 36 + 10 + 19 + 61 + 60


def test_registered_configs_equal_reference_values():
    for fam in ("vit", "swin", "convnext", "efficientnet", "resnet"):
        table = json.loads((ZOO / f"{fam}.json").read_text())
        for name, fields in table.items():
            cfg = registry.model_config(name)
            assert type(cfg).__name__ == fields["__config__"]
            assert registry.model_class(name).__name__ == fields["__class__"]
            for k, v in fields.items():
                if k.startswith("__"):
                    continue
                got = getattr(cfg, k)
                got = json.loads(json.dumps(got))  # tuples -> lists
                assert got == v, (name, k, got, v)


def test_list_models_filters_and_natural_sort():
    names = tfimm.list_models("vit_base_patch*_224", exclude_filters="*sam*")
    assert names == ["vit_base_patch8_224", "vit_base_patch16_224", "vit_base_patch32_224"]  # 8 < 16 < 32
    assert tfimm.list_models("resnet*", module="vit") == []
    both = tfimm.list_models(["vit_tiny*", "deit_tiny*"], exclude_filters="*384")
    assert "vit_tiny_patch16_224" in both and "deit_tiny_patch16_224" in both and "vit_tiny_patch16_384" not in both
    assert "vit_large_patch32_224" not in tfimm.list_models(pretrained=True) or registry.model_config("vit_large_patch32_224").url
    assert set(registry.list_modules()) == {"vit", "swin", "convnext", "efficientnet", "resnet"}
    assert registry.is_model_in_modules("resnet50", ["resnet"]) and not registry.is_model_in_modules("resnet50", ["vit"])


def test_register_model_contract():
    from dataclasses import dataclass

    from tfimm.architectures.vit import ViT, ViTConfig

    def wrong_name():
        return ViT, ViTConfig(name="something_else")

    with pytest.raises(ValueError):
        registry.register_model(wrong_name)

    def vit_cpu_test_model():
        return ViT, ViTConfig(name="vit_cpu_test_model", input_size=(32, 32), patch_size=16, embed_dim=32, nb_blocks=1,
                              nb_heads=1, nb_classes=5)

    registry.register_model(vit_cpu_test_model)
    assert registry.is_model("vit_cpu_test_model")
    cfg = registry.model_config("vit_cpu_test_model")
    cfg.nb_classes = 7  # the registry stores a deep copy at registration ...
    m = tfimm.create_model("vit_cpu_test_model", device="cpu")
    assert m.cfg.nb_classes in (5, 7)  # ... and create_model deep-copies again
    assert m.name == m.cfg.name == "vit_cpu_test_model"


def test_create_model_errors_and_overrides(caplog):
    with pytest.raises(RuntimeError, match="Unknown model"):
        tfimm.create_model("not_a_model")
    with pytest.raises(ValueError, match="Unknown model"):
        tfimm.create_preprocessing("not_a_model")
    with caplog.at_level(logging.WARNING):
        m = tfimm.create_model("vit_tiny_patch16_224", device="cpu", nb_classes=10, nb_blocks=2, not_a_field=1, name="foo")
    assert "does not have field `not_a_field`" in caplog.text
    assert m.cfg.nb_classes == 10 and m.cfg.nb_blocks == 2 and m.name == "foo"
    assert registry.model_config("vit_tiny_patch16_224").nb_blocks == 12  # registered config untouched
    assert m.params["head/kernel"].shape == (192, 10)
    m0 = tfimm.create_model("vit_tiny_patch16_224", device="cpu", nb_classes=0, nb_blocks=1)
    assert "head/kernel" not in m0.params
    with pytest.raises(NotImplementedError):
        tfimm.create_model("vit_tiny_patch16_224", device="cpu", nb_blocks=1)(np.zeros((1, 224, 224, 3)), training=True)


def test_every_registration_constructs():
    """All 186 registrations build their variables (meta device: shapes only) -- none is left unimplemented."""
    names = [n for fam in ("vit", "swin", "convnext", "efficientnet", "resnet")
             for n in json.loads((ZOO / f"{fam}.json").read_text())]  # (other tests register scratch models)
    assert len(names) == 186
    for name in names:
        m = tfimm.create_model(name, device="meta")
        assert m.count_params() > 0, name


def test_no_cpu_fallback():
    from tfimm.backend.lib import KernelLibraryError

    m = tfimm.create_model("vit_tiny_patch16_224", device="cpu", nb_blocks=1)
    with pytest.raises(KernelLibraryError, match="no CPU fallback"):
        m(m.dummy_inputs)


@pytest.mark.parametrize("name", ["vit_tiny_patch16_224", "swin_tiny_patch4_window7_224", "convnext_tiny", "efficientnet_b0", "resnet18"])
def test_weight_names_follow_reference_convention(name):
    m = tfimm.create_model(name, device="cpu")
    assert m.name == m.cfg.name
    for w in m.weights:
        assert w.name.startswith(m.name + "/") and w.name.endswith(":0")
    assert tuple(m.dummy_inputs.shape) == (1, *m.cfg.input_size, m.cfg.in_channels)


@pytest.mark.parametrize("in_channels", [1, 3, 5, 6])
@pytest.mark.parametrize("dtype", ["float32", "float16"])
def test_preprocessing(in_channels, dtype):
    """reference tests/models/test_factory.py:127-137 plus the values."""
    pre = tfimm.create_preprocessing("resnet18", in_channels=in_channels, dtype=dtype)
    img = np.random.default_rng(0).integers(0, 255, size=(11, 13, in_channels)).astype(np.uint8)
    out = pre(img)
    assert out.shape == img.shape and out.dtype == np.dtype(dtype)
    batch = pre(img[None])
    assert batch.shape == (1, *img.shape)
    mean = (list(tfimm.utils.IMAGENET_DEFAULT_MEAN) * 3)[:in_channels]
    std = (list(tfimm.utils.IMAGENET_DEFAULT_STD) * 3)[:in_channels]
    ref = (img.astype(np.float64) / 255.0 - mean) / std
    assert np.abs(out.astype(np.float64) - ref).max() < (1e-5 if dtype == "float32" else 5e-3)
    tout = pre(torch.from_numpy(img))
    assert isinstance(tout, torch.Tensor) and np.abs(tout.numpy().astype(np.float64) - ref).max() < 5e-3


def test_transfer_weights_classifier_and_first_conv():
    """reference tests/models/test_factory.py:37-90 (the weight bookkeeping part)."""
    src = tfimm.create_model("resnet18", device="cpu", seed=1)
    dst = tfimm.create_model("resnet18", device="cpu", seed=2, nb_classes=10, in_channels=1)
    fc_before = dst.params["remove/fc/kernel"].clone()
    transfer_weights(src, dst)
    assert torch.equal(dst.params["remove/fc/kernel"], fc_before)          # different class count: kept
    assert torch.allclose(dst.params["conv1/kernel"], src.params["conv1/kernel"].sum(dim=2, keepdim=True))
    assert torch.equal(dst.params["layer1/0/conv1/kernel"], src.params["layer1/0/conv1/kernel"])
    dst6 = tfimm.create_model("resnet18", device="cpu", seed=3, in_channels=6)
    transfer_weights(src, dst6)
    k = src.params["conv1/kernel"]
    assert torch.allclose(dst6.params["conv1/kernel"], torch.cat([k, k], dim=2) * 0.5)
    assert torch.equal(dst6.params["remove/fc/kernel"], src.params["remove/fc/kernel"])  # same classes: copied


def test_transfer_weights_interpolates_pos_embed():
    src = tfimm.create_model("vit_tiny_patch16_224", device="cpu", nb_blocks=1, seed=1)
    src.load_weights_dict({"pos_embed": torch.randn(1, 197, 192)}, strict=False)
    dst = tfimm.create_model("vit_tiny_patch16_224", device="cpu", nb_blocks=1, input_size=(384, 384), seed=2)
    transfer_weights(src, dst)
    assert dst.params["pos_embed"].shape == (1, 1 + 24 * 24, 192)
    assert torch.equal(dst.params["pos_embed"][:, :1], src.params["pos_embed"][:, :1])


def test_save_and_reload_weights(tmp_path):
    from tfimm.models import save_weights

    m = tfimm.create_model("convnext_tiny", device="cpu", seed=5, nb_blocks=(1, 1, 1, 1))
    path = str(tmp_path / "w.npz")
    save_weights(m, path)
    tfimm.set_model_cache("convnext_tiny", path)
    try:
        assert tfimm.cached_model_path("convnext_tiny") == path and tfimm.list_cached_models() == ["convnext_tiny"]
        with pytest.raises(ValueError):  # registered depths (3,3,9,3) need more weights than the file holds
            tfimm.create_model("convnext_tiny", pretrained=True, device="cpu")
    except AttributeError:
        pass
    finally:
        tfimm.clear_model_cache("convnext_tiny")
    m2 = tfimm.create_model("convnext_tiny", device="cpu", seed=6, nb_blocks=(1, 1, 1, 1))
    m2.load_weights_dict(dict(np.load(path)))
    for k in m.params:
        assert torch.equal(m.params[k], m2.params[k])


def test_cache_dir(monkeypatch, tmp_path):
    monkeypatch.delenv("TFIMM_HOME", raising=False)
    monkeypatch.setenv("XDG_CACHE_HOME", "/some/cache")
    assert tfimm.get_dir() == "/some/cache/tfimm"
    monkeypatch.setenv("TFIMM_HOME", "/other")
    assert tfimm.get_dir() == "/other"
    tfimm.set_dir(str(tmp_path))
    try:
        assert tfimm.get_dir() == str(tmp_path)
        (tmp_path / "resnet18").mkdir()
        assert tfimm.cached_model_path("resnet18") == str(tmp_path / "resnet18")
        assert tfimm.cached_model_path("resnet50") is None
    finally:
        tfimm.set_dir(None)


def test_etc_helpers():
    from tfimm.utils import make_divisible, to_2tuple

    assert to_2tuple(3) == (3, 3) and to_2tuple((1, 2, 3)) == (1, 2)
    assert [make_divisible(v, 8) for v in (32 * 1.4, 16 * 1.4, 24 * 1.4, 1280 * 1.4, 10, 3)] == [48, 24, 32, 1792, 16, 8]
    assert make_divisible(2048 * 0.0625, 8, round_limit=0.0) == 128


def test_c_abi_library_exports_every_declared_symbol():
    """The .so loads without a GPU and exports exactly what include/tfimm_b200.h declares."""
    from tfimm.backend import lib

    handle = lib.load()
    header = (ROOT / "include" / "tfimm_b200.h").read_text()
    declared = set(re.findall(r"\b(tfimm_b200_[a-z0-9_]+)\s*\(", header))
    assert declared == set(lib.exported_symbols()), declared ^ set(lib.exported_symbols())
    nm = subprocess.run(["nm", "-D", "--defined-only", str(lib.LIB_PATH)], capture_output=True, text=True).stdout
    exported = set(re.findall(r"\sT\s+(tfimm_b200_[a-z0-9_]+)", nm))
    assert declared <= exported, declared - exported
    assert handle.tfimm_b200_version().decode().startswith("tfimm_b200")
    # arity of every binding matches the header's parameter list
    for name, argtypes in lib.SIGNATURES.items():
        m = re.search(name + r"\s*\(([^;]*?)\)\s*;", header, re.S)
        assert m, name
        params = [p.strip() for p in m.group(1).split(",") if p.strip() and p.strip() != "void"]
        assert len(params) == len(argtypes), (name, len(params), len(argtypes))
        # ... and so does the kind of every parameter (pointer / int / long / float): a float passed as int, or a
        # 64-bit stride passed as int, would be silent garbage through ctypes
        import ctypes

        for p, ct in zip(params, argtypes):
            want = ctypes.c_void_p if "*" in p else ctypes.c_float if p.startswith("float") else \
                ctypes.c_long if p.startswith("long") else ctypes.c_int
            assert ct is want, (name, p, ct)


def test_every_kernel_of_the_library_belongs_to_a_bench_family():
    """bench.py's roofline table and tools/ncu_traffic.py group launches by kernel family: every __global__ function of
    the built library must map to one (a new kernel without a family would silently drop out of `roofline.traffic`)."""
    import re
    import shutil
    import subprocess
    import sys
    from pathlib import Path

    if shutil.which("cuobjdump") is None or shutil.which("c++filt") is None:
        pytest.skip("cuobjdump / c++filt not available")
    root = Path(__file__).resolve().parent.parent
    lib = root / "tensorflow-image-models_b200" / "tfimm" / "backend" / "libtfimm_b200.so"
    if not lib.exists():
        pytest.skip("library not built")
    out = subprocess.run(["cuobjdump", "--dump-resource-usage", str(lib)], capture_output=True, text=True).stdout
    names = sorted(set(re.findall(r"Function (\S+?):", out)))
    assert len(names) > 100, len(names)
    dem = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
    sys.path.insert(0, str(root / "tools"))
    import ncu_traffic

    unmapped = [d for d in dem if ncu_traffic.family_of(d).startswith("other:")]
    assert not unmapped, unmapped[:5]


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU stand-in the driver times beside the GPU arm) runs without a GPU and prints
    one JSON line with the contract's keys."""
    import sys
    from pathlib import Path

    root = Path(__file__).resolve().parent.parent
    res = subprocess.run([sys.executable, str(root / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--ref-batch", "2", "--model", "vit_tiny_patch16_224"], capture_output=True, text=True,
                         timeout=600, cwd=str(root))
    assert res.returncode == 0, res.stderr[-2000:]
    line = [ln for ln in res.stdout.splitlines() if ln.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "images/sec"
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["value"] > 0


def test_bench_dump_outputs_writes_the_timed_logits(tmp_path, monkeypatch):
    """`--dump-outputs DIR` writes the last timed step's logits (seeded inputs: the same on every run) as float32 .npy,
    and keeps a fixed sample of rows when the outputs exceed the size limit."""
    import sys

    root = Path(__file__).resolve().parent.parent
    dumps = []
    for run in ("a", "b"):
        res = subprocess.run([sys.executable, str(root / "bench.py"), "--impl", "reference", "--steps", "2", "--warmup",
                              "1", "--ref-batch", "2", "--model", "vit_tiny_patch16_224", "--dump-outputs",
                              str(tmp_path / run)], capture_output=True, text=True, timeout=600, cwd=str(root))
        assert res.returncode == 0, res.stderr[-2000:]
        assert sorted(p.name for p in (tmp_path / run).iterdir()) == ["vit_tiny_patch16_224.npy"]
        dumps.append(np.load(tmp_path / run / "vit_tiny_patch16_224.npy"))
    assert dumps[0].dtype == np.float32 and dumps[0].shape == (2, 1000)
    assert np.array_equal(dumps[0], dumps[1])
    from oracle import params
    from oracle import vit as ovit

    cfg = tfimm.models.model_config("vit_tiny_patch16_224")
    want = ovit.forward(cfg, params.random_params(ovit.param_shapes(cfg), seed=0), params.test_images(2, 224, 224))
    assert np.abs(dumps[0] - want.numpy()).max() <= 1e-4 * np.abs(want.numpy()).max()

    sys.path.insert(0, str(root))
    import bench

    monkeypatch.setattr(bench, "DUMP_BYTES", 4096)
    big = torch.arange(400 * 4, dtype=torch.float64).reshape(400, 4)
    for run in ("c", "d"):
        bench.dump_outputs(tmp_path / run, {"big": big, "small": torch.ones(3, 2)})
    a = np.load(tmp_path / "c" / "big.npy")
    assert a.dtype == np.float32 and a.shape == (128, 4) and np.array_equal(a, np.load(tmp_path / "d" / "big.npy"))
    assert np.all(np.diff(a[:, 0]) > 0) and np.all(a[:, 0] % 4 == 0)  # whole rows of the original, in order
    assert np.array_equal(np.load(tmp_path / "c" / "small.npy"), np.ones((3, 2), np.float32))
