"""Writes tests/golden/reference_pin/ FROM THE REFERENCE ITSELF: what the UNMODIFIED reference code computes for every
comparison in tests/test_reference_pin_cpu.py (the cases, seeds and digests are that module's).

The reference runs on the torch-CPU TensorFlow shim through ``oracle/ref_runner.py``; each result is checked against
the oracle / engine on the spot with the test's own tolerance before it is stored.  Needs a checkout of the
reference (tfimm 0.2.14); run from the repo root:

    python tools/make_reference_pin_golden.py [--reference DIR]
"""
import argparse
import dataclasses
import importlib
import importlib.util
import json
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tensorflow-image-models_b200"))

import tfimm  # noqa: E402
from oracle import params  # noqa: E402
from oracle import ref_runner as rr  # noqa: E402

_spec = importlib.util.spec_from_file_location("reference_pin", ROOT / "tests" / "test_reference_pin_cpu.py")
T = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(T)


def _json(obj):
    return np.array(json.dumps(obj))


def shim_float64():
    out = {}
    rr.set_floatx("float64")
    try:
        for i, (family, name, overrides) in enumerate(T.CASES):
            omod = importlib.import_module(f"oracle.{family}")
            ref = rr.create_model(name, **overrides)
            cfg = T._engine_cfg(name, overrides)
            w = params.random_params(omod.param_shapes(cfg), seed=31, dtype=torch.float64)
            ref.assign(w, ignore_missing=T.IGNORE)
            x = params.test_images(2, *cfg.input_size, cfg.in_channels).double()
            y_ref, f_ref = ref(x, return_features=True)
            assert y_ref.dtype == torch.float64
            with torch.no_grad():
                y_or, f_or = omod.forward(cfg, w, x, return_features=True)
            assert T._nerr(y_or, y_ref) < 1e-12, name
            out[f"c{i}_meta"] = _json({"model": name, "overrides": overrides,
                                       "weight_shapes": {k: list(v) for k, v in ref.weight_shapes().items()},
                                       "logits_shape": list(y_ref.shape),
                                       "features": [[k, list(v.shape)] for k, v in f_ref.items()]})
            out[f"c{i}_logits"] = T.digest(y_ref, T.LOGIT_SAMPLES)
            out[f"c{i}_features"] = np.concatenate([T.digest(v, T.FEATURE_SAMPLES) for v in f_ref.values()])
            print(f"shim case {i} {name}: oracle vs reference {T._nerr(y_or, y_ref):.1e}")
    finally:
        rr.set_floatx("float32")
    return out


def vit_logits():
    from oracle import vit as ovit

    ref = rr.create_model("vit_tiny_patch16_224")
    cfg = T._engine_cfg("vit_tiny_patch16_224", {})
    w = params.random_params(ovit.param_shapes(cfg), seed=3)
    ref.assign(w)
    y32 = ref(params.test_images(1, 224, 224))
    assert y32.dtype == torch.float32
    assert T._nerr(ovit.forward(cfg, w, params.test_images(1, 224, 224)), y32) < 2e-6

    ov = {"input_size": (64, 64), "nb_blocks": 1, "interpolate_input": True}
    rr.set_floatx("float64")
    try:
        ref = rr.create_model("vit_tiny_patch16_224", **ov)
        cfg = T._engine_cfg("vit_tiny_patch16_224", ov)
        w = params.random_params(ovit.param_shapes(cfg), seed=4, dtype=torch.float64)
        ref.assign(w)
        x = params.test_images(1, 96, 128).double()
        y64 = ref(x)
    finally:
        rr.set_floatx("float32")
    assert T._nerr(ovit.forward(cfg, w, x), y64) < 1e-6
    return {"float32_224": y32.numpy(), "interpolate_input_float64": y64.numpy()}


def initial_values():
    ranges = {}
    for name, ov in T.INITIAL_VALUE_CASES:
        ranges[name] = {k: [float(v.min()), float(v.max())] for k, v in rr.create_model(name, **ov).weights_dict().items()}
    return {"meta": _json(ranges)}


def registry():
    with rr._reference_modules():
        mods = rr._import_reference()
        configs = {n: dataclasses.asdict(mods["registry"].model_config(n)) for n in T.REGISTRY_CONFIGS}
    return {"meta": _json({"list_models": {fam: rr.list_models(module=fam) for fam in rr.FAMILIES},
                           "configs": configs})}


def preprocessing():
    img = np.random.default_rng(0).integers(0, 256, (2, 16, 16, 3)).astype(np.uint8)
    out = {}
    for name in T.PREPROCESSING_MODELS:
        ref = rr.create_preprocessing(name, dtype="float32")
        with rr._reference_modules():
            a = ref(img)
        out[name] = np.asarray(a.numpy() if hasattr(a, "numpy") else a, dtype=np.float32)
    try:
        rr.create_preprocessing("not_a_model")
        raised = None
    except Exception as e:  # noqa: BLE001 -- the type is what is recorded
        raised = type(e).__name__
    out["meta"] = _json({"unknown_model_raises": raised})
    return out


def transfer_weights():
    out = {}
    for name, ov in T.TRANSFER_MODELS:
        fam = {"resnet18": "resnet", "vit_tiny_patch16_224": "vit", "convnext_tiny": "convnext"}[name]
        omod = importlib.import_module(f"oracle.{fam}")
        w = params.random_params(omod.param_shapes(T._engine_cfg(name, ov)), seed=17)
        for j, change in enumerate(T.TRANSFER_CHANGES):
            src_ref = rr.create_model(name, **ov)
            src_ref.assign(w, ignore_missing=T.IGNORE)
            dst_ref = rr.create_model(name, **ov, **change)
            before = dst_ref.weights_dict()
            rr.transfer_weights(src_ref, dst_ref)
            after = dst_ref.weights_dict()
            meta, digests = [], []
            for k, v in after.items():
                if any(p in k for p in T.IGNORE):
                    continue
                if np.array_equal(v, before[k]):
                    meta.append([k, "unchanged"])
                elif k in w and np.array_equal(v, w[k].numpy()):
                    meta.append([k, "source"])
                else:
                    meta.append([k, list(v.shape)])
                    digests.append(T.digest(v, T.FEATURE_SAMPLES))
            out[f"{name}_{j}_meta"] = _json(meta)
            out[f"{name}_{j}_digests"] = np.concatenate(digests) if digests else np.zeros(0)
            print(f"transfer {name} {change}: {sum(1 for _, h in meta if not isinstance(h, str))} digests")
    return out


def state_dict_conversion():
    out = {}
    for arch in T.CONVERSION_ARCHS:
        name, ov, sd = T.conversion_case(arch)
        ref = rr.create_model(name, **ov)
        rr.load_pytorch_weights(ref, {k: v.clone() for k, v in sd.items()})
        out[arch] = _json({k: T.array_hash(v) for k, v in ref.weights_dict().items()
                           if not any(p in k for p in T.IGNORE)})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", type=Path, default=rr.REFERENCE, help="checkout of the reference repository")
    args = ap.parse_args()
    rr.REFERENCE = args.reference
    if not rr.available():
        raise SystemExit(f"{args.reference} is not a checkout of the reference (tfimm/architectures/vit.py missing)")
    out_dir = ROOT / "tests" / "golden" / "reference_pin"
    out_dir.mkdir(parents=True, exist_ok=True)
    for make in (shim_float64, vit_logits, initial_values, registry, preprocessing, transfer_weights,
                 state_dict_conversion):
        path = out_dir / f"{make.__name__}.npz"
        np.savez_compressed(path, **make())
        print(path.name, f"{path.stat().st_size / 1024:.0f} KB")


if __name__ == "__main__":
    main()
