"""TEST INFRASTRUCTURE ONLY -- the launch census: every distinct kernel launch the model zoo produces.

The host side (``tfimm/architectures/*.py``) decides every launch shape, and the C++ dispatch picks a kernel from
that shape.  So the set of distinct launches over all registrations is the set of kernel paths the zoo can reach.
This module defines what makes two launches "the same" (``signature``), how a registration is run for the census
(``build_model``, ``images``, ``forward``) and how every launcher of ``tfimm.backend.ops`` is intercepted
(``intercepted_launchers``).  ``tools/make_launch_census.py`` writes the census with it: on a GPU from the real
launchers (``tests/golden/launch_census.json``), or with ``--host`` on CPU from the emulated launchers for
``HOST_NAMES`` without strides (``tests/golden/launch_census_host.json``, read by ``tests/test_launch_census_cpu.py``).
"""
import importlib
import inspect
import json
from contextlib import contextmanager, nullcontext
from pathlib import Path

import torch

from . import emulate_bf16, params

GOLDEN = Path(__file__).resolve().parent.parent / "tests" / "golden"
CENSUS_PATH = GOLDEN / "launch_census.json"
# One small registration per family: its host-side launches (without strides) are checked on CPU.
HOST_CENSUS_PATH = GOLDEN / "launch_census_host.json"
HOST_NAMES = ("vit_tiny_patch16_224", "deit_tiny_distilled_patch16_224", "swin_tiny_patch4_window7_224", "convnext_tiny",
              "efficientnet_b0", "resnet18", "seresnext26d_32x4d")

# An odd batch: the implicit conv puts two images in one tile, window counts become odd and the per-image gates of
# the squeeze-excite GEMM need more than one image and an uneven split.
BATCH = 3
WEIGHT_SEED = 7
MODES = ("bf16", "bf16_uint8", "bf16_features", "fp32")

# Every launching function of tfimm.backend.ops (the shape predicates launch nothing).
LAUNCHERS = tuple(n for n in emulate_bf16._EMULATED if n != "mlp_fused_supported")

_DT = {torch.float32: "f32", torch.bfloat16: "bf16", torch.uint8: "u8", torch.int32: "i32", torch.int64: "i64",
       torch.float64: "f64"}


def run_key(name, mode):
    return f"{name}/{mode}"


def bind(launcher, args, kwargs):
    """Arguments of one launch by parameter name, defaults filled in (the emulation has the launchers' signatures)."""
    ba = inspect.signature(getattr(emulate_bf16, launcher)).bind(*args, **kwargs)
    ba.apply_defaults()
    return dict(ba.arguments)


def _fmt(v, strides):
    if isinstance(v, torch.Tensor):
        s = f"{_DT[v.dtype]}[{','.join(map(str, v.shape))}]"
        return s + "{" + ",".join(map(str, v.stride())) + "}" if strides else s
    if isinstance(v, torch.dtype):
        return _DT[v]
    if isinstance(v, float):
        return repr(v)          # shortest round-trip form: distinct scales / eps stay distinct signatures
    if isinstance(v, (tuple, list)):
        return "(" + ",".join(_fmt(x, strides) for x in v) + ")"
    return repr(v)


def signature(launcher, bound, strides=True):
    """The launcher, every argument by name (tensors as dtype, shape and -- with ``strides`` -- strides; scalars by
    value) and whether ``out`` aliases ``residual``.  In-place launchers are told apart by their name."""
    body = ", ".join(f"{k}={_fmt(v, strides)}" for k, v in bound.items())
    out, res = bound.get("out"), bound.get("residual")
    alias = out is not None and res is not None and out.data_ptr() == res.data_ptr()
    return f"{launcher}({body})" + (" out=residual" if alias else "")


def launches(launcher, bound):
    """False for the calls that return without a kernel (a cast to the tensor's own dtype)."""
    return not (launcher == "cast" and bound["x"].dtype == bound["dtype"])


@contextmanager
def intercepted_launchers(hook):
    """Inside the block ``ops.<launcher>(*a, **k)`` calls ``hook(launcher, real_function, a, k)`` instead."""
    from tfimm.backend import ops

    saved = {n: getattr(ops, n) for n in LAUNCHERS}
    for n, f in saved.items():
        setattr(ops, n, (lambda n, f: lambda *a, **k: hook(n, f, a, k))(n, f))
    try:
        yield
    finally:
        for n, f in saved.items():
            setattr(ops, n, f)


def oracle_module(model):
    return importlib.import_module("oracle." + type(model).__module__.rsplit(".", 1)[-1])


def build_model(name, mode, device, weights=None):
    """The registration at the precision of ``mode`` with seeded random weights (pass ``weights`` to reuse them)."""
    import tfimm

    model = tfimm.create_model(name, precision="fp32" if mode == "fp32" else "bf16", device=device)
    if weights is None:
        weights = params.random_params(oracle_module(model).param_shapes(model.cfg), seed=WEIGHT_SEED)
    model.load_weights_dict(weights)
    return model, weights


def images(model, mode):
    cfg = model.cfg
    x = params.test_images(BATCH, *cfg.input_size, cfg.in_channels)
    if mode == "bf16_uint8":
        x = (x * 256.0).clamp(max=255.0).to(torch.uint8)
    return x


def forward(model, mode, x):
    with torch.no_grad():
        if mode == "bf16_features":
            return model(x, return_features=True)
        return model(x)


def load_census(path=CENSUS_PATH):
    with open(path) as f:
        return json.load(f)


def collect(names, modes=MODES, device="cuda", strides=True, emulate=False, log=None):
    """{run_key: [signature, ...]} (distinct, in first-launch order) for every registration in ``names`` and mode.
    ``emulate``: run the host orchestration on CPU with the float32 emulation of every launcher instead of kernels."""
    runs, current = {}, []

    def hook(launcher, real, a, k):
        bound = bind(launcher, a, k)
        if launches(launcher, bound):
            sig = signature(launcher, bound, strides)
            if sig not in current:
                current.append(sig)
        return real(*a, **k)

    with host_plan_on_cpu() if emulate else nullcontext():
        for name in names:
            weights = None
            for mode in modes:
                model, weights = build_model(name, mode, device, weights)
                current = runs.setdefault(run_key(name, mode), [])
                ctx = emulate_bf16.emulated_ops(torch.float32) if emulate else nullcontext()
                with ctx, intercepted_launchers(hook):
                    forward(model, mode, images(model, mode))
                del model
                if log:
                    log(f"{run_key(name, mode)}: {len(current)} signatures")
    return runs


@contextmanager
def host_plan_on_cpu():
    """Inside the block models on a CPU device compile their launch plan instead of refusing to run: the product path
    has no CPU fallback, but the host-side plan is device-agnostic, and with ``emulate_bf16.emulated_ops`` every
    launch it makes runs in torch."""
    from tfimm.models.model import Model

    def ensure_plan(self):
        if self._plan is None:
            self._plan = self._compile()
        return self._plan

    saved, Model._ensure_plan = Model._ensure_plan, ensure_plan
    try:
        yield
    finally:
        Model._ensure_plan = saved


def census_from_runs(runs):
    """The census file's content: each signature once, owned by the first run (registration-major, then MODES)
    that produces it, with every registration that produces it."""
    sigs, index = [], {}
    out_runs = {}
    for key, run_sigs in runs.items():
        name = key.split("/")[0]
        ids = []
        for s in run_sigs:
            if s not in index:
                index[s] = len(sigs)
                sigs.append({"sig": s, "owner": key, "registrations": []})
            entry = sigs[index[s]]
            if name not in entry["registrations"]:
                entry["registrations"].append(name)
            ids.append(index[s])
        out_runs[key] = ids
    return {"batch": BATCH, "weight_seed": WEIGHT_SEED, "modes": list(MODES), "runs": out_runs, "signatures": sigs}


def dumps(census):
    """The census as JSON with one run and one signature per line (reviewable diffs)."""
    head = ",\n".join(f"{json.dumps(k)}: {json.dumps(census[k])}" for k in ("batch", "weight_seed", "modes"))
    runs = ",\n".join(f"{json.dumps(k)}: {json.dumps(v)}" for k, v in census["runs"].items())
    sigs = ",\n".join(json.dumps(e) for e in census["signatures"])
    return "{\n" + head + ',\n"runs": {\n' + runs + '\n},\n"signatures": [\n' + sigs + "\n]\n}\n"
