"""Regenerate tests/golden/launch_census.json: every distinct kernel launch of every registration (needs a B200).

    python tools/make_launch_census.py [--out PATH] [--only NAME ...]
    python tools/make_launch_census.py --host        # CPU: tests/golden/launch_census_host.json

Each registration runs one forward per mode of ``oracle.launch_census.MODES`` (bf16 with float32 images, bf16 with
uint8 images, bf16 with ``return_features=True``, fp32) at batch 3 with seeded random weights, on the real
launchers: their ``ldc``-padded outputs give strides the CPU emulation does not reproduce.  The output depends only
on the host-side code, so a rerun on the same tree writes the same bytes.

``--host`` runs ``oracle.launch_census.HOST_NAMES`` on CPU instead, with the float32 emulation of every launcher, and
records the signatures without strides (the emulation returns contiguous tensors where the kernels return padded
views).  tests/test_launch_census_cpu.py checks the host orchestration against that file.
"""
import argparse
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
for p in (str(ROOT), str(ROOT / "tensorflow-image-models_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)


def main():
    import torch

    import tfimm
    from oracle import launch_census as lc

    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--only", nargs="*", default=None, help="registrations to run (default: all)")
    ap.add_argument("--host", action="store_true", help="CPU, emulated launchers, no strides, HOST_NAMES")
    args = ap.parse_args()
    t0 = time.time()
    log = lambda s: print(f"[{time.time() - t0:6.0f}s] {s}", flush=True)  # noqa: E731
    if args.host:
        out = args.out or str(lc.HOST_CENSUS_PATH)
        runs = lc.collect(args.only or lc.HOST_NAMES, device="cpu", strides=False, emulate=True, log=log)
    else:
        assert torch.cuda.is_available(), "the census records the real launchers: it needs a CUDA device"
        out = args.out or str(lc.CENSUS_PATH)
        runs = lc.collect(args.only or tfimm.list_models(), device="cuda", log=log)
    census = lc.census_from_runs(runs)
    text = lc.dumps(census)
    Path(out).write_text(text)
    print(f"{len(census['signatures'])} signatures from {len(runs)} runs -> {out} ({len(text) / 1e6:.1f} MB)")


if __name__ == "__main__":
    main()
