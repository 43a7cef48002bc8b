"""What the host side launches, and which kernels the library holds, checked without a GPU.

* ``tests/golden/launch_census_host.json``: the host orchestration of one small registration per family
  (``oracle.launch_census.HOST_NAMES``), run in each of the four census modes at batch 3 on CPU with the emulated
  launchers, produces exactly the committed launch signatures (launcher, tensor dtypes and shapes, scalar arguments,
  ``out``/``residual`` aliasing; strides are left out because the emulation returns contiguous tensors where the
  kernels return ``ldc``-padded views).  A host-side change that alters what is launched -- a shape, a fused path
  taken or dropped, a different activation or block_n -- shows up here before any GPU run; regenerate the file with
  ``python tools/make_launch_census.py --host`` when the change is intended.
* ``tests/golden/kernel_symbols.txt`` lists the ``__global__`` functions of the library built from this tree (the
  ``Function :`` headers of ``cuobjdump -sass``, demangled), so that an added or dropped kernel instantiation is a
  visible change of that file.
"""
import shutil
import subprocess
from pathlib import Path

import pytest

from oracle import launch_census as lc

GOLDEN = Path(__file__).resolve().parent / "golden"
LIB = Path(__file__).resolve().parent.parent / "tensorflow-image-models_b200" / "tfimm" / "backend" / "libtfimm_b200.so"


@pytest.fixture(scope="module")
def host_census():
    return lc.load_census(lc.HOST_CENSUS_PATH)


def test_host_census_is_well_formed(host_census):
    assert host_census["batch"] == lc.BATCH and host_census["modes"] == list(lc.MODES)
    assert list(host_census["runs"]) == [lc.run_key(n, m) for n in lc.HOST_NAMES for m in lc.MODES]
    sigs = [e["sig"] for e in host_census["signatures"]]
    assert len(set(sigs)) == len(sigs)
    for i, e in enumerate(host_census["signatures"]):
        producers = [k for k, ids in host_census["runs"].items() if i in ids]
        assert e["owner"] == producers[0], e["sig"]              # the first run that produces it, in run order
        assert e["registrations"] == list(dict.fromkeys(k.split("/")[0] for k in producers)), e["sig"]


def test_host_orchestration_launches_the_committed_signatures(host_census):
    runs = lc.collect(lc.HOST_NAMES, device="cpu", strides=False, emulate=True)
    assert list(runs) == list(host_census["runs"])
    for key, sigs in runs.items():
        committed = [host_census["signatures"][i]["sig"] for i in host_census["runs"][key]]
        assert sigs == committed, (key, sorted(set(sigs) ^ set(committed))[:4])


def test_signature_records_aliasing_and_skips_no_op_casts():
    import torch

    a = torch.zeros(4, 8, dtype=torch.bfloat16)
    w = torch.zeros(16, 8, dtype=torch.bfloat16)
    r = torch.zeros(4, 16)
    aliased = lc.signature("gemm", lc.bind("gemm", (a, w), {"residual": r, "out": r}))
    separate = lc.signature("gemm", lc.bind("gemm", (a, w), {"residual": r, "out": r.clone()}))
    assert aliased.endswith(" out=residual") and not separate.endswith(" out=residual")
    assert "a=bf16[4,8]{8,1}" in separate and "a=bf16[4,8]," in lc.signature("gemm", lc.bind("gemm", (a, w), {}),
                                                                                strides=False)
    qkv = torch.zeros(6, 3 * 2 * 64, dtype=torch.bfloat16)
    s1, s2 = (lc.signature("attention", lc.bind("attention", (qkv, 2, 3, 2, 64, sc), {})) for sc in (0.125, 0.1250000001))
    assert s1 != s2                                      # scalars are kept to full precision
    assert not lc.launches("cast", lc.bind("cast", (r, torch.float32), {}))
    assert lc.launches("cast", lc.bind("cast", (r, torch.bfloat16), {}))


def _tool(name):
    found = shutil.which(name)
    if found is None and (Path("/usr/local/cuda/bin") / name).exists():
        found = str(Path("/usr/local/cuda/bin") / name)
    return found


def library_kernel_symbols(lib=LIB):
    """Demangled names of the ``__global__`` functions in ``lib`` (the ``Function :`` headers of ``cuobjdump -sass``)."""
    sass = subprocess.run([_tool("cuobjdump"), "-sass", str(lib)], capture_output=True, text=True, check=True).stdout
    mangled = sorted({line.split("Function :", 1)[1].strip() for line in sass.splitlines() if "Function :" in line})
    demangled = subprocess.run([_tool("cu++filt")], input="\n".join(mangled) + "\n", capture_output=True, text=True,
                               check=True).stdout
    return sorted({s.strip() for s in demangled.splitlines() if s.strip()})


@pytest.mark.skipif(_tool("cuobjdump") is None or _tool("cu++filt") is None, reason="cuobjdump / cu++filt not found")
def test_kernel_symbol_table_matches_the_library():
    committed = (GOLDEN / "kernel_symbols.txt").read_text().splitlines()
    assert library_kernel_symbols() == committed
