import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_collection_modifyitems(config, items):
    """`gpu`-marked tests need a CUDA device: skip them (instead of failing with 'no NVIDIA driver') on a box
    that has nvcc but no GPU, so that `pytest -x` on the CPU suite never stops on them."""
    try:
        import torch
        have = torch.cuda.is_available()
    except Exception:
        have = False
    if have:
        return
    skip = pytest.mark.skip(reason="needs a CUDA device (the product has no CPU fallback)")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


@pytest.fixture(scope="session")
def built_lib():
    """Build libvatlq.so if needed (nvcc cross-compiles without a GPU)."""
    import __graft_entry__ as g
    g.build()
    import vatlq
    return vatlq


def load_golden(name):
    """The arrays of tests/golden/<name>, with the heat maps and features that oracle/golden_inputs.py rebuilds from
    seeds put back under their names."""
    from oracle import golden_inputs as G
    z = dict(np.load(os.path.join(GOLD, name), allow_pickle=False))
    if name == "scan.npz":
        z["H"] = G.scan_inputs()[0]
    elif name == "next.npz":
        z["H"] = G.next_inputs()[0]
        z["clu_X"], z["iid_X"] = G.next_features(True), G.next_features(False)
    elif name == "peaks.npz":
        z["H"] = G.peaks_inputs()
    elif name == "coreset.npz":
        z.update({f"{tag}/X": X for tag, X in G.coreset_features().items()})
    return z


@pytest.fixture(scope="session")
def gold_scan():
    return load_golden("scan.npz")


@pytest.fixture(scope="session")
def gold_wpu():
    return load_golden("wpu.npz")


@pytest.fixture(scope="session")
def gold_fuse():
    return load_golden("fuse.npz")


@pytest.fixture(scope="session")
def gold_next():
    return load_golden("next.npz")


@pytest.fixture(scope="session")
def gold_coreset():
    z = load_golden("coreset.npz")
    cases = {}
    for key in z:
        tag, field = key.split("/")
        cases.setdefault(tag, {})[field] = z[key]
    return cases


def ae_weights_from_gold(z):
    return [(z[f"W{k}"], z[f"b{k}"]) for k in range(8)]
