import importlib
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def po():
    """CPU oracle front-end (test infrastructure)."""
    from oracle import pyoracle
    pyoracle.build()
    return pyoracle


@pytest.fixture(scope="session")
def ref_data(po, tmp_path_factory):
    """A data directory laid out like the reference's (AlexNet/Bin.Files, AlexNet/imagenet_mean.single.bin, Bmp.Files,
    Cls.Names) with the reference's outputs on it (tests/golden): the reference's shipped files where they are staged
    under oracle/_ref/data, else the seeded stand-in written by pyoracle.stage_synth_data."""
    import numpy as np
    if po.have_alexnet() and os.path.isdir(os.path.join(po.REF_DATA, "Bmp.Files")):
        d, shipped = po.REF_DATA, True
        bmps = [os.path.join(d, "Bmp.Files", "ILSVRC2012_val_%08d.BMP" % i) for i in range(1, 11)]
        kat, bmp = "alexnet_kat.npz", "bmp_top5.npz"
    else:
        d, shipped = str(tmp_path_factory.mktemp("ref_data")), False
        bmps = po.stage_synth_data(d)
        kat, bmp = "synth_alexnet_kat.npz", "synth_bmp_top5.npz"
    gold = os.path.join(ROOT, "tests", "golden")
    return dict(dir=d, model_dir=os.path.join(d, "AlexNet", "Bin.Files"), shipped=shipped, bmps=bmps,
                mean=os.path.join(d, "AlexNet", "imagenet_mean.single.bin"),
                kat=np.load(os.path.join(gold, kat)), bmp=np.load(os.path.join(gold, bmp)))


@pytest.fixture(scope="session")
def qcnn():
    """The product binding; the shared library must have been built (no fallback)."""
    return importlib.import_module("quantized-cnn_b200")


@pytest.fixture(scope="session")
def ctx(qcnn):
    import torch
    assert torch.cuda.is_available(), "gpu-marked test started without a GPU"
    c = qcnn.Context(0)
    yield c
    c.close()
