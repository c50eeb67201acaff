"""CPU-side checks of the product library: it loads without a GPU, exports every symbol include/qcnn.h declares,
its file-format code agrees with the oracle and the reference's golden byte images, and compute entry points fail
loudly (no CPU fallback) when no device is present."""
import ctypes as C
import os
import re

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_library_exports_every_declared_symbol(qcnn):
    text = open(qcnn.HEADER_PATH).read()
    declared = sorted(set(re.findall(r"QCNN_API[^;(]*?\b(qcnn_[a-z0-9_]+)\s*\(", text)))
    assert len(declared) >= 40
    lib = C.CDLL(qcnn.LIB_PATH)
    missing = [n for n in declared if not hasattr(lib, n)]
    assert not missing, missing
    # the binding knows every declared symbol too (no silently unbound entry point)
    assert sorted(qcnn.EXPORTS) == declared
    assert b"sm_100a" in qcnn.lib.qcnn_version()


def test_no_cpu_fallback_without_gpu(qcnn):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(qcnn.QcnnError) as e:
        qcnn.Context(0)
    assert "no CPU fallback" in str(e.value)


def test_product_never_links_the_oracle(qcnn):
    import subprocess
    out = subprocess.run(["ldd", qcnn.LIB_PATH], capture_output=True, text=True).stdout
    assert "pq_oracle" not in out and "qcnn_ref" not in out
    syms = subprocess.run(["nm", "-D", qcnn.LIB_PATH], capture_output=True, text=True).stdout
    assert "pqo_" not in syms and "ref_net" not in syms


def test_cbn_and_bin_formats_match_reference_bytes(qcnn, tmp_path):
    g = np.load(os.path.join(GOLD, "cbn_vectors.npz"))
    for key in sorted(k[:-5] for k in g.files if k.endswith("_idx0")):
        idx0, blob = g[key + "_idx0"], g[key + "_file"]
        bits = int(key[1])
        ref_path = str(tmp_path / (key + ".cbn"))
        blob.tofile(ref_path)
        got, b = qcnn.read_cbn_u8(ref_path)
        assert b == bits
        assert got.shape == idx0.shape and np.array_equal(got, idx0)     # bit-exact assignment decoding
        mine = str(tmp_path / (key + ".w.cbn"))
        qcnn.write_cbn_u8(mine, idx0, bits)
        assert np.array_equal(np.fromfile(mine, np.uint8), blob)          # byte-identical files
    p = str(tmp_path / "t.bin")
    g["bin_file"].tofile(p)
    assert np.array_equal(qcnn.read_bin_f32(p), g["bin_arr"])
    qcnn.write_bin_f32(p + "2", g["bin_arr"])
    assert np.array_equal(np.fromfile(p + "2", np.uint8), g["bin_file"])


def test_cbn_edge_cases_against_oracle(qcnn, po, tmp_path):
    rng = np.random.RandomState(0)
    for bits in range(1, 9):
        per_block = 4096 * 8 // bits
        for n in (1, per_block - 1, per_block, per_block + 1, 2 * per_block + 17):
            idx0 = rng.randint(0, 1 << bits, size=n).astype(np.uint8)
            a = str(tmp_path / "a.cbn")
            b = str(tmp_path / "b.cbn")
            qcnn.write_cbn_u8(a, idx0, bits)
            po.write_cbn(b, idx0, bits)
            assert np.array_equal(np.fromfile(a, np.uint8), np.fromfile(b, np.uint8))
            assert os.path.getsize(a) == 4 + 4 + 4 + 4096 * ((n + per_block - 1) // per_block)
            got, gb = qcnn.read_cbn_u8(b)
            assert gb == bits and np.array_equal(got, idx0)
            got2, _ = po.read_cbn(a)
            assert np.array_equal(got2, idx0)


def test_shipped_alexnet_files_decode_identically(qcnn, po, ref_data):
    """The AlexNet parameter files of the ref_data fixture: the reference's shipped ones where they are staged."""
    layers = po.alexnet_layers()
    params = po.load_model(ref_data["model_dir"], po.ALEXNET_PFX, layers)
    for l, p in params.items():
        base = os.path.join(ref_data["model_dir"], po.ALEXNET_PFX)
        a, bits = qcnn.read_cbn_u8("%s.asmtLst.%02d.cbn" % (base, l + 1))
        assert bits == p["bits"] and np.array_equal(a, p["asmt"])
        S, K, d = p["ctrd"].shape
        assert int(a.max()) == K - 1 and int(a.min()) == 0
        assert np.array_equal(qcnn.read_bin_f32("%s.ctrdLst.%02d.bin" % (base, l + 1)), p["ctrd"])
        assert np.array_equal(qcnn.read_bin_f32("%s.biasVec.%02d.bin" % (base, l + 1)).reshape(-1), p["bias"])


def test_missing_file_reports_error(qcnn):
    with pytest.raises(qcnn.QcnnError):
        qcnn.read_bin_f32("/nonexistent/file.bin")
