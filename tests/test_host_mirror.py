"""The C++ host layer that keeps the reference's class API (CaffeEvaWrapper / CaffeEva / CaffePara / BmpImgIO):
CPU-side pieces are checked here against golden data produced by the compiled reference; the GPU-side end-to-end
classification of ten BMP fixtures is gpu-marked.  The data directory is the ref_data fixture's: the reference's
shipped model, mean image and BMPs where they are staged, else a seeded stand-in with the reference's outputs on it."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
PKG = os.path.join(ROOT, "quantized-cnn_b200")


def hostlib():
    lib = C.CDLL(os.path.join(PKG, "libqcnn_host.so"))
    return lib


def test_layer_tables_match_reference_counts():
    lib = hostlib()
    chw = (C.c_int * 3)()
    types = (C.c_int * 64)()
    # (layerCnt, input size) of reference src/CaffePara.cc:20-237
    expect = {"AlexNet": (23, 227), "CaffeNet": (23, 227), "VggCnnS": (22, 224), "VGG16": (39, 224),
              "CaffeNetFGB": (23, 227), "CaffeNetFGD": (23, 227)}
    for name, (cnt, size) in expect.items():
        n = lib.qcnn_host_layer_table(name.encode(), chw, types, 64)
        assert n == cnt and tuple(chw) == (3, size, size), name
    n = lib.qcnn_host_layer_table(b"AlexNet", chw, types, 64)
    # Conv ReLU LoRN Pool ... SMax in ENUM_LyrType order (0 Conv, 1 Pool, 2 FCnt, 3 ReLU, 4 LoRN, 5 Drpt, 6 SMax)
    assert list(types[:n]) == [0, 3, 4, 1, 0, 3, 4, 1, 0, 3, 0, 3, 0, 3, 1, 2, 3, 5, 2, 3, 5, 2, 6]
    n = lib.qcnn_host_layer_table(b"CaffeNet", chw, types, 64)
    assert list(types[:4]) == [0, 3, 1, 4]          # pooling before LRN
    assert lib.qcnn_host_layer_table(b"ResNet", chw, types, 64) == -1


def test_bmp_preprocessing_matches_reference_bit_for_bit(ref_data):
    lib = hostlib()
    g = ref_data["bmp"]
    mean = ref_data["mean"].encode()
    for i, path in enumerate(ref_data["bmps"], 1):
        bmp = path.encode()
        out = np.zeros(3 * 227 * 227, np.float32)
        n = lib.qcnn_host_load_bmp_alexnet(mean, bmp, out.ctypes.data_as(C.c_void_p), out.size)
        assert n == out.size
        assert np.array_equal(out[:64], g["img_head_%02d" % i])
        a = out.astype(np.float64)
        cks = np.array([a.sum(), np.sqrt((a * a).sum()), a.max(), a.min()])
        assert np.allclose(cks, g["img_cks_%02d" % i], rtol=1e-12, atol=0)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["strict", "default"])
def test_wrapper_classifies_reference_bmps_like_the_reference(mode, ref_data):
    """quancnn_b200 classify == UnitTest::UT_CaffeEvaWrapper (reference src/UnitTest.cc:67-124) on the ten fixtures;
    expected top-5 from the compiled reference (tests/golden/bmp_top5.npz == SURVEY.md Appendix B for the shipped
    fixtures, tests/golden/synth_bmp_top5.npz for the stand-in)."""
    g = ref_data["bmp"]
    data = ref_data["dir"]
    bmps = ref_data["bmps"]
    cmd = [os.path.join(PKG, "quancnn_b200"), "classify", data, os.path.join(data, "Cls.Names", "class_names.txt"),
           os.path.join(data, "Cls.Names", "image_labels.txt"), "5"] + bmps
    # strict: LUT + gather kernels only (QCNN_NO_DECTC / QCNN_FC_TC=0), probabilities within 2e-5 of the reference;
    # default: decode-at-use tensor-core kernels allowed, within 2e-4 (tolerances: tests/test_gpu_net.py)
    env = dict(os.environ)
    ptol = 2e-4
    if mode == "strict":
        env["QCNN_NO_DECTC"] = "1"
        env["QCNN_FC_TC"] = "0"
        ptol = 2e-5
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("RESULT ")]
    assert len(lines) == 10
    for i, line in enumerate(lines, 1):
        head, tail = line.split("|")
        pairs = [p.split(":") for p in tail.split()]
        idx = np.array([int(p[0]) for p in pairs])
        prob = np.array([float(p[1]) for p in pairs], np.float32)
        assert "gt=-" not in head
        ref_idx, ref_prob = g["top5_idx_%02d" % i], g["top5_prob_%02d" % i]
        assert np.abs(prob - ref_prob).max() <= ptol, (i, prob, ref_prob)
        gaps = ref_prob[:-1] - ref_prob[1:]
        if gaps.min() > max(1e-4, 4 * ptol):
            assert np.array_equal(idx, ref_idx), (i, idx, ref_idx)
        else:
            assert idx[0] == ref_idx[0]


@pytest.mark.gpu
def test_per_layer_members_agree_with_fused_network(ref_data):
    """CaffeEva::CalcFeatMap_* driven layer by layer with host matrices (the reference executor's calling pattern)
    reproduces the fused device-resident forward pass."""
    out = subprocess.run([os.path.join(PKG, "quancnn_b200"), "layers", ref_data["dir"]], capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("LAYERS")][0]
    # the reference's class for LCG image 12345 (533 with the shipped model: SURVEY.md Appendix B synthetic KAT)
    assert "argmax0=%d " % int(ref_data["kat"]["top5_0"][0]) in line
    # probabilities of the layer-by-layer run (host matrices between layers, un-fused kernels) vs the fused device pass
    err = float(line.split("max|layerwise-fused|=")[1])
    assert err <= 2e-5, line


@pytest.mark.gpu
def test_host_executor_shards_over_all_gpus(ref_data):
    """CaffeEva::SetDeviceCount(n): ExecForwardPass through qcnn_multi_* (n = every GPU of the box, 1 included)."""
    import torch
    n = max(1, min(torch.cuda.device_count(), 8))
    out = subprocess.run([os.path.join(PKG, "quancnn_b200"), "layers", ref_data["dir"], str(n)], capture_output=True,
                         text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("LAYERS")][0]
    assert "argmax0=%d " % int(ref_data["kat"]["top5_0"][0]) in line
