"""Generates the committed golden vectors from the COMPILED REFERENCE (oracle/_ref/libqcnn_ref.so, built from the
unmodified /root/reference sources by oracle/Makefile).  Run here (needs /root/reference); the outputs travel with
the repo so the oracle can be pinned on boxes where the reference tree does not exist.

    python tests/golden/make_golden.py

Outputs (all small):
  alexnet_kat.npz   shipped quantized AlexNet on the SURVEY.md 8(d) LCG images seed 12345/12346: logits, probs,
                    top-5, per-layer (sum, l2, max) checksums of featMapLst
  synth_layers.npz  reference CalcFeatMap outputs of small synthetic conv / FC / LRN / pool / softmax layers
                    (inputs + parameters stored alongside)
  bmp_top5.npz      top-5 of CaffeEvaWrapper::Proc on the ten shipped BMPs + fingerprints of BmpImgIO::Load outputs
  cbn_vectors.npz   byte images of .cbn / .bin files written by the reference's own FileIO for 4/5/7/8-bit tables
  synth_alexnet_kat.npz, synth_bmp_top5.npz
                    the same as alexnet_kat.npz / bmp_top5.npz for the seeded data directory of
                    pyoracle.stage_synth_data (synthetic AlexNet, mean image and BMPs): what the tests compare against
                    where the reference's shipped files are not staged
  live_ref.npz      reference GetInPdMat outputs and reference forward passes of seeded random conv / FC layers
                    (fixed samples of the outputs + float64 checksums; inputs are regenerated from the seeds)
  alexnet_live_ref.npz
                    the reference's CaffeEva on LCG image 777, shipped and synthetic AlexNet: probabilities, samples +
                    checksums of every feature map, SHA-256 of every decoded parameter buffer
"""
import hashlib
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import pyoracle as po  # noqa: E402
from test_oracle_vs_reference import LUT_CASES, RANDOM_LAYER_CASES  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def alexnet_kat(dirpath=po.ALEXNET_DIR, name="alexnet_kat.npz"):
    net = po.RefNet(dirpath, po.ALEXNET_PFX)
    imgs = po.lcg_images(2, 12345)
    out = {}
    for i in range(2):
        prob = net.forward(imgs[i])
        logits = net.featmap(22).reshape(-1)
        idx, val = po.topk(prob, 5)
        cks = []
        for l in range(24):
            m = net.featmap(l).astype(np.float64).reshape(-1)
            cks.append([m.sum(), np.sqrt((m * m).sum()), m.max()])
        out["prob%d" % i] = prob
        out["logits%d" % i] = logits
        out["top5_%d" % i] = idx
        out["cks%d" % i] = np.array(cks)
        # a thin slice of every PQ layer's output (first 64 values) for localisation
        for l in (1, 5, 9, 11, 13, 16, 19, 22):
            out["fm%d_%d" % (l, i)] = net.featmap(l).reshape(-1)[:64].copy()
    net.close()
    np.savez_compressed(os.path.join(OUT, name), **out)


def synth_layers():
    rng = np.random.RandomState(2016)
    out = {}
    cases = {
        # name: (layers, in_chw, pq)
        "convA": ([po.conv(1, 3, 32, 1, 1)], (16, 7, 9), {0: (2, 16, 8)}),
        "convB": ([po.conv(2, 5, 32, 2, 1)], (12, 9, 9), {0: (2, 32, 4)}),       # groups, d<Cg/S... partial last
        "convC": ([po.conv(0, 7, 16, 1, 3)], (3, 23, 23), {0: (1, 64, 8)}),      # strided, d > Cin
        "fcA": ([po.fcnt(40)], (24, 1, 1), {0: (6, 16, 4)}),
        "fcB": ([po.fcnt(24)], (10, 1, 1), {0: (3, 32, 4)}),                     # Din % d != 0
        "misc": ([po.relu(), po.lorn(5, 1e-4, 0.75, 1.0), po.pool(0, 3, 2)], (8, 9, 9), {}),
        "tiny": ([po.conv(1, 3, 16, 1, 1), po.relu(), po.pool(0, 2, 2), po.fcnt(16), po.relu(), po.drpt(0.5),
                  po.fcnt(8), po.smax()], (4, 6, 6), {0: (1, 16, 4), 3: (36, 16, 4), 6: (4, 8, 4)}),
    }
    with tempfile.TemporaryDirectory() as tmp:
        # NOTE: the reference's gather loops are unrolled by 8 (CaffeEva.cc:849-858, 1008-1017), so it needs
        # Cout/grp % 8 == 0 and Dout % 8 == 0 -- other sizes overrun its buffers.
        for ci, (name, (layers, chw, pq)) in enumerate(sorted(cases.items())):
            params = po.synth_model(layers, chw, pq, seed=100 + ci, ctrd_std=0.3)
            po.save_model(tmp, name, params)
            net = po.RefNet(tmp, name, layers=layers, in_chw=chw)
            img = (rng.randn(*chw) * 3).astype(np.float32)
            prob = net.forward(img)
            out[name + "_img"] = img
            out[name + "_out"] = prob
            for l, p in params.items():
                out["%s_bias%d" % (name, l)] = p["bias"]
                out["%s_ctrd%d" % (name, l)] = p["ctrd"]
                out["%s_asmt%d" % (name, l)] = p["asmt"]
            for l in range(len(layers) + 1):
                out["%s_fm%d" % (name, l)] = net.featmap(l)
            net.close()
    np.savez_compressed(os.path.join(OUT, "synth_layers.npz"), **out)


def cbn_vectors():
    import ctypes as C
    rng = np.random.RandomState(5)
    out = {}
    R = po.ref()
    with tempfile.TemporaryDirectory() as tmp:
        for bits, shape in [(4, (5, 700)), (5, (3, 2300)), (7, (4, 3, 3, 130)), (8, (9000,)), (7, (4681,)), (7, (4682,))]:
            K = 1 << bits
            # 8-bit tables: index 255 is excluded on purpose.  Its 1-based form wraps to 0 and the reference WRITER
            # then computes (0 - 1) >> 8 == -1 as an int and ORs 0xFF over the previous element's byte
            # (FileIO.h:327-333) -- a reference bug our writer does not reproduce (covered by a live round-trip test).
            hi = K - 1 if bits == 8 else K
            idx0 = rng.randint(0, hi, size=shape).astype(np.uint8)
            idx0.reshape(-1)[:2] = [hi - 1, 0]
            path = os.path.join(tmp, "t.cbn")
            one = (idx0.astype(np.int32) + 1).astype(np.uint8)   # 1-based as the reference writer expects (wraps at 256)
            dims = (C.c_int * idx0.ndim)(*idx0.shape)
            assert R.ref_write_cbn(path.encode(), idx0.ndim, dims, one.ctypes.data_as(C.c_void_p), bits) == 0
            key = "b%d_%s" % (bits, "x".join(map(str, shape)))
            out[key + "_idx0"] = idx0
            out[key + "_file"] = np.fromfile(path, np.uint8)
        arr = rng.randn(3, 4, 5).astype(np.float32)
        path = os.path.join(tmp, "t.bin")
        dims = (C.c_int * 3)(*arr.shape)
        assert R.ref_write_bin_f32(path.encode(), 3, dims, arr.ctypes.data_as(C.c_void_p)) == 0
        out["bin_arr"] = arr
        out["bin_file"] = np.fromfile(path, np.uint8)
    np.savez_compressed(os.path.join(OUT, "cbn_vectors.npz"), **out)


def bmp_top5(d=po.REF_DATA, bmps=None, name="bmp_top5.npz"):
    """CaffeEvaWrapper::Proc (reference src/CaffeEvaWrapper.cc:153-209) on the ten shipped BMPs + a fingerprint of
    BmpImgIO::Load's output tensor for each."""
    import ctypes as C
    R = po.ref()
    R.ref_wrapper_create.restype = C.c_void_p
    if bmps is None:
        bmps = ["%s/Bmp.Files/ILSVRC2012_val_%08d.BMP" % (d, i) for i in range(1, 11)]
    h = C.c_void_p(R.ref_wrapper_create(d.encode(), (d + "/Cls.Names/class_names.txt").encode(),
                                        (d + "/Cls.Names/image_labels.txt").encode()))
    assert h.value
    out = {}
    for i, path in enumerate(bmps, 1):
        bmp = path.encode()
        idx = np.zeros(5, np.int32)
        pr = np.zeros(5, np.float32)
        assert R.ref_wrapper_proc(h, bmp, 5, idx.ctypes.data_as(C.c_void_p), pr.ctypes.data_as(C.c_void_p)) == 0
        img = np.zeros(3 * 227 * 227, np.float32)
        assert R.ref_wrapper_load_bmp(h, bmp, img.ctypes.data_as(C.c_void_p), img.size) == img.size
        a = img.astype(np.float64)
        out["top5_idx_%02d" % i] = idx
        out["top5_prob_%02d" % i] = pr
        out["img_cks_%02d" % i] = np.array([a.sum(), np.sqrt((a * a).sum()), a.max(), a.min()])
        out["img_head_%02d" % i] = img[:64].copy()
    np.savez_compressed(os.path.join(OUT, name), **out)


def synth_data():
    """alexnet_kat / bmp_top5 on the seeded stand-in of the reference's data directory."""
    with tempfile.TemporaryDirectory() as tmp:
        bmps = po.stage_synth_data(tmp)
        alexnet_kat(os.path.join(tmp, "AlexNet", "Bin.Files"), "synth_alexnet_kat.npz")
        bmp_top5(tmp, bmps, "synth_bmp_top5.npz")


def alexnet_live_ref():
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        po.stage_synth_data(tmp)
        for key, dirpath in (("shipped", po.ALEXNET_DIR), ("synth", os.path.join(tmp, "AlexNet", "Bin.Files"))):
            net = po.RefNet(dirpath, po.ALEXNET_PFX)
            out[key + "_prob"] = net.forward(po.lcg_images(1, 777)[0])
            for l in range(24):
                out["%s_fm%d_idx" % (key, l)], out["%s_fm%d_val" % (key, l)], out["%s_fm%d_cks" % (key, l)] = \
                    sample(net.featmap(l), 64)
            for l in po.ALEXNET_PQ:
                for which, name in ((0, "bias"), (1, "ctrd"), (2, "asmt")):
                    a, _ = net.param(l, which)
                    out["%s_%s%d_sha256" % (key, name, l)] = np.array(hashlib.sha256(a.tobytes()).hexdigest())
            net.close()
    np.savez_compressed(os.path.join(OUT, "alexnet_live_ref.npz"), **out)


def sample(a, n=512):
    """A fixed sample of a flattened output (indices, values) and its float64 (sum, l2, max)."""
    a = np.ascontiguousarray(a, np.float32).reshape(-1)
    idx = np.sort(np.random.RandomState(a.size).choice(a.size, min(n, a.size), replace=False))
    m = a.astype(np.float64)
    return idx, a[idx], np.array([m.sum(), np.sqrt((m * m).sum()), m.max()])


def live_ref():
    """Inputs of tests/test_oracle_vs_reference.py's LUT-stage and random-layer tests (same seeds, same order), through
    the reference."""
    out = {}
    rng = np.random.RandomState(11)
    for c, (P, D, S, K, d) in enumerate(LUT_CASES):
        data = (rng.randn(P, D) * 10).astype(np.float32)
        ctrd = (rng.randn(S, K, d) * 0.1).astype(np.float32)
        out["lut%d_idx" % c], out["lut%d_val" % c], out["lut%d_cks" % c] = sample(po.ref_get_inpd(data, ctrd))
    rng = np.random.RandomState(99)
    with tempfile.TemporaryDirectory() as tmp:
        for ci, (layers, chw, pq) in enumerate(RANDOM_LAYER_CASES):
            params = po.synth_model(layers, chw, pq, seed=ci, ctrd_std=0.2)
            d = os.path.join(tmp, "m%d" % ci)
            po.save_model(d, "rnd", params)
            net = po.RefNet(d, "rnd", layers=layers, in_chw=chw)
            a, _ = net.param(0, 2)
            out["rnd%d_asmt_sha256" % ci] = np.array(hashlib.sha256(a.tobytes()).hexdigest())
            for j in range(2):
                img = (rng.randn(*chw) * 5).astype(np.float32)
                out["rnd%d_%d_idx" % (ci, j)], out["rnd%d_%d_val" % (ci, j)], out["rnd%d_%d_cks" % (ci, j)] = \
                    sample(net.forward(img))
            net.close()
    np.savez_compressed(os.path.join(OUT, "live_ref.npz"), **out)


if __name__ == "__main__":
    assert po.have_ref(), "build oracle/_ref first (make -C oracle ref data)"
    po.build()
    alexnet_kat()
    synth_layers()
    cbn_vectors()
    bmp_top5()
    synth_data()
    live_ref()
    alexnet_live_ref()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))
