"""Pins the CPU oracle (oracle/pq_oracle.c) bit-for-bit against golden vectors generated from the compiled reference
(tests/golden/make_golden.py; the reference is built from its unmodified sources by oracle/Makefile, and the vectors
travel with the repository).  No GPU, no product code."""
import hashlib
import os

import numpy as np
import pytest

from oracle import pyoracle

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden(name):
    return np.load(os.path.join(GOLD, name))


SYNTH = {
    # must mirror tests/golden/make_golden.py
    "convA": ("conv", (1, 3, 32, 1, 1), (16, 7, 9)),
    "convB": ("conv", (2, 5, 32, 2, 1), (12, 9, 9)),
    "convC": ("conv", (0, 7, 16, 1, 3), (3, 23, 23)),
    "fcA": ("fc", 40, (24, 1, 1)),
    "fcB": ("fc", 24, (10, 1, 1)),
}


@pytest.mark.parametrize("name", sorted(SYNTH))
def test_oracle_single_layer_matches_reference_golden(name, po):
    g = golden("synth_layers.npz")
    kind, spec, chw = SYNTH[name]
    img = g[name + "_img"][None]
    ctrd, asmt, bias = g[name + "_ctrd0"], g[name + "_asmt0"], g[name + "_bias0"]
    x = po.nchw_to_nhwc(img)
    assert np.array_equal(x, g[name + "_fm0"])
    if kind == "conv":
        y = po.conv_aprx(x, po.conv(*spec), ctrd, asmt, bias)
    else:
        y = po.fc_aprx(po.nhwc_to_nchw(x).reshape(1, -1), ctrd, asmt, bias)
    assert np.array_equal(y.reshape(-1), g[name + "_fm1"].reshape(-1))


def test_oracle_misc_layers_match_reference_golden(po):
    g = golden("synth_layers.npz")
    x = g["misc_fm0"]
    r = po.relu_f(x)
    assert np.array_equal(r, g["misc_fm1"])
    n = po.lrn_f(r, 5, 1e-4, 0.75, 1.0)
    assert np.array_equal(n, g["misc_fm2"])
    p = po.pool_f(n, 3, 0, 2)
    assert np.array_equal(p, g["misc_fm3"])


def test_oracle_tiny_net_matches_reference_golden(po):
    g = golden("synth_layers.npz")
    layers = [po.conv(1, 3, 16, 1, 1), po.relu(), po.pool(0, 2, 2), po.fcnt(16), po.relu(), po.drpt(0.5),
              po.fcnt(8), po.smax()]
    params = {l: dict(bias=g["tiny_bias%d" % l], ctrd=g["tiny_ctrd%d" % l], asmt=g["tiny_asmt%d" % l]) for l in (0, 3, 6)}
    prob, maps = po.net_forward(layers, params, g["tiny_img"][None], keep=True)
    assert np.array_equal(prob.reshape(-1), g["tiny_out"])
    for l in (0, 1, 2, 4, 5, 6, 7, 8):  # featMapLst[3] is left in NCHW element order by the reference
        assert np.array_equal(maps[l].reshape(-1), g["tiny_fm%d" % l].reshape(-1)), l
    assert np.array_equal(po.nhwc_to_nchw(maps[3]).reshape(-1), g["tiny_fm3"].reshape(-1))
    assert abs(float(prob.sum()) - 1.0) < 1e-5


def test_oracle_file_formats_match_reference_bytes(po, tmp_path):
    g = golden("cbn_vectors.npz")
    keys = sorted(k[:-5] for k in g.files if k.endswith("_idx0"))
    assert len(keys) == 6
    for key in keys:
        idx0, blob = g[key + "_idx0"], g[key + "_file"]
        bits = int(key[1])
        ref_path = str(tmp_path / (key + ".ref.cbn"))
        blob.tofile(ref_path)
        got, b = po.read_cbn(ref_path)
        assert b == bits and np.array_equal(got, idx0)
        mine = str(tmp_path / (key + ".mine.cbn"))
        po.write_cbn(mine, idx0, bits)
        assert np.array_equal(np.fromfile(mine, np.uint8), blob)
    p = str(tmp_path / "t.bin")
    g["bin_file"].tofile(p)
    assert np.array_equal(po.read_bin(p), g["bin_arr"])
    po.write_bin(p + "2", g["bin_arr"])
    assert np.array_equal(np.fromfile(p + "2", np.uint8), g["bin_file"])


def test_lcg_image_generator(po):
    img = po.lcg_images(1, 12345).reshape(-1)
    s = 12345
    exp = []
    for _ in range(8):
        s = (s * 1664525 + 1013904223) & 0xFFFFFFFF
        exp.append(((s >> 8) & 0xFFFF) / 65536.0 * 256.0 - 128.0)
    assert np.array_equal(img[:8], np.array(exp, np.float32))
    assert img.min() >= -128 and img.max() < 128


def test_oracle_alexnet_kat_matches_reference_golden(po, ref_data):
    """AlexNet through the oracle port: the reference's shipped parameter files where they are staged under
    oracle/_ref/data, else the seeded synthetic AlexNet of pyoracle.stage_synth_data."""
    g = ref_data["kat"]
    layers = po.alexnet_layers()
    params = po.load_model(ref_data["model_dir"], po.ALEXNET_PFX, layers)
    imgs = po.lcg_images(2, 12345)
    for i in range(2):
        prob, maps = po.net_forward(layers, params, imgs[i:i + 1], keep=True)
        assert np.array_equal(prob[0], g["prob%d" % i])
        assert np.array_equal(maps[22].reshape(-1), g["logits%d" % i])
        idx, _ = po.topk(prob[0], 5)
        assert np.array_equal(idx, g["top5_%d" % i])
        for l in (1, 5, 9, 11, 13, 16, 19, 22):
            assert np.array_equal(maps[l].reshape(-1)[:64], g["fm%d_%d" % (l, i)])
        cks = g["cks%d" % i]
        for l in range(24):
            m = maps[l].astype(np.float64).reshape(-1)
            assert np.allclose([m.sum(), np.sqrt((m * m).sum()), m.max()], cks[l], rtol=1e-12, atol=0)
    if ref_data["shipped"]:
        # SURVEY.md Appendix B: seed 12345 -> class 533, p = 0.621259
        assert int(g["top5_0"][0]) == 533 and abs(float(g["prob0"][533]) - 0.621259) < 1e-6


# ---- seeded cases whose reference outputs are stored in tests/golden/live_ref.npz (make_golden.py: live_ref) ----
LUT_CASES = [(50, 48, 6, 128, 8), (7, 3, 1, 128, 8), (3, 10, 3, 32, 4), (2, 4096, 4096, 16, 1)]
RANDOM_LAYER_CASES = [
    ([pyoracle.conv(1, 3, 64, 2, 1)], (32, 13, 13), {0: (4, 64, 4)}),
    ([pyoracle.conv(2, 5, 48, 1, 2)], (6, 17, 15), {0: (2, 128, 4)}),      # d > remaining dims in last subspace
    ([pyoracle.conv(0, 11, 32, 1, 4)], (3, 51, 51), {0: (1, 128, 8)}),
    ([pyoracle.fcnt(64)], (30, 2, 2), {0: (30, 32, 4)}),
    ([pyoracle.fcnt(1000)], (100, 1, 1), {0: (100, 16, 1)}),
]


def assert_matches_sample(out, g, key):
    """out bit-identical to the reference at the stored sample positions, and its float64 (sum, l2, max) equal."""
    out = out.reshape(-1)
    assert np.array_equal(out[g[key + "_idx"]], g[key + "_val"]), key
    m = out.astype(np.float64)
    assert np.allclose([m.sum(), np.sqrt((m * m).sum()), m.max()], g[key + "_cks"], rtol=1e-12, atol=0), key


def test_oracle_lut_stage_matches_live_reference(po):
    g = golden("live_ref.npz")
    rng = np.random.RandomState(11)
    for c, (P, D, S, K, d) in enumerate(LUT_CASES):
        data = (rng.randn(P, D) * 10).astype(np.float32)
        ctrd = (rng.randn(S, K, d) * 0.1).astype(np.float32)
        assert_matches_sample(po.get_inpd(data, ctrd), g, "lut%d" % c)


def test_oracle_random_layers_match_live_reference(po, tmp_path):
    """Seeded random conv / FC shapes against the reference's own CalcFeatMap_ConvAprx / _FCntAprx."""
    g = golden("live_ref.npz")
    rng = np.random.RandomState(99)
    for ci, (layers, chw, pq) in enumerate(RANDOM_LAYER_CASES):
        params = po.synth_model(layers, chw, pq, seed=ci, ctrd_std=0.2)
        d = str(tmp_path / ("m%d" % ci))
        po.save_model(d, "rnd", params)
        # decoded parameters identical (bit-exact assignment indexing): the oracle reads back what the reference read
        a, _ = po.read_cbn(os.path.join(d, "rnd.asmtLst.01.cbn"))
        assert np.array_equal(a, params[0]["asmt"])
        assert hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest() == str(g["rnd%d_asmt_sha256" % ci])
        for j in range(2):
            img = (rng.randn(*chw) * 5).astype(np.float32)
            assert_matches_sample(po.net_forward(layers, params, img[None]), g, "rnd%d_%d" % (ci, j))


def test_alexnet_live_reference_vs_oracle(po, ref_data):
    """The reference's CaffeEva on LCG image 777 (tests/golden/alexnet_live_ref.npz, for the shipped and the synthetic
    AlexNet of the ref_data fixture): probabilities, every feature map and every decoded parameter buffer."""
    g = golden("alexnet_live_ref.npz")
    key = "shipped" if ref_data["shipped"] else "synth"
    layers = po.alexnet_layers()
    params = po.load_model(ref_data["model_dir"], po.ALEXNET_PFX, layers)
    mine, maps = po.net_forward(layers, params, po.lcg_images(1, 777), keep=True)
    assert np.array_equal(mine[0], g[key + "_prob"])
    for l in range(24):
        if l == 15:
            continue  # reference leaves featMapLst[15] in NCHW order (CaffeEva.cc:246-253)
        assert_matches_sample(maps[l], g, "%s_fm%d" % (key, l))
    for l in params:
        for name in ("bias", "ctrd", "asmt"):
            a = np.ascontiguousarray(params[l][name])
            assert hashlib.sha256(a.tobytes()).hexdigest() == str(g["%s_%s%d_sha256" % (key, name, l)]), (l, name)
