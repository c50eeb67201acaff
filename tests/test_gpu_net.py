"""Whole-network parity of the device executor (C ABI: qcnn_net_*) against the CPU oracle / compiled reference.

Two configurations, each with its stated tolerance (metric of test_gpu_layers.close: error relative to
max(1, |ref|, 0.1 max|ref|)):
  strict   tensor_core = 0 on every PQ layer: LUT + gather kernels, fp32 adds.  Feature maps / logits RTOL = 1e-4
           (measured 1.6e-5 through all 23 layers), softmax probabilities 2e-5 absolute (measured 9e-6).
  default  the autotuner may run any layer as a decode-at-use GEMM on the tensor cores (3xTF32, accumulation inside the
           tensor core).  Feature maps / logits 5e-4 (measured 2e-4 chained), probabilities 2e-4 absolute (measured 5e-5).
Identical top-5 ordering wherever the reference's own top-5 probabilities are separated by more than the tolerance."""
import numpy as np
import pytest

from test_gpu_layers import RTOL, close

MODES = {"strict": (RTOL, 2e-5), "default": (5e-4, 2e-4)}


def set_mode(net, mode):
    if mode == "strict":
        for l in range(net.layer_count):
            pl = net.pq_layer(l)
            if pl is not None:
                pl.set_param("tensor_core", 0)


def top5_consistent(p_gpu, p_ref, po, atol=2e-5):
    ig, _ = po.topk(p_gpu, 5)
    ir, vr = po.topk(p_ref, 5)
    srt = np.sort(p_ref)[::-1]
    gaps = srt[:5] - srt[1:6]
    if gaps.min() > 4 * atol:
        return np.array_equal(ig, ir)
    return set(ig[:1]) == set(ir[:1]) or gaps[0] <= 4 * atol


@pytest.fixture(scope="module")
def synth_dir(po, tmp_path_factory):
    d = str(tmp_path_factory.mktemp("synth_alexnet"))
    params = po.synth_alexnet(seed=1)
    po.save_model(d, "synth", params)
    return d, params


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["strict", "default"])
def test_alexnet_synthetic_weights_all_feature_maps(po, qcnn, ctx, synth_dir, mode):
    import torch
    d, params = synth_dir
    layers = po.alexnet_layers()
    net = qcnn.Net(ctx, d, "synth", "AlexNet")
    assert net.layer_count == 23 and net.out_len == 1000
    set_mode(net, mode)
    RT, PT = MODES[mode]
    N = 3
    img = po.lcg_images(N, 4242)
    ref_prob, ref_maps = po.net_forward(layers, params, img, keep=True)
    imgd = torch.from_numpy(img).cuda()
    # (a) un-fused: every featMapLst entry is materialised and compared
    net.set_keep_maps(True)
    logits = torch.empty((N, 1000), dtype=torch.float32, device="cuda")
    prob_d = net.forward(imgd, logits=logits)   # keep alive: featMapLst[23] lives in this caller-owned tensor
    prob = prob_d.cpu().numpy()
    for l in range(24):
        fm = net.featmap(l, N)
        assert fm is not None, l
        e = close(fm.cpu().numpy().reshape(-1), ref_maps[l].reshape(-1))
        assert e <= RT, (l, e)
    assert close(logits.cpu().numpy(), ref_maps[22]) <= RT
    assert np.abs(prob - ref_prob).max() <= PT
    # (b) fused production path gives the same answer
    net.set_keep_maps(False)
    prob_f = net.forward(imgd, logits=logits).cpu().numpy()
    assert close(logits.cpu().numpy(), ref_maps[22]) <= RT
    assert np.abs(prob_f - ref_prob).max() <= PT
    assert net.launch_count() < 23          # fusion really happened
    for i in range(N):
        assert top5_consistent(prob_f[i], ref_prob[i], po, atol=PT)
    # (c) batch invariance: per-image results do not depend on batch composition (tilings -- hence the fp32
    #     summation order -- are chosen per batch size, so "same" means within the parity tolerance)
    p1 = net.forward(imgd[1:2].contiguous()).cpu().numpy()
    assert np.abs(p1[0] - prob_f[1]).max() <= PT
    # (c2) small batches on a non-default stream are replayed from a captured CUDA graph after two eager passes
    side = torch.cuda.Stream()
    one = imgd[1:2].contiguous()
    pg = torch.empty((1, 1000), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        for _ in range(5):
            net.forward(one, prob=pg)
            side.synchronize()
            assert np.abs(pg.cpu().numpy()[0] - p1[0]).max() <= 1e-7
        assert net.launch_count() > 0
    # (d) host-buffer entry point (H2D + chunked pipeline + D2H) == device entry point
    #     (chunks of 2 + 1 images run with their own tilings / kernel families, hence the mode's tolerance)
    net.set_chunk(2)
    ph = net.forward_host(img)
    HT = PT
    assert np.abs(ph - prob_f).max() <= HT
    pin = torch.from_numpy(img).pin_memory()
    out = torch.empty((N, 1000), dtype=torch.float32).pin_memory()
    net.forward_host(pin, out)
    assert np.abs(out.numpy() - prob_f).max() <= HT
    net.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["strict", "default"])
def test_alexnet_shipped_weights_vs_golden_and_live_reference(po, qcnn, ctx, mode, ref_data):
    """The reference's own quantized AlexNet files, loaded unchanged through the C ABI, against the reference's outputs
    (tests/golden/alexnet_kat.npz); where they are not staged, the seeded synthetic AlexNet of the ref_data fixture
    against tests/golden/synth_alexnet_kat.npz."""
    import torch
    g = ref_data["kat"]
    model_dir = ref_data["model_dir"]
    net = qcnn.Net(ctx, model_dir, po.ALEXNET_PFX, "AlexNet")
    set_mode(net, mode)
    RT, PT = MODES[mode]
    img = po.lcg_images(2, 12345)
    logits = torch.empty((2, 1000), dtype=torch.float32, device="cuda")
    prob = net.forward(torch.from_numpy(img).cuda(), logits=logits).cpu().numpy()
    lg = logits.cpu().numpy()
    for i in range(2):
        assert close(lg[i], g["logits%d" % i]) <= RT
        assert np.abs(prob[i] - g["prob%d" % i]).max() <= PT
        assert top5_consistent(prob[i], g["prob%d" % i], po, atol=PT)
    if ref_data["shipped"]:
        assert int(prob[0].argmax()) == 533 and abs(float(prob[0][533]) - 0.621259) < PT   # SURVEY.md Appendix B KAT
    # decoded device assignment tables are bit-identical to the reference's asmtBuf
    params = po.load_model(model_dir, po.ALEXNET_PFX, po.alexnet_layers())
    for l, p in params.items():
        a = p["asmt"]
        want = np.transpose(a, (1, 2, 3, 0)) if a.ndim == 4 else a.T
        assert np.array_equal(net.pq_layer(l).read_asmt(a.size), want.reshape(-1)), l
    if po.have_ref():
        ref = po.RefNet(model_dir, po.ALEXNET_PFX)
        imgs = po.lcg_images(4, 999)
        pg = net.forward(torch.from_numpy(imgs).cuda()).cpu().numpy()
        for i in range(4):
            pr = ref.forward(imgs[i])
            assert np.abs(pg[i] - pr).max() <= PT
            assert top5_consistent(pg[i], pr, po, atol=PT)
        ref.close()
    net.close()


@pytest.mark.gpu
def test_custom_layer_table_pool_before_lrn(po, qcnn, ctx, tmp_path):
    """CaffeNet ordering (pool -> LRN, not fused) and a net that does not end in softmax, via qcnn_net_create_custom."""
    import torch
    layers = [po.conv(1, 3, 32, 1, 1), po.relu(), po.pool(0, 3, 2), po.lorn(5, 1e-4, 0.75, 1.0),
              po.conv(1, 3, 32, 2, 1), po.relu(), po.fcnt(64), po.relu(), po.drpt(0.5), po.fcnt(24)]
    chw = (8, 15, 15)
    pq = {0: (2, 64, 4), 4: (4, 32, 4), 6: (49 * 8, 32, 4), 9: (16, 16, 4)}
    params = po.synth_model(layers, chw, pq, seed=3, ctrd_std=0.2)
    d = str(tmp_path)
    po.save_model(d, "c", params)
    infos = [qcnn.LayerInfo(L["type"], L.get("pad", 0), L.get("k", 0), L.get("cnt", 0), L.get("grp", 0),
                            L.get("stride", 0), L.get("nod", 0), L.get("size", 0), L.get("alpha", 0.0),
                            L.get("beta", 0.0), L.get("kini", 0.0), L.get("ratio", 0.0)) for L in layers]
    net = qcnn.Net(ctx, d, "c", layers=infos, in_chw=chw)
    rng = np.random.RandomState(1)
    img = (rng.randn(5, *chw) * 4).astype(np.float32)
    ref = po.net_forward(layers, params, img)
    out = net.forward(torch.from_numpy(img).cuda()).cpu().numpy()
    assert close(out, ref) <= MODES["default"][0]
    set_mode(net, "strict")
    out = net.forward(torch.from_numpy(img).cuda()).cpu().numpy()
    assert close(out, ref) <= RTOL
    net.close()


@pytest.mark.gpu
def test_error_reporting(qcnn, ctx, tmp_path):
    with pytest.raises(qcnn.QcnnError) as e:
        qcnn.Net(ctx, str(tmp_path), "nothing", "AlexNet")
    assert "could not load" in str(e.value)
    with pytest.raises(qcnn.QcnnError) as e:
        qcnn.Net(ctx, str(tmp_path), "nothing", "ResNet")
    assert "unrecognized caffe model name" in str(e.value)
    bad = np.full((8, 4), 200, np.uint8)
    with pytest.raises(qcnn.QcnnError) as e:
        qcnn.FcLayer(ctx, 16, np.zeros((4, 32, 4), np.float32), bad, np.zeros(8, np.float32))
    assert "not < K" in str(e.value)
