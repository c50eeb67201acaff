"""The steps either side of the PQ path on the device (SURVEY.md 8(f1), 8(f2)): BmpImgIO's ReszImg / RmMeanImg / CropImg
(qcnn_preproc_*), the uint8 entry points of the network, and the k-fold arg-max (qcnn_topk).

Bars: preprocessing BIT-IDENTICAL to the CPU path (the C++ host port, itself pinned bit-for-bit to the compiled reference
by tests/test_host_mirror.py, and the reference fingerprints in tests/golden/bmp_top5.npz, or synth_bmp_top5.npz for
the seeded stand-in of the ref_data fixture); top-k identical to the
oracle's restatement of CaffeEvaWrapper::Proc, ties included; uint8 entry == fp32 entry on (float)pixel - mean, bit for bit."""
import ctypes as C
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "quantized-cnn_b200")


def decode_bmp(path):
    """24-bpp uncompressed BMP -> uint8 [H, W, 3] in the file's B, G, R order, top row first."""
    raw = np.fromfile(path, np.uint8)
    off = int(raw[10:14].view("<u4")[0])
    wid = int(raw[18:22].view("<i4")[0])
    hei = int(raw[22:26].view("<i4")[0])
    assert raw[0] == ord("B") and raw[1] == ord("M") and int(raw[28:30].view("<u2")[0]) == 24
    row = (wid * 3 + 3) & ~3
    h = abs(hei)
    rows = raw[off:off + row * h].reshape(h, row)[:, :wid * 3].reshape(h, wid, 3)
    return np.ascontiguousarray(rows[::-1] if hei > 0 else rows)


def resz_crop_numpy(img, mean, full, crop, relaxed, mean_full):
    """numpy restatement of BmpImgIO::Load (reference src/BmpImgIO.cc:105-224) with its float / double steps."""
    f32 = np.float32
    hs, ws = img.shape[:2]
    sh = f32(hs - 1) / f32(full - 1)
    sw = f32(ws - 1) / f32(full - 1)
    hd = wd = full
    if relaxed:
        sh = min(sh, sw)
        sw = min(sh, sw)
        hd = int(np.float64(f32(hs - 1) / sh) + 0.0000001) + 1
        wd = int(np.float64(f32(ws - 1) / sw) + 0.0000001) + 1
    yo, xo = (hd - crop) // 2, (wd - crop) // 2
    ys = np.arange(yo, yo + crop)
    xs = np.arange(xo, xo + crop)
    yc = (sh * ys.astype(f32)).astype(f32)
    yl = np.maximum(0, yc.astype(np.int32))
    yh = np.minimum(hs - 1, yl + 1)
    wyl = (1.0 - (yc - yl.astype(f32)).astype(f32).astype(np.float64)).astype(f32)
    wyh = (1.0 - (yh.astype(f32) - yc).astype(f32).astype(np.float64)).astype(f32)
    xc = (sw * xs.astype(f32)).astype(f32)
    xl = np.maximum(0, xc.astype(np.int32))
    xh = np.minimum(ws - 1, xl + 1)
    wxl = (1.0 - (xc - xl.astype(f32)).astype(f32).astype(np.float64)).astype(f32)
    wxh = (1.0 - (xh.astype(f32) - xc).astype(f32).astype(np.float64)).astype(f32)
    wLT, wRT = wyl[:, None] * wxl[None, :], wyl[:, None] * wxh[None, :]
    wLB, wRB = wyh[:, None] * wxl[None, :], wyh[:, None] * wxh[None, :]
    wsum = ((wLT + wRT) + wLB) + wRB
    src = img.astype(f32)
    out = np.empty((3, crop, crop), f32)
    for c in range(3):
        a, b = src[yl][:, xl, c], src[yl][:, xh, c]
        e, f = src[yh][:, xl, c], src[yh][:, xh, c]
        v = ((a * wLT + b * wRT) + e * wLB) + f * wRB
        v = v / wsum
        m = mean[c][np.ix_(ys, xs)] if mean_full else mean[c]
        out[c] = v - m
    return out


@pytest.mark.gpu
def test_device_bmp_preprocessing_is_bit_identical_to_the_cpu_path(po, qcnn, ctx, ref_data):
    host = C.CDLL(os.path.join(PKG, "libqcnn_host.so"))
    g = ref_data["bmp"]
    mean_path = ref_data["mean"]
    mean = po.read_bin(mean_path)
    assert mean.shape == (3, 256, 256)
    pp = qcnn.Preproc(ctx, mean)           # AlexNet recipe of CaffeEvaWrapper::SetModel: Strict 256x256, full mean, crop 227
    paths = ref_data["bmps"]
    imgs = [decode_bmp(p) for p in paths]
    assert len({im.shape for im in imgs}) > 1          # pictures of different sizes in ONE launch
    got = pp.run(imgs).cpu().numpy()
    for i, p in enumerate(paths, 1):
        want = np.empty(3 * 227 * 227, np.float32)
        n = host.qcnn_host_load_bmp_alexnet(mean_path.encode(), p.encode(), want.ctypes.data_as(C.c_void_p), want.size)
        assert n == want.size
        assert np.array_equal(got[i - 1].reshape(-1), want), i            # bit-identical to the C++ host port
        assert np.array_equal(got[i - 1].reshape(-1)[:64], g["img_head_%02d" % i])   # and to the compiled reference
        a = got[i - 1].astype(np.float64)
        assert np.allclose([a.sum(), np.sqrt((a * a).sum()), a.max(), a.min()], g["img_cks_%02d" % i], rtol=1e-12, atol=0)
        assert np.array_equal(got[i - 1], resz_crop_numpy(imgs[i - 1], mean, 256, 227, False, True))
    pp.close()


@pytest.mark.gpu
def test_device_preprocessing_relaxed_resize_and_crop_mean(qcnn, ctx):
    """The VggCnnS recipe (Relaxed resize keeps the aspect ratio, crop-size mean, crop 224) on synthetic pictures."""
    rng = np.random.RandomState(9)
    mean = (rng.rand(3, 224, 224) * 120).astype(np.float32)
    pp = qcnn.Preproc(ctx, mean, 256, 256, 224, 224, resz_type=1, mean_type=1)
    imgs = [rng.randint(0, 256, size=s + (3,)).astype(np.uint8) for s in [(256, 256), (300, 400), (517, 333), (1024, 768), (240, 700)]]
    got = pp.run(imgs).cpu().numpy()
    for i, im in enumerate(imgs):
        assert np.array_equal(got[i], resz_crop_numpy(im, mean, 256, 224, True, False)), im.shape
    pp.close()
    with pytest.raises(qcnn.QcnnError):
        qcnn.Preproc(ctx, mean, 256, 256, 224, 224, resz_type=1, mean_type=0)     # full-size mean needs a Strict resize


@pytest.mark.gpu
def test_topk_on_device(po, qcnn, ctx):
    import torch
    rng = np.random.RandomState(4)
    p = rng.rand(37, 1000).astype(np.float32)
    p[3, 10] = p[3, 700] = 2.0            # tie for the maximum: the lower index wins, then the other one
    p[5] = 0.0                            # all equal: index 0 every time (the zeroed winner is still a first maximum)
    p[6, :] = -1.0                        # nothing above zero: after the first winner is zeroed IT wins again
    idx, val = ctx.topk(torch.from_numpy(p).cuda(), 5)
    idx, val = idx.cpu().numpy(), val.cpu().numpy()
    for n in range(p.shape[0]):
        ri, rv = po.topk(p[n], 5)
        assert np.array_equal(idx[n], ri) and np.array_equal(val[n], rv), n
    assert list(idx[3][:2]) == [10, 700] and list(idx[5]) == [0, 0, 0, 0, 0]
    # mode 1 = CaffeEva::CvtFeatMapToLablVec: the scan starts from (FLT_MIN, index 0)
    idx1, _ = ctx.topk(torch.from_numpy(p).cuda(), 5, mode=1)
    idx1 = idx1.cpu().numpy()
    assert np.array_equal(idx1[:3], idx[:3]) and list(idx1[5]) == [0, 0, 0, 0, 0] and list(idx1[6]) == [0, 0, 0, 0, 0]


@pytest.mark.gpu
def test_uint8_entry_points_equal_the_fp32_entry(po, qcnn, ctx, tmp_path):
    import torch
    d = str(tmp_path)
    po.save_model(d, "s", po.synth_alexnet(seed=2))
    net = qcnn.Net(ctx, d, "s", "AlexNet")
    rng = np.random.RandomState(1)
    N = 70
    net.set_chunk(32)                           # host entries run a pipeline of 8 + 32 + 30 images
    pix = rng.randint(0, 256, size=(N, 227, 227, 3)).astype(np.uint8)
    mean = (rng.rand(3, 227, 227) * 120 + 60).astype(np.float32)
    x = np.ascontiguousarray(np.transpose(pix, (0, 3, 1, 2))).astype(np.float32) - mean[None]     # (float)pixel - mean
    net.set_input_mean(mean)
    want = net.forward(torch.from_numpy(x).cuda()).cpu().numpy()
    got = net.forward_u8(torch.from_numpy(pix).cuda()).cpu().numpy()
    assert np.array_equal(got, want)
    # host entries: identical probabilities (chunked exactly like the fp32 host entry) and on-device top-5
    ph = net.forward_host(x)
    assert np.array_equal(net.forward_u8_host(pix), ph)
    idx, val = net.forward_u8_host(torch.from_numpy(pix).pin_memory(), k=5)
    idx2, val2 = net.forward_topk_host(x, 5)
    for n in range(N):
        ri, rv = po.topk(ph[n], 5)
        assert np.array_equal(idx[n], ri) and np.array_equal(val[n], rv)
        assert np.array_equal(idx2[n], ri) and np.array_equal(val2[n], rv)
    # asynchronous form, two steps in flight (the second slot's pixels travel while the first step computes)
    pin = [torch.from_numpy(pix).pin_memory(), torch.from_numpy(pix[::-1].copy()).pin_memory()]
    wants = [want, net.forward_u8(pin[1].cuda()).cpu().numpy()]
    oi = [torch.empty((N, 5), dtype=torch.int32).pin_memory() for _ in range(2)]
    ov = [torch.empty((N, 5), dtype=torch.float32).pin_memory() for _ in range(2)]
    op = [torch.empty((N, 1000), dtype=torch.float32).pin_memory() for _ in range(2)]
    tickets = []
    for step in range(5):
        b = step & 1
        if step >= 2:
            net.wait(tickets[step - 2])
            assert np.array_equal(op[b].numpy(), wants[b])
        tickets.append(net.submit_u8_host(pin[b], k=5, idx_h=oi[b], val_h=ov[b], prob_h=op[b]))
    net.wait(tickets[-2])
    net.wait(tickets[-1])
    assert np.array_equal(op[0].numpy(), wants[0]) and np.array_equal(op[1].numpy(), wants[1])
    for n in range(N):
        ri, rv = po.topk(want[n], 5)
        assert np.array_equal(oi[0].numpy()[n], ri) and np.array_equal(ov[0].numpy()[n], rv)
    net.set_input_mean(None)
    assert np.array_equal(net.forward_u8(torch.from_numpy(pix).cuda()).cpu().numpy(),
                          net.forward(torch.from_numpy(np.ascontiguousarray(np.transpose(pix, (0, 3, 1, 2))).astype(np.float32)).cuda()).cpu().numpy())
    net.close()
