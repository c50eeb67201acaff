"""TEST INFRASTRUCTURE ONLY: ctypes/numpy front-end to the CPU oracle.

Two libraries sit behind this module, both built by ``oracle/Makefile``:

* ``oracle/_build/libpq_oracle.so`` -- our plain-C restatement (``oracle/pq_oracle.c``) of the reference's
  PQ forward path (``src/CaffeEva.cc:760-868, 968-1025, 1261-1296`` ...), the *port*.
* ``oracle/_ref/libqcnn_ref.so``    -- the UNMODIFIED reference sources compiled in place plus
  ``oracle/ref_harness.cc``, the *reference* (only present where it was prebuilt).

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs import
this module.  The product (``quantized-cnn_b200``) never does.
"""
import ctypes as C
import os
import subprocess
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(HERE, "_build", "libpq_oracle.so")
REF_SO = os.path.join(HERE, "_ref", "libqcnn_ref.so")
REF_DATA = os.path.join(HERE, "_ref", "data")
ALEXNET_DIR = os.path.join(REF_DATA, "AlexNet", "Bin.Files")
ALEXNET_PFX = "bvlc_alexnet_aCaF"

# ENUM_LyrType order of include/CaffePara.h:26
CONV, POOL, FCNT, RELU, LORN, DRPT, SMAX = range(7)


def build(force=False):
    """Compile the oracle (and, where /root/reference exists, the reference + staged fixtures)."""
    if force or not os.path.exists(ORACLE_SO) or \
            os.path.getmtime(ORACLE_SO) < os.path.getmtime(os.path.join(HERE, "pq_oracle.c")):
        subprocess.check_call(["make", "-s", "-C", HERE, "oracle"])
    if os.path.isdir("/root/reference/src"):
        subprocess.check_call(["make", "-s", "-C", HERE, "ref", "data"])


_oracle = None
_ref = None


def oracle():
    global _oracle
    if _oracle is None:
        build()
        L = C.CDLL(ORACLE_SO)
        L.pqo_read_bin.restype = C.c_long
        L.pqo_read_cbn.restype = C.c_long
        _oracle = L
    return _oracle


def have_ref():
    return os.path.exists(REF_SO)


def have_alexnet():
    return os.path.exists(os.path.join(ALEXNET_DIR, ALEXNET_PFX + ".asmtLst.22.cbn"))


def ref():
    global _ref
    if _ref is None:
        L = C.CDLL(REF_SO)
        L.ref_net_create.restype = C.c_void_p
        L.ref_net_create_custom.restype = C.c_void_p
        L.ref_net_time_forward.restype = C.c_double
        _ref = L
    return _ref


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _u8(a):
    return np.ascontiguousarray(a, dtype=np.uint8)


# ------------------------------------------------------------------------------------------------
# model description (Python mirror of CaffePara::ConfigLayer_AlexNet, src/CaffePara.cc:20-52)
# ------------------------------------------------------------------------------------------------
def conv(pad, k, cnt, grp, stride):
    return dict(type=CONV, pad=pad, k=k, cnt=cnt, grp=grp, stride=stride)


def pool(pad, k, stride):
    return dict(type=POOL, pad=pad, k=k, stride=stride)


def fcnt(n):
    return dict(type=FCNT, nod=n)


def relu():
    return dict(type=RELU)


def lorn(size, alpha, beta, k):
    return dict(type=LORN, size=size, alpha=alpha, beta=beta, kini=k)


def drpt(r):
    return dict(type=DRPT, ratio=r)


def smax():
    return dict(type=SMAX)


def alexnet_layers():
    return [conv(0, 11, 96, 1, 4), relu(), lorn(5, 1e-4, 0.75, 1.0), pool(0, 3, 2),
            conv(2, 5, 256, 2, 1), relu(), lorn(5, 1e-4, 0.75, 1.0), pool(0, 3, 2),
            conv(1, 3, 384, 1, 1), relu(), conv(1, 3, 384, 2, 1), relu(), conv(1, 3, 256, 2, 1), relu(),
            pool(0, 3, 2), fcnt(4096), relu(), drpt(0.5), fcnt(4096), relu(), drpt(0.5), fcnt(1000), smax()]


ALEXNET_IN = (3, 227, 227)
# (S, K, d) of the shipped quantized AlexNet, file index = layerInd + 1 (SURVEY.md A.3)
ALEXNET_PQ = {0: (1, 128, 8), 4: (6, 128, 8), 8: (32, 128, 8), 10: (24, 128, 8), 12: (24, 128, 8),
              15: (2304, 32, 4), 18: (1024, 32, 4), 21: (4096, 16, 1)}


def infer_shapes(layers, in_chw):
    """NHWC shapes (H, W, C) after every layer (CaffeEva::PrepFeatMap, src/CaffeEva.cc:328-392)."""
    c, h, w = in_chw
    shapes = [(h, w, c)]
    for L in layers:
        h, w, c = shapes[-1]
        if L["type"] == CONV:
            ho = (h + 2 * L["pad"] - L["k"]) // L["stride"] + 1
            wo = (w + 2 * L["pad"] - L["k"]) // L["stride"] + 1
            shapes.append((ho, wo, L["cnt"]))
        elif L["type"] == POOL:
            ho = int(np.ceil((h + 2 * L["pad"] - L["k"]) / float(L["stride"]))) + 1
            wo = int(np.ceil((w + 2 * L["pad"] - L["k"]) / float(L["stride"]))) + 1
            shapes.append((ho, wo, c))
        elif L["type"] == FCNT:
            shapes.append((1, 1, L["nod"]))
        else:
            shapes.append((h, w, c))
    return shapes


# ------------------------------------------------------------------------------------------------
# file formats
# ------------------------------------------------------------------------------------------------
def read_bin(path, dtype=np.float32):
    L = oracle()
    dims = (C.c_int * 4)()
    n = L.pqo_read_bin(path.encode(), dims, None, C.c_long(0), C.c_int(np.dtype(dtype).itemsize))
    if n < 0:
        raise IOError(path)
    out = np.empty(n, dtype)
    L.pqo_read_bin(path.encode(), dims, _p(out), C.c_long(n), C.c_int(out.itemsize))
    with open(path, "rb") as f:
        dc = np.frombuffer(f.read(4), np.int32)[0]
    return out.reshape([dims[i] for i in range(dc)])


def read_cbn(path):
    """0-based indices as CaffePara holds them after LoadLayerPara, plus the bit width."""
    L = oracle()
    dims = (C.c_int * 4)()
    bits = C.c_int(0)
    n = L.pqo_read_cbn(path.encode(), dims, None, C.c_long(0), C.byref(bits))
    if n < 0:
        raise IOError(path)
    out = np.empty(n, np.uint8)
    L.pqo_read_cbn(path.encode(), dims, _p(out), C.c_long(n), C.byref(bits))
    with open(path, "rb") as f:
        dc = np.frombuffer(f.read(4), np.int32)[0]
    return out.reshape([dims[i] for i in range(dc)]), bits.value


def write_bin(path, arr):
    arr = np.ascontiguousarray(arr)
    dims = (C.c_int * arr.ndim)(*arr.shape)
    if oracle().pqo_write_bin(path.encode(), arr.ndim, dims, _p(arr), arr.itemsize) != 0:
        raise IOError(path)


def write_cbn(path, idx0, bits):
    idx0 = _u8(idx0)
    dims = (C.c_int * idx0.ndim)(*idx0.shape)
    if oracle().pqo_write_cbn(path.encode(), idx0.ndim, dims, _p(idx0), bits) != 0:
        raise IOError(path)


def bits_for(K):
    """CaffePara::CalcBitCntPerEle on the 1-based maximum K (src/CaffePara.cc:360-378)."""
    b, m = 0, K - 1
    while m:
        m //= 2
        b += 1
    return b


# ------------------------------------------------------------------------------------------------
# per-layer oracle calls (numpy in / numpy out)
# ------------------------------------------------------------------------------------------------
def get_inpd(data, ctrd):
    data = _f32(data)
    ctrd = _f32(ctrd)
    P, D = data.shape
    S, K, d = ctrd.shape
    out = np.empty((P, S, K), np.float32)
    oracle().pqo_get_inpd(_p(data), C.c_long(P), D, _p(ctrd), S, K, d, _p(out))
    return out


def conv_aprx(src, L, ctrd, asmt, bias):
    """src NHWC [N,H,W,C]; ctrd [S,K,d]; asmt [Cout,k,k,S] 0-based (file order)."""
    src = _f32(src)
    ctrd = _f32(ctrd)
    asmt = _u8(asmt)
    bias = _f32(bias)
    N, H, W, Cin = src.shape
    S, K, d = ctrd.shape
    ho = (H + 2 * L["pad"] - L["k"]) // L["stride"] + 1
    wo = (W + 2 * L["pad"] - L["k"]) // L["stride"] + 1
    dst = np.empty((N, ho, wo, L["cnt"]), np.float32)
    oracle().pqo_conv_aprx(_p(src), N, H, W, Cin, L["cnt"], L["k"], L["pad"], L["stride"], L["grp"],
                           _p(ctrd), S, K, d, _p(asmt), _p(bias), _p(dst))
    return dst


def fc_aprx(src, ctrd, asmt, bias):
    """src [N,Din]; ctrd [S,K,d]; asmt [Dout,S] 0-based (file order)."""
    src = _f32(src)
    ctrd = _f32(ctrd)
    asmt = _u8(asmt)
    bias = _f32(bias)
    N, Din = src.shape
    S, K, d = ctrd.shape
    Dout = asmt.shape[0]
    dst = np.empty((N, Dout), np.float32)
    oracle().pqo_fc_aprx(_p(src), N, Din, Dout, _p(ctrd), S, K, d, _p(asmt), _p(bias), _p(dst))
    return dst


def relu_f(x):
    x = _f32(x)
    y = np.empty_like(x)
    oracle().pqo_relu(_p(x), C.c_long(x.size), _p(y))
    return y


def lrn_f(x, size, alpha, beta, k):
    x = _f32(x)
    y = np.empty_like(x)
    oracle().pqo_lrn(_p(x), C.c_long(x.size // x.shape[-1]), x.shape[-1], size, C.c_float(alpha),
                     C.c_float(beta), C.c_float(k), _p(y))
    return y


def pool_f(x, ksz, pad, stride):
    x = _f32(x)
    N, H, W, Cc = x.shape
    ho = int(np.ceil((H + 2 * pad - ksz) / float(stride))) + 1
    wo = int(np.ceil((W + 2 * pad - ksz) / float(stride))) + 1
    y = np.empty((N, ho, wo, Cc), np.float32)
    oracle().pqo_pool(_p(x), N, H, W, Cc, ksz, pad, stride, _p(y))
    return y


def softmax_f(x):
    x = _f32(x)
    y = np.empty_like(x)
    oracle().pqo_softmax(_p(x), x.shape[0], x.shape[1], _p(y))
    return y


def nchw_to_nhwc(x):
    x = _f32(x)
    N, Cc, H, W = x.shape
    y = np.empty((N, H, W, Cc), np.float32)
    oracle().pqo_nchw_to_nhwc(_p(x), N, Cc, H, W, _p(y))
    return y


def nhwc_to_nchw(x):
    x = _f32(x)
    N, H, W, Cc = x.shape
    y = np.empty((N, Cc, H, W), np.float32)
    oracle().pqo_nhwc_to_nchw(_p(x), N, H, W, Cc, _p(y))
    return y


def topk(prob, k=5):
    prob = _f32(prob)
    idx = np.empty(k, np.int32)
    val = np.empty(k, np.float32)
    oracle().pqo_topk(_p(prob), prob.size, k, _p(idx), _p(val))
    return idx, val


def lcg_images(n, seed0=12345, chw=ALEXNET_IN):
    """SURVEY.md 8(d) synthetic images: image i uses seed seed0 + i."""
    out = np.empty((n,) + tuple(chw), np.float32)
    per = int(np.prod(chw))
    for i in range(n):
        oracle().pqo_lcg_fill(C.c_uint32((seed0 + i) & 0xFFFFFFFF), _p(out[i]), C.c_long(per))
    return out


# ------------------------------------------------------------------------------------------------
# model parameter sets
# ------------------------------------------------------------------------------------------------
def load_model(dirpath, pfx, layers):
    """{layerInd: dict(bias, ctrd [S,K,d], asmt (file order, 0-based), bits)} for conv/FC layers."""
    params = {}
    for l, L in enumerate(layers):
        if L["type"] in (CONV, FCNT):
            base = os.path.join(dirpath, pfx)
            asmt, bits = read_cbn("%s.asmtLst.%02d.cbn" % (base, l + 1))
            params[l] = dict(bias=read_bin("%s.biasVec.%02d.bin" % (base, l + 1)).reshape(-1),
                             ctrd=read_bin("%s.ctrdLst.%02d.bin" % (base, l + 1)), asmt=asmt, bits=bits)
    return params


def synth_model(layers, in_chw, pq, seed=0, ctrd_std=0.05, bias_std=0.1):
    """Random-init parameters of a given architecture: ctrd ~ N(0, std^2), asmt ~ U{0..K-1}, bias ~ N(0, .1^2).

    ``pq`` maps layerInd -> (S, K, d).  As in the shipped conv1 file (d=8 of which 3 are used), codebook columns
    beyond the layer's input width stay in the file but are never read.
    """
    rng = np.random.RandomState(seed)
    shapes = infer_shapes(layers, in_chw)
    params = {}
    for l, L in enumerate(layers):
        if L["type"] not in (CONV, FCNT):
            continue
        S, K, d = pq[l]
        h, w, c = shapes[l]
        if L["type"] == CONV:
            asmt = rng.randint(0, K, size=(L["cnt"], L["k"], L["k"], S)).astype(np.uint8)
            nout = L["cnt"]
            fan = L["k"] * L["k"] * (c // L["grp"])
        else:
            asmt = rng.randint(0, K, size=(L["nod"], S)).astype(np.uint8)
            nout = L["nod"]
            fan = h * w * c
        std = ctrd_std if ctrd_std is not None else 1.0 / np.sqrt(fan)
        params[l] = dict(bias=(rng.randn(nout) * bias_std).astype(np.float32),
                         ctrd=(rng.randn(S, K, d) * std).astype(np.float32), asmt=asmt, bits=bits_for(K))
    return params


def synth_alexnet(seed=0):
    """AlexNet-shaped random model with He-style codebook scale so activations stay O(1..100) through 8 layers."""
    params = synth_model(alexnet_layers(), ALEXNET_IN, ALEXNET_PQ, seed=seed, ctrd_std=None, bias_std=0.05)
    # keep the logits well inside expf's range: the reference softmax does not subtract the maximum (CaffeEva.cc:1107)
    params[21]["ctrd"] = (params[21]["ctrd"] * np.float32(0.25)).astype(np.float32)
    return params


def save_model(dirpath, pfx, params):
    """Write parameters in the reference's on-disk formats (.bin / .cbn), readable by CaffePara::LoadLayerPara."""
    os.makedirs(dirpath, exist_ok=True)
    for l, p in params.items():
        base = os.path.join(dirpath, pfx)
        write_bin("%s.biasVec.%02d.bin" % (base, l + 1), p["bias"].astype(np.float32))
        write_bin("%s.ctrdLst.%02d.bin" % (base, l + 1), p["ctrd"].astype(np.float32))
        write_cbn("%s.asmtLst.%02d.cbn" % (base, l + 1), p["asmt"], p["bits"])


# ------------------------------------------------------------------------------------------------
# seeded stand-in for the reference's data directory
# ------------------------------------------------------------------------------------------------
SYNTH_BMP_SHAPES = [(375, 500), (333, 500), (500, 375), (256, 256), (227, 301), (480, 640), (301, 227), (257, 383),
                    (400, 299), (281, 421)]      # (H, W): several row paddings, up- and down-scaling


def write_bmp(path, pix):
    """uint8 [H, W, 3] (B, G, R, top row first) -> 24-bpp uncompressed bottom-up BMP."""
    h, w, _ = pix.shape
    row = (w * 3 + 3) & ~3
    body = np.zeros((h, row), np.uint8)
    body[:, :w * 3] = pix[::-1].reshape(h, w * 3)
    head = np.zeros(54, np.uint8)
    head[0:2] = [ord("B"), ord("M")]
    head[2:6] = np.frombuffer(np.uint32(54 + body.size).tobytes(), np.uint8)
    head[10:14] = np.frombuffer(np.uint32(54).tobytes(), np.uint8)
    head[14:18] = np.frombuffer(np.uint32(40).tobytes(), np.uint8)
    head[18:26] = np.frombuffer(np.array([w, h], "<i4").tobytes(), np.uint8)
    head[26:30] = np.frombuffer(np.array([1, 24], "<u2").tobytes(), np.uint8)
    head[34:38] = np.frombuffer(np.uint32(body.size).tobytes(), np.uint8)
    np.concatenate([head, body.reshape(-1)]).tofile(path)


def stage_synth_data(dirpath, seed=1):
    """Writes the layout CaffeEvaWrapper reads (AlexNet/Bin.Files/<ALEXNET_PFX>.*, AlexNet/imagenet_mean.single.bin,
    Cls.Names/class_names.txt, Cls.Names/image_labels.txt) plus ten BMPs under Bmp.Files/, all from seeds: the AlexNet
    of synth_alexnet(seed), a random mean image and random pictures of the sizes in SYNTH_BMP_SHAPES.  Returns the list
    of BMP paths."""
    rng = np.random.RandomState(seed + 1000)
    save_model(os.path.join(dirpath, "AlexNet", "Bin.Files"), ALEXNET_PFX, synth_alexnet(seed))
    write_bin(os.path.join(dirpath, "AlexNet", "imagenet_mean.single.bin"),
              (rng.rand(3, 256, 256) * 120 + 60).astype(np.float32))
    os.makedirs(os.path.join(dirpath, "Bmp.Files"), exist_ok=True)
    os.makedirs(os.path.join(dirpath, "Cls.Names"), exist_ok=True)
    paths = []
    for i, (h, w) in enumerate(SYNTH_BMP_SHAPES, 1):
        paths.append(os.path.join(dirpath, "Bmp.Files", "SYNTH_%08d.BMP" % i))
        write_bmp(paths[-1], rng.randint(0, 256, size=(h, w, 3)).astype(np.uint8))
    with open(os.path.join(dirpath, "Cls.Names", "class_names.txt"), "w") as f:
        f.write("".join("class %d\n" % c for c in range(1000)))
    with open(os.path.join(dirpath, "Cls.Names", "image_labels.txt"), "w") as f:
        f.write("".join("SYNTH_%08d.JPEG %d\n" % (i, (37 * i) % 1000) for i in range(1, len(paths) + 1)))
    return paths


# ------------------------------------------------------------------------------------------------
# whole-network oracle (the port): CaffeEva::ExecForwardPass(img, prob), src/CaffeEva.cc:213-261
# ------------------------------------------------------------------------------------------------
def net_forward(layers, params, img_nchw, keep=False):
    """Returns probs [N, C] (and, with keep=True, the list featMapLst[0..L] in the reference's element order)."""
    x = nchw_to_nhwc(img_nchw)
    maps = [x]
    first_fc = True
    for l, L in enumerate(layers):
        t = L["type"]
        if t == CONV:
            p = params[l]
            x = conv_aprx(x, L, p["ctrd"], p["asmt"], p["bias"])
        elif t == FCNT:
            p = params[l]
            if first_fc and x.ndim == 4:
                x = nhwc_to_nchw(x)  # CaffeEva.cc:236-238
            first_fc = False
            x = fc_aprx(x.reshape(x.shape[0], -1), p["ctrd"], p["asmt"], p["bias"])
        elif t == RELU:
            x = relu_f(x)
        elif t == LORN:
            x = lrn_f(x, L["size"], L["alpha"], L["beta"], L["kini"])
        elif t == POOL:
            x = pool_f(x, L["k"], L["pad"], L["stride"])
        elif t == DRPT:
            x = x.copy()  # CaffeEva.cc:1091-1096: identity
        elif t == SMAX:
            x = softmax_f(x.reshape(x.shape[0], -1))
        maps.append(x)
    return (x, maps) if keep else x


# ------------------------------------------------------------------------------------------------
# the compiled reference
# ------------------------------------------------------------------------------------------------
class _Spec(C.Structure):
    _fields_ = [("type", C.c_int), ("padSiz", C.c_int), ("knlSiz", C.c_int), ("knlCnt", C.c_int),
                ("grpCnt", C.c_int), ("stride", C.c_int), ("nodCnt", C.c_int), ("lrnSiz", C.c_int),
                ("lrnAlp", C.c_float), ("lrnBet", C.c_float), ("lrnIni", C.c_float), ("drpRat", C.c_float)]


def _spec(L):
    return _Spec(L["type"], L.get("pad", 0), L.get("k", 0), L.get("cnt", 0), L.get("grp", 0), L.get("stride", 0),
                 L.get("nod", 0), L.get("size", 0), L.get("alpha", 0.0), L.get("beta", 0.0), L.get("kini", 0.0),
                 L.get("ratio", 0.0))


class RefNet(object):
    """The reference's own CaffeEva object (batch size 1), driven through oracle/ref_harness.cc."""

    def __init__(self, dirpath, pfx, layers=None, in_chw=ALEXNET_IN, model="AlexNet"):
        R = ref()
        if layers is None:
            self.h = R.ref_net_create(dirpath.encode(), pfx.encode(), model.encode(), 1)
            layers = alexnet_layers()
        else:
            arr = (_Spec * len(layers))(*[_spec(L) for L in layers])
            self.h = R.ref_net_create_custom(dirpath.encode(), pfx.encode(), len(layers), arr, in_chw[0], in_chw[1],
                                             in_chw[2], 1)
        if not self.h:
            raise RuntimeError("reference failed to load %s/%s" % (dirpath, pfx))
        self.h = C.c_void_p(self.h)
        self.layers = layers
        self.in_chw = in_chw
        self.shapes = infer_shapes(layers, in_chw)

    def forward(self, img_chw):
        img = _f32(img_chw).reshape(-1)
        n_out = int(np.prod(self.shapes[-1]))
        prob = np.empty(n_out, np.float32)
        ref().ref_net_forward(self.h, _p(img), _p(prob), n_out)
        return prob

    def featmap(self, idx):
        dims = (C.c_int * 4)()
        n = ref().ref_net_featmap(self.h, idx, dims, None, 0)
        out = np.empty(n, np.float32)
        ref().ref_net_featmap(self.h, idx, dims, _p(out), n)
        return out.reshape([dims[i] for i in range(4)])

    def layer_forward(self, l, src):
        src = _f32(src).reshape(-1)
        n_out = int(np.prod(self.shapes[l + 1]))
        dst = np.empty(n_out, np.float32)
        r = ref().ref_net_layer_forward(self.h, l, _p(src), src.size, _p(dst), n_out)
        if r != n_out:
            raise RuntimeError("reference layer %d: size mismatch (%d vs %d)" % (l, r, n_out))
        return dst.reshape((1,) + tuple(self.shapes[l + 1]))

    def param(self, l, which):
        dims = (C.c_int * 4)()
        n = ref().ref_net_param(self.h, l, which, dims, None, 0)
        dt = np.uint8 if which == 2 else np.float32
        out = np.empty(n, dt)
        ref().ref_net_param(self.h, l, which, dims, _p(out), out.nbytes)
        return out, [dims[i] for i in range(4)]

    def time_forward(self, imgs, warmup, iters):
        imgs = _f32(imgs)
        each = np.zeros(iters, np.float64)
        tot = ref().ref_net_time_forward(self.h, _p(imgs), imgs.shape[0], warmup, iters, _p(each))
        return tot, each

    def close(self):
        if self.h:
            ref().ref_net_destroy(self.h)
            self.h = None


def ref_get_inpd(data, ctrd_skd):
    """Reference GetInPdMat; ctrd given in FILE order [S,K,d] (permuted here like PrepCtrdBuf does)."""
    data = _f32(data)
    S, K, d = ctrd_skd.shape
    buf = _f32(np.transpose(ctrd_skd, (0, 2, 1)))
    P, D = data.shape
    out = np.empty((P, S, K), np.float32)
    ref().ref_get_inpd(_p(data), P, D, _p(buf), S, d, K, _p(out))
    return out
