"""Device Canny edge map of the Gated-SCNN forward (kdcc_canny, kdcc.functional.canny_edges; DESIGN.md 4.3f).

The contract is bit-exactness with models/gscnn/gscnn.py:284-288: numpy's uint8 cast, then cv2.Canny(img, low, high)
with aperture 3 and the L1 gradient.  CPU: argument validation of the C ABI, the numpy reference (canny_oracle.py)
against cv2 itself and against the frozen cv2 output of tests/golden/canny.npz, and the cast rule byte by byte.  GPU:
the kernels against the reference, bit for bit, in fp32 and bf16, NCHW and channels_last."""
import ctypes
import math
import os

import numpy as np
import pytest
import torch

import canny_oracle as orc

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "canny.npz")
THRESHOLDS = [(10, 100), (50, 150), (100, 10), (0, 0), (30.7, 30.2)]


@pytest.fixture(scope="module")
def kdcc():
    import __graft_entry__ as entry
    entry.build()
    import kdcc as pkg
    return pkg


def random_u8(rs, H, W, C, kind):
    if kind == "noise":
        return rs.randint(0, 256, (H, W, C)).astype(np.uint8)
    if kind == "smooth":
        from scipy import ndimage
        return np.clip(ndimage.gaussian_filter(rs.rand(H, W, C) * 255, (2, 2, 0)), 0, 255).astype(np.uint8)
    img = np.zeros((H, W, C), np.uint8)
    yy, xx = np.mgrid[:H, :W]
    for _ in range(3):
        cy, cx, r = rs.randint(0, H), rs.randint(0, W), rs.randint(1, 30)
        img[(yy - cy) ** 2 + (xx - cx) ** 2 < r * r] = rs.randint(0, 256, C)
    return img


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def test_abi_validation(kdcc):
    L = kdcc._abi.lib()
    NCHW, NHWC, F32, BF16 = kdcc._abi.NCHW, kdcc._abi.NHWC, kdcc._abi.F32, kdcc._abi.BF16
    p = ctypes.c_void_p(256)   # never dereferenced: validation returns before any CUDA call
    ws = L.kdcc_canny_workspace_bytes(2, 64, 64)
    assert ws > 0
    assert L.kdcc_canny_workspace_bytes(2, 64, 128) > ws and L.kdcc_canny_workspace_bytes(4, 64, 128) > L.kdcc_canny_workspace_bytes(2, 64, 128)

    def call(img=p, edges=p, work=p, nbytes=ws, N=2, C=3, H=64, W=64, layout=NCHW, dtype=F32, low=10.0, high=100.0):
        return L.kdcc_canny(img, edges, work, nbytes, N, C, H, W, layout, dtype, low, high, None)

    assert call(img=None) == -1 and call(edges=None) == -1 and call(work=None) == -1
    for dims in ({"N": 0}, {"H": 0}, {"W": 0}, {"N": -1}, {"H": -5}, {"W": -2}):
        assert call(**dims) == -1, dims
    assert call(C=1) == -2 and call(C=4) == -2
    assert call(layout=7) == -1 and call(layout=2) == -1 and call(dtype=5) == -1 and call(dtype=-1) == -1
    assert call(low=float("nan")) == -1
    assert call(nbytes=ws - 1) == -3
    big = L.kdcc_canny_workspace_bytes(2, 1 << 15, 1 << 15)        # N*H*W = 2^31
    assert call(N=2, H=1 << 15, W=1 << 15, nbytes=big) == -2
    assert call(N=1, H=1 << 15, W=1 << 15, layout=NHWC, dtype=BF16) == -3   # 2^30 pixels: shape accepted, workspace short


def test_cast_rule_bytes():
    x = np.array([-1.5, 0.7, 256.2, 300, -200, 1e10, -1e10, np.nan, np.inf, -np.inf, 255.9, -0.9, 2147483520.0, -2147483648.0,
                  2147483648.0, -2.1, 2.6], np.float32)
    want = [255, 0, 0, 44, 56, 0, 0, 0, 0, 0, 255, 0, 128, 0, 0, 254, 2]
    assert orc.to_uint8_like_numpy(x).tolist() == want
    v = np.random.RandomState(0).uniform(-1000, 1000, 10000).astype(np.float32)   # in int32 range: numpy agrees everywhere
    assert np.array_equal(orc.to_uint8_like_numpy(v), v.astype(np.int32).astype(np.uint8))
    v = np.random.RandomState(1).uniform(0, 256, 10000).astype(np.float32)
    assert np.array_equal(orc.to_uint8_like_numpy(v), v.astype(np.uint8))


@pytest.mark.parametrize("threads", [1, None])
def test_oracle_matches_cv2_sweep(threads):
    cv2 = pytest.importorskip("cv2")
    prev = cv2.getNumThreads()
    if threads is not None:
        cv2.setNumThreads(threads)
    try:
        rs = np.random.RandomState(11 if threads else 12)
        sizes = [(1, 1), (1, 7), (9, 1), (2, 2), (3, 5)] + [(rs.randint(1, 90), rs.randint(1, 130)) for _ in range(55)]
        for k, (H, W) in enumerate(sizes):
            C = 3 if k % 3 else 1
            img = random_u8(rs, H, W, C, ("noise", "smooth", "shapes")[k % 3])
            if C == 1:
                img = img[:, :, 0]
            for lo, hi in THRESHOLDS:
                assert np.array_equal(orc.canny(img, lo, hi), cv2.Canny(img, lo, hi)), (H, W, C, lo, hi)
    finally:
        cv2.setNumThreads(prev)


def test_oracle_matches_cv2_full_size():
    cv2 = pytest.importorskip("cv2")
    img = random_u8(np.random.RandomState(5), 1024, 2048, 3, "smooth")
    img[::7] = np.random.RandomState(6).randint(0, 256, img[::7].shape)
    assert np.array_equal(orc.canny(img, 10, 100), cv2.Canny(img, 10, 100))


def test_oracle_matches_golden():
    g = np.load(GOLD)
    n = len([k for k in g.files if k.startswith("img_")])
    assert n >= 5
    for k in range(n):
        lo, hi = g["thr_%d" % k]
        assert np.array_equal(orc.canny(g["img_%d" % k], lo, hi), g["edges_%d" % k]), k


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def device_input(x, dtype, channels_last):
    """(N, 3, H, W) float numpy -> device tensor; returns it and the fp32 values the device sees (bf16 rounded)."""
    t = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).cuda().to(dtype)
    if channels_last:
        t = t.contiguous(memory_format=torch.channels_last)
    return t, t.float().cpu().numpy()


def check(kdcc, x, lo=10, hi=100, dtype=torch.float32, channels_last=False, cv2_too=True):
    t, seen = device_input(x, dtype, channels_last)
    got = kdcc.functional.canny_edges(t, lo, hi)
    assert got.dtype == torch.float32 and got.shape == (x.shape[0], 1, x.shape[2], x.shape[3]) and got.is_contiguous()
    assert got.grad_fn is None
    got = got.cpu().numpy()
    want = orc.gscnn_canny(seen, lo, hi)
    assert np.array_equal(got, want), "%d of %d pixels differ" % (int((got != want).sum()), got.size)
    if cv2_too:
        try:
            import cv2
        except ImportError:
            return got
        im = orc.to_uint8_like_numpy(seen.transpose(0, 2, 3, 1))
        for i in range(x.shape[0]):
            assert np.array_equal(got[i, 0], cv2.Canny(im[i], lo, hi)), i
    return got


FORMATS = [(torch.float32, False), (torch.float32, True), (torch.bfloat16, False), (torch.bfloat16, True)]
FORMAT_IDS = ["f32-nchw", "f32-cl", "bf16-nchw", "bf16-cl"]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype,cl", FORMATS, ids=FORMAT_IDS)
@pytest.mark.parametrize("H,W", [(1, 1), (1, 300), (300, 1), (7, 13), (33, 65), (129, 257), (1023, 2047)])
def test_sizes_dtypes_layouts(kdcc, H, W, dtype, cl):
    rs = np.random.RandomState(H * 7919 + W)
    N = 2 if H * W < 10 ** 6 else 1
    x = np.stack([random_u8(rs, H, W, 3, kind).transpose(2, 0, 1) for kind in ("smooth", "shapes")[:N]]).astype(np.float32)
    x += rs.uniform(-0.9, 0.9, x.shape).astype(np.float32)           # fractions truncate toward zero
    flat = x.reshape(-1)
    pos = rs.randint(0, flat.size, 12)
    flat[pos] = np.array([-1.5, 300, -200, 1e10, np.nan, np.inf, -np.inf, 256.2, -0.5, 511, -255, 2.6], np.float32)
    for lo, hi in THRESHOLDS:
        check(kdcc, x, lo, hi, dtype, cl, cv2_too=(lo, hi) == (10, 100))


def structured_images():
    H = W = 96
    yy, xx = np.mgrid[:H, :W].astype(np.float64)
    out = {}
    angles = np.arange(0, 180.001, 3.75)
    steps, lines = [], []
    for k, a in enumerate(angles):
        t = math.radians(a)
        d = (xx - W / 2 + 0.3) * math.cos(t) + (yy - H / 2 + 0.1) * math.sin(t)
        ramp = np.clip(d * 0.7 + 0.5, 0, 1)               # anti-aliased step: directions around every sector bound
        steps.append(np.stack([ramp * 200 + 20, ramp * (90 + k) + 40, (1 - ramp) * 160 + 10]))
        line = np.clip(1.5 - np.abs(d), 0, 1)
        lines.append(np.stack([line * 230, line * 120 + 30, line * (70 + 3 * k)]))
    out["steps"] = np.stack(steps)
    out["lines"] = np.stack(lines)
    circles = []
    for r in (3, 7.5, 15, 30, 45):
        disc = np.clip(r + 0.5 - np.hypot(yy - 47.3, xx - 48.6), 0, 1)
        circles.append(np.stack([disc * 255, disc * 128, 255 - disc * 200]))
    out["circles"] = np.stack(circles)
    checks = []
    for s in (1, 2, 3, 8):
        cb = (((yy // s) + (xx // s)) % 2) * 255
        checks.append(np.stack([cb, 255 - cb, cb * 0.5]))
    out["checkerboards"] = np.stack(checks)
    rs = np.random.RandomState(3)
    from scipy import ndimage
    q = []
    for levels in (2, 3, 4):
        base = ndimage.gaussian_filter(rs.rand(H, W), 3)
        base = np.floor((base - base.min()) / (np.ptp(base) + 1e-9) * levels) * (255 // levels)
        q.append(np.stack([base, base, base]))                          # equal channels: every magnitude ties
        q.append(np.stack([base, base[::-1], base.T]))
    out["quantised"] = np.stack(q)
    out["constant"] = np.full((2, 3, H, W), 77.0)
    return {k: v.astype(np.float32) for k, v in out.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("cl", [False, True], ids=["nchw", "cl"])
@pytest.mark.parametrize("kind", ["steps", "lines", "circles", "checkerboards", "quantised", "constant"])
def test_structured_images(kdcc, kind, cl):
    x = structured_images()[kind]
    for lo, hi in THRESHOLDS:
        got = check(kdcc, x, lo, hi, torch.float32, cl)
        if kind == "constant":
            assert not got.any()
        if kind in ("steps", "circles") and (lo, hi) == (10, 100):
            assert got.any()


def serpentine(strong):
    """A 1024 x 2048 band of value 5 that snakes through every 16-row tile band and every 128-column tile, whose
    one-pixel contour (|grad| = 20: weak at thresholds (10, 100)) is one 8-connected candidate component.  With `strong`
    the band's first 8 x 2 pixels are 40: a few strong candidates at one end of the contour."""
    H, W = 1024, 2048
    img = np.zeros((H, W), np.float32)
    for k, y in enumerate(range(4, H, 16)):
        img[y:y + 8, 8:W - 8] = 5
        if y + 24 <= H:
            x = W - 16 if k % 2 == 0 else 8
            img[y:y + 24, x:x + 8] = 5
    if strong:
        img[4:12, 8:10] = 40
    return np.broadcast_to(img, (1, 3, H, W)).copy()


@pytest.mark.gpu
def test_cross_tile_hysteresis(kdcc):
    x = serpentine(True)
    got = check(kdcc, x, 10, 100)[0, 0] > 0
    cand = orc.gscnn_canny(x, 10, 10)[0, 0] > 0                  # low == high: every candidate is strong
    assert cand.sum() > 250000
    assert np.array_equal(got, cand)                             # the whole winding contour is lit
    assert got.reshape(64, 16, 16, 128).any(axis=(1, 3)).all()   # ... in every 16 x 128 tile
    assert not check(kdcc, serpentine(False), 10, 100).any()


@pytest.mark.gpu
def test_full_size_gscnn(kdcc):
    rs = np.random.RandomState(8)
    x = np.stack([random_u8(rs, 1024, 2048, 3, "smooth").transpose(2, 0, 1), random_u8(rs, 1024, 2048, 3, "shapes").transpose(2, 0, 1)])
    x = x.astype(np.float32) + rs.uniform(0, 0.99, x.shape).astype(np.float32)
    x[1, :, ::5] = rs.uniform(0, 255, x[1, :, ::5].shape)
    got = check(kdcc, x)
    try:
        import cv2
    except ImportError:
        cv2 = None
    if cv2 is not None:   # the forward's own lines
        inp = torch.from_numpy(x).cuda()
        N, _, H, W = inp.shape
        im_arr = inp.cpu().numpy().transpose((0, 2, 3, 1)).astype(np.uint8)
        canny = np.zeros((N, 1, H, W))
        for i in range(N):
            canny[i] = cv2.Canny(im_arr[i], 10, 100)
        canny = torch.from_numpy(canny).cuda().float()
        assert torch.equal(kdcc.functional.canny_edges(inp, 10, 100), canny)
    # ImageNet-normalised input, as the reference loop feeds it: values in about [-2.1, 2.6] cast to 254, 255, 0, 1, 2
    mean = np.array([0.485, 0.456, 0.406], np.float32)[None, :, None, None]
    std = np.array([0.229, 0.224, 0.225], np.float32)[None, :, None, None]
    xn = ((x / 255 - mean) / std).astype(np.float32)
    got = check(kdcc, xn)
    assert got.any()


@pytest.mark.gpu
def test_repeatable_graph_and_side_stream(kdcc):
    rs = np.random.RandomState(9)
    x = torch.from_numpy(rs.uniform(0, 255, (2, 3, 256, 512)).astype(np.float32)).cuda()
    f = kdcc.functional.canny_edges
    a, b = f(x, 10, 100), f(x, 10, 100)
    assert torch.equal(a, b)
    assert np.array_equal(a.cpu().numpy(), orc.gscnn_canny(x, 10, 100))

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        c = f(x, 10, 100)
    torch.cuda.current_stream().wait_stream(s)
    assert torch.equal(a, c)

    static_in = x.clone()
    g = torch.cuda.CUDAGraph()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        f(static_in, 10, 100)                                    # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(s)
    with torch.cuda.graph(g, stream=s):
        static_out = f(static_in, 10, 100)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(static_out, a)
    y = torch.from_numpy(rs.uniform(0, 255, (2, 3, 256, 512)).astype(np.float32)).cuda()
    static_in.copy_(y)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(static_out, f(y, 10, 100))
