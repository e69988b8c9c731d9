"""Test-time windows of inference_test on the device (kdcc_tta_windows, kdcc.functional.tta_windows,
kdcc.tta.prepare_windows; DESIGN.md 4.3h).

The contract is bit-exactness with the host preparation of utils/tta_process.py:52-117 as kdcc.tta's host mirror runs
it: ToPILImage, PIL resize BILINEAR, FLIP_LEFT_RIGHT, ToTensor + Normalize and the window crops.  CPU: the numpy
restatement (tta_prep_oracle.py) against Pillow's resize, torch's cast and the host mirror's windows, and argument
validation of the C ABI.  GPU: the kernels against the host mirror with torch.equal, in fp32 and bf16."""
import ctypes
import math

import numpy as np
import pytest
import torch

import tta_prep_oracle as orc

MEAN_STD = ([0.485, 0.456, 0.406], [0.229, 0.224, 0.225])
SCALES = [1.0, 0.5, 0.75, 1.25, 1.75]


@pytest.fixture(scope="module")
def kdcc():
    import __graft_entry__ as entry
    entry.build()
    import kdcc as pkg
    return pkg


def host_windows(x, scales, crop, overlap=1 / 3):
    """inference_test's host preparation of one image: (ori_size, mapping, windows) on the host.  bf16 goes through
    ToPILImage's `pic.mul(255).byte()` form (torchvision up to 0.15); the installed torchvision converts through numpy,
    which has no bf16, and for fp32 the two forms give the same bytes (test_oracle_cast_matches_torch)."""
    from PIL import Image
    from torchvision import transforms
    from kdcc import tta
    x = x.cpu()
    if x.dtype == torch.bfloat16:
        image = Image.fromarray(x.mul(255).byte().permute(1, 2, 0).numpy(), "RGB")
    else:
        image = transforms.ToPILImage()(x)
    data = tta.scale_and_flip_image(image, MEAN_STD, scales)
    return tta.get_crops_image(data, scales, crop_size=crop, overlap=overlap)


def make_image(rs, H, W, kind, specials=False):
    """(3, H, W) fp32: [0, 1] data, or ImageNet-normalised data (what inference_test is fed), optionally with NaN /
    +-inf / 1e10 / -1e10 sprinkled in."""
    x = rs.uniform(0, 1, (3, H, W)).astype(np.float32)
    if kind == "imagenet":
        x = (x - np.float32(MEAN_STD[0]).reshape(3, 1, 1)) / np.float32(MEAN_STD[1]).reshape(3, 1, 1)
    if specials:
        flat = x.reshape(-1)
        idx = rs.choice(flat.size, min(flat.size, 40), replace=False)
        flat[idx] = rs.choice([np.nan, np.inf, -np.inf, 1e10, -1e10, 300.0 / 255, -1.7 / 255], idx.size)
    return torch.from_numpy(x)


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def _resize_cases():
    rs = np.random.RandomState(21)
    cases = []
    for H, W in [(1, 1), (1, 37), (53, 1), (1, 90), (90, 1), (7, 5), (13, 89)]:
        for s in (0.25, 0.5, 1.3, 2.0):
            cases.append((H, W, max(int(W * s), 1), max(int(H * s), 1)))
    for _ in range(40):   # odd sizes, random up- and downscales
        H, W = rs.randint(1, 91), rs.randint(1, 91)
        s = rs.uniform(0.25, 2.0)
        cases.append((H, W, max(int(W * s), 1), max(int(H * s), 1)))
    for _ in range(10):   # int(w * s) just below and just above an integer
        H, W, k = rs.randint(5, 91), rs.randint(5, 91), rs.randint(2, 60)
        for d in (-1e-3, 1e-3):
            s = (k + d) / W
            cases.append((H, W, int(W * s), max(int(H * s), 1)))
    for _ in range(10):   # downscale to a quarter: four-pixel support
        H, W = rs.randint(8, 91), rs.randint(8, 91)
        cases.append((H, W, int(W * 0.25), int(H * 0.25)))
    for _ in range(6):    # one axis unchanged
        H, W = rs.randint(2, 91), rs.randint(2, 91)
        cases += [(H, W, W, rs.randint(1, 120)), (H, W, rs.randint(1, 120), H)]
    return cases


def test_oracle_resize_matches_pillow():
    from PIL import Image
    rs = np.random.RandomState(3)
    for H, W, w, h in _resize_cases():
        img = rs.randint(0, 256, (H, W, 3)).astype(np.uint8)
        want = np.asarray(Image.fromarray(img).resize((w, h), Image.BILINEAR))
        assert np.array_equal(orc.pil_resize(img, w, h), want), (H, W, w, h)


def test_oracle_cast_matches_torch():
    rs = np.random.RandomState(4)
    specials = np.float32([2.2, -1.7, 300 / 255, np.nan, np.inf, -np.inf, 1e10, -1e10, 0.0, -0.0, 1.0, 255.9 / 255,
                           2147483520.0 / 255, 8.4e6, -8.4e6, 2.64, -2.1179])
    imagenet = make_image(rs, 64, 64, "imagenet").numpy().reshape(-1)
    x = np.concatenate([specials, imagenet, rs.standard_normal(20000).astype(np.float32) * 4,
                        rs.uniform(0, 1, 20000).astype(np.float32)])
    t = torch.from_numpy(x)
    assert np.array_equal(orc.to_pil_bytes(x), t.mul(255).byte().numpy())
    with np.errstate(invalid="ignore"):   # the installed ToPILImage's numpy form
        assert np.array_equal(orc.to_pil_bytes(x), (x * 255).astype(np.uint8))
    tb = t.bfloat16()
    assert np.array_equal(orc.to_pil_bytes(tb.float().numpy(), bf16=True), tb.mul(255).byte().numpy())
    assert orc.to_pil_bytes(np.float32([2.2]), bf16=True)[0] == 48 and orc.to_pil_bytes(np.float32([2.2]))[0] == 49
    assert orc.to_pil_bytes(np.float32([-1.7 / 255, 300 / 255]))[:].tolist() == [255, 44]


@pytest.mark.parametrize("kind", ["unit", "imagenet"])
def test_oracle_windows_match_host_mirror(kind):
    pytest.importorskip("torchvision")
    rs = np.random.RandomState(5)
    for H, W, crop, s, bf16 in [(36, 60, 24, 1.0, False), (41, 67, 32, 0.75, True), (29, 53, 16, 1.25, False),
                                (24, 30, 64, 0.5, False), (50, 45, 24, 1.75, True), (1, 33, 2, 1.3, False)]:
        x = make_image(rs, H, W, kind, specials=True)
        if bf16:
            x = x.bfloat16()
        ori, mapping, want = host_windows(x, [s], crop)
        (w, h, boxes), = mapping
        tile = int(s * crop)
        stride = math.ceil(tile * (1 - 1 / 3))
        got = orc.tta_windows(x.float().numpy(), h, w, tile, stride, *MEAN_STD, bf16=bf16)
        assert ori == (W, H) and orc.window_boxes(w, h, tile, stride) == boxes
        assert got.shape == tuple(want.shape) and np.array_equal(got.view(np.uint32), want.numpy().view(np.uint32))


def test_window_count_matches_window_coordinates(kdcc):
    for w, h, tile in [(60, 36, 24), (2048, 1024, 1024), (1536, 768, 768), (30, 20, 64), (100, 7, 13), (5, 5, 1)]:
        stride = math.ceil(tile * (1 - 1 / 3))
        assert kdcc.functional.tta_window_count(w, h, tile, stride) == len(kdcc.tta.window_coordinates(w, h, tile))
    assert kdcc.functional.tta_window_count(10, 10, 40, 27) == 0 and kdcc.tta.window_coordinates(10, 10, 40) == []


def test_abi_validation_and_workspace(kdcc):
    L = kdcc._abi.lib()
    F32, BF16 = kdcc._abi.F32, kdcc._abi.BF16
    p = ctypes.c_void_p(256)   # never dereferenced: validation returns before any CUDA call
    ws = L.kdcc_tta_windows_workspace_bytes(64, 96, 48, 72)
    assert ws >= 3 * 64 * 72                                      # the horizontal pass's uint8 intermediate
    assert L.kdcc_tta_windows_workspace_bytes(64, 96, 64, 96) == 0   # scale 1: a plain copy, no workspace
    assert 0 < L.kdcc_tta_windows_workspace_bytes(64, 96, 48, 96) < 3 * 64 * 96   # vertical pass only: weights
    assert L.kdcc_tta_windows_workspace_bytes(64, 96, 48, 73) > ws
    assert L.kdcc_tta_windows_workspace_bytes(0, 96, 48, 72) == 0

    def call(img=p, H=64, W=96, dtype=F32, h=48, w=72, tile=32, stride=22, out=p, work=p, nbytes=ws):
        return L.kdcc_tta_windows(img, H, W, dtype, h, w, tile, stride, 0.5, 0.5, 0.5, 0.25, 0.25, 0.25, out, work,
                                  nbytes, None)

    assert call(img=None) == -1 and call(out=None) == -1 and call(work=None) == -1
    for dims in ({"H": 0}, {"W": -1}, {"h": 0}, {"w": -3}, {"tile": 0}, {"stride": 0}, {"stride": -4}):
        assert call(**dims) == -1, dims
    assert call(dtype=2) == -1 and call(dtype=5) == -1 and call(dtype=-1) == -1   # code 2 is pointwise-only
    assert call(nbytes=ws - 1) == -3
    assert call(H=1 << 15, W=1 << 15, h=64, w=64, dtype=BF16) == -2              # 3 * 2^30 image elements
    big = L.kdcc_tta_windows_workspace_bytes(1 << 14, 1 << 14, 64, 1 << 13)
    assert big > 3 * (1 << 27)
    assert call(H=1 << 14, W=1 << 14, h=64, w=1 << 13, nbytes=big - 1) == -3      # 3 * 2^28: accepted, workspace short
    assert call(H=1000, W=1000, h=1000, w=1000, tile=100, stride=1, work=None, nbytes=0) == -2   # 4.9e10 outputs
    # no window (the tile overhangs the image by a stride or more): nothing to write, no CUDA call
    assert call(H=10, W=10, h=10, w=10, tile=40, stride=27, work=None, nbytes=0) == 0


def test_entry_points_refuse_host_tensors_and_mismatched_scales(kdcc):
    x = torch.rand(3, 20, 30)
    with pytest.raises(kdcc.KdccError):
        kdcc.functional.tta_windows(x, 20, 30, 16, 11, *MEAN_STD)
    with pytest.raises(kdcc.KdccError):
        kdcc.tta.prepare_windows(x, [1.0], 16, MEAN_STD)
    with pytest.raises(RuntimeError, match="Sizes of tensors must match"):   # torch.cat's rule, before any kernel
        kdcc.tta.prepare_windows(x, [1.0, 0.5], 16, MEAN_STD)
    with pytest.raises(RuntimeError):
        kdcc.tta.prepare_windows(x, [1.0], 80, MEAN_STD)                     # no window: torch.stack([]) raises
    with pytest.raises(ValueError):
        kdcc.tta.prepare_windows(x, [0.01], 16, MEAN_STD)                    # PIL refuses an empty image


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _device_windows(kdcc, x, s, crop):
    H, W = x.shape[1:]
    tile = int(s * crop)
    return kdcc.functional.tta_windows(x, int(H * s), int(W * s), tile, math.ceil(tile * (1 - 1 / 3)), *MEAN_STD)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("kind", ["unit", "imagenet"])
@pytest.mark.parametrize("s", SCALES)
def test_windows_match_host_mirror(kdcc, dtype, kind, s):
    rs = np.random.RandomState(int(s * 100) + (7 if kind == "unit" else 8))
    for H, W, crop in [(97, 161, 64), (64, 64, 32), (33, 250, 48), (30, 24, 64), (2, 90, 2), (90, 2, 2)]:
        x = make_image(rs, H, W, kind, specials=(H == 97))
        if dtype == "bf16":
            x = x.bfloat16()
        ori, mapping, want = host_windows(x, [s], crop)
        got = _device_windows(kdcc, x.cuda(), s, crop)
        assert torch.equal(got.cpu(), want), (H, W, crop)
        ori2, mapping2, got2 = kdcc.tta.prepare_windows(x.cuda(), [s], crop, MEAN_STD)
        assert (ori2, mapping2) == (ori, mapping) and torch.equal(got2, got)


@pytest.mark.gpu
@pytest.mark.parametrize("s", [1.0, 0.75])
def test_full_frame_matches_host_mirror(kdcc, s):
    rs = np.random.RandomState(31)
    for kind, dtype in [("imagenet", torch.float32), ("unit", torch.bfloat16)]:
        x = make_image(rs, 1024, 2048, kind).to(dtype)
        ori, mapping, want = host_windows(x, [s], 1024)
        ori2, mapping2, got = kdcc.tta.prepare_windows(x.cuda(), [s], 1024, MEAN_STD)
        assert (ori2, mapping2) == (ori, mapping)
        assert got.shape == want.shape and torch.equal(got.cpu(), want), kind


@pytest.mark.gpu
def test_prepare_windows_several_scales_in_one_batch(kdcc):
    rs = np.random.RandomState(12)
    # every scale gives the same window size, as the reference's torch.cat needs
    for H, W, crop, scales in [(36, 60, 24, [1.0, 1.03, 1.01]), (100, 150, 4, [1.0, 1.2, 1.1, 1.05]),
                               (24, 30, 64, [1.0])]:
        x = make_image(rs, H, W, "imagenet", specials=True)
        ori, mapping, want = host_windows(x, scales, crop)
        ori2, mapping2, got = kdcc.tta.prepare_windows(x.cuda(), scales, crop, MEAN_STD)
        assert (ori2, mapping2) == (ori, mapping) and torch.equal(got.cpu(), want), (H, W, scales)


@pytest.mark.gpu
def test_inference_test_matches_host_prepared_path(kdcc):
    """inference_test with device preparation against the same loop fed by the host preparation (its previous form)."""
    from kdcc import tta
    torch.manual_seed(0)
    net = torch.nn.Conv2d(3, 5, 1).cuda()
    for data, args in [(torch.rand(2, 3, 36, 60, device="cuda"), {"scales": [1.0], "crop_size": 24}),
                       (torch.randn(1, 3, 53, 81, device="cuda"), {"scales": [0.75], "crop_size": 32}),
                       (torch.randn(2, 3, 40, 64, device="cuda").bfloat16(), {"scales": [1.0, 1.03], "crop_size": 24})]:
        out = tta.inference_test(lambda w: net(w.float()), data, args)
        for n in range(data.shape[0]):
            ori, mapping, windows = host_windows(data[n], args["scales"], args["crop_size"])
            with torch.no_grad():
                want = tta.reverse_mapping(mapping, net(windows.cuda()), ori).mean(dim=0)
            assert torch.equal(out[n], want)


@pytest.mark.gpu
def test_no_sync_repeatable_and_graph_replay(kdcc):
    rs = np.random.RandomState(13)
    x = make_image(rs, 256, 384, "imagenet").cuda()
    f = lambda img, s: _device_windows(kdcc, img, s, 128)
    for s in (1.0, 0.75):
        f(x, s)                                   # library and workspace in place before the checked calls
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        a = {s: f(x, s) for s in (1.0, 0.75)}
        kdcc.tta.prepare_windows(x, [0.75], 128, MEAN_STD)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    for s in (1.0, 0.75):
        assert torch.equal(a[s], f(x, s))

    s = torch.cuda.Stream()
    static_in = x.clone()
    g = torch.cuda.CUDAGraph()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        f(static_in, 0.75)                        # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(s)
    with torch.cuda.graph(g, stream=s):
        static_out = f(static_in, 0.75)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(static_out, a[0.75])
    y = make_image(rs, 256, 384, "unit").cuda()
    static_in.copy_(y)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(static_out, f(y, 0.75))
