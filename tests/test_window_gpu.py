"""Sliding-window inference in the predict step: the window gather kernel against torch slicing, the overlap-averaging
predict epilogue against an fp64 evaluation of the window semantics, and predict_mask(window=, stride=) against its
torch composition on the bf16 and FP8 models, chunked and above the single-forward bound."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from iswm_b200 import ops
from tests.test_model_gpu import build, report

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _labels(B, H, W, seed, dtype=torch.int64):
    g = torch.Generator().manual_seed(seed)
    y = (torch.rand((B, H, W), generator=g) < 0.3).long()
    y[torch.rand((B, H, W), generator=g) < 0.05] = 255
    return y.to(dtype).to(DEV)


def _counts(y, pred):
    t, p = y.long().cpu().numpy().ravel(), pred.long().cpu().numpy().ravel()
    ok = (t == 0) | (t == 1)
    return np.bincount(t[ok] * 2 + p[ok], minlength=4)


def _grid(H, W, window, stride):
    (wh, ys), (ww, xs) = ops.window_offsets(H, window[0], stride[0]), ops.window_offsets(W, window[1], stride[1])
    return (wh, ww), [(y0, x0) for y0 in ys for x0 in xs]


# ----------------------------------------------------------------------------- gather
@pytest.mark.parametrize("shape,window,stride", [((2, 3, 70, 93), (32, 40), (20, 27)), ((3, 2, 64, 64), (32, 32), (32, 32)),
                                                 ((2, 3, 50, 130), (80, 48), (60, 16)), ((1, 3, 40, 30), (64, 64), (48, 48))])
def test_gather_matches_torch_slicing(shape, window, stride):
    g = torch.Generator().manual_seed(shape[2] + shape[3])
    x = torch.randn(shape, generator=g).to(DEV)
    (wh, ww), offs = _grid(shape[2], shape[3], window, stride)
    ref = torch.cat([x[b:b + 1, :, y0:y0 + wh, x0:x0 + ww] for b in range(shape[0]) for y0, x0 in offs])
    got = ops.window_gather_f32(x, window, stride)
    assert torch.equal(got, ref)
    # sub-ranges into batch slices of a larger buffer, the rest untouched
    N = ref.shape[0]
    for first, n in ((0, 1), (1, N - 2), (N - 3, 3), (N // 2, N - N // 2)):
        if first < 0 or n < 1 or first + n > N:
            continue
        buf = torch.full((n + 2,) + tuple(ref.shape[1:]), float("nan"), device=DEV)
        ops.window_gather_f32(x, window, stride, first, n, out=buf[1:n + 1])
        assert torch.equal(buf[1:n + 1], ref[first:first + n]) and bool(buf[0].isnan().all()) and bool(buf[-1].isnan().all())
    with pytest.raises(ValueError):
        ops.window_gather_f32(x, window, stride, N - 1, 2)


# ----------------------------------------------------------------------------- epilogue
def _p1_reference(lo, B, H, W, window, stride):
    """fp64 evaluation of the window semantics on the same low-resolution logits."""
    (wh, ww), offs = _grid(H, W, window, stride)
    s = torch.zeros((B, H, W), dtype=torch.float64)
    c = torch.zeros((B, H, W), dtype=torch.float64)
    up = F.interpolate(lo.double().cpu().permute(0, 3, 1, 2), size=(wh, ww), mode="bilinear", align_corners=False)
    p = torch.softmax(up, 1)[:, 1]
    for b in range(B):
        for k, (y0, x0) in enumerate(offs):
            s[b, y0:y0 + wh, x0:x0 + ww] += p[b * len(offs) + k]
            c[b, y0:y0 + wh, x0:x0 + ww] += 1
    return (s / c).numpy()


# (B, H, W, window, stride): stride == window, a snapped last window, s = w/4 (5 windows per axis over a pixel),
# W % 4 != 0, a scene smaller than the window on one axis
_EPI = [(2, 64, 96, (32, 32), (32, 32)), (1, 70, 90, (32, 32), (24, 24)), (1, 80, 80, (32, 32), (8, 8)),
        (2, 45, 61, (24, 20), (18, 15)), (2, 20, 75, (32, 32), (16, 16))]


@pytest.mark.parametrize("case", range(len(_EPI)))
@pytest.mark.parametrize("ldt", [torch.int64, torch.uint8])
def test_epilogue_against_fp64_semantics(case, ldt):
    B, H, W, window, stride = _EPI[case]
    (wh, ww), offs = _grid(H, W, window, stride)
    g = torch.Generator().manual_seed(case)
    lo = (torch.randn((B * len(offs), (wh + 3) // 4, (ww + 3) // 4, 2), generator=g) * 1.5).to(DEV)
    y = _labels(B, H, W, case, ldt)
    p1 = _p1_reference(lo, B, H, W, window, stride)
    for thr in (0.2, 0.5, 0.7):
        cm, pred, conf = ops.predict_window_epilogue(lo, H, W, window, stride, y, threshold=thr)
        pn = pred.cpu().numpy()
        bad = (pn != (p1 > thr)) & (np.abs(p1 - thr) > 1e-5)
        assert not bad.any(), f"thr {thr}: {int(bad.sum())} decisions away from the threshold differ"
        d = np.abs(conf.cpu().numpy().astype(int) - (p1 * 255).astype(int))
        at_edge = np.abs(p1 * 255 - np.round(p1 * 255)) <= 255 * 1e-5
        assert d.max() <= 1 and not ((d == 1) & ~at_edge).any()
        assert cm[:4].cpu().tolist() == _counts(y, pred).tolist()
    # without labels, and into given batch slices
    pred_s = torch.full((B + 1, H, W), 7, dtype=torch.uint8, device=DEV)
    conf_s = torch.full((B + 1, H, W), 7, dtype=torch.uint8, device=DEV)
    cm0, _, _ = ops.predict_window_epilogue(lo, H, W, window, stride, None, threshold=0.7, pred=pred_s[1:], conf=conf_s[1:])
    assert cm0 is None
    assert torch.equal(pred_s[1:], pred) and torch.equal(conf_s[1:], conf) and int(pred_s[0].min()) == int(conf_s[0].max()) == 7
    report("window_epilogue", case=case, windows=lo.shape[0], conf_max_dev=float(np.abs(conf.cpu().numpy() / 255.0 - p1).max()))


def test_epilogue_rejects_bad_shapes():
    lo = torch.zeros((5, 8, 8, 2), device=DEV)
    with pytest.raises(ValueError):
        ops.predict_window_epilogue(lo, 64, 64, (32, 32), (16, 16))             # 9 windows per scene, 5 given
    with pytest.raises(RuntimeError):
        ops.predict_window_epilogue(torch.zeros((9, 8, 8, 3), device=DEV), 64, 64, (32, 32), (16, 16))     # C != 2
    with pytest.raises(ValueError):
        ops.predict_window_epilogue(lo, 64, 64, (32, 32), (33, 16))             # stride above the window


# ----------------------------------------------------------------------------- predict_mask end to end
def _check_against_composition(model, x, y, window, stride, name):
    from iswm_b200.metrics import StreamMetrics
    from iswm_b200.predict import predict_mask
    m_f, m_r = StreamMetrics(2, device=DEV, shape_metrics=False), StreamMetrics(2, device=DEV, shape_metrics=False)
    pf, cf = predict_mask(model, x, 0.5, y, m_f, window=window, stride=stride)
    pr, cr = predict_mask(model, x, 0.5, y, m_r, fused=False, window=window, stride=stride)
    dis = pf != pr
    report(name, disagree=int(dis.sum()), conf_differ=int((cf != cr).sum()),
           conf_max_dev=int((cf.int() - cr.int()).abs().max()), cm_fused=m_f._cm()[:4].tolist(), cm_ref=m_r._cm()[:4].tolist())
    assert torch.equal(pf, pr) and torch.equal(cf, cr)
    assert torch.equal(m_f._cm(), m_r._cm())
    assert m_f._cm()[:4].tolist() == _counts(y, pf).tolist()
    return pf, cf


@pytest.mark.parametrize("backbone,os_", [("resnet50", 16), ("resnet101", 8)])
@pytest.mark.parametrize("shape,window,stride", [((1, 300, 452), 128, 96), ((2, 257, 450), (128, 160), (100, 120))])
def test_predict_mask_window_against_torch_composition(backbone, os_, shape, window, stride):
    m, _ = build(backbone, os_)
    m.to(DEV).eval()
    B, H, W = shape
    g = torch.Generator(device=DEV).manual_seed(H + W)
    x = torch.randn((B, 3, H, W), device=DEV, generator=g)
    _check_against_composition(m, x, _labels(B, H, W, B, torch.uint8), window, stride, f"window_{backbone}_os{os_}_{B}x{H}x{W}")


def test_predict_mask_window_fp8():
    from iswm_b200.quant import quantize_fp8
    m, _ = build("resnet50", 16)
    m.to(DEV).eval()
    g = torch.Generator(device=DEV).manual_seed(3)
    x = torch.randn((2, 3, 257, 450), device=DEV, generator=g)
    qm = quantize_fp8(m, x[:, :, :128, :160].contiguous())
    _check_against_composition(qm, x, _labels(2, 257, 450, 4, torch.int64), (128, 160), (100, 120), "window_fp8_r50_os16_2x257x450")


@pytest.mark.parametrize("shape", [(2, 96, 128), (1, 90, 118)])
def test_single_window_equals_the_plain_path(shape):
    """A window covering the whole scene is the default single-forward path, bit for bit."""
    from iswm_b200.metrics import StreamMetrics
    from iswm_b200.predict import predict_mask
    m, _ = build("resnet50", 16)
    m.to(DEV).eval()
    B, H, W = shape
    g = torch.Generator(device=DEV).manual_seed(W)
    x = torch.randn((B, 3, H, W), device=DEV, generator=g)
    y = _labels(B, H, W, 1, torch.int64)
    m0, m1, m2 = (StreamMetrics(2, device=DEV, shape_metrics=False) for _ in range(3))
    p0, c0 = predict_mask(m, x, 0.5, y, m0)
    p1, c1 = predict_mask(m, x, 0.5, y, m1, window=(H, W))
    p2, c2 = predict_mask(m, x, 0.5, y, m2, window=512, stride=16)
    for p, c, mm in ((p1, c1, m1), (p2, c2, m2)):
        assert torch.equal(p0, p) and torch.equal(c0, c) and torch.equal(m0._cm(), mm._cm())


def test_chunked_equals_unchunked(monkeypatch):
    """Window lists larger than the per-forward bound run in chunks (windows of different scenes sharing a forward):
    the same maps and counts, bit for bit, as one forward."""
    from iswm_b200 import predict
    from iswm_b200.metrics import StreamMetrics
    m, _ = build("resnet50", 16)
    m.to(DEV).eval()
    g = torch.Generator(device=DEV).manual_seed(5)
    x = torch.randn((2, 3, 257, 450), device=DEV, generator=g)
    y = _labels(2, 257, 450, 6, torch.uint8)
    m0, m1 = StreamMetrics(2, device=DEV, shape_metrics=False), StreamMetrics(2, device=DEV, shape_metrics=False)
    launches = []
    real = m.forward_lowres
    monkeypatch.setattr(m, "forward_lowres", lambda xv: (launches.append(tuple(xv.shape)), real(xv))[1])
    p0, c0 = predict.predict_mask(m, x, 0.5, y, m0, window=(128, 160), stride=(100, 120))
    assert launches == [(24, 3, 128, 160)], launches
    launches.clear()
    monkeypatch.setattr(predict, "MAX_FORWARD_PIXELS", 5 * 128 * 160 + 7)       # 12 windows per scene: chunks of 5
    p1, c1 = predict.predict_mask(m, x, 0.5, y, m1, window=(128, 160), stride=(100, 120))
    assert launches == [(5, 3, 128, 160)] * 4 + [(4, 3, 128, 160)], launches
    assert torch.equal(p0, p1) and torch.equal(c0, c1) and torch.equal(m0._cm(), m1._cm())


def test_scene_above_the_forward_bound():
    """One 6144^2 scene (37.7 M px, above MAX_FORWARD_PIXELS as a single forward) in windows of 512 / stride 384."""
    from iswm_b200 import predict
    m, _ = build("resnet50", 16)
    m.to(DEV).eval()
    assert 6144 * 6144 > predict.MAX_FORWARD_PIXELS
    g = torch.Generator(device=DEV).manual_seed(6144)
    x = torch.randn((1, 3, 6144, 6144), device=DEV, generator=g)
    _check_against_composition(m, x, _labels(1, 6144, 6144, 7, torch.uint8), 512, 384, "window_r50_os16_1x6144x6144")


def test_predict_mask_window_rejects_bad_requests():
    from iswm_b200.network import modeling
    from iswm_b200.predict import predict_mask
    m, _ = build("resnet50", 16)
    m.to(DEV).eval()
    x = torch.zeros((1, 3, 64, 64), device=DEV)
    for kw in (dict(window=15), dict(window=(32, 8)), dict(window=32, stride=0), dict(window=32, stride=33),
               dict(window=32, scales=(0.75, 1.0)), dict(window=32, flip=True), dict(stride=16)):
        with pytest.raises(ValueError):
            predict_mask(m, x, **kw)
    m3 = modeling.deeplabv3plus_resnet50(num_classes=3, output_stride=16, pretrained_backbone=False).to(DEV).eval()
    with pytest.raises(ValueError):
        predict_mask(m3, x, window=32)
    with pytest.raises(RuntimeError):
        predict_mask(m, x.cpu(), window=32)
