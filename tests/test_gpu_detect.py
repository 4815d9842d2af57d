"""Object boxes on the GPU (b200seg.detect_objects, b200seg.overlay) against cv2 itself, the library the reference's
overlay_predictions (inference.py:48-146) calls: cv2.resize(INTER_NEAREST), cv2.morphologyEx(MORPH_CLOSE),
cv2.connectedComponentsWithStats(connectivity=8) and cv2.addWeighted.  Every comparison is exact: label images, stats rows,
float64 centroids and blended bytes."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

cv2 = pytest.importorskip("cv2")

import b200seg  # noqa: E402
from oracle import unet_oracle as O  # noqa: E402
from util import expand_aliases, f2_meta, f2_sd  # noqa: E402

DEV = torch.device("cuda", 0)


# ------------------------------------------------------------------------------------------ the cv2 recipe
def cv_planes(mask, classes, H, W, close):
    """Per frame, per class: (closed plane, label image, stats, centroids) from cv2."""
    out = []
    for m in mask:
        r = cv2.resize(m, (W, H), interpolation=cv2.INTER_NEAREST)
        planes = []
        for c in classes:
            p = (r == c).astype(np.uint8)
            if close > 1:
                p = cv2.morphologyEx(p, cv2.MORPH_CLOSE, np.ones((close, close), np.uint8))
            n, lab, st, cen = cv2.connectedComponentsWithStats(p, connectivity=8)
            planes.append((p, lab, st, cen))
        out.append(planes)
    return out


def cv_rows(planes, classes, min_area):
    rows = []
    for (p, lab, st, cen), c in zip(planes, classes):
        for l in range(1, st.shape[0]):
            if st[l, 4] >= min_area:
                rows.append(((c, l) + tuple(int(v) for v in st[l, :5]), (float(cen[l, 0]), float(cen[l, 1]))))
    return rows


def check_against_cv2(mask_np, classes, size=None, close=5, min_area=0, max_objects=None):
    """Run detect_objects with labels and compare everything with cv2; returns (detections, cv2 planes)."""
    B, Hm, Wm = mask_np.shape
    W, H = size if size is not None else (Wm, Hm)
    planes = cv_planes(mask_np, classes, H, W, close)
    rows = [cv_rows(p, classes, min_area) for p in planes]
    M = max_objects if max_objects is not None else max(1, max(len(r) for r in rows))
    det = b200seg.detect_objects(torch.from_numpy(mask_np).to(DEV), classes, size=size, close=close, min_area=min_area,
                                 max_objects=M, labels=True)
    lab = det.labels.cpu().numpy()
    cnt = det.count.cpu().numpy()
    st = det.stats.cpu().numpy()
    cen = det.centroid.cpu().numpy()
    for b in range(B):
        for k in range(len(classes)):
            assert np.array_equal(lab[b, k], planes[b][k][1]), (b, classes[k])
        assert cnt[b] == len(rows[b]), (b, cnt[b], len(rows[b]))
        n = min(len(rows[b]), M)
        want_st = np.array([r[0] for r in rows[b][:n]], dtype=np.int32).reshape(n, 7)
        want_cen = np.array([r[1] for r in rows[b][:n]], dtype=np.float64).reshape(n, 2)
        assert np.array_equal(st[b, :n], want_st), b
        assert np.array_equal(cen[b, :n], want_cen), b            # exact float64: same sums, same division
        assert not st[b, n:].any() and not cen[b, n:].any()       # rows past the count are zero
    return det, planes


# ------------------------------------------------------------------------------------------ 1. resize + close
@pytest.mark.parametrize("hm,wm,h,w", [(128, 256, 540, 960), (256, 512, 128, 200), (64, 96, 64, 96), (37, 53, 101, 77),
                                       (1, 40, 1, 97), (40, 1, 97, 1), (5, 7, 1, 33), (9, 3, 40, 1)])
@pytest.mark.parametrize("close", [1, 3, 5, 7])
def test_resize_and_close_match_cv2(hm, wm, h, w, close):
    rng = np.random.default_rng(hm * 1000 + wm + close)
    # blobs plus salt: the close both fills holes and bridges gaps
    m = rng.integers(0, 4, (2, hm, wm), dtype=np.uint8)
    m[rng.random((2, hm, wm)) < 0.6] = 0
    classes = [1, 2, 3]
    det = b200seg.detect_objects(torch.from_numpy(m).to(DEV), classes, size=(w, h), close=close, labels=True)
    lab = det.labels.cpu().numpy()
    planes = cv_planes(m, classes, h, w, close)
    for b in range(2):
        for k in range(3):
            assert np.array_equal(lab[b, k] > 0, planes[b][k][0] > 0), (b, k)


def test_close_of_the_largest_element_and_a_frame_border():
    """k = 15 on a plane smaller than the element in one direction; foreground touching every border."""
    rng = np.random.default_rng(3)
    m = (rng.random((1, 11, 70)) < 0.3).astype(np.uint8)
    m[0, 0, :] = 1
    m[0, :, -1] = 1
    check_against_cv2(m, [1], close=15)
    check_against_cv2(m, [0, 1], size=(141, 23), close=9)


# ------------------------------------------------------------------------------------------ 2. labels and stats
def _spiral(n):
    """A one-pixel path winding inward with one-pixel gaps: one component whose blocks chain over the whole plane."""
    p = np.zeros((n, n), np.uint8)
    y, x, d = 0, 0, 0
    dirs = [(0, 1), (1, 0), (0, -1), (-1, 0)]
    p[0, 0] = 1
    inside = lambda yy, xx: 0 <= yy < n and 0 <= xx < n
    while True:
        for _ in range(2):                        # go on, or turn once
            dy, dx = dirs[d]
            ny, nx = y + dy, x + dx
            if inside(ny, nx) and not p[ny, nx] and not (inside(ny + dy, nx + dx) and p[ny + dy, nx + dx]):
                y, x = ny, nx
                p[y, x] = 1
                break
            d = (d + 1) % 4
        else:
            return p


def _diagonals(h, w):
    p = np.zeros((h, w), np.uint8)
    for c in range(-h, w, 7):                     # one-pixel lines, connected only through diagonal neighbours
        for y in range(h):
            if 0 <= y + c < w:
                p[y, y + c] = 1
    for c in range(3, w + h, 11):
        for y in range(h):
            if 0 <= c - y < w:
                p[y, c - y] = 1
    return p


@pytest.mark.parametrize("name", ["sparse", "sparse_odd", "dense", "checker", "block_checker", "diagonals", "spiral", "full",
                                  "empty", "isolated_pixels"])
def test_labels_stats_and_centroids_match_cv2(name):
    rng = np.random.default_rng(len(name))
    if name == "sparse":
        p = (rng.random((200, 300)) < 0.08).astype(np.uint8)              # thousands of components
    elif name == "sparse_odd":
        p = (rng.random((101, 77)) < 0.15).astype(np.uint8)
    elif name == "dense":
        p = (rng.random((241, 163)) < 0.45).astype(np.uint8)              # near percolation: long, branching unions
    elif name == "checker":
        yy, xx = np.mgrid[:63, :97]
        p = ((yy + xx) % 2).astype(np.uint8)
    elif name == "block_checker":
        yy, xx = np.mgrid[:65, :99]
        p = ((yy // 2 + xx // 2) % 2).astype(np.uint8)                    # 2x2 blocks touching only at corners
    elif name == "diagonals":
        p = _diagonals(121, 143)
    elif name == "spiral":
        p = _spiral(201)
    elif name == "full":
        p = np.ones((257, 511), np.uint8)                                 # one component, every lane on one root
    elif name == "empty":
        p = np.zeros((33, 45), np.uint8)
    else:
        p = np.zeros((99, 131), np.uint8)
        p[::2, ::2] = 1                                                   # one component per block
    m = np.stack([p * 3, (1 - p) * 3]).astype(np.uint8)                 # the plane and its complement
    det, planes = check_against_cv2(m, [3], close=1)
    if name == "full":
        assert det.count.cpu().tolist() == [1, 0]
    if name == "empty":
        assert det.count.cpu().tolist() == [0, 1]


def test_many_planes_in_one_call():
    """16 classes, odd frame, 3 frames: every plane labelled independently, rows in (class position, label) order."""
    rng = np.random.default_rng(16)
    m = rng.integers(0, 20, (3, 67, 91), dtype=np.uint8)
    classes = [7, 0, 15, 3, 19, 1, 2, 4, 5, 6, 8, 9, 10, 11, 12, 13]
    check_against_cv2(m, classes, size=(183, 135), close=3)


# ------------------------------------------------------------------------------------------ 3. rows
def test_min_area_row_order_and_capacity():
    rng = np.random.default_rng(21)
    m = rng.integers(0, 4, (2, 96, 128), dtype=np.uint8)
    m[rng.random(m.shape) < 0.5] = 0
    classes = [2, 1]
    det, planes = check_against_cv2(m, classes, size=(200, 150), close=3, min_area=6)
    full = [cv_rows(p, classes, 6) for p in planes]
    assert all(len(r) > 20 for r in full)
    assert [r[0][0] for r in full[0]] == sorted([r[0][0] for r in full[0]], key=classes.index)   # class position order
    # capacity: count keeps counting, the rows are the first max_objects in order, nothing else is written
    det, _ = check_against_cv2(m, classes, size=(200, 150), close=3, min_area=6, max_objects=9)
    assert all(int(c) > 9 for c in det.count.cpu())
    rows = det.to_list()
    assert [len(r) for r in rows] == [9, 9]
    assert rows[0] == [r[0] + r[1] for r in full[0][:9]]


# ------------------------------------------------------------------------------------------ 4. the real flow
def test_f2_network_masks_give_the_cv2_objects_and_contour_boxes():
    """predict_mask of the trained F2 network on road-scene frames, then detect_objects at the reference's 960x540 frame
    size, classes 1..9: equal to cv2 run on the same mask, and every cv2.boundingRect of the closed plane's external
    contours (the reference's "contours, boxes") is the box of a returned component."""
    sd, meta = f2_sd(), f2_meta()["full"]
    b, h, w = meta["shape"]
    x, _ = O.road_scene_batch(b, h, w, seed=meta["seed"])
    m = b200seg.MobileNetV2UNet(output_channels=10)
    full = dict(m.state_dict())
    full.update(expand_aliases(sd))
    m.load_state_dict(full, strict=True)
    m = m.to(DEV).bfloat16().eval()
    with torch.no_grad():
        mask = m.predict_mask(x.to(DEV).bfloat16())
    classes = list(range(1, 10))
    mnp = mask.cpu().numpy()
    det, planes = check_against_cv2(mnp, classes, size=(960, 540), close=5, min_area=0)
    assert int(det.count.sum()) >= 6                       # the six rectangles per frame, at least
    rows = det.to_list()
    for bi in range(b):
        boxes = {(r[0], r[2], r[3], r[4], r[5]) for r in rows[bi]}
        for k, c in enumerate(classes):
            contours, _ = cv2.findContours(planes[bi][k][0], cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE)
            for ct in contours:
                assert (c,) + tuple(cv2.boundingRect(ct)) in boxes


# ------------------------------------------------------------------------------------------ 5. capture, determinism
def test_detect_and_overlay_capture_in_a_cuda_graph():
    rng = np.random.default_rng(5)
    def inputs(seed):
        r = np.random.default_rng(seed)
        mk = r.integers(0, 6, (2, 64, 128), dtype=np.uint8)
        mk[r.random(mk.shape) < 0.4] = 0
        fr = r.integers(0, 256, (2, 135, 240, 3), dtype=np.uint8)
        return torch.from_numpy(mk).to(DEV), torch.from_numpy(fr).to(DEV)
    pal = torch.from_numpy(rng.integers(0, 256, (6, 3), dtype=np.uint8)).to(DEV)
    mask, frames = inputs(1)
    kw = dict(size=(240, 135), close=5, min_area=3, max_objects=64, labels=True)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):                                         # warm-up outside the capture
        b200seg.detect_objects(mask, [1, 2, 5], **kw)
        b200seg.overlay(frames, mask, pal, 0.7, 0.3)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        det_g = b200seg.detect_objects(mask, [1, 2, 5], **kw)
        vis_g = b200seg.overlay(frames, mask, pal, 0.7, 0.3)
    m2, f2 = inputs(2)
    mask.copy_(m2)
    frames.copy_(f2)
    g.replay()
    e1 = b200seg.detect_objects(m2, [1, 2, 5], **kw)
    e2 = b200seg.detect_objects(m2, [1, 2, 5], **kw)
    v1 = b200seg.overlay(f2, m2, pal, 0.7, 0.3)
    torch.cuda.synchronize()
    for a, b_ in ((e1, e2), (e1, det_g)):
        assert torch.equal(a._buf, b_._buf) and torch.equal(a.labels, b_.labels)
    assert torch.equal(v1, vis_g)
    assert int(e1.count.sum()) > 10


# ------------------------------------------------------------------------------------------ 6. overlay
@pytest.mark.parametrize("abg", [(0.7, 0.3, 0.0), (0.65, 0.35, 0.0), (0.3, 0.7, 10.0)])
@pytest.mark.parametrize("shape", [(2, 128, 256, 540, 960), (3, 37, 53, 101, 77)])
def test_overlay_matches_cv2_add_weighted(abg, shape):
    a, bt, gm = abg
    B, hm, wm, h, w = shape
    rng = np.random.default_rng(h + w)
    frames = rng.integers(0, 256, (B, h, w, 3), dtype=np.uint8)
    mask = rng.integers(0, 14, (B, hm, wm), dtype=np.uint8)                # values 10..13 have no palette row
    pal = rng.integers(0, 256, (10, 3), dtype=np.uint8)
    got = b200seg.overlay(torch.from_numpy(frames).to(DEV), torch.from_numpy(mask).to(DEV), torch.from_numpy(pal).to(DEV),
                          a, bt, gm).cpu().numpy()
    ext = np.zeros((256, 3), np.uint8)
    ext[:10] = pal
    for b in range(B):
        col = ext[cv2.resize(mask[b], (w, h), interpolation=cv2.INTER_NEAREST)]
        want = cv2.addWeighted(frames[b], a, col, bt, gm)
        assert np.array_equal(got[b], want), (b, int((got[b] != want).sum()))


def test_gpu_argument_errors():
    m = torch.zeros(1, 8, 8, dtype=torch.uint8, device=DEV)
    with pytest.raises(ValueError):
        b200seg.detect_objects(m.float(), [1])
    with pytest.raises(ValueError):
        b200seg.detect_objects(m, [1, 1])
    with pytest.raises(ValueError):
        b200seg.detect_objects(m, [1], close=4)
    with pytest.raises(RuntimeError, match="CUDA"):
        b200seg.detect_objects(m.cpu(), [1])
    with pytest.raises(ValueError):
        b200seg.overlay(torch.zeros(2, 8, 8, 3, dtype=torch.uint8, device=DEV), m, [[0, 0, 0]], 0.5, 0.5)
