"""Case generators for the detector post-processing edge tests: tests/test_gpu_detect_edges.py (CUDA kernels) and
tests/test_detect_edges_hostemu.py (the same cases through the host emulation of the kernel bodies).

Every generator returns, beside its inputs, what is needed to check in numpy that the edge it is for is actually hit:
the tests assert that coverage instead of trusting the construction."""
import numpy as np

from oracle import detect as odet

NMS_NMAX = 3049                 # the largest frame dd_nms accepts: dd_nms_smem_bytes(3049) fits 227 KB of shared memory
BIG_COUNTS = (0, 1, 1024, 1025, 1056, 1537, 2048, 3049, 5000)     # 5000 > nmax: the kernel clamps it to nmax
BIG_THRS = (0.6, 0.3, 0.9)
FRAC_THRS = (0.6, 0.0, -0.1, 1.0)       # 0.0 is the boundary of "disjoint never suppresses", < 0 turns it off
EXACT_THRS = (0.3, 0.5, 0.6, 0.75)
F32 = np.float32


# ----------------------------------------------------------------------------------------------- NMS
def overlap(bi, bj):
    """fl(inter(i, j) / area(j)) evaluated like oracle.detect.non_max_suppression (f64, +1 px); broadcasts."""
    bi, bj = np.asarray(bi, float), np.asarray(bj, float)
    x2i, y2i = bi[..., 2] + bi[..., 0], bi[..., 3] + bi[..., 1]
    x2j, y2j = bj[..., 2] + bj[..., 0], bj[..., 3] + bj[..., 1]
    w = np.maximum(0, np.minimum(x2i, x2j) - np.maximum(bi[..., 0], bj[..., 0]) + 1)
    h = np.maximum(0, np.minimum(y2i, y2j) - np.maximum(bi[..., 1], bj[..., 1]) + 1)
    area = (x2j - bj[..., 0] + 1) * (y2j - bj[..., 1] + 1)
    with np.errstate(divide="ignore", invalid="ignore"):
        return (w * h) / area


def nms_batches(boxes, scores, thr, batch=32):
    """The lazy batches of dd_nms_frame replayed in numpy: the next `batch` candidates (in rank order) not yet removed
    are gathered 32 ranks at a time from a cursor; when a batch fills inside such a window the cursor resumes after
    its last member.  Returns (keep list, number of such resumes)."""
    order = np.argsort(scores, kind="stable")[::-1]
    b = np.asarray(boxes, float)[order]
    n = len(b)
    removed = np.zeros(n, bool)
    keep, cursor, resumes = [], 0, 0
    while True:
        sel = []
        while len(sel) < batch and cursor < n:
            win = np.arange(cursor, min(cursor + 32, n))
            alive = win[~removed[win]]
            if len(sel) + len(alive) > batch:
                alive = alive[:batch - len(sel)]
                cursor = int(alive[-1]) + 1
                resumes += 1
            else:
                cursor += 32
            sel.extend(int(r) for r in alive)
        if not sel:
            return keep, resumes
        for r in sel:
            if removed[r]:
                continue
            keep.append(int(order[r]))
            removed[r + 1:] |= overlap(b[r], b[r + 1:]) > thr


def clustered_boxes(rng, n, integer=True, size_scale=1.0):
    """n tlwh boxes around n/6 cluster centres on a canvas that grows with n (many suppressions, many survivors)."""
    side = 25.0 * np.sqrt(max(n, 1)) + 200
    k = max(1, n // 6)
    cx, cy = rng.uniform(0, side, k), rng.uniform(0, side * 0.75, k)
    p = rng.integers(0, k, n)
    b = np.stack([cx[p] + rng.normal(0, 7, n), cy[p] + rng.normal(0, 7, n),
                  rng.uniform(10, 60, n) * size_scale, rng.uniform(20, 120, n) * size_scale], 1)
    return np.floor(b) if integer else b


def unique_scores(rng, n):
    """Distinct f32 scores in [0.25, 1) in random order."""
    return (0.25 + 0.75 * (rng.permutation(n) + rng.uniform(0.1, 0.9, n)) / max(n, 1)).astype(F32)


def big_batch(rng):
    """One [len(BIG_COUNTS), NMS_NMAX] batch of clustered integer frames; the last count exceeds nmax."""
    B = len(BIG_COUNTS)
    boxes = np.zeros((B, NMS_NMAX, 4))
    scores = np.zeros((B, NMS_NMAX), F32)
    for f, c in enumerate(BIG_COUNTS):
        n = min(c, NMS_NMAX)
        boxes[f, :n] = clustered_boxes(rng, n)
        scores[f, :n] = unique_scores(rng, n)
    return boxes, scores, np.array(BIG_COUNTS, np.int32)


def fractional_frames(rng):
    """Frames that leave the integer fast path of the row builder: non-integer boxes (n = 17 .. 2048), an integer frame
    with one fractional box, integer boxes beyond 2^20 and negative ones, nested boxes (overlap exactly 1.0), touching
    boxes (overlap width exactly 0), slivers (overlap width 2^-30) and degenerate boxes (zero / negative area)."""
    frames = {}
    for n in (17, 100, 1024, 2048):
        frames["frac%d" % n] = (clustered_boxes(rng, n, integer=False), unique_scores(rng, n))
    b = clustered_boxes(rng, 300)
    b[150, 0] += 0.5
    frames["one_frac"] = (b, unique_scores(rng, 300))
    b = clustered_boxes(rng, 400)
    b[:200, :2] += 2 ** 20                        # isint needs |coord| < 2^20 for its int32 disjointness test
    frames["huge"] = (b, unique_scores(rng, 400))
    b = clustered_boxes(rng, 400)
    b[:, :2] -= 3000
    frames["negative"] = (b, unique_scores(rng, 400))
    # hand-made edges on a grid of 200 px cells: per cell a reference box R and one partner P of lower score
    cells = []
    for k in range(96):
        x, y = 200.0 * (k % 12), 200.0 * (k // 12)
        w, h = rng.integers(20, 80), rng.integers(20, 80)
        if k % 4 == 0:            # P nested inside R: inter == area(P), overlap exactly 1.0
            P = (x + 3, y + 4, w - 9, h - 9)
        elif k % 4 == 1:          # P touching R on the right: overlap width exactly 0
            P = (x + w + 1, y, 30, h)
        elif k % 4 == 2:          # P overlapping R by a 2^-30 px sliver
            P = (x + w + 1 - 2.0 ** -30, y + 0.25, 30.5, h)
        else:                     # degenerate P: zero area (w = -1) or negative area (w = -3)
            P = (x + 5, y + 5, -1.0 if k % 8 == 3 else -3.0, h)
        cells += [(x, y, float(w), float(h)), P]
    b = np.array(cells, float)
    s = np.empty(len(b), F32)
    s[0::2] = unique_scores(rng, len(b) // 2) + F32(1.0)
    s[1::2] = unique_scores(rng, len(b) // 2)
    frames["edges"] = (b, s)
    return frames


def exact_geometries(thr, side=40):
    """All (W, H, iw, ih) with sides < `side` and fl(iw * ih / (W * H)) == thr: an integer box J of W x H pixels
    (+1 convention) overlapped by iw x ih pixels."""
    v = np.arange(1, side)
    W, H, iw, ih = (a.ravel() for a in np.meshgrid(v, v, v, v, indexing="ij"))
    ok = (iw <= W) & (ih <= H) & ((iw * ih).astype(float) / (W * H).astype(float) == thr)
    return np.stack([W[ok], H[ok], iw[ok], ih[ok]], 1)


def _pair(X, Y, W, H, iw, ih, ax, ay):
    """J = W x H pixels at (X, Y); I covers J's bottom-right iw x ih pixels and extends ax, ay beyond it."""
    return (X + W - iw, Y + H - ih, iw - 1 + ax, ih - 1 + ay), (X, Y, W - 1, H - 1)


def ulps(r, thr):
    """Signed distance of f64 overlap values r from thr in units in the last place (r, thr > 0)."""
    return np.asarray(r, np.float64).view(np.int64) - np.float64(thr).view(np.int64)


def near_fractional_pair(rng, thr, ox, oy, lo, hi):
    """A fractional pair (I, J) at cell offset (ox, oy) whose f64 overlap is lo..hi ulp from thr: within the 2^-40
    guard band of dd_nms_suppresses, where the division decides.  Found by search: J random, I covering the lower part
    of J (fractional height ih) and overlapping it by about thr * area / ih, then walked one ulp of its left edge at a
    time (the fractional ih makes the rounded overlaps land on every ulp near thr, also for thr = 0.5)."""
    for attempt in range(100):
        m = 256
        X, Y = ox + rng.uniform(0, 50, m), oy + rng.uniform(1, 50, m)
        W, H = rng.uniform(8, 40, m), rng.uniform(8, 40, m)
        J = np.stack([X, Y, W, H], 1)
        x2j, y2j = W + X, H + Y
        yi = Y + rng.uniform(0, 0.3, m) * H
        x1 = x2j + 1 - thr * ((x2j - X + 1) * (y2j - Y + 1)) / (y2j - yi + 1)
        for step in range(-4, 5):
            xi = x1.copy()
            for _ in range(abs(step)):
                xi = np.nextafter(xi, np.inf if step > 0 else -np.inf)
            I = np.stack([xi, yi, x2j + 5 - xi, y2j + 2 - yi], 1)
            d = ulps(overlap(I, J), thr)
            hit = np.nonzero((d >= lo) & (d <= hi))[0]
            if len(hit):
                return tuple(I[hit[0]]), tuple(J[hit[0]])
    raise AssertionError("no pair within %d..%d ulp of %r" % (lo, hi, thr))


def exact_frames(rng, thr):
    """Two frames of non-interacting pairs (I picked first, J tested against thr): frame 0 <= 1024 boxes (the register
    path) with integer pairs exactly on thr and their +-1 px neighbours; frame 1 > 1024 boxes with more exact pairs and
    fractional pairs within 2 ulp of thr.  Returns (boxes [2,nmax,4], scores, counts, pairs per frame [(I, J)])."""
    geo = exact_geometries(thr)
    geo = geo[rng.permutation(len(geo))]
    frames = []
    for f, (n_exact, n_near) in enumerate(((256, 0), (600, 240))):
        g = geo[f * 256:f * 256 + n_exact]
        pairs = []
        for W, H, iw, ih in g:
            ax, ay = (int(v) for v in rng.integers(0, 5, 2))
            pairs.append(_pair(0, 0, int(W), int(H), int(iw), int(ih), ax, ay))
            iw2 = int(iw) + (1 if (iw < W and rng.random() < 0.5) or iw == 1 else -1)       # +-1 px neighbour
            pairs.append(_pair(0, 0, int(W), int(H), iw2, int(ih), ax, ay))

        def cell(k):                                    # one pair per 100 px cell (a pair spans < 96 px)
            return 100.0 * (k % 48), 100.0 * (k // 48)
        boxes = []
        for k, (I, J) in enumerate(pairs):
            ox, oy = cell(k)
            boxes += [(I[0] + ox, I[1] + oy, I[2], I[3]), (J[0] + ox, J[1] + oy, J[2], J[3])]
        for k in range(len(pairs), len(pairs) + n_near):   # fractional pairs are built in place: an offset would round
            lo, hi = ((-2, -1), (0, 0), (1, 2))[k % 3]
            I, J = near_fractional_pair(rng, thr, *cell(k), lo, hi)
            boxes += [I, J]
        pairs = [(boxes[2 * k], boxes[2 * k + 1]) for k in range(len(boxes) // 2)]
        s = rng.permutation(len(pairs)).astype(np.float64)
        scores = np.stack([2 * s + 1, 2 * s], 1).ravel() / (2 * len(pairs))
        frames.append((np.array(boxes, float), (0.25 + 0.75 * scores).astype(F32), pairs))
    nmax = max(len(b) for b, _, _ in frames)
    B = np.zeros((2, nmax, 4))
    S = np.zeros((2, nmax), F32)
    for f, (b, s, _) in enumerate(frames):
        B[f, :len(b)], S[f, :len(b)] = b, s
    return B, S, np.array([len(b) for b, _, _ in frames], np.int32), [p for _, _, p in frames]


def pair_overlaps(pairs):
    """overlap(I, J) of every pair, in numpy (the exactness check of exact_frames)."""
    I = np.array([p[0] for p in pairs], float)
    J = np.array([p[1] for p in pairs], float)
    return overlap(I, J)


TIE_SIZES = (17, 40, 300, 1100, 1500)


def tied_frames(rng):
    """Clustered integer frames whose scores take only 8 distinct values (ties at n > 16 and n > 1024)."""
    levels = np.array([0.3, 0.4, 0.45, 0.5, 0.6, 0.7, 0.8, 0.9], F32)
    return [(clustered_boxes(rng, n), levels[rng.integers(0, 8, n)]) for n in TIE_SIZES]


# ----------------------------------------------------------------------------------------------- YOLOv5 rows
YOLO_NC = 80
YOLO_NAMES = ["c%02d" % i for i in range(YOLO_NC)]
YOLO_WANTED = [YOLO_NAMES[i] for i in range(YOLO_NC) if i % 3 != 2]         # class 2, 5, 8, ... unwanted
YOLO_MASK = np.array([0 if i % 3 == 2 else 1 for i in range(YOLO_NC)], np.uint8)


def _row(rng, obj):
    r = np.zeros(5 + YOLO_NC, F32)
    r[0:2] = rng.uniform(0.1, 0.9, 2)
    r[2:4] = rng.uniform(0.02, 0.2, 2)
    r[4] = obj
    r[5:] = rng.uniform(0.0, 0.3, YOLO_NC)
    return r


def yolo_edge_head(rng, na=640, thr=0.25):
    """f32 head [na, 85] for score threshold `thr` = 0.25: background rows plus rows with obj * cls exactly on the
    threshold and one f32 ulp either side, rows whose top class is tied (raw values, or equal products of different
    raw values) between a wanted and an unwanted class in both orders, and rows with NaN objectness or a NaN class
    score (np.argmax returns the first NaN, whose score fails the threshold).  Returns (head, kinds {name: rows})."""
    assert thr == 0.25
    h = np.stack([_row(rng, rng.uniform(0.0, 0.4)) for _ in range(na)])
    kinds = {k: [] for k in ("exact", "below", "above", "tie", "nan")}
    slots = iter(rng.permutation(na))

    def put(kind, r):
        i = next(slots)
        h[i] = r
        kinds[kind].append(int(i))

    half = F32(0.5)
    for k in range(24):
        c = int(rng.choice(np.nonzero(YOLO_MASK)[0]))
        r = _row(rng, half); r[5 + c] = half; put("exact", r)                          # 0.5 * 0.5 == 0.25
        r = _row(rng, F32(0.25)); r[5 + c] = F32(1.0); put("exact", r)                 # 0.25 * 1 == 0.25
        r = _row(rng, half); r[5 + c] = np.nextafter(half, F32(0)); put("below", r)    # one ulp below 0.25
        r = _row(rng, half); r[5 + c] = np.nextafter(half, F32(1)); put("above", r)    # one ulp above 0.25
    # product ties: two different raw class values whose f32 products with obj round to the same value
    obj = F32(0.7)
    a = F32(0.8)
    while obj * np.nextafter(a, F32(1)) != obj * a:
        a = np.nextafter(a, F32(1))
    b = np.nextafter(a, F32(1))
    for k in range(24):
        wc = 3 * int(rng.integers(0, YOLO_NC // 3))            # wanted class
        uc = wc + 2                                            # unwanted class (i % 3 == 2)
        first, second = (wc, uc) if k % 2 == 0 else (uc, wc)
        r = _row(rng, F32(0.9)); r[5 + first] = r[5 + second] = F32(0.6); put("tie", r)
        r = _row(rng, obj); r[5 + first], r[5 + second] = (a, b) if k % 4 < 2 else (b, a); put("tie", r)
    for k in range(12):
        r = _row(rng, F32(np.nan) if k % 3 == 0 else F32(0.9))
        r[5 + 3] = F32(0.9)                                    # a passing wanted class ...
        if k % 3 == 1:
            r[5 + 40] = F32(np.nan)                            # ... and a NaN class after it
        elif k % 3 == 2:
            r[5 + 0] = F32(np.nan)                             # ... and a NaN class before it
        put("nan", r)
    return h, kinds


def yolo_products(head):
    """obj * cls in f32, like the decode (rows x classes)."""
    return head[:, 5:] * head[:, 4:5]


def yolo_tie_rows(head, thr, rows=None):
    """Rows whose top product is reached by two or more classes and passes thr (NaN-free rows only)."""
    p = yolo_products(head)
    ok = ~np.isnan(p).any(axis=1)
    m = np.where(ok[:, None], p, 0).max(axis=1)
    ok = ok & (m >= F32(thr)) & ((p == m[:, None]).sum(axis=1) >= 2)
    idx = np.nonzero(ok)[0]
    return idx if rows is None else np.intersect1d(idx, rows)


def yolo_reference(head, thr, frame=(640, 480)):
    """oracle decode + box filter for one frame -> (int boxes f64, score, cls, anchor)."""
    tlwh, cls, score, anchor = odet.yolo_decode(head, frame[0], frame[1], YOLO_NAMES, YOLO_WANTED, thr)
    ib, kept = odet.box_filter(list(tlwh), frame[0], frame[1])
    return ib.astype(float).reshape(-1, 4), score[kept], cls[kept], anchor[kept]


def yolo_u8_edge_head(rng, na=2000):
    """u8 head [na, 85] for scale = 2^-8, zero point 0, threshold 0.25 (products q_cls * q_obj / 2^16 are exact in f32):
    rows with q_cls * q_obj == 16384 (128 * 128, exactly on the threshold), 16383 (129 * 127, just below) and 16385
    (145 * 113, just above); 256 levels over 80 classes make tied top classes common.  Returns (q, kinds)."""
    q = rng.integers(0, 200, (na, 5 + YOLO_NC)).astype(np.uint8)
    q[:, 4] = rng.integers(0, 256, na)
    kinds = {"exact": [], "below": [], "above": []}
    rows = rng.permutation(na)[:60]
    for k, i in enumerate(rows):
        c = int(rng.choice(np.nonzero(YOLO_MASK)[0]))
        q[i, 5:] = rng.integers(0, 40, YOLO_NC)
        kind, (qc, qo) = (("exact", (128, 128)), ("below", (129, 127)), ("above", (145, 113)))[k % 3]
        q[i, 5 + c], q[i, 4] = qc, qo
        kinds[kind].append(int(i))
    return q, kinds


def u8_scale():
    return F32(2.0 ** -8)


# ----------------------------------------------------------------------------------------------- Keras YOLOv3
Y3_NAMES = ["person", "bicycle", "car", "dog"]
Y3_WANTED = ["person", "bicycle", "car"]
Y3_ANCHORS = [[116, 90, 156, 198, 373, 326], [30, 61, 62, 45, 59, 119], [10, 13, 16, 30, 33, 23]]
Y3_NET = 64


def _sig(x):
    return odet._sigmoid_f32(np.asarray(x, F32))


def yolo3_edge_maps(rng):
    """Raw output maps (grids 2, 4, 8 for a 64 x 64 input, 4 classes) with ~30 confident, overlapping boxes in the
    middle of the finest grid, and a score threshold equal to one box's class-1 probability sigmoid(obj) *
    sigmoid(cls): that probability sits exactly on the threshold (zeroed by the `>` of decode_netout) while its class 0
    is well above it; one more box has only that probability.  Returns (maps, thr, (box index, class) on thr)."""
    nc = len(Y3_NAMES)
    maps = []
    for g in (Y3_NET // 32, Y3_NET // 16, Y3_NET // 8):
        o = np.empty((g, g, 3, 5 + nc), F32)
        o[..., 0:2] = rng.normal(0, 1, (g, g, 3, 2))
        o[..., 2:4] = rng.uniform(-0.5, 0.5, (g, g, 3, 2))
        o[..., 4] = -9.0
        o[..., 5:] = -6.0
        maps.append(o)
    o = maps[2]
    cells = [(y, x, b) for y in range(2, 6) for x in range(2, 6) for b in range(3)]
    hot = [cells[i] for i in rng.permutation(len(cells))[:30]]
    obj = F32(3.0)
    c1 = F32(-0.8)
    thr = float(_sig(obj) * _sig(c1))
    for k, (y, x, b) in enumerate(hot):
        o[y, x, b, 4] = obj
        o[y, x, b, 5 + int(rng.integers(0, 3))] = rng.uniform(2.0, 4.0)
    y, x, b = hot[0]
    o[y, x, b, 5 + 1] = c1                                  # class 0..2 above thr (its main class) + class 1 on thr
    o[y, x, b, 5 + 0] = F32(3.5)
    y, x, b = hot[1]
    o[y, x, b, 5:] = -6.0
    o[y, x, b, 5 + 1] = c1                                  # only class 1, exactly on thr
    return [m.reshape(m.shape[0], m.shape[1], -1) for m in maps], thr


def yolo3_probabilities(maps):
    """sigmoid(obj) * sigmoid(cls) of every box and class, like decode_netout (f32)."""
    out = []
    for m in maps:
        o = m.reshape(-1, 5 + len(Y3_NAMES)).astype(F32)
        out.append(_sig(o[:, 4])[:, None] * _sig(o[:, 5:]))
    return np.concatenate(out)


def y3_iou(p, q):
    """bbox_iou of tools/yolo.py on (xmin, ymin, xmax, ymax) int boxes (interval overlap without +1)."""
    def ov(a1, a2, b1, b2):
        if b1 < a1:
            return 0 if b2 < a1 else min(a2, b2) - a1
        return 0 if a2 < b1 else min(a2, b2) - b1
    inter = ov(p[0], p[2], q[0], q[2]) * ov(p[1], p[3], q[1], q[3])
    union = (p[2] - p[0]) * (p[3] - p[1]) + (q[2] - q[0]) * (q[3] - q[1]) - inter
    return float(inter) / union if union else None


def yolo3_reference(maps, thr, nms_thresh):
    return odet.yolo3_detect(maps, Y3_ANCHORS, Y3_NAMES, Y3_WANTED, thr, 640, 480, Y3_NET, Y3_NET, nms_thresh)


def yolo3_exact_iou(maps, thr):
    """An nms_thresh equal to the IoU of a pair of returned boxes at which the reference's `>=` decides the output:
    its result differs from the one at the next larger double.  The pairs are read back from the reference's output
    without suppression (boxes come back transposed: x = ymin, y = xmin)."""
    b, _, _ = yolo3_reference(maps, thr, 2.0)
    boxes = [(y, x, y + h, x + w) for x, y, w, h in b.tolist()]
    vals = sorted({v for i in range(len(boxes)) for j in range(i + 1, len(boxes))
                   for v in [y3_iou(boxes[i], boxes[j])] if v is not None and 0.2 < v < 0.9})
    for v in vals:
        lo, hi = yolo3_reference(maps, thr, v), yolo3_reference(maps, thr, float(np.nextafter(v, 1.0)))
        if len(lo[0]) != len(hi[0]):
            return v
    raise AssertionError("no pair of boxes whose IoU decides the output")


# ----------------------------------------------------------------------------------------------- coverage, in numpy
def fractional_coverage(frames):
    """Which edges of fractional_frames are present (every value must be True)."""
    def nonint(b):
        x2, y2 = b[:, 2] + b[:, 0], b[:, 3] + b[:, 1]
        return ((b[:, :2] != np.floor(b[:, :2])).any(axis=1) | (x2 != np.floor(x2)) | (y2 != np.floor(y2)))
    b = frames["edges"][0]
    R, P = b[0::2], b[1::2]
    ov = overlap(R, P)
    iw = np.minimum(R[:, 2] + R[:, 0], P[:, 2] + P[:, 0]) - np.maximum(R[:, 0], P[:, 0]) + 1
    hb, nb = frames["huge"][0], frames["negative"][0]
    return dict(
        frac_big=len(frames["frac2048"][0]) > 1024 and nonint(frames["frac2048"][0]).all(),
        one_frac=int(nonint(frames["one_frac"][0]).sum()) == 1,
        huge=(np.abs(hb[:, :2]) >= 2 ** 20).any() and not nonint(hb).any(),
        negative=(nb[:, :2] < 0).all() and not nonint(nb).any(),
        nested=int((ov == 1.0).sum()) >= 20,
        touching=int((iw == 0).sum()) >= 20,
        sliver=int(((iw > 0) & (iw < 1e-8)).sum()) >= 20,
        degenerate=int(((P[:, 2] + P[:, 0]) - P[:, 0] + 1 <= 0).sum()) >= 20)


def exact_coverage(pairs, thr):
    """(pairs exactly on thr, pairs 1-2 ulp below, pairs 1-2 ulp above) over both frames of exact_frames."""
    d = np.concatenate([ulps(pair_overlaps(p), thr) for p in pairs])
    return int((d == 0).sum()), int(((d >= -2) & (d < 0)).sum()), int(((d > 0) & (d <= 2)).sum())


def assert_yolo_coverage(head, kinds, thr, step=None):
    """The rows yolo_edge_head / yolo_u8_edge_head built are what they claim to be: top products exactly on thr and
    one step below / above it (one f32 ulp, or the quantization step of a u8 head)."""
    p = yolo_products(head)
    with np.errstate(invalid="ignore"):
        m = p.max(axis=1)
    t = F32(thr)
    below, above = (np.nextafter(t, F32(0)), np.nextafter(t, F32(1))) if step is None else (t - F32(step), t + F32(step))
    assert len(kinds["exact"]) >= 20 and (m[kinds["exact"]] == t).all()
    assert len(kinds["below"]) >= 20 and (m[kinds["below"]] == below).all()
    assert len(kinds["above"]) >= 20 and (m[kinds["above"]] == above).all()
    assert len(yolo_tie_rows(head, thr, kinds.get("tie"))) >= 20
    if "nan" in kinds:
        assert np.isnan(p[kinds["nan"]]).any(axis=1).all()
