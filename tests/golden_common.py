"""Helpers shared by tests/golden/make_golden.py (reference side) and the tests (oracle / CUDA side)."""
import numpy as np

TRACK_KEYS = ("age", "hits", "hit_streak", "time_since_update", "lost_frames")


def pack_tracks(frames_out):
    """list (per frame) of list[dict] -> flat arrays."""
    rows = []
    traj_last, traj_len = [], []
    for f, tracks in enumerate(frames_out):
        for t in tracks:
            rows.append([f, int(t["track_id"][1:]), *np.asarray(t["bbox"], np.float64), float(t["confidence"]),
                         1.0 if t["status"] == "predicted" else 0.0, *[t[k] for k in TRACK_KEYS],
                         float(t["is_lost"]), *np.asarray(t["velocity"], np.float64), float(t["motion_confidence"]),
                         float(t["is_stable_motion"]), float(t["speed"]), float(t["direction"])])
            tr = np.asarray(t["trajectory"], np.float64).reshape(-1, 2)
            traj_len.append(len(tr))
            pad = np.zeros((30, 2)); pad[:len(tr)] = tr
            traj_last.append(pad)
    cols = ["frame", "id", "x1", "y1", "x2", "y2", "confidence", "predicted", *TRACK_KEYS, "is_lost",
            "vx", "vy", "motion_confidence", "is_stable_motion", "speed", "direction"]
    return np.asarray(rows, np.float64).reshape(-1, len(cols)), cols, np.asarray(traj_len), np.asarray(traj_last)



def synth_pred(seed, B, nc, A, frac=0.15, wh=(4, 60), span=600):
    """(B, 4+nc, A) xywh + class scores with clustered boxes so that suppression happens."""
    g = np.random.default_rng(seed)
    nclu = max(1, A // 6)
    centers = g.uniform(20, span, (B, nclu, 2))
    which = g.integers(0, nclu, (B, A))
    xy = np.take_along_axis(centers, which[..., None].repeat(2, -1), 1) + g.normal(0, 3, (B, A, 2))
    whs = g.uniform(*wh, (B, A, 2))
    sc = g.uniform(0, 1, (B, A, nc)) ** 6
    sc *= (g.random((B, A, 1)) < frac * 3)
    return np.concatenate([xy, whs, sc], 2).transpose(0, 2, 1).astype(np.float32)




# ---------------------------------------------------------------------------------------------------------------------
# "same detection set" with a stated exclusion band (north_star: post-NMS boxes within 1e-2 relative of the fp32 reference,
# the same detection set at the same conf / iou thresholds; SURVEY.md H1: borderline items need an explicit band)
# ---------------------------------------------------------------------------------------------------------------------
BAND_LOGIT = 0.12      # class-logit perturbation (uniform +-) the band covers: bf16 storage of the activations moves the logits of
                       # candidates by 0.017 (median) / 0.088 (99 %) / 0.117 (max over 2096 candidates, fp32 vs bf16 oracle)
BAND_BOX = 0.10        # box-coordinate perturbation in pixels (uniform +-): measured 0.005 (median) / 0.03 (99 %) / 0.07 (max)
BAND_TRIALS = 128
BOX_RTOL = 1e-2        # box tolerance, relative to the largest coordinate of the reference row


def _iou_matrix(b):
    x1, y1 = np.maximum(b[:, None, 0], b[None, :, 0]), np.maximum(b[:, None, 1], b[None, :, 1])
    x2, y2 = np.minimum(b[:, None, 2], b[None, :, 2]), np.minimum(b[:, None, 3], b[None, :, 3])
    inter = np.clip(x2 - x1, 0, None) * np.clip(y2 - y1, 0, None)
    area = (b[:, 2] - b[:, 0]) * (b[:, 3] - b[:, 1])
    return inter / (area[:, None] + area[None, :] - inter)


def _logit(p):
    p = np.clip(np.asarray(p, np.float64), 1e-9, 1 - 1e-9)
    return np.log(p / (1 - p))


def _greedy_keep(boxes, scores, cls, alive, iou_thres):
    """Exact greedy NMS (per class) over the candidates with alive[i]; returns the kept mask."""
    keep = np.zeros(len(boxes), bool)
    iou = _iou_matrix(boxes)
    same = cls[:, None] == cls[None, :]
    dead = ~alive
    for i in np.argsort(-scores, kind="stable"):
        if dead[i]:
            continue
        keep[i] = True
        dead |= same[i] & (iou[i] > iou_thres)
    return keep


def detection_set_report(dets, ref, cand, conf, iou_thres, seed=0, frame_hw=None):
    """Compare engine detections ``dets`` (k,6) with the fp32 reference's ``ref`` (n,6), given the candidate list ``cand`` (m,6)
    the reference's NMS saw (every row of ``ref`` is a row of ``cand``; ``cand`` boxes are NOT clipped to the frame -- NMS
    runs before clip_boxes -- while ``dets`` / ``ref`` are: pass ``frame_hw`` so that rows are matched on the clipped boxes).

    Exclusion band: the reference's own NMS is re-run BAND_TRIALS times on its candidates with every class logit moved by
    up to +-BAND_LOGIT and every box coordinate by up to +-BAND_BOX px (seeded) -- the size of change bf16 storage of the
    activations produces.  A candidate is DECIDED if it is kept in every trial or suppressed / below ``conf`` in every trial;
    the engine must keep every decided-kept candidate (box within BOX_RTOL, score within 5e-2) and none of the
    decided-suppressed ones.  Candidates whose fate flips between trials (near-ties of the greedy order, IoUs at the
    threshold, scores at ``conf``) are the band: reported, not judged.
    Returns a dict with counts; ``errors`` lists violations (empty == same detection set outside the band)."""
    cand = np.asarray(cand, np.float64)
    ref = np.asarray(ref, np.float64)
    dets = np.asarray(dets, np.float64)
    m = len(cand)
    g = np.random.default_rng(seed)
    kept_count = np.zeros(m, int)
    lg = _logit(cand[:, 4]) if m else np.zeros(0)
    lconf = float(_logit(conf))
    for _ in range(BAND_TRIALS if m else 0):
        l2 = lg + g.uniform(-BAND_LOGIT, BAND_LOGIT, m)
        b2 = cand[:, :4] + g.uniform(-BAND_BOX, BAND_BOX, (m, 4))
        kept_count += _greedy_keep(b2, l2, cand[:, 5], l2 > lconf, iou_thres)
    always, never = kept_count == BAND_TRIALS, kept_count == 0

    cand_m = cand.copy()                                          # what a candidate looks like in the output: clipped to the frame
    if frame_hw is not None and m:
        cand_m[:, [0, 2]] = cand_m[:, [0, 2]].clip(0, frame_hw[1])
        cand_m[:, [1, 3]] = cand_m[:, [1, 3]].clip(0, frame_hw[0])

    def cand_index(row):
        """index of the reference candidate this row corresponds to (same class, box within BOX_RTOL; boxes clipped to the same
        frame border can coincide, then the closest score decides), or -1"""
        if not m:
            return -1
        e = np.abs(cand_m[:, :4] - row[:4]).max(1) / max(np.abs(row[:4]).max(), 1.0)
        e[cand[:, 5] != row[5]] = np.inf
        if not e.min() < BOX_RTOL:
            return -1
        near = np.nonzero(e <= e.min() + 1e-3)[0]               # coinciding boxes: the closest score decides
        return int(near[np.abs(cand[near, 4] - row[4]).argmin()])

    ref_idx = [cand_index(r) for r in ref]
    assert all(k >= 0 for k in ref_idx), "every reference detection must be one of the reference candidates"
    errors = []
    got = set()
    for d in dets:
        k = cand_index(d)
        if k < 0:
            if _logit(d[4]) > lconf + BAND_LOGIT:
                errors.append(("engine detection matches no reference candidate", d.tolist()))
            continue
        got.add(k)
        if never[k]:
            errors.append(("engine kept a box the reference decidedly suppresses", d.tolist()))
        elif abs(d[4] - cand[k, 4]) > 5e-2:
            errors.append(("score differs by more than 5e-2", d.tolist(), cand[k].tolist()))
    for k in np.nonzero(always)[0]:
        if k not in got:
            errors.append(("decided reference detection missing", cand[k].tolist()))
    n_strict = int(sum(always[k] for k in ref_idx))
    n_matched = int(sum(k in got for k in ref_idx))              # reference rows the engine also reports (band or not), box within BOX_RTOL
    return {"n_ref": len(ref), "n_det": len(dets), "n_ref_strict": n_strict, "n_ref_in_band": len(ref) - n_strict, "n_ref_matched": n_matched,
            "n_det_not_in_ref": int(len(dets) - sum(1 for k in got if k in set(ref_idx))),
            "n_cand": m, "n_cand_in_band": int((~always & ~never).sum()), "errors": errors}


def bytetrack_script(n_frames=90, n_targets=14, seed=5, hw=(512, 640)):
    """Scripted detections for the ByteTrack goldens: targets on straight lines with jitter, per-frame scores that wander across
    the high / low thresholds (0.25 / 0.1), misses (a target undetected for a few frames -> lost -> re-found), crossings
    (overlapping boxes) and clutter.  Returns a list of (n, 6) float32 arrays [x1, y1, x2, y2, conf, cls] per frame."""
    g = np.random.default_rng(seed)
    H, W = hw
    pos = np.stack([g.uniform(40, W - 40, n_targets), g.uniform(40, H - 40, n_targets)], 1)
    vel = g.normal(0, 2.0, (n_targets, 2))
    size = g.uniform(8, 40, (n_targets, 2))
    base = g.uniform(0.2, 0.9, n_targets)
    cls = g.integers(0, 3, n_targets)
    off_until = np.zeros(n_targets, int)
    frames = []
    for f in range(n_frames):
        pos += vel
        for k in range(n_targets):
            for a, lim in ((0, W), (1, H)):
                if pos[k, a] < 20 or pos[k, a] > lim - 20:
                    vel[k, a] = -vel[k, a]
        rows = []
        for k in range(n_targets):
            if f >= off_until[k] and g.random() < 0.04:
                off_until[k] = f + int(g.integers(2, 12))
            if f < off_until[k]:
                continue
            c = pos[k] + g.normal(0, 0.6, 2)
            s = size[k] * (1 + g.normal(0, 0.03, 2))
            conf = float(np.clip(base[k] + g.normal(0, 0.12), 0.02, 0.99))
            rows.append([c[0] - s[0] / 2, c[1] - s[1] / 2, c[0] + s[0] / 2, c[1] + s[1] / 2, conf, cls[k]])
        for _ in range(int(g.integers(0, 4))):
            c = np.array([g.uniform(10, W - 10), g.uniform(10, H - 10)])
            s = g.uniform(6, 30, 2)
            rows.append([c[0] - s[0] / 2, c[1] - s[1] / 2, c[0] + s[0] / 2, c[1] + s[1] / 2, float(g.uniform(0.05, 0.6)), int(g.integers(0, 3))])
        arr = np.asarray(rows, dtype=np.float32).reshape(-1, 6)
        frames.append(arr[g.permutation(len(arr))])
    return frames


def botsort_scene(n_frames=50, seed=9, hw=(256, 320)):
    """Frames + detections for the BoT-SORT goldens: a fixed textured world (sum of random Gaussian spots: plenty of corners for
    goodFeaturesToTrack) seen through a window that shakes a few pixels per frame (global camera motion for the GMC), and the
    scripted detections of bytetrack_script shifted by the same offsets.  Returns (frames [n] of (h, w, 3) uint8, dets [n] of (k, 6))."""
    g = np.random.default_rng(seed)
    h, w = hw
    pad = 40
    world = np.zeros((h + 2 * pad, w + 2 * pad), np.float32)
    yy, xx = np.mgrid[0:world.shape[0], 0:world.shape[1]]
    for _ in range(500):
        cx, cy, s, a = g.uniform(0, world.shape[1]), g.uniform(0, world.shape[0]), g.uniform(1.5, 4.0), g.uniform(20, 90)
        x0, x1, y0, y1 = int(max(cx - 4 * s, 0)), int(min(cx + 4 * s + 1, world.shape[1])), int(max(cy - 4 * s, 0)), int(min(cy + 4 * s + 1, world.shape[0]))
        world[y0:y1, x0:x1] += a * np.exp(-((xx[y0:y1, x0:x1] - cx) ** 2 + (yy[y0:y1, x0:x1] - cy) ** 2) / (2 * s * s))
    world = np.clip(world + 20, 0, 255).astype(np.uint8)
    dets = bytetrack_script(n_frames, 10, seed + 1, hw)
    off = np.zeros(2, int)
    frames, out = [], []
    for f in range(n_frames):
        off = np.clip(off + g.integers(-3, 4, 2), -pad + 2, pad - 2)
        if f in (20, 21, 35):
            off = np.clip(off + g.integers(-12, 13, 2), -pad + 2, pad - 2)          # a camera jolt
        win = world[pad + off[1]:pad + off[1] + h, pad + off[0]:pad + off[0] + w]
        frames.append(np.ascontiguousarray(np.stack([win, win, win], -1)))
        d = dets[f].copy()
        d[:, [0, 2]] -= off[0]
        d[:, [1, 3]] -= off[1]
        out.append(d)
    return frames, out


def motion_frames_scene(n_frames=60, seed=13, hw=(256, 320)):
    """Frames + detections for the frame-driven path of the camera-motion tracker (N1): the textured world of botsort_scene seen
    through a window that drifts a pixel or two per frame and JOLTS by 35-75 px at a few frames (global motion above the detector's
    30 / 50 px thresholds, twice in the same direction on consecutive frames), detections shifted by the same offsets.
    Returns (frames [n] (h, w, 3) uint8, dets [n] list of [x1, y1, x2, y2, conf] python floats)."""
    g = np.random.default_rng(seed)
    h, w = hw
    pad = 220
    world = np.zeros((h + 2 * pad, w + 2 * pad), np.float32)
    yy, xx = np.mgrid[0:world.shape[0], 0:world.shape[1]]
    for _ in range(420):                                             # broad spots: pyramidal LK must follow 60-px displacements
        cx, cy, s, a = g.uniform(0, world.shape[1]), g.uniform(0, world.shape[0]), g.uniform(10.0, 26.0), g.uniform(12, 45)
        x0, x1, y0, y1 = int(max(cx - 4 * s, 0)), int(min(cx + 4 * s + 1, world.shape[1])), int(max(cy - 4 * s, 0)), int(min(cy + 4 * s + 1, world.shape[0]))
        world[y0:y1, x0:x1] += a * np.exp(-((xx[y0:y1, x0:x1] - cx) ** 2 + (yy[y0:y1, x0:x1] - cy) ** 2) / (2 * s * s))
    world = np.clip(world + 20, 0, 255).astype(np.uint8)
    dets = bytetrack_script(n_frames, 8, seed + 1, hw)
    jolts = {12: (38, 0), 24: (58, 10), 25: (61, 8), 26: (40, 5), 40: (-70, -30), 41: (-66, -25), 52: (0, 75)}
    off = np.zeros(2, int)
    frames, out = [], []
    for f in range(n_frames):
        off = off + g.integers(-2, 3, 2)
        if f in jolts:
            off = off + np.array(jolts[f])
        off = np.clip(off, -pad + 2, pad - 2)
        win = world[pad + off[1]:pad + off[1] + h, pad + off[0]:pad + off[0] + w]
        frames.append(np.ascontiguousarray(np.stack([win, win, win], -1)))
        d = dets[f].astype(np.float64).copy()
        d = d[d[:, 4] > 0.2]
        d[:, [0, 2]] -= off[0]
        d[:, [1, 3]] -= off[1]
        out.append([[float(v) for v in r[:5]] for r in d])
    return frames, out


def overlay_scene(n_frames=14, h=240, w=320):
    """Scripted input of the track-overlay test (tests/golden/overlay.npz): per frame (image, tracks, detections, frame_info) with a
    tracked target, a coasting one that blinks, one at the right / bottom edges (captions flip), long trails and fast targets."""
    yy, xx = np.mgrid[0:h, 0:w]
    base = np.stack([(xx * 255 // w), (yy * 255 // h), ((xx + yy) * 255 // (w + h))], axis=-1).astype(np.uint8)
    frames = []
    for f in range(n_frames):
        trail_a = [(40 + 3 * k, 60 + 2 * k) for k in range(f + 1)]
        trail_b = [(200 - 2 * k, 120 + k) for k in range(30)][: 2 * f + 3]
        tracks = [
            {"track_id": 1, "bbox": [30.4 + 3 * f, 50.9 + 2 * f, 52.2 + 3 * f, 68.1 + 2 * f], "status": "detected", "time_since_update": 0,
             "confidence": 0.91 - 0.01 * f, "trajectory": trail_a, "velocity": (3.0, 2.0)},
            {"track_id": 7, "bbox": [190.0 - 2 * f, 110.0 + f, 214.5 - 2 * f, 131.5 + f], "status": "predicted", "time_since_update": f + 1,
             "confidence": 0.6 * 0.95 ** f, "trajectory": trail_b, "velocity": (-2.0, 1.0)},
            {"track_id": "12", "bbox": np.array([w - 40.0, h - 18.0, w - 8.0, h - 2.0], dtype=np.float32), "status": "detected",
             "confidence": 1.0, "trajectory": [(w - 24, h - 10)], "velocity": (0.3, -0.4)},
            {"track_id": 20, "bbox": (5, 200, 25, 236), "status": "predicted", "time_since_update": 3},
        ]
        dets = [[31.0 + 3 * f, 51.0 + 2 * f, 52.0 + 3 * f, 68.0 + 2 * f, 0.88], [100.0, 20.0, 112.0, 29.0, 0.42, 0.0], [1, 2, 3, 4]] if f % 3 else []
        info = None if f == 2 else ({"frame_number": f, "state_changes": f // 4} if f % 2 else {"frame_number": f})
        frames.append((base.copy(), tracks, dets, info))
    return frames


PLOT_KWARGS = ({}, {"conf": False}, {"labels": False}, {"line_width": 1}, {"line_width": 5}, {"color_mode": "instance"}, {"boxes": False})


def results_exports(make):
    """Results.summary / save_txt / plot over fixed boxes, with and without track ids (tests/golden/results_exports.npz):
    ``make(img, path, names, data)`` builds a Results (the reference's or this package's).  Returns {key: str}: summaries as
    JSON, save_txt files verbatim, plots as "shape dtype sha256" of their pixels -- boxes at the top / right edges, every
    palette colour class, tracked and untracked rows, the plot switches, an image-scaled line width."""
    import hashlib
    import json
    import os
    import tempfile

    def digest(a):
        return f"{a.shape} {a.dtype} " + hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()

    out = {}
    img = np.zeros((96, 128, 3), np.uint8)
    names = {0: "aircraft", 1: "bird"}
    for data in (np.array([[10.5, 12.25, 30.0, 40.75, 0.912345, 0.0], [50.0, 20.0, 70.125, 44.0, 0.4, 1.0]], np.float32),
                 np.array([[10.5, 12.25, 30.0, 40.75, 7.0, 0.912345, 0.0], [50.0, 20.0, 70.125, 44.0, 12.0, 0.4, 1.0]], np.float32)):
        r, n = make(img, "a.jpg", names, data.copy()), data.shape[1]
        out[f"summary_{n}"] = json.dumps(r.summary())
        out[f"summary_normalized_{n}"] = json.dumps(r.summary(normalize=True, decimals=3))
        for save_conf in (False, True):
            with tempfile.TemporaryDirectory() as d:
                p = os.path.join(d, "r.txt")
                r.save_txt(p, save_conf=save_conf)
                with open(p) as fh:
                    out[f"txt_{n}_conf{int(save_conf)}"] = fh.read()
    out["summary_empty"] = json.dumps(make(img, "a.jpg", names, np.zeros((0, 6), np.float32)).summary())
    frame = np.random.default_rng(3).integers(0, 255, (240, 320, 3), dtype=np.uint8)
    many = {c: f"class{c}" for c in range(24)}
    xy = np.array([[4.2, 3.9, 60.0, 40.0], [250.5, 100.0, 318.0, 160.7], [100.0, 120.0, 101.0, 121.0], [-5.0, 200.0, 40.0, 260.0]], np.float32)
    for tracked in (False, True):
        rows = []
        for c in range(24):
            b = xy[c % 4] + np.float32(3 * (c // 4))
            rows.append(np.concatenate([b, [100.0 + c] if tracked else [], [0.05 + 0.04 * c, float(c)]]))
        r = make(frame, "a.jpg", many, np.array(rows, np.float32))
        for j, kw in enumerate(PLOT_KWARGS):
            out[f"plot_tracked{int(tracked)}_{j}"] = digest(r.plot(**kw))
        out[f"plot_tracked{int(tracked)}_big"] = digest(r.plot(img=np.zeros((720, 1280, 3), np.uint8)))
    return out
