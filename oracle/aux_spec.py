"""NumPy restatement of the steps either side of the develop path (SURVEY.md section 8f): flat-field correction and
hot-pixel detection before it, camera-space HDR fusion after it.

TEST INFRASTRUCTURE ONLY.  Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s CPU-baseline leg may import this
module; the product (`pysp_b200/`) never does.

Parity status: PINNED against the reference itself -- `tests/golden/make_golden_aux.py` runs the unmodified reference
(raw_correction.py, raw_bad_pixel_corr.py, raw_hdr.py) and stores its outputs in `tests/golden/aux_*.npz`;
`tests/test_oracle_aux.py` checks this restatement against them bit for bit.

Third-party arithmetic restated here: NumPy's float32 `np.mean` (pairwise summation, numpy/_core/src/umath/
loops_utils.h.src `@TYPE@_pairwise_sum`, numpy==2.2.4 in requirements.txt:4; 2.3.5 here) at raw_correction.py:45, and
NumPy's NEP-50 scalar promotion at raw_hdr.py:61-75.
"""
import numpy as np

from oracle.ahd_spec import join_planes, mat3_f64, split_planes

f32 = np.float32


# ----------------------------------------------------------------------------------------------------------------
# np.mean of a float32 colour plane (raw_correction.py:45)
# ----------------------------------------------------------------------------------------------------------------
def pairwise_leaves(a, offs, n):
    """NumPy's unrolled block sum of n <= 128 float32 values, for the blocks a[o:o+n] of every o in `offs` at once: eight
    strided partial sums, a fixed combine, then the tail."""
    v = a[offs[:, None] + np.arange(n)]
    if n < 8:
        res = np.zeros(len(offs), dtype=f32)
        for i in range(n):
            res = (res + v[:, i]).astype(f32)
        return res
    m = n - (n % 8)
    r = v[:, :m].reshape(len(offs), -1, 8)
    acc = r[:, 0].copy()
    for k in range(1, r.shape[1]):
        acc = (acc + r[:, k]).astype(f32)
    res = (((acc[:, 0] + acc[:, 1]) + (acc[:, 2] + acc[:, 3])) + ((acc[:, 4] + acc[:, 5]) + (acc[:, 6] + acc[:, 7]))).astype(f32)
    for i in range(m, n):
        res = (res + v[:, i]).astype(f32)
    return res


def _pairwise_level(a, groups):
    """Sums of the runs of one recursion depth, {length: start offsets} -> {length: sums}.  The runs of the next depth are
    grouped by length across parents, so every depth costs a few vector operations however many runs it has."""
    nxt, plan, res = {}, [], {}
    for n, offs in groups.items():
        if n <= 128:
            res[n] = pairwise_leaves(a, offs, n)
            continue
        n2 = n // 2
        n2 -= n2 % 8
        kids = []
        for cn, co in ((n2, offs), (n - n2, offs + n2)):
            parts = nxt.setdefault(cn, [])
            kids.append((cn, sum(len(q) for q in parts)))
            parts.append(co)
        plan.append((n, len(offs), kids))
    if nxt:
        sub = _pairwise_level(a, {cn: np.concatenate(parts) for cn, parts in nxt.items()})
        for n, k, ((ln, ls), (rn, rs)) in plan:
            res[n] = (sub[ln][ls:ls + k] + sub[rn][rs:rs + k]).astype(f32)
    return res


def pairwise_sum(a):
    """float32 sum in NumPy's order: recursive halving (left half rounded down to a multiple of 8) down to blocks of
    at most 128 elements, each half summed before the two are added.  `a` is the plane in row-major order: bayer_to_rgbg's
    planes are strided views whose two axes coalesce (bayer_chan_mixer.py:13-21), so np.mean sees one run of h*w
    elements."""
    a = np.ascontiguousarray(a, dtype=f32).ravel()
    n = a.shape[0]
    return _pairwise_level(a, {n: np.zeros(1, dtype=np.int64)})[n][0]


def plane_mean(p):
    """np.mean: the float32 sum divided by the integer count in float64, rounded to float32 once (numpy/_core/_methods.py,
    _mean).  A float32 divisor gives the same bits only up to 2^24 elements, where float32(p.size) is still p.size."""
    return f32(np.float64(pairwise_sum(p)) / p.size)


# ----------------------------------------------------------------------------------------------------------------
# flat_frame_correction (raw_correction.py:25-63)
# ----------------------------------------------------------------------------------------------------------------
def flat_frame_correction(sensor, flat, clamp_high=False):
    """Per CFA plane: out = (chan * mean(flat_chan)) / flat_chan in float32; +inf -> largest finite value of the plane;
    negative -> 0; optional clamp at 1; a plane whose quotient is +-inf everywhere is left untouched."""
    outs = []
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        for chan, chan_flat in zip(split_planes(np.asarray(sensor, dtype=f32)), split_planes(np.asarray(flat, dtype=f32))):
            mean_chan = plane_mean(chan_flat)
            output = ((chan * mean_chan).astype(f32) / chan_flat).astype(f32)
            if np.isinf(output).all():
                outs.append(np.copy(chan))
                continue
            finite = np.isfinite(output)
            # no finite value at all (e.g. a 0/0 plane): the reference's masked maximum is undefined; +inf -> NaN here
            max_output = output[finite].max() if finite.any() else f32(np.nan)
            output[output == np.inf] = max_output
            output[output < 0] = 0
            if clamp_high:
                output[output > 1] = 1
            outs.append(output)
    return join_planes(*outs)


# ----------------------------------------------------------------------------------------------------------------
# find_erroneous_pixels_threshold (raw_bad_pixel_corr.py:30-65)
# ----------------------------------------------------------------------------------------------------------------
def find_erroneous_pixels_threshold(sensor, min_delta=0.025, min_neighbour_count=5):
    """Per CFA plane: a photosite is hot when (value - min_delta) exceeds more than `min_neighbour_count` of its eight
    same-colour neighbours (np.pad mode="reflect", i.e. no edge duplication)."""
    masks = []
    for chan in split_planes(np.asarray(sensor, dtype=f32)):
        padded = np.pad(chan, (1, 1), mode="reflect")
        h, w = chan.shape
        ref = (chan - f32(min_delta)).astype(f32)
        cnt = np.zeros((h, w), dtype=np.int32)
        for dy in range(3):
            for dx in range(3):
                if dy == 1 and dx == 1:
                    continue
                cnt += ref > padded[dy:dy + h, dx:dx + w]
        masks.append(cnt > min_neighbour_count)
    return masks


# ----------------------------------------------------------------------------------------------------------------
# fuse_exposures_from_debayer (raw_hdr.py:7-83)
# ----------------------------------------------------------------------------------------------------------------
def fuse_exposures_from_debayer(images, evs, wb, m_cam_to_srgb, wb_normalized=None, target_ev=None):
    """Camera-space HDR fusion of demosaiced exposures (float32 [H,W,3], white balance applied).  Returns
    (linear sRGB f32, contribution count int32 [H,W,3], the images as the reference leaves them after its
    wb_undo()/wb_apply() round trip)."""
    wb = np.asarray(wb, dtype=f32)[:3]
    evs = [float(e) for e in evs]
    if wb_normalized is None:
        wb_normalized = [False] * len(images)
    if target_ev is None:
        target_ev = 0
        for e in evs:
            target_ev += e
        target_ev /= len(evs)
    offs = [2 ** (e - target_ev) for e in evs]
    sum_pixel = np.zeros(images[0].shape, dtype=f32)
    sum_weight = np.zeros(images[0].shape, dtype=f32)
    count = np.zeros(images[0].shape, dtype=np.int32)
    off_max = np.max(offs)                       # np.float64: NOT a weak scalar (raw_hdr.py:52, 75)
    max_exposure = None
    left = []
    for img, off, norm in zip(images, offs, wb_normalized):
        img = np.asarray(img, dtype=f32)
        if norm:                                 # base_types/image_base.py:56-57
            img = (img * max(wb)).astype(f32)
        undone = (img.astype(np.float64) / wb).astype(f32)                 # wb_undo, image_base.py:58
        weights = (f32(0.5) - np.abs(undone - f32(0.5))).astype(f32)        # raw_hdr.py:59
        weights = (weights * f32(1.6 ** (-0.1 * off))).astype(f32)          # Python float: weak scalar -> float32
        sum_weight += weights
        applied = (undone * wb).astype(f32)                                 # wb_apply, image_base.py:48
        left.append(applied)
        if off == off_max:
            max_exposure = applied
        sum_pixel += ((applied * weights).astype(f32) * f32(off)).astype(f32)
        count[weights > 0] += 1
    max_exposure = np.multiply(max_exposure, off_max)                       # float64 array
    with np.errstate(divide="ignore", invalid="ignore"):
        q = np.divide(sum_pixel, sum_weight)
    fused = np.where(sum_weight == 0, max_exposure, q).astype(f32)
    return mat3_f64(fused, m_cam_to_srgb), count, left
