"""The detection half of the IR (640x480) tracker (track/irtrackextractor.py:324-389,391-492,789-818): components of the
background-subtracted frame through ``detect_objects_ir`` on the device, then the rectangle merging that glues the
fragments of one animal together.  (The reference's ``IRTrackExtractor._process_frame`` itself cannot run as written --
with ``DO_SALIENCY = False`` it evaluates ``np.amin(None)`` -- so only the pieces with defined behaviour are mirrored.)

``detect_ir_regions_batch`` and ``ir_clip_regions`` run the same composition for a whole clip on the device: the components of
every frame in one call (csrc/detect_kernels.cu) and the merging in one launch (csrc/ir_kernels.cu)."""
import numpy as np

from ..ml_tools.imageprocessing import detect_objects_ir
from ..ml_tools.tools import eucl_distance_sq


def rect_distance(r_a, r_b):
    """Gap between two [x, y, w, h, ...] rectangles: 0 along an axis on which they overlap (irtrackextractor.py:789-818)."""
    x_1 = x_2 = y_1 = y_2 = 0
    if r_a[2] + r_b[2] > max(r_a[0] + r_a[2], r_b[2] + r_b[0]) - min(r_a[0], r_b[0]):
        pass
    elif r_a[0] < r_b[0]:
        x_1, x_2 = r_a[0] + r_a[2], r_b[0]
    else:
        x_1, x_2 = r_b[0] + r_b[2], r_a[0]
    if r_a[3] + r_b[3] > max(r_a[1] + r_a[3], r_b[1] + r_b[3]) - min(r_a[1], r_b[1]):
        pass
    elif r_a[1] < r_b[1]:
        y_1, y_2 = r_a[1] + r_a[3], r_b[1]
    else:
        y_1, y_2 = r_b[1] + r_b[3], r_a[1]
    return eucl_distance_sq((x_1, y_1), (x_2, y_2)) ** 0.5


def merge_limits(scale=None):
    """(min_mass, min_size, max_gap) of merge_components for ``scale`` (irtrackextractor.py:324-331)."""
    min_mass, min_size, max_gap = 10 * 4, 16, 40
    if scale:
        min_mass = int(min_mass * scale)
        min_size = int(min_size * scale)
        max_gap *= scale
    return min_mass, min_size, max_gap


def merge_components(rectangles, scale=None):
    """Merge stats rows [x, y, w, h, area] that overlap or lie within MAX_GAP of each other, largest first, until nothing
    merges any more (irtrackextractor.py:324-389; the reference's arithmetic is kept as written, including the bottom edge
    it derives from the x extent)."""
    min_mass, min_size, max_gap = merge_limits(scale)
    rectangles = [r for r in rectangles if r[4] > min_mass or (r[2] > min_size and r[3] > min_size)]
    rectangles = sorted(rectangles, key=lambda s: s[4], reverse=True)
    rectangles = [(r, r.copy()) for r in rectangles]  # merge on the original rectangle, not on the grown one
    rect_i = 0
    while rect_i < len(rectangles):
        rect, merged_r = rectangles[rect_i]
        merged = False
        index = 0
        while index < len(rectangles):
            within = False
            r_2 = rectangles[index][0]
            if r_2[0] == rect[0]:
                index += 1
                continue
            if r_2[2] + rect[2] > max(r_2[0] + r_2[2], rect[2] + rect[0]) - min(r_2[0], rect[0]):
                within = r_2[3] + rect[3] > max(r_2[1] + r_2[3], rect[1] + rect[3]) - min(r_2[1], rect[1])
            if rect_distance(rect, r_2) < max_gap or within:
                cur_right = merged_r[0] + merged_r[2]
                merged_r[0] = min(merged_r[0], r_2[0])
                merged_r[1] = min(merged_r[1], r_2[1])
                merged_r[2] = max(cur_right, r_2[0] + r_2[2])
                merged_r[3] = max(merged_r[1] + merged_r[3], r_2[1] + r_2[3])
                merged_r[2] -= merged_r[0]
                merged_r[3] -= merged_r[1]
                merged_r[4] += r_2[4]
                merged = True
                del rectangles[index]
            else:
                index += 1
        rect_i = 0 if merged else rect_i + 1
    return [rect[1] for rect in rectangles]


def detect_ir_regions(filtered, scale=None):
    """What ``IRTrackExtractor._process_frame`` does with a background-subtracted frame (irtrackextractor.py:453-455):
    ``detect_objects_ir(filtered, threshold=0)`` -> stats rows without the background -> ``merge_components``.
    Returns (labels, merged rectangles)."""
    _, mask, component_details = detect_objects_ir(filtered, threshold=0)
    return mask, merge_components(list(component_details[1:]), scale=scale)


def _used_rows(d_rows, d_counts, counts):
    """Rows [t][:counts[t]] of a [N][R][5] CUDA tensor, copied back in one piece and split per frame."""
    import torch

    top = int(counts.max()) if counts.size else 0
    used = torch.arange(top, device=d_rows.device)[None, :] < d_counts[:, None]
    flat = d_rows[:, :top][used].cpu().numpy()
    return np.split(flat, np.cumsum(counts)[:-1]) if counts.size else []


def detect_ir_regions_batch(frames, scale=None, threshold=0, labels=False):
    """``detect_ir_regions`` for every frame of frames [N][H][W] uint8 (a host array or a CUDA tensor) in one components
    call and one merge launch.  Returns (stats, merged), or (stats, merged, labels) with labels=True: per frame the
    ``detect_objects_ir`` stats rows (background first) and the merged [x, y, w, h, area] rows as int32 host arrays, and
    the int32 label images [N][H][W].  A frame with more than ``detect.MAX_COMPONENTS`` components raises, as
    ``detect_ir_regions`` does on it."""
    import torch

    from .. import engine, native
    from ..ml_tools import detect

    eng = engine.get_engine()
    if isinstance(frames, torch.Tensor):
        if frames.dtype != torch.uint8 or not frames.is_cuda:
            raise ValueError("detect_ir_regions_batch takes uint8 frames (a host array or a CUDA tensor)")
        d = frames.contiguous()
    else:
        frames = np.ascontiguousarray(frames)
        if frames.dtype != np.uint8:
            raise ValueError("detect_ir_regions_batch takes uint8 frames (a host array or a CUDA tensor)")
        d = torch.from_numpy(frames).to(eng.device)
    if d.dim() != 3:
        raise ValueError("detect_ir_regions_batch takes frames [N][H][W]")
    n, h, w = d.shape
    if n == 0:
        return ([], [], np.zeros((0, h, w), np.int32)) if labels else ([], [])
    mc = detect.MAX_COMPONENTS
    i32 = dict(dtype=torch.int32, device=d.device)
    eng.ctx.use_torch_stream()
    d_counts, d_stats = torch.empty(n, **i32), torch.empty((n, mc + 1, 5), **i32)
    d_labels = torch.empty((n, h, w), **i32) if labels else None
    eng.ctx.detect_objects_batch(d, n, w, h, threshold, native.DETECT_OPEN_GRAY, mc, d_counts, d_stats, None, d_labels)
    d_merged_counts, d_merged = torch.empty(n, **i32), torch.empty((n, mc, 5), **i32)
    min_mass, min_size, max_gap = merge_limits(scale)
    eng.ctx.ir_merge_components(d_stats, d_counts, n, mc, min_mass, min_size, max_gap, d_merged, d_merged_counts)
    counts, merged_counts = torch.stack([d_counts, d_merged_counts]).cpu().numpy()
    over = np.nonzero(counts - 1 > mc)[0]
    if over.size:
        t = int(over[0])
        raise native.NativeError("frame {}: {} components exceed max_components {}".format(t, int(counts[t]) - 1, mc))
    out = (_used_rows(d_stats, d_counts, counts), _used_rows(d_merged, d_merged_counts, merged_counts))
    return out + (d_labels.cpu().numpy(),) if labels else out


def ir_clip_regions(frames, background=None, learning_rate=-1, scale=None):
    """Regions of every frame of one IR clip: frames [N][H][W] grey uint8 (a host array or a CUDA tensor) through
    ``background.update_backgrounds`` (a new ``MOG2Background`` when None; ``learning_rate`` a number or one per frame)
    and ``detect_ir_regions_batch`` on its masks, which stay on the device.  Returns (stats, merged) as
    ``detect_ir_regions_batch`` does."""
    from .cliptracker import MOG2Background

    if background is None:
        background = MOG2Background()
    masks = background.update_backgrounds(background._to_device(frames), learning_rate)
    return detect_ir_regions_batch(masks, scale=scale)
