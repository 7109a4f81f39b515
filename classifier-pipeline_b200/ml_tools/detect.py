"""``detect_objects`` / ``detect_objects_ir`` / ``detect_objects_both`` on the device for one image of any size
(ml_tools/imageprocessing.py:185-248): uint8 cast -> grey morphology / GaussianBlur -> threshold (optionally Otsu) ->
binary morphology with the tuple kernel -> connectedComponentsWithStats."""
import numpy as np

from .. import engine as _engine
from .. import native

MAX_COMPONENTS = 8192
BLUR_SIZES = (3, 5, 7, 15)  # cv2.GaussianBlur kernels whose 8-bit fixed-point taps are built (csrc/detect_kernels.cu)


def _blur_size(kernel):
    kernel = tuple(kernel)
    if len(kernel) != 2 or kernel[0] != kernel[1] or kernel[0] not in BLUR_SIZES:
        # cv2.GaussianBlur derives sigma and fixed-point taps from the kernel size
        raise NotImplementedError("GaussianBlur kernel {}: only square kernels of {} are built".format(kernel, BLUR_SIZES))
    return kernel[0]


def _run(image, threshold, blur, steps, or_mask=None, stats_only=False):
    import torch

    image = np.uint8(image)  # numpy's cast, exactly as the reference
    if image.ndim != 2:
        raise ValueError("detect_objects: single-channel image expected")
    H, W = image.shape
    eng = _engine.get_engine()
    eng.ctx.use_torch_stream()
    d_img = torch.from_numpy(np.ascontiguousarray(image)).to(eng.device)
    d_or = None
    if or_mask is not None:
        d_or = torch.from_numpy(np.ascontiguousarray(np.uint8(or_mask))).to(eng.device)
    d_labels = torch.empty((H, W), dtype=torch.int32, device=eng.device)
    d_stats = torch.empty((MAX_COMPONENTS + 1, 5), dtype=torch.int32, device=eng.device)
    d_cent = torch.empty((MAX_COMPONENTS + 1, 2), dtype=torch.float64, device=eng.device)
    n, _ = eng.ctx.detect_objects(d_img, W, H, threshold, blur, steps, MAX_COMPONENTS, d_labels, d_stats, d_cent, d_or_mask=d_or)
    return n, d_labels.cpu().numpy(), d_stats[:n].cpu().numpy(), d_cent[:n].cpu().numpy()


def detect_objects(image, otsus=False, threshold=30, kernel=(15, 15)):
    """Returns (n_labels, labels int32 (H, W), stats int32 (n, 5), centroids float64 (n, 2)), row 0 = background.
    A tuple ``kernel`` reaches cv2.morphologyEx as a 2x1 structuring element whatever its values."""
    steps = native.DETECT_CLOSE | (native.DETECT_OTSU if otsus else 0)
    return _run(image, threshold, _blur_size(kernel), steps)


def detect_objects_ir(image, otsus=False, threshold=100, kernel=(15, 15)):
    """imageprocessing.py:185-199: morphological open of the grey image, threshold, components.
    Returns (n_labels, labels, stats) like the reference."""
    tuple(kernel)
    steps = native.DETECT_OPEN_GRAY | (native.DETECT_OTSU if otsus else 0)
    n, labels, stats, _ = _run(image, threshold, 0, steps)
    return n, labels, stats


def _binary_mask(image, threshold, steps):
    import torch

    image = np.uint8(image)
    H, W = image.shape
    eng = _engine.get_engine()
    eng.ctx.use_torch_stream()
    d_img = torch.from_numpy(np.ascontiguousarray(image)).to(eng.device)
    d_mask = torch.empty((H, W), dtype=torch.uint8, device=eng.device)
    eng.ctx.detect_objects(d_img, W, H, threshold, 0, steps | native.DETECT_MASK_ONLY, 1, None, None, None, d_mask_out=d_mask)
    return d_mask.cpu().numpy()


def detect_objects_both(salicencyMap, backsub, threshold=30, kernel=(15, 15), otsus=False):
    """imageprocessing.py:202-238: the saliency map (open, threshold) OR-ed into the background-subtraction mask (blur,
    threshold, dilate, close), then components.  Returns (n_labels, labels, stats)."""
    or_mask = None
    if salicencyMap is not None:
        or_mask = _binary_mask(salicencyMap, threshold, native.DETECT_OPEN_GRAY | (native.DETECT_OTSU if otsus else 0))
    steps = native.DETECT_DILATE | native.DETECT_CLOSE | (native.DETECT_OTSU if otsus else 0)
    n, labels, stats, _ = _run(backsub, threshold, _blur_size(kernel), steps, or_mask=or_mask)
    return n, labels, stats
