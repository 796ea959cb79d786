"""Reference for the contrast re-read (INTEGRATION.md section 10), built on the unchanged oracle.

``contrast_grey`` and ``adjust_contrast_grey`` are EasyOCR's (easyocr/utils.py), verbatim, on numpy with a live
``np.percentile``.  ``contrast_params`` / ``stretch_table`` / ``adjust_crop`` are the colour extension the engine
computes: the grey percentiles of a 128 x 32 crop in the caller's channel order drive one 256-entry map applied to all
three channels.  ``keep_second`` is the selection rule; ``image_to_data_contrast`` runs the oracle's path and re-reads
the words the rule picks.
"""
from __future__ import annotations

import cv2
import numpy as np
import torch

from oracle import tuatara_ref as R
from scores_ref import word_scores

# cv2.cvtColor(COLOR_BGR2GRAY) on 8-bit pixels: (B * 3735 + G * 19235 + R * 9798 + 2^14) >> 15
GREY_COEF = (3735, 19235, 9798)
GREY_SHIFT = 15


def contrast_grey(img):
    high = np.percentile(img, 90)
    low = np.percentile(img, 10)
    return (high - low) / np.maximum(10, high + low), high, low


def adjust_contrast_grey(img, target=0.4):
    contrast, high, low = contrast_grey(img)
    if contrast < target:
        img = img.astype(int)
        ratio = 200. / np.maximum(10, high - low)
        img = (img - low + 25) * ratio
        img = np.maximum(np.full(img.shape, 0), np.minimum(np.full(img.shape, 255), img)).astype(np.uint8)
    return img


def grey(crop: np.ndarray) -> np.ndarray:
    return cv2.cvtColor(np.ascontiguousarray(crop), cv2.COLOR_BGR2GRAY)


def grey_formula(bgr: np.ndarray) -> np.ndarray:
    """The device's grey of uint8 [..., 3] pixels."""
    v = bgr.astype(np.int64)
    b, g, r = GREY_COEF
    return (v[..., 0] * b + v[..., 1] * g + v[..., 2] * r + (1 << (GREY_SHIFT - 1))) >> GREY_SHIFT


def contrast_params(crop: np.ndarray, adjust_contrast: float):
    """-> (low contrast?, low, high) of a uint8 [32, 128, 3] crop; adjust_contrast is compared as the float32 it is
    passed as."""
    contrast, high, low = contrast_grey(grey(crop))
    return bool(contrast < float(np.float32(adjust_contrast))), float(low), float(high)


def stretch_table(low: float, high: float) -> np.ndarray:
    """adjust_contrast_grey's map as a table: entry v is what a pixel of value v becomes."""
    ratio = 200. / np.maximum(10, high - low)
    v = np.arange(256).astype(int)
    return np.maximum(np.full(256, 0), np.minimum(np.full(256, 255), (v - low + 25) * ratio)).astype(np.uint8)


def adjust_crop(crop: np.ndarray, adjust_contrast: float):
    """-> (the crop as the second read sees it, stretched?): every channel through the grey map when low contrast."""
    low_contrast, low, high = contrast_params(crop, adjust_contrast)
    if not low_contrast:
        return crop.copy(), False
    return stretch_table(low, high)[crop], True


def keep_second(conf1: float, conf2: float) -> bool:
    """The second read replaces the first only when its conf is strictly greater (float32; ties and NaN keep the first)."""
    return bool(np.float32(conf2) > np.float32(conf1))


def reread_words(conf, crops: np.ndarray, contrast_ths: float, adjust_contrast: float):
    """-> (indices of the words read again, their stretched crops): conf below contrast_ths and a low-contrast crop."""
    idx, out = [], []
    for i, (c, crop) in enumerate(zip(conf, crops)):
        if not np.float32(c) < np.float32(contrast_ths):
            continue
        adj, stretched = adjust_crop(crop, adjust_contrast)
        if stretched:
            idx.append(i)
            out.append(adj)
    return idx, (np.stack(out) if out else np.zeros((0, 32, 128, 3), np.uint8))


def image_to_data_contrast(image: np.ndarray, craft_model, parseq_model, contrast_ths: float, adjust_contrast: float = 0.5,
                           **kw):
    """The oracle's image_to_data with the contrast re-read: items carry text, bbox, conf, char_conf and reread (whether
    the word was read again, whichever read won)."""
    st = R.Stages()
    out = R.image_to_data(image, craft_model, parseq_model, stages=st, **kw)
    if not out:
        return out
    tok = R.Tokenizer()

    def scored(logits):
        probs, ids = torch.softmax(logits, -1).max(-1)
        texts = [R.truncate_at_eos(t) for t in tok.decode(torch.softmax(logits, -1))]
        return texts, [word_scores(p, i, tok.eos_id) for p, i in zip(probs.numpy(), ids.numpy())]

    _, sc = scored(torch.from_numpy(st.logits))
    for item, s in zip(out, sc):
        item.update(conf=s[0], char_conf=s[1], reread=False)
    idx, crops = reread_words([s[0] for s in sc], st.crops_u8, contrast_ths, adjust_contrast)
    if idx:
        texts2, sc2 = scored(R.run_parseq(parseq_model, crops))
        for k, i in enumerate(idx):
            out[i]["reread"] = True
            if keep_second(out[i]["conf"], sc2[k][0]):
                out[i].update(text=texts2[k], conf=sc2[k][0], char_conf=sc2[k][1])
    return out
