"""Reference for rotation candidates (INTEGRATION.md section 8), built on the unchanged oracle.

``candidate_crop`` is candidate a of a box with ``rectify = 0``: ``cv2.resize(cv2.rotate(roi, code_a), (128, 32))`` on the
clamped boundingRect ROI of ``crop_rect``, channels as the oracle hands them to PARSeq.  ``candidate_quad`` is the
``rectify = 1`` quad, ``rect_to_quad``'s corners shifted cyclically by a / 90.  ``select`` is the choice rule over the
section 6 conf of ``scores_ref.word_scores``; ``image_to_data_oriented`` runs the oracle's whole path once per candidate
and keeps the winner of every word.
"""
from __future__ import annotations

import math

import cv2
import numpy as np
import torch

from oracle import tuatara_ref as R
from scores_ref import word_scores

ANGLES = (0, 90, 180, 270)
CODES = {90: cv2.ROTATE_90_COUNTERCLOCKWISE, 180: cv2.ROTATE_180, 270: cv2.ROTATE_90_CLOCKWISE}


def candidate_set(rotation_info) -> list[int]:
    """0 and the requested angles, in the order 0, 90, 180, 270."""
    return [a for a in ANGLES if a == 0 or a in set(rotation_info)]


def rotate(img: np.ndarray, angle: int) -> np.ndarray:
    """img turned `angle` degrees counter-clockwise."""
    return img if angle == 0 else cv2.rotate(np.ascontiguousarray(img), CODES[angle])


def candidate_crop(image: np.ndarray, rect_xywh, angle: int) -> np.ndarray:
    """uint8 [32, 128, 3] in the image's channel order; a rect with no area gives the black crop."""
    x, y, w, h = rect_xywh
    if w <= 0 or h <= 0:
        return np.zeros((32, 128, 3), np.uint8)
    return cv2.resize(rotate(image[y:y + h, x:x + w], angle), (128, 32))


def candidate_quad(rect, angle: int) -> np.ndarray:
    q = R.rect_to_quad(rect)
    return np.roll(q, -(angle // 90), axis=0)


def conf_of(ids: np.ndarray, p: np.ndarray) -> float:
    """Section 6 conf of one crop: product of p[0..e] in double, rounded once to float32 (e = first id 0, else 25)."""
    z = np.flatnonzero(ids == 0)
    e = int(z[0]) if len(z) else len(ids) - 1
    return float(np.float32(math.prod(float(v) for v in p[:e + 1])))


def select(confs) -> int:
    """Index of the winner: a later candidate replaces the best only when its conf is strictly greater (float32)."""
    best = 0
    for r in range(1, len(confs)):
        if np.float32(confs[r]) > np.float32(confs[best]):
            best = r
    return best


def image_to_data_oriented(image: np.ndarray, craft_model, parseq_model, rotation_info, **kw):
    """The oracle's image_to_data where every word is read at each candidate angle (rectify = 0) and the candidate with
    the highest conf is kept: items carry text, bbox, conf, char_conf and angle."""
    st = R.Stages()
    out = R.image_to_data(image, craft_model, parseq_model, stages=st, **kw)
    if not out:
        return out
    cands = candidate_set(rotation_info)
    eos_id = R.Tokenizer().eos_id
    tok = R.Tokenizer()
    per = []
    for a in cands:
        crops = np.stack([candidate_crop(image, r, a) for r in st.crop_rects])
        logits = R.run_parseq(parseq_model, crops)
        probs, ids = torch.softmax(logits, -1).max(-1)
        texts = [R.truncate_at_eos(t) for t in tok.decode(torch.softmax(logits, -1))]
        per.append((texts, probs.numpy(), ids.numpy(), logits.numpy()))
    for i, item in enumerate(out):
        scored = [word_scores(p[1][i], p[2][i], eos_id) for p in per]
        b = select([s[0] for s in scored])
        item.update(text=per[b][0][i], conf=scored[b][0], char_conf=scored[b][1], angle=cands[b],
                    logits=[p[3][i] for p in per])
    return out
