"""tuatara_b200: B200-native implementation of the Tuatara OCR hot path.

Python here is only the host-side mirror of the reference's interface
(``bindings/python.cpp:43-58``: ``image_to_data(image, weights_dir, outputs_dir)``) plus thin
stage-level wrappers used by the parity tests and the benchmark.  Every call goes through
the C ABI of ``libtuatara_b200.so``; nothing is computed in Python and nothing falls back
to the CPU.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native
from ._native import TuataraError, check, lib, ptr

__all__ = [
    "TuataraError", "Engine", "image_to_data", "images_to_data", "image_to_data_scored", "images_to_data_scored",
    "default_config", "resize_plan", "preprocess", "postprocess", "crop_resize", "contrast_adjust", "decode_ids", "decode_scores", "tokenizer_table",
    "char_filter_mask", "Lexicon", "min_area_rect", "convex_hull",
    "rect_points", "rect_bounding", "adjust_rect", "rect_to_bbox", "launch_count",
]


def default_config() -> _native.tt_config:
    cfg = _native.tt_config()
    lib().tt_config_default(C.byref(cfg))
    return cfg


def launch_count() -> int:
    return int(lib().tt_launch_count())


# --------------------------------------------------------------------------- host logic
def resize_plan(rows: int, cols: int, canvas_size: float = 1024.0, mag_ratio: float = 1.0):
    """-> (target_h, target_w, h32, w32, ratio)  (tuatara.cpp:211-226)."""
    th, tw, h32, w32, ratio = C.c_int(), C.c_int(), C.c_int(), C.c_int(), C.c_float()
    check(lib().tt_resize_plan(rows, cols, canvas_size, mag_ratio, C.byref(th), C.byref(tw), C.byref(h32),
                               C.byref(w32), C.byref(ratio)), "tt_resize_plan")
    return th.value, tw.value, h32.value, w32.value, np.float32(ratio.value)


def tokenizer_table():
    buf = C.create_string_buffer(128)
    eos, bos, pad = C.c_int(), C.c_int(), C.c_int()
    check(lib().tt_tokenizer_table(buf, C.byref(eos), C.byref(bos), C.byref(pad)), "tt_tokenizer_table")
    return buf.value.decode("latin-1"), eos.value, bos.value, pad.value


def _filter_bytes(v, name: str):
    if v is None:
        return None
    if not isinstance(v, str):
        raise TypeError(f"{name}: expected str or None")
    return v.encode()


def char_filter_mask(allow: str | None = None, block: str | None = None) -> np.ndarray:
    """Class mask of a character filter (tt_char_filter_mask): uint32 [4], bit c & 31 of word c >> 5 set when class c may
    be produced.  Classes 0 and 88 (they print nothing) are always set; word 3 is 0."""
    f = _native.tt_char_filter(_filter_bytes(allow, "allow"), _filter_bytes(block, "block"))
    out = np.zeros(4, np.uint32)
    check(lib().tt_char_filter_mask(C.byref(f), ptr(out)), "tt_char_filter_mask")
    return out


def _filters(allowlist, blocklist, n_pages: int):
    """allowlist / blocklist keywords -> a tt_char_filter array (None: no filter).  Each is None, a str for every page, or
    a list with one str or None per page."""
    if allowlist is None and blocklist is None:
        return None
    per_page = isinstance(allowlist, (list, tuple)) or isinstance(blocklist, (list, tuple))
    n = n_pages if per_page else 1
    cols = []
    for v, name in ((allowlist, "allowlist"), (blocklist, "blocklist")):
        if isinstance(v, (list, tuple)):
            if len(v) != n_pages:
                raise ValueError(f"{name}: expected one entry per page ({n_pages}), got {len(v)}")
            cols.append([_filter_bytes(x, name) for x in v])
        else:
            cols.append([_filter_bytes(v, name)] * n)
    return (_native.tt_char_filter * n)(*[_native.tt_char_filter(a, b) for a, b in zip(*cols)])


class Lexicon:
    """A reusable word list (tt_lexicon, INTEGRATION.md section 9): every word recognised under it is one of its words.
    words: an iterable of str, each 1..25 characters that PARSeq can print (no ']', '~', control or non-ASCII
    characters); duplicates count once.  Build it once and pass it as ``lexicon=`` to as many calls as needed."""

    def __init__(self, words):
        if isinstance(words, (str, bytes)) or not hasattr(words, "__iter__"):
            raise TypeError("Lexicon: expected an iterable of str")
        ws = list(words)
        for i, w in enumerate(ws):
            if not isinstance(w, str):
                raise TypeError(f"Lexicon: word {i} is a {type(w).__name__}, expected str")
            if "\0" in w:
                raise TuataraError(f"tt_lexicon_create: word {i} holds byte 0x00, which no class prints")
        arr = (C.c_char_p * max(len(ws), 1))(*[w.encode() for w in ws])
        self._h = C.c_void_p()
        check(lib().tt_lexicon_create(arr, len(ws), C.byref(self._h)), "tt_lexicon_create")

    def info(self) -> tuple[int, int]:
        """-> (distinct words, states of the trie)."""
        nw, ns = C.c_int(), C.c_int()
        check(lib().tt_lexicon_info(self._h, C.byref(nw), C.byref(ns)), "tt_lexicon_info")
        return nw.value, ns.value

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().tt_lexicon_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close


def _is_words(v) -> bool:
    return not isinstance(v, (str, bytes, Lexicon)) and v is not None and hasattr(v, "__iter__")


def _lexicon_arg(lexicon, n_pages: int, strict: bool):
    """lexicon keyword -> (a list of Lexicon or None, one entry or one per page) or None.  It is a Lexicon or an iterable
    of str (one lexicon for every page), or a list with one entry per page, each None or one of those (strict: each None
    or a Lexicon, so that a list of str is always one word list)."""
    if lexicon is None:
        return None
    if isinstance(lexicon, Lexicon):
        return [lexicon]
    if isinstance(lexicon, (str, bytes)) or not hasattr(lexicon, "__iter__"):
        raise TypeError("lexicon: expected a Lexicon, an iterable of str or a list with one entry per page")
    vals = list(lexicon)
    if all(isinstance(v, str) for v in vals):
        return [Lexicon(vals)]
    ok = (lambda v: v is None or isinstance(v, Lexicon)) if strict else (lambda v: v is None or isinstance(v, Lexicon) or _is_words(v))
    if not isinstance(lexicon, (list, tuple)) or not all(ok(v) for v in vals):
        raise TypeError("lexicon: a list with one entry per page holds " +
                        ("Lexicon objects or None" if strict else "None, Lexicon objects or iterables of str") +
                        ", and a word list holds only str")
    if len(vals) != n_pages:
        raise ValueError(f"lexicon: expected one entry per page ({n_pages}), got {len(vals)}")
    return [v if v is None or isinstance(v, Lexicon) else Lexicon(v) for v in vals]


def _engine_lexicon(lexicon, n_pages: int):
    """The module functions' lexicon keyword (word lists allowed per page) -> what Engine.ocr_pages takes."""
    lex = _lexicon_arg(lexicon, n_pages, strict=False)
    return lex[0] if lex is not None and len(lex) == 1 and lex[0] is not None else lex


def decode_ids(ids: np.ndarray) -> list[str]:
    ids = np.ascontiguousarray(ids, np.int32)
    n, ln = ids.shape
    out = np.zeros((n, 64), np.uint8)
    check(lib().tt_decode(ptr(ids), n, ln, ptr(out), 64), "tt_decode")
    return [bytes(row).split(b"\0", 1)[0].decode("latin-1") for row in out]


def decode_scores(ids: np.ndarray, pmax: np.ndarray):
    """decode_ids with scores (host only): ids int32 [n, len], pmax float32 [n, len] (the largest softmax probability
    per position) -> (texts, conf float32 [n], char_conf: list of float32 arrays, one value per character)."""
    ids = np.ascontiguousarray(ids, np.int32)
    pmax = np.ascontiguousarray(pmax, np.float32)
    n, ln = ids.shape
    if pmax.shape != ids.shape:
        raise ValueError("decode_scores: ids and pmax differ in shape")
    out = np.zeros((n, 64), np.uint8)
    conf = np.empty(n, np.float32)
    cc = np.empty((n, ln), np.float32)
    check(lib().tt_decode_scores(ptr(ids), ptr(pmax), n, ln, ptr(out), 64, ptr(conf), ptr(cc)), "tt_decode_scores")
    texts = [bytes(row).split(b"\0", 1)[0].decode("latin-1") for row in out]
    return texts, conf, [cc[i, :len(t)].copy() for i, t in enumerate(texts)]


def convex_hull(points: np.ndarray) -> np.ndarray:
    n = len(points)
    idx = np.zeros(max(n, 1), np.int32)
    n_out = C.c_int()
    if points.dtype.kind == "f":
        p = np.ascontiguousarray(points, np.float32)
        check(lib().tt_convex_hull_f32(ptr(p), n, ptr(idx), C.byref(n_out)), "tt_convex_hull_f32")
    else:
        p = np.ascontiguousarray(points, np.int32)
        check(lib().tt_convex_hull_i32(ptr(p), n, ptr(idx), C.byref(n_out)), "tt_convex_hull_i32")
    return idx[: n_out.value].copy()


def _rect_tuple(r: np.ndarray):
    return ((float(r[0]), float(r[1])), (float(r[2]), float(r[3])), float(r[4]))


def _rect_array(rect) -> np.ndarray:
    (cx, cy), (w, h), a = rect
    return np.array([cx, cy, w, h, a], np.float32)


def min_area_rect(points: np.ndarray):
    """cv2.minAreaRect-compatible: ((cx, cy), (w, h), angle)."""
    out = np.zeros(5, np.float32)
    if points.dtype.kind == "f":
        p = np.ascontiguousarray(points, np.float32).reshape(-1, 2)
        check(lib().tt_min_area_rect_f32(ptr(p), len(p), ptr(out)), "tt_min_area_rect_f32")
    else:
        p = np.ascontiguousarray(points, np.int32).reshape(-1, 2)
        check(lib().tt_min_area_rect_i32(ptr(p), len(p), ptr(out)), "tt_min_area_rect_i32")
    return _rect_tuple(out)


def rect_points(rect) -> np.ndarray:
    out = np.zeros((4, 2), np.float32)
    check(lib().tt_rect_points(ptr(_rect_array(rect)), ptr(out)), "tt_rect_points")
    return out


def rect_bounding(rect):
    out = np.zeros(4, np.int32)
    check(lib().tt_rect_bounding(ptr(_rect_array(rect)), ptr(out)), "tt_rect_bounding")
    return tuple(int(v) for v in out)


def adjust_rect(rect, ratio_w, ratio_h, ratio_net=2.0):
    out = np.zeros(5, np.float32)
    check(lib().tt_adjust_rect(ptr(_rect_array(rect)), float(ratio_w), float(ratio_h), float(ratio_net), ptr(out)),
          "tt_adjust_rect")
    return _rect_tuple(out)


def rect_to_bbox(rect) -> list[float]:
    out = np.zeros(4, np.float32)
    check(lib().tt_rect_to_bbox(ptr(_rect_array(rect)), ptr(out)), "tt_rect_to_bbox")
    return [float(v) for v in out]


# ------------------------------------------------------------------- GPU stages (host buffers)
def preprocess(image: np.ndarray, canvas_size: float = 1024.0, mag_ratio: float = 1.0):
    """Channel swap + resize + pad on the GPU -> (uint8 [h32, w32, 3], ratio)."""
    _th, _tw, h32, w32, ratio = resize_plan(image.shape[0], image.shape[1], canvas_size, mag_ratio)
    out = np.empty((h32, w32, 3), np.uint8)
    im = _native.image_struct(image)
    check(lib().tt_preprocess(C.byref(im), canvas_size, mag_ratio, ptr(out)), "tt_preprocess")
    return out, ratio


def postprocess(maps: np.ndarray, cfg: _native.tt_config | None = None, want_labels: bool = True):
    """get_detected_boxes on the GPU.  maps: float32 [H, W, 2].
    -> dict(n_labels, labels [H,W] int32, stats [n_labels,5] int32, rects [list of cv2-style tuples], rect_labels)."""
    maps = np.ascontiguousarray(maps, np.float32)
    H, W, _ = maps.shape
    cap = H * W // 2 + 2
    labels = np.empty((H, W), np.int32) if want_labels else None
    stats = np.zeros((cap, 5), np.int32)
    rects = np.zeros((cap, 5), np.float32)
    rlabels = np.zeros(cap, np.int32)
    n_labels, n_rects = C.c_int(), C.c_int()
    check(lib().tt_postprocess(ptr(maps), H, W, C.byref(cfg) if cfg is not None else None, ptr(labels), ptr(stats),
                               cap, C.byref(n_labels), ptr(rects), ptr(rlabels), cap, C.byref(n_rects)),
          "tt_postprocess")
    return dict(n_labels=n_labels.value, labels=labels, stats=stats[: n_labels.value].copy(),
                rects=[_rect_tuple(r) for r in rects[: n_rects.value]],
                rect_labels=rlabels[: n_rects.value].copy())


def crop_resize(image: np.ndarray, rects_xywh, angles=None) -> np.ndarray:
    """Batched crop + 128x32 bilinear resize on the GPU -> uint8 [n, 32, 128, 3].  angles: None, or one angle per rect
    from {0, 90, 180, 270}: the crop is turned that many degrees counter-clockwise before the resize
    (tt_crop_resize_rotated, cv2.resize(cv2.rotate(roi, code), (128, 32)))."""
    r = np.ascontiguousarray(np.asarray(rects_xywh, np.int32).reshape(-1, 4))
    out = np.empty((len(r), 32, 128, 3), np.uint8)
    im = _native.image_struct(image)
    if angles is None:
        check(lib().tt_crop_resize(C.byref(im), ptr(r), len(r), ptr(out)), "tt_crop_resize")
    else:
        a = np.ascontiguousarray(np.asarray(angles, np.int32).reshape(-1))
        if len(a) != len(r):
            raise ValueError(f"crop_resize: {len(r)} rects but {len(a)} angles")
        check(lib().tt_crop_resize_rotated(C.byref(im), ptr(r), ptr(a), len(r), ptr(out)), "tt_crop_resize_rotated")
    return out


def contrast_adjust(crops, adjust_contrast: float = 0.5):
    """The contrast stretch of the contrast re-read (tt_contrast_adjust, INTEGRATION.md section 10) on the GPU.  crops:
    uint8 [n, 32, 128, 3] (crop_resize's output) -> (uint8 [n, 32, 128, 3], stretched bool [n]): each crop whose grey
    contrast is below adjust_contrast stretched by EasyOCR's adjust_contrast_grey map on all three channels, the rest
    unchanged."""
    x = np.ascontiguousarray(crops, np.uint8)
    if x.ndim != 4 or x.shape[1:] != (32, 128, 3):
        raise ValueError(f"contrast_adjust: expected crops of shape (n, 32, 128, 3), got {x.shape}")
    out = np.empty_like(x)
    flags = np.empty(len(x), np.int32)
    check(lib().tt_contrast_adjust(ptr(x), len(x), float(adjust_contrast), ptr(out), ptr(flags)), "tt_contrast_adjust")
    return out, flags.astype(bool)


def rect_to_quad(rect) -> np.ndarray:
    """The quadrilateral tt_config.rectify warps for a RotatedRect: float32 [4, 2] (tl, tr, br, bl)."""
    out = np.zeros(8, np.float32)
    check(lib().tt_rect_to_quad(ptr(_rect_array(rect)), ptr(out)), "tt_rect_to_quad")
    return out.reshape(4, 2)


def crop_warp(image: np.ndarray, quads) -> np.ndarray:
    """Rectified crops on the GPU (cv2.getPerspectiveTransform + cv2.warpPerspective semantics) -> uint8 [n, 32, 128, 3]."""
    q = np.ascontiguousarray(np.asarray(quads, np.float32).reshape(-1, 8))
    out = np.empty((len(q), 32, 128, 3), np.uint8)
    im = _native.image_struct(image)
    check(lib().tt_crop_warp(C.byref(im), ptr(q), len(q), ptr(out)), "tt_crop_warp")
    return out


# --------------------------------------------------------------------------------- engine
class Engine:
    """Weights resident on the GPU(s) + streams + workspaces (tt_engine_*)."""

    def __init__(self, weights_dir: str, devices=None, cfg: _native.tt_config | None = None):
        """devices: list of CUDA device indices, "all", or None (= the TT_DEVICES environment variable, else device 0)."""
        self._h = C.c_void_p()
        dev = None
        n = 0
        if isinstance(devices, str) and devices == "all":
            devices = list(range(lib().tt_device_count()))
        if devices is not None:
            n = len(devices)
            dev = (C.c_int * n)(*devices)
        check(lib().tt_engine_create(str(weights_dir).encode(), dev, n, C.byref(cfg) if cfg is not None else None,
                                     C.byref(self._h)), "tt_engine_create")

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().tt_engine_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close

    def ocr_pages(self, images: list, score_override: list | None = None, detect_only: bool = False,
                  scores: bool = False, *, allowlist=None, blocklist=None, rotation_info=None,
                  lexicon=None, contrast_ths: float = 0.0, adjust_contrast: float = 0.5) -> list[list[dict]]:
        """images: uint8 [H,W,3] numpy arrays (host) or torch CUDA tensors (already on the device).
        score_override: optional per-page float32 [h32/2, w32/2, 2] maps (numpy or CUDA tensors, or
        None entries) that replace CRAFT's output after CRAFT has run (benchmark / parity tests).
        scores: every item also carries conf (word confidence 0..1, None when not recognised), det_score (the
        detection score of its box) and char_conf (one probability per character of text); see tt_item_scores.
        allowlist / blocklist: character filters (tt_char_filter): recognition only produces characters in
        allowlist and not in blocklist.  Each is None, a str for every page, or a list with one str or None per page.
        rotation_info: an iterable of angles from {90, 180, 270}: each word is also read turned
        that many degrees counter-clockwise and the candidate with the highest word confidence wins; every item then
        carries "angle" (0, 90, 180 or 270; -1 when not recognised).  An empty iterable reads every word upright.
        lexicon: every recognised word is one of a word list (INTEGRATION.md section 9): a Lexicon or an iterable of
        str for every page, or a list with one Lexicon or None per page (None: the page decodes as without lexicon).
        contrast_ths / adjust_contrast: a word whose confidence is below contrast_ths and whose crop's contrast is below
        adjust_contrast is read again from a contrast-stretched crop and the more confident read is kept (INTEGRATION.md
        section 10; 0 = off, EasyOCR's readtext uses 0.1 and 0.5)."""
        n = len(images)
        on_dev = n > 0 and not isinstance(images[0], np.ndarray)
        if on_dev:
            structs = [_native.tt_image(t.data_ptr(), t.shape[0], t.shape[1], t.shape[2], t.stride(0)) for t in images]
        else:
            structs = [_native.image_struct(im) for im in images]
        arr = (_native.tt_image * n)(*structs)
        if n and any(isinstance(im, np.ndarray) == on_dev for im in images):
            raise TuataraError("ocr_pages: host and device pages cannot be mixed in one call")
        opt = _native.tt_ocr_options(int(on_dev), 0, None, int(detect_only), int(scores))
        keep = []
        if score_override is not None:
            ov_dev = any(m is not None and not isinstance(m, np.ndarray) for m in score_override)
            ptrs = (C.c_void_p * n)()
            for i, m in enumerate(score_override):
                if m is None:
                    ptrs[i] = None
                    continue
                if isinstance(m, np.ndarray):
                    m = np.ascontiguousarray(m, np.float32)
                keep.append(m)
                ptrs[i] = ptr(m)
            opt.override_on_device = int(ov_dev)
            opt.score_override = ptrs
        res = C.POINTER(_native.tt_result)()
        filters = _filters(allowlist, blocklist, n)
        rot = None if rotation_info is None else _rotations(rotation_info)
        lex = _lexicon_arg(lexicon, n, strict=True)
        if contrast_ths != 0.0 or adjust_contrast != 0.5:
            handles = None if lex is None else (C.c_void_p * len(lex))(*[None if x is None else x._h.value for x in lex])
            check(lib().tt_ocr_pages_contrast(self._h, arr, n, C.byref(opt), filters or None, len(filters) if filters else 0,
                                              rot, len(rot) if rot is not None else 0, handles, len(lex) if lex else 0,
                                              float(contrast_ths), float(adjust_contrast), C.byref(res)),
                  "tt_ocr_pages_contrast")
        elif lex is None:
            check(lib().tt_ocr_pages_oriented(self._h, arr, n, C.byref(opt), filters or None, len(filters) if filters else 0,
                                              rot, len(rot) if rot is not None else 0, C.byref(res)), "tt_ocr_pages_oriented")
        else:
            handles = (C.c_void_p * len(lex))(*[None if x is None else x._h.value for x in lex])
            check(lib().tt_ocr_pages_lexicon(self._h, arr, n, C.byref(opt), filters or None, len(filters) if filters else 0,
                                             rot, len(rot) if rot is not None else 0, handles, len(lex), C.byref(res)),
                  "tt_ocr_pages_lexicon")
        try:
            out = []
            for p in range(res.contents.n_pages):
                page = res.contents.pages[p]
                out.append([dict(text=page.items[i].text.decode("latin-1"), bbox=[float(v) for v in page.items[i].bbox])
                            for i in range(page.n_items)])
                if scores:
                    for i, item in enumerate(out[-1]):
                        item.update(_item_scores(res, p, i))
                if rot is not None:
                    for i, item in enumerate(out[-1]):
                        item["angle"] = _item_angle(res, p, i) if len(rot) else (-1 if detect_only else 0)
            return out
        finally:
            lib().tt_result_free(res)

    def craft_forward(self, craft_input: np.ndarray) -> np.ndarray:
        """craft_input: uint8 [h32, w32, 3] from preprocess() -> float32 [h32/2, w32/2, 2]."""
        x = np.ascontiguousarray(craft_input, np.uint8)
        h32, w32, _ = x.shape
        out = np.empty((h32 // 2, w32 // 2, 2), np.float32)
        check(lib().tt_craft_forward(self._h, ptr(x), h32, w32, ptr(out)), "tt_craft_forward")
        return out

    def craft_tap(self, name: str) -> np.ndarray:
        """A named activation of the last craft_forward() as float32 [H, W, C] (per-slice parity tests)."""
        dims = (C.c_int * 3)()
        check(lib().tt_craft_tap(self._h, name.encode(), None, 0, dims), "tt_craft_tap")
        out = np.empty((dims[0], dims[1], dims[2]), np.float32)
        check(lib().tt_craft_tap(self._h, name.encode(), ptr(out), out.size, dims), "tt_craft_tap")
        return out

    def parseq_forward_scores(self, crops_u8: np.ndarray, class_masks: np.ndarray | None = None):
        """crops_u8: uint8 [n, 32, 128, 3] -> (ids int32 [n, 26], pmax float32 [n, 26]): parseq_forward's ids and the
        largest softmax probability of the refinement logits at each position.  class_masks: as in parseq_forward
        (pmax is then renormalised over each crop's allowed classes)."""
        x = np.ascontiguousarray(crops_u8, np.uint8)
        n = x.shape[0]
        ids = np.empty((n, 26), np.int32)
        pmax = np.empty((n, 26), np.float32)
        if class_masks is None:
            check(lib().tt_parseq_forward_scores(self._h, ptr(x), n, ptr(ids), ptr(pmax)), "tt_parseq_forward_scores")
        else:
            m = _class_masks(class_masks, n)
            check(lib().tt_parseq_forward_masked(self._h, ptr(x), n, None, ptr(m), None, ptr(ids), ptr(pmax)),
                  "tt_parseq_forward_masked")
        return ids, pmax

    def parseq_forward(self, crops_u8: np.ndarray, forced_tokens: np.ndarray | None = None,
                       class_masks: np.ndarray | None = None):
        """crops_u8: uint8 [n, 32, 128, 3] -> (logits float32 [n, 26, 95], ids int32 [n, 26]).
        class_masks: uint32 [n, 4] per-crop class masks (char_filter_mask): every greedy choice runs over the crop's
        allowed classes (tt_parseq_forward_masked); the logits stay unmasked."""
        x = np.ascontiguousarray(crops_u8, np.uint8)
        n = x.shape[0]
        logits = np.empty((n, 26, 95), np.float32)
        ids = np.empty((n, 26), np.int32)
        ft = None if forced_tokens is None else np.ascontiguousarray(forced_tokens, np.int32)
        if class_masks is None:
            check(lib().tt_parseq_forward(self._h, ptr(x), n, ptr(ft), ptr(logits), ptr(ids)), "tt_parseq_forward")
        else:
            m = _class_masks(class_masks, n)
            check(lib().tt_parseq_forward_masked(self._h, ptr(x), n, ptr(ft), ptr(m), ptr(logits), ptr(ids), None),
                  "tt_parseq_forward_masked")
        return logits, ids

    def parseq_forward_lexicon(self, crops_u8: np.ndarray, lexicon: Lexicon, forced_tokens: np.ndarray | None = None):
        """parseq_forward with every crop walking one lexicon's trie (tt_parseq_forward_lexicon)
        -> (logits float32 [n, 26, 95], ids int32 [n, 26], pmax float32 [n, 26])."""
        x = np.ascontiguousarray(crops_u8, np.uint8)
        n = x.shape[0]
        logits = np.empty((n, 26, 95), np.float32)
        ids = np.empty((n, 26), np.int32)
        pmax = np.empty((n, 26), np.float32)
        ft = None if forced_tokens is None else np.ascontiguousarray(forced_tokens, np.int32)
        check(lib().tt_parseq_forward_lexicon(self._h, ptr(x), n, ptr(ft), lexicon._h, ptr(logits), ptr(ids), ptr(pmax)),
              "tt_parseq_forward_lexicon")
        return logits, ids, pmax


def _class_masks(class_masks, n: int) -> np.ndarray:
    m = np.ascontiguousarray(class_masks, np.uint32)
    if m.shape != (n, 4):
        raise ValueError(f"class_masks: expected shape ({n}, 4), got {m.shape}")
    return m


def _rotations(rotation_info):
    """rotation_info keyword -> an int32 ctypes array (the values are checked by tt_ocr_pages_oriented)."""
    if isinstance(rotation_info, (str, bytes)) or not hasattr(rotation_info, "__iter__"):
        raise TypeError("rotation_info: expected an iterable of ints from {90, 180, 270}")
    vals = list(rotation_info)
    if not all(isinstance(v, (int, np.integer)) and not isinstance(v, bool) for v in vals):
        raise TypeError(f"rotation_info: expected ints, got {vals!r}")
    return (C.c_int * len(vals))(*[int(v) for v in vals])


def _item_angle(res, page: int, item: int) -> int:
    a = C.c_int()
    check(lib().tt_item_angle(res, page, item, C.byref(a)), "tt_item_angle")
    return a.value


def _item_scores(res, page: int, item: int) -> dict:
    conf, det = C.c_float(), C.c_float()
    cc, n = C.POINTER(C.c_float)(), C.c_int()
    check(lib().tt_item_scores(res, page, item, C.byref(conf), C.byref(det), C.byref(cc), C.byref(n)), "tt_item_scores")
    return dict(conf=None if conf.value < 0 else conf.value, det_score=det.value,
                char_conf=[cc[k] for k in range(n.value)])


_engines: dict = {}


def _engine_for(weights_dir: str) -> Engine:
    key = str(weights_dir)
    if key not in _engines:
        import os
        # like include/tuatara.h: TT_DEVICES when set, else every visible GPU
        _engines[key] = Engine(key, devices=None if os.environ.get("TT_DEVICES") else "all")
    return _engines[key]


def image_to_data(image: np.ndarray, weights_dir: str, outputs_dir: str, *, allowlist: str | None = None,
                  blocklist: str | None = None, rotation_info=None, lexicon=None, contrast_ths: float = 0.0,
                  adjust_contrast: float = 0.5) -> list[dict]:
    """Same call as the reference's ``pytuatara.image_to_data`` (bindings/python.cpp:43-57):
    uint8 [H, W, 3] in, list of ``dict(text=str, bbox=[4 floats])`` out.  Empty directory
    strings print to stderr and return [] like tuatara.cpp:315-323.  allowlist / blocklist: recognition only produces
    characters in allowlist and not in blocklist (INTEGRATION.md section 7).  rotation_info: angles from {90, 180, 270}
    at which each word is also read; items then carry "angle" (INTEGRATION.md section 8).  lexicon: a Lexicon or an
    iterable of str; every recognised word is one of its words (INTEGRATION.md section 9).  contrast_ths /
    adjust_contrast: low-confidence words on low-contrast crops are read again from a stretched crop (INTEGRATION.md
    section 10; 0 = off)."""
    return _one_page(image, weights_dir, outputs_dir, allowlist=allowlist, blocklist=blocklist,
                     rotation_info=rotation_info, lexicon=lexicon, contrast_ths=contrast_ths,
                     adjust_contrast=adjust_contrast)


def images_to_data(images: list[np.ndarray], weights_dir: str, outputs_dir: str = ".", *, allowlist=None,
                   blocklist=None, rotation_info=None, lexicon=None, contrast_ths: float = 0.0,
                   adjust_contrast: float = 0.5) -> list[list[dict]]:
    """Additive batch API: one call, many pages (sharded over the engine's GPUs).  allowlist / blocklist: None, a str
    for every page, or a list with one str or None per page.  lexicon: a Lexicon or an iterable of str for every page,
    or a list with one entry per page, each None, a Lexicon or an iterable of str."""
    images = list(images)
    return _engine_for(weights_dir).ocr_pages(images, allowlist=allowlist, blocklist=blocklist,
                                              rotation_info=rotation_info,
                                              lexicon=_engine_lexicon(lexicon, len(images)), contrast_ths=contrast_ths,
                                              adjust_contrast=adjust_contrast)


def image_to_data_scored(image: np.ndarray, weights_dir: str, outputs_dir: str, *, allowlist: str | None = None,
                         blocklist: str | None = None, rotation_info=None, lexicon=None, contrast_ths: float = 0.0,
                         adjust_contrast: float = 0.5) -> list[dict]:
    """image_to_data whose items also carry ``conf`` (word confidence 0..1), ``det_score`` (the detection score of the
    box) and ``char_conf`` (one probability per character of ``text``).  Same inputs, errors and soft failures;
    ``text`` and ``bbox`` are what image_to_data returns."""
    return _one_page(image, weights_dir, outputs_dir, scores=True, allowlist=allowlist, blocklist=blocklist,
                     rotation_info=rotation_info, lexicon=lexicon, contrast_ths=contrast_ths,
                     adjust_contrast=adjust_contrast)


def images_to_data_scored(images: list[np.ndarray], weights_dir: str, outputs_dir: str = ".", *, allowlist=None,
                          blocklist=None, rotation_info=None, lexicon=None, contrast_ths: float = 0.0,
                          adjust_contrast: float = 0.5) -> list[list[dict]]:
    """Batch variant of image_to_data_scored."""
    images = list(images)
    return _engine_for(weights_dir).ocr_pages(images, scores=True, allowlist=allowlist, blocklist=blocklist,
                                              rotation_info=rotation_info,
                                              lexicon=_engine_lexicon(lexicon, len(images)), contrast_ths=contrast_ths,
                                              adjust_contrast=adjust_contrast)


def _one_page(image: np.ndarray, weights_dir: str, outputs_dir: str, **kw) -> list[dict]:
    """image_to_data and image_to_data_scored: empty directory strings print to stderr and return [] like
    tuatara.cpp:315-323; else the page's items from Engine.ocr_pages(**kw)."""
    import sys

    if not weights_dir:
        print("Please provide a value for weights_dir", file=sys.stderr)
        return []
    if not outputs_dir:
        print("Please provide a value for outputs_dir", file=sys.stderr)
        return []
    if image.ndim != 3:
        raise RuntimeError("Input array should have 3 dimensions")
    kw["lexicon"] = _engine_lexicon(kw.get("lexicon"), 1)
    return _engine_for(weights_dir).ocr_pages([image], **kw)[0]
