"""Reference scores for the tests of tt_ocr_options.with_scores (INTEGRATION.md section 6), computed from what the oracle
already keeps of a run (oracle/tuatara_ref.py's Stages): the PARSeq logits and the CCL labels with the normalised text
map.  Not reference behaviour: the reference drops the probabilities at tuatara.cpp:101-106."""
import math

import numpy as np
import torch

from oracle import tuatara_ref as R


def word_scores(probs: np.ndarray, ids: np.ndarray, eos_id: int = 88):
    """The scores of one crop from the max / argmax of the softmax at its 26 positions.  End position e = the first
    position of id 0 (itos[0] = ']', where the decoded text is cut, tuatara.cpp:497-502), else the last;
    conf = prod(probs[0..e]) in double, rounded once to float32; char_conf = probs of the positions that produce a
    character of the text: before the first id 0 (every position when there is none) and id != eos_id."""
    zero = np.flatnonzero(ids == 0)
    e = int(zero[0]) if len(zero) else len(ids) - 1
    conf = float(np.float32(math.prod(float(x) for x in probs[:e + 1])))
    stop = e if len(zero) else len(ids)
    char_conf = [float(probs[t]) for t in range(stop) if int(ids[t]) != eos_id]
    return conf, char_conf


def image_to_data_scored(image: np.ndarray, craft_model, parseq_model, stages: R.Stages | None = None, **kw):
    """R.image_to_data, and per item conf / char_conf from the softmax the reference takes (tuatara.cpp:486) and
    det_score = maxVal of the item's component (tuatara.cpp:151-152), as the oracle computes it."""
    st = stages if stages is not None else R.Stages()
    out = R.image_to_data(image, craft_model, parseq_model, stages=st, **kw)
    if not out:
        return out
    probs, ids = torch.softmax(torch.from_numpy(st.logits), -1).max(-1)   # the tokenizer's max (:101-106)
    dbg = st.det_debug
    eos_id = R.Tokenizer().eos_id
    for i, item in enumerate(out):
        item["conf"], item["char_conf"] = word_scores(probs[i].numpy(), ids[i].numpy(), eos_id)
        k = dbg.mapper[i]   # the component of box i
        item["det_score"] = float(np.float32(dbg.text_norm[dbg.labels == k].max()))
    return out
