"""ctypes binding of tests/lcd_oracle.c, the CPU restatement of the loop-closure candidates and word weights.

The C source is compiled on first use with the flags of oracle/Makefile's pinned build into a per-user directory
under the system's temporary directory (the tree may be read-only), keyed on the source's hash."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lcd_oracle.c")
FLAGS = ["-std=gnu11", "-O2", "-fwrapv", "-ffp-contract=off", "-fPIC", "-shared"]
_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    src = open(SRC, "rb").read()
    tag = hashlib.sha256(src + " ".join(FLAGS).encode()).hexdigest()[:16]
    d = os.path.join(tempfile.gettempdir(), "mv_lcd_oracle_%d" % os.getuid())
    os.makedirs(d, exist_ok=True)
    so = os.path.join(d, "liblcd_oracle_%s.so" % tag)
    if not os.path.exists(so):
        tmp = "%s.%d.tmp" % (so, os.getpid())
        subprocess.run(["gcc"] + FLAGS + ["-o", tmp, SRC, "-lm"], check=True, capture_output=True)
        os.replace(tmp, so)
    L = C.CDLL(so)
    vp, i32 = C.c_void_p, C.c_int
    L.orc_lcd_candidates.argtypes = [i32, i32, i32, i32, vp, vp, vp, i32, i32, i32, vp, vp]
    L.orc_lcd_candidates.restype = None
    L.orc_lcd_word_weights.argtypes = [i32, i32, i32, vp, vp, vp]
    L.orc_lcd_word_weights.restype = None
    _lib = L
    return L


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def candidates(word, q_count, n_words, weight, min_gap, k, min_score, first_frame):
    """-> (cand int32 [n, k], score int32 [n, k]), mv_loop_candidates' outputs."""
    word = np.ascontiguousarray(word, np.int32)
    q_count = np.ascontiguousarray(q_count, np.int32)
    weight = None if weight is None else np.ascontiguousarray(weight, np.int8)
    n, top_n = word.shape
    cand = np.zeros((n, k), np.int32)
    score = np.zeros((n, k), np.int32)
    load().orc_lcd_candidates(n, first_frame, top_n, n_words, _p(word), _p(q_count), _p(weight), min_gap, k,
                              min_score, _p(cand), _p(score))
    return cand, score


def word_weights(word, q_count, n_words):
    """-> int8 [n_words], mv_lcd_word_weights' output."""
    word = np.ascontiguousarray(word, np.int32)
    q_count = np.ascontiguousarray(q_count, np.int32)
    n, top_n = word.shape
    out = np.zeros(n_words, np.int8)
    load().orc_lcd_word_weights(n, top_n, n_words, _p(word), _p(q_count), _p(out))
    return out
