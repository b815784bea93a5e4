"""TEST INFRASTRUCTURE ONLY -- ctypes front end of the CPU oracle (oracle/ctc_oracle.cpp).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module.  The product package never does.

The oracle mirrors the call shape of the reference (``pyctcdecode/decoder.py:730-945``):
``OracleDecoder.decode_beams(logits, ...)`` returns a list of
``(text, text_frames, logit_score, lm_score)`` tuples, ``decode`` the top text with history
pruning on (decoder.py:888).
"""
import ctypes as C
import os
import re
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "liboracle.so")
REF_DIR = os.path.join(_HERE, "_ref")
_lib = None


def build(force=False):
    """Compile liboracle.so with g++ (building the checker is not using it)."""
    src = os.path.join(_HERE, "ctc_oracle.cpp")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s", "-B", "liboracle.so"])
    return _LIB_PATH


def install_reference():
    """pip-install the UNMODIFIED reference package into oracle/_ref (git-ignored) for bench.py's reference arm.
    The checkout of kensho-technologies/pyctcdecode 0.6.0 is named by $PYCTCDECODE_REFERENCE; without it nothing is
    installed and bench.py times the C++ port instead.  Installed from a copy: pip builds in the source tree.
    Best effort: when the install cannot run (no pip, no setuptools, not a checkout) it warns and installs nothing,
    since the product and its tests do not need it."""
    import shutil
    import sys
    import tempfile
    src = os.environ.get("PYCTCDECODE_REFERENCE")
    if not src or os.path.isdir(os.path.join(REF_DIR, "pyctcdecode")):
        return
    if not os.path.isdir(os.path.join(src, "pyctcdecode")):
        print("oracle/_ref: PYCTCDECODE_REFERENCE=%s is not a pyctcdecode checkout; not installed" % src, file=sys.stderr)
        return
    with tempfile.TemporaryDirectory() as tmp:
        copy = os.path.join(tmp, "reference")
        shutil.copytree(src, copy, ignore=shutil.ignore_patterns(".git"))
        cmd = [sys.executable, "-m", "pip", "install", "--no-index", "--no-build-isolation", "--no-deps", "--no-cache-dir",
               "--quiet", "--target", REF_DIR, copy]
        log = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if log.returncode != 0:
        shutil.rmtree(REF_DIR, ignore_errors=True)       # no partial install for bench.py to find
        print("oracle/_ref: installing the reference failed, bench.py times the C++ port:\n" + log.stdout[-2000:],
              file=sys.stderr)


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        L = C.CDLL(_LIB_PATH)
        vp, cp, i32, f64 = C.c_void_p, C.c_char_p, C.c_int, C.c_double
        L.orc_lm_load.restype = vp
        L.orc_lm_load.argtypes = [cp]
        L.orc_lm_free.argtypes = [vp]
        L.orc_lm_order.argtypes = [vp]
        L.orc_lm_contains.argtypes = [vp, cp]
        L.orc_state_new.restype = vp
        L.orc_state_new.argtypes = [vp, i32]
        L.orc_state_empty.restype = vp
        L.orc_state_free.argtypes = [vp]
        L.orc_state_len.argtypes = [vp]
        L.orc_state_get.argtypes = [vp, C.POINTER(C.c_uint32), C.POINTER(C.c_float)]
        L.orc_base_score.restype = C.c_float
        L.orc_base_score.argtypes = [vp, vp, cp, vp]
        L.orc_decoder_new.restype = vp
        L.orc_decoder_new.argtypes = [C.POINTER(cp), i32, i32, vp, C.POINTER(cp), i32, f64, f64, f64, i32]
        L.orc_decoder_free.argtypes = [vp]
        L.orc_decoder_set_params.argtypes = [vp, f64, f64, f64, i32]
        L.orc_decode.restype = vp
        L.orc_decode.argtypes = [vp, vp, i32, i32, i32, i32, f64, f64, i32, C.POINTER(cp), i32, f64, vp]
        L.orc_decode_batch.argtypes = [vp, C.POINTER(vp), C.POINTER(i32), i32, i32, i32, i32, f64, f64, i32,
                                       C.POINTER(cp), i32, f64, i32, C.POINTER(vp)]
        L.orc_result_free.argtypes = [vp]
        L.orc_result_nbeams.argtypes = [vp]
        L.orc_result_text.restype = cp
        L.orc_result_text.argtypes = [vp, i32]
        L.orc_result_logit.restype = f64
        L.orc_result_logit.argtypes = [vp, i32]
        L.orc_result_lm.restype = f64
        L.orc_result_lm.argtypes = [vp, i32]
        L.orc_result_nwords.argtypes = [vp, i32]
        L.orc_result_word.restype = cp
        L.orc_result_word.argtypes = [vp, i32, i32]
        L.orc_result_frames.restype = C.POINTER(i32)
        L.orc_result_frames.argtypes = [vp, i32]
        L.orc_result_state.restype = vp
        L.orc_result_state.argtypes = [vp, i32]
        L.orc_token_order.argtypes = [C.POINTER(i32), i32, i32, C.POINTER(i32)]
        L.orc_pairwise_sum_f32.restype = C.c_float
        L.orc_pairwise_sum_f32.argtypes = [vp, C.c_long]
        L.orc_pairwise_sum_f64.restype = f64
        L.orc_pairwise_sum_f64.argtypes = [vp, C.c_long]
        L.orc_looks_like_probs.argtypes = [vp, i32, i32, i32]
        L.orc_normalise.argtypes = [vp, i32, i32, i32, vp]
        _lib = L
    return _lib


# --------------------------------------------------------------------------------------
# label normalisation, restated from reference alphabet.py:22-148 (kept local so the oracle
# does not depend on the product's host code)
# --------------------------------------------------------------------------------------
_BPE = "▁"
_UNK = "⁇"
_UNK_BPE = _BPE + _UNK + _BPE
_BLANK_PTN = re.compile(r"^[<\[]pad[>\]]$", flags=re.IGNORECASE)
_UNK_PTN = re.compile(r"^[<\[]unk[>\]]$", flags=re.IGNORECASE)
_SPECIAL_PTN = re.compile(r"^[<\[].+[>\]]$")


def normalize_labels(labels):
    labels = list(labels)
    is_bpe = any(s.startswith("##") for s in labels) or any(s.startswith(_BPE) for s in labels)
    if len(labels) != len(set(labels)):
        raise ValueError("duplicate labels")
    if is_bpe and any(" " in s for s in labels):
        raise ValueError("space in BPE vocabulary")
    out = labels[:]
    if is_bpe:
        if any(s.startswith("##") for s in labels):
            conv = []
            for tok in out:
                if tok.startswith("##"):
                    conv.append(tok[2:])
                elif _SPECIAL_PTN.match(tok) or tok in ("", _BPE, _UNK_BPE, "<unk>"):
                    conv.append(tok)
                else:
                    conv.append(_BPE + tok)
            out = conv
        out = ["" if _BLANK_PTN.match(t) else t for t in out]
        if "" not in out:
            out.append("")
        out = [_UNK_BPE if _UNK_PTN.match(t) else t for t in out]
    else:
        if "|" in out and " " not in out:
            out[out.index("|")] = " "
        out = ["" if _BLANK_PTN.match(t) else t for t in out]
        if "_" in out and "" not in out:
            out[out.index("_")] = ""
        if "" not in out:
            out.append("")
        out = [_UNK if _UNK_PTN.match(t) else t for t in out]
    return out, is_bpe


def _cstr_array(strings):
    arr = (C.c_char_p * max(1, len(strings)))()
    for i, s in enumerate(strings):
        arr[i] = s.encode("utf-8")
    return arr


class OracleNgram:
    """kenlm.Model look-alike backed by the oracle's n-gram engine."""

    def __init__(self, path):
        self.path = os.path.abspath(path).encode("utf-8")
        self._h = lib().orc_lm_load(self.path)
        if not self._h:
            raise OSError("cannot load ARPA %s" % path)
        self.order = lib().orc_lm_order(self._h)

    def __contains__(self, word):
        return bool(lib().orc_lm_contains(self._h, word.encode("utf-8")))

    def start_state(self, bos=True):
        return OracleState(lib().orc_state_new(self._h, 1 if bos else 0))

    def base_score(self, in_state, word, out_state=None):
        out_state = out_state or OracleState(lib().orc_state_empty())
        s = lib().orc_base_score(self._h, in_state._h, word.encode("utf-8"), out_state._h)
        return float(s), out_state


class OracleState:
    def __init__(self, handle):
        self._h = handle

    def __del__(self):
        if self._h and _lib is not None:
            _lib.orc_state_free(self._h)
            self._h = None

    def get(self):
        n = lib().orc_state_len(self._h)
        w = (C.c_uint32 * max(1, n))()
        b = (C.c_float * max(1, n))()
        lib().orc_state_get(self._h, w, b)
        return list(w[:n]), list(b[:n])


def _as_input(logits):
    arr = np.asarray(logits)
    if arr.dtype == np.float32:
        return np.ascontiguousarray(arr), 0
    return np.ascontiguousarray(arr, dtype=np.float64), 1


class OracleDecoder:
    def __init__(self, labels, kenlm_model_path=None, unigrams=None, alpha=0.5, beta=1.5,
                 unk_score_offset=-10.0, lm_score_boundary=True, normalized=False, is_bpe=None):
        if normalized:
            self.labels = list(labels)
            self.is_bpe = bool(is_bpe)
        else:
            self.labels, self.is_bpe = normalize_labels(labels)
        self.ngram = OracleNgram(kenlm_model_path) if kenlm_model_path else None
        if self.ngram is not None and unigrams is None and kenlm_model_path.endswith(".arpa"):
            unigrams = load_unigrams_from_arpa(kenlm_model_path)
        lab = _cstr_array(self.labels)
        if unigrams is None:
            uni, n_uni = _cstr_array([]), -1
        else:
            ulist = list(unigrams)
            uni, n_uni = _cstr_array(ulist), len(ulist)
        self._h = lib().orc_decoder_new(lab, len(self.labels), int(self.is_bpe),
                                        self.ngram._h if self.ngram else None, uni, n_uni,
                                        alpha, beta, unk_score_offset, int(lm_score_boundary))

    def reset_params(self, alpha, beta, unk_score_offset, lm_score_boundary):
        lib().orc_decoder_set_params(self._h, alpha, beta, unk_score_offset, int(lm_score_boundary))

    def _collect(self, res, with_state=False):
        L = lib()
        out = []
        for i in range(L.orc_result_nbeams(res)):
            nw = L.orc_result_nwords(res, i)
            fr = L.orc_result_frames(res, i)
            frames = [(L.orc_result_word(res, i, w).decode("utf-8"), (fr[2 * w], fr[2 * w + 1])) for w in range(nw)]
            item = (L.orc_result_text(res, i).decode("utf-8"), frames, L.orc_result_logit(res, i), L.orc_result_lm(res, i))
            if with_state:
                st = L.orc_result_state(res, i)
                item = item + (OracleState(st) if st else None,)
            out.append(item)
        L.orc_result_free(res)
        return out

    def decode_beams(self, logits, beam_width=100, beam_prune_logp=-10.0, token_min_logp=-5.0,
                     prune_history=False, hotwords=None, hotword_weight=10.0, lm_start_state=None,
                     with_state=False):
        arr, dt = _as_input(logits)
        if arr.ndim != 2 or arr.shape[1] != len(self.labels):
            raise ValueError("bad logits shape %s" % (arr.shape,))
        hot = list(hotwords or [])
        res = lib().orc_decode(self._h, arr.ctypes.data, arr.shape[0], arr.shape[1], dt, beam_width,
                               beam_prune_logp, token_min_logp, int(prune_history), _cstr_array(hot), len(hot),
                               hotword_weight, lm_start_state._h if lm_start_state is not None else None)
        if not res:
            raise ValueError("oracle decode failed")
        return self._collect(res, with_state)

    def decode(self, logits, **kw):
        kw["prune_history"] = True
        return self.decode_beams(logits, **kw)[0][0]

    def decode_beams_batch(self, logits_list, n_threads=1, beam_width=100, beam_prune_logp=-10.0,
                           token_min_logp=-5.0, prune_history=False, hotwords=None, hotword_weight=10.0):
        arrs = [_as_input(x) for x in logits_list]
        if not arrs:
            return []
        dt = arrs[0][1]
        assert all(a[1] == dt for a in arrs), "mixed dtypes"
        B = len(arrs)
        ptrs = (C.c_void_p * B)(*[a[0].ctypes.data for a in arrs])
        Ts = (C.c_int * B)(*[a[0].shape[0] for a in arrs])
        results = (C.c_void_p * B)()
        hot = list(hotwords or [])
        lib().orc_decode_batch(self._h, ptrs, Ts, B, len(self.labels), dt, beam_width, beam_prune_logp,
                               token_min_logp, int(prune_history), _cstr_array(hot), len(hot), hotword_weight,
                               n_threads, results)
        return [self._collect(results[i]) for i in range(B)]

    def decode_batch(self, logits_list, n_threads=1, **kw):
        kw["prune_history"] = True
        return [b[0][0] for b in self.decode_beams_batch(logits_list, n_threads=n_threads, **kw)]


def load_unigrams_from_arpa(path):
    """reference language_model.py:67-84"""
    unigrams = set()
    with open(path, encoding="utf-8") as fh:
        on = False
        for line in fh:
            line = line.strip()
            if line == "\\1-grams:":
                on = True
            elif line == "\\2-grams:":
                break
            if on and line:
                parts = line.split("\t")
                if len(parts) == 3:
                    unigrams.add(parts[1])
    return unigrams


def token_order(selected_sorted, argmax):
    sel = (C.c_int * max(1, len(selected_sorted)))(*selected_sorted)
    out = (C.c_int * (len(selected_sorted) + 1))()
    n = lib().orc_token_order(sel, len(selected_sorted), int(argmax), out)
    return list(out[:n])


def normalise(logits):
    arr, dt = _as_input(logits)
    out = np.empty(arr.shape, dtype=np.float64)
    lib().orc_normalise(arr.ctypes.data, arr.shape[0], arr.shape[1], dt, out.ctypes.data)
    return out


def looks_like_probs(logits):
    arr, dt = _as_input(logits)
    return bool(lib().orc_looks_like_probs(arr.ctypes.data, arr.shape[0], arr.shape[1], dt))
