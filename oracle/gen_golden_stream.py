"""TEST INFRASTRUCTURE ONLY (build container only: needs /root/reference).

Streaming goldens: runs the UNMODIFIED reference's get_starting_state / partial_decode_beams
(decoder.py:669-728, exercised by its tests/test_decoder.py:515-698) chunk by chunk and records
the LMBeam list every call returns -> tests/golden/stream_cases.json (+ stream_arrays.npz for
inputs that are not in arrays.npz).  The GPU box has no /root/reference; the parity tests read
these committed vectors.

    python oracle/gen_golden_stream.py
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, "refshim"))
sys.path.insert(0, "/root/reference")
sys.path.insert(0, ROOT)

import logging  # noqa: E402

logging.disable(logging.CRITICAL)

from pyctcdecode import build_ctcdecoder  # noqa: E402  (the reference)
from pyctcdecode.language_model import HotwordScorer  # noqa: E402

from tests import goldens, synth  # noqa: E402

REF_TESTS = "/root/reference/pyctcdecode/tests"
OUT = os.path.join(ROOT, "tests", "golden")


def beams_json(beams):
    return [{"text": b.text, "next_word": b.next_word, "partial_word": b.partial_word, "last_char": b.last_char,
             "text_frames": [[int(s), int(e)] for s, e in b.text_frames],
             "partial_frames": [int(b.partial_frames[0]), int(b.partial_frames[1])],
             "logit_score": float(b.logit_score), "lm_score": float(b.lm_score)} for b in beams]


def main():
    base = goldens.load_arrays(OUT)
    extra, cases = {}, []
    toy = os.path.join(REF_TESTS, "sample_data", "bugs_bunny_kenlm.arpa")
    SAMPLE_LABELS = [" ", "b", "g", "n", "s", "u", "y", ""]
    bpe_labels = ["▁bugs", "▁bun", "ny", ""]
    libri_bpe_labels = ["▁⁇▁", "▁"] + ["##" + c for c in synth.LIBRI_LABELS[1:]]

    def run(name, labels, arr_name, x, bounds, lm=None, calls=None, **common):
        """bounds: chunk end indices; calls: per-chunk overrides (hotwords, hotword_weight, force_next_word)."""
        kw = {}
        if lm is not None:
            kw = {k: v for k, v in lm.items() if k not in ("arpa_kind", "workload")}
            if lm["arpa_kind"] == "toy":
                kw["kenlm_model_path"] = toy
        dec = build_ctcdecoder(labels, **kw)
        beams, cached_lm, cached_p = dec.get_starting_state()
        start, steps = 0, []
        for i, end in enumerate(bounds):
            c = dict((calls or {}).get(i, {}))
            hot = c.get("hotwords")
            scorer = HotwordScorer.build_scorer(hot, weight=c.get("hotword_weight", 10.0)) if hot is not None else None
            is_end = i == len(bounds) - 1
            out = dec.partial_decode_beams(x[start:end], cached_lm, cached_p, beams, start, hotword_scorer=scorer,
                                           force_next_word=bool(c.get("force_next_word", False)), is_end=is_end, **common)
            steps.append({"start": start, "end": end, "call": c, "is_end": is_end, "beams": beams_json(out)})
            beams, start = out, end
        lm_json = None if lm is None else {k: (list(v) if k == "unigrams" and v is not None else v)
                                           for k, v in lm.items() if k != "kenlm_model_path"}
        cases.append({"name": name, "labels": labels, "array": arr_name, "lm": lm_json, "common": common, "steps": steps})

    tl = base["test_logits"]
    toy_lm = dict(arpa_kind="toy")
    # reference tests/test_decoder.py:515-584 (test_partial_decode, test_partial_decode_with_lm)
    run("test_logits_nolm", SAMPLE_LABELS, "test_logits", tl, [3, 8, len(tl)])
    run("test_logits_lm", SAMPLE_LABELS, "test_logits", tl, [3, 8, len(tl)], toy_lm)
    run("test_logits_lm_unigrams", SAMPLE_LABELS, "test_logits", tl, [1, 2, 5, 9, len(tl)], dict(toy_lm, unigrams=["bugs", "bunny"]))
    run("test_logits_whole", SAMPLE_LABELS, "test_logits", tl, [len(tl)], toy_lm)
    # :586-618 hotwords, :620-698 different scorers per chunk
    hb = {i: dict(hotwords=["bugs"], hotword_weight=25.0) for i in range(3)}
    run("test_logits_hot", SAMPLE_LABELS, "test_logits", tl, [3, 8, len(tl)], calls=hb)
    run("test_logits_hot_switch", SAMPLE_LABELS, "test_logits", tl, [3, 8, len(tl)],
        calls={0: dict(hotwords=["bugs"], hotword_weight=15.0), 1: dict(hotwords=["bunny"], hotword_weight=15.0), 2: {}})
    run("test_logits_hot_switch2", SAMPLE_LABELS, "test_logits", tl, [3, 8, len(tl)],
        calls={0: dict(hotwords=["bugs"], hotword_weight=15.0), 1: dict(hotwords=["bugs"], hotword_weight=15.0),
               2: dict(hotwords=["bunny"], hotword_weight=15.0)})
    run("test_logits_force", SAMPLE_LABELS, "test_logits", tl, [5, 9, len(tl)], toy_lm, calls={0: dict(force_next_word=True)})
    run("bpe_frames", bpe_labels, "bpe_frames", base["bpe_frames"], [2, 4, 6])
    libri = base["libri"]
    b50 = list(range(50, len(libri), 50)) + [len(libri)]
    run("libri_50", synth.LIBRI_LABELS, "libri", libri, b50)
    run("libri_50_history_beam20", synth.LIBRI_LABELS, "libri", libri, b50, beam_width=20, prune_history=True)
    run("libri_ragged_force", synth.LIBRI_LABELS, "libri", libri, [7, 8, 100, 101, 250, len(libri)],
        calls={2: dict(force_next_word=True)}, beam_width=30)
    run("libri_bpe_64", libri_bpe_labels, "libri_bpe", base["libri_bpe"], list(range(64, len(libri), 64)) + [len(libri)], beam_width=25)
    run("libri_hot", synth.LIBRI_LABELS, "libri", libri, b50, calls={i: dict(hotwords=["goodeal", "set my"], hotword_weight=8.0) for i in range(len(b50))},
        beam_width=40)
    # seeded synthetic with n-gram models
    fams = {
        "B_3gram": (dict(kind="char", vocab="B", n_words=300, lm_order=3), dict(alpha=0.5, beta=1.0)),
        "A_2gram": (dict(kind="char", vocab="A", n_words=300, lm_order=2), dict()),
        "C_bpe_4gram": (dict(kind="bpe", n_words=300, lm_order=4), dict(alpha=0.7, beta=2.0)),
        "B_nolm": (dict(kind="char", vocab="B", n_words=300, lm_order=0), {}),
    }
    for fam, (wkw, lmkw) in fams.items():
        wl = synth.make_workload(wkw)
        for i, regime in enumerate(["peaky", "diffuse"]):
            T = 120 if wl.V <= 64 else 48
            x = wl.utterance(7100 + i, T, regime)
            name = "stream_%s_%d" % (fam, i)
            extra[name] = x
            lm = dict(lmkw, arpa_kind="synth", workload=wkw, kenlm_model_path=wl.arpa, unigrams=wl.words) if wl.arpa else None
            step = 37 if wl.V <= 64 else 13
            bounds = list(range(step, T, step)) + [T]
            calls = {1: dict(force_next_word=True)} if i == 1 else {}
            if i == 0:
                calls = {j: dict(hotwords=[wl.words[3], wl.words[10]], hotword_weight=6.0) for j in range(len(bounds))}
            run(name, wl.labels, name, x, bounds, lm, calls=calls, beam_width=[24, 100][i], prune_history=bool(i))

    np.savez_compressed(os.path.join(OUT, "stream_arrays.npz"), **extra)
    with open(os.path.join(OUT, "stream_cases.json"), "w", encoding="utf-8") as fh:
        json.dump({"cases": cases, "generator": "oracle/gen_golden_stream.py",
                   "reference": "pyctcdecode 0.6.0 partial_decode_beams, numpy %s" % np.__version__}, fh, ensure_ascii=False, indent=0)
    print("wrote %d streaming cases (%d calls)" % (len(cases), sum(len(c["steps"]) for c in cases)))


if __name__ == "__main__":
    main()
