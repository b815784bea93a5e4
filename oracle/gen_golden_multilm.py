"""TEST INFRASTRUCTURE ONLY (build container only: needs /root/reference).

MultiLanguageModel goldens: the UNMODIFIED reference's BeamSearchDecoderCTC over a MultiLanguageModel
(language_model.py:455-502; its own test: tests/test_decoder.py:386-401) on seeded inputs
-> tests/golden/multilm_cases.json (+ multilm_arrays.npz).

    python oracle/gen_golden_multilm.py
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

import kenlm  # noqa: E402  (the stand-in of oracle/refshim)
from pyctcdecode import BeamSearchDecoderCTC, LanguageModel  # noqa: E402  (the reference)
from pyctcdecode.language_model import MultiLanguageModel  # noqa: E402
from pyctcdecode.alphabet import Alphabet  # noqa: E402

from tests import goldens, synth  # noqa: E402

REF_TESTS = "/root/reference/pyctcdecode/tests"
OUT = os.path.join(ROOT, "tests", "golden")


def beams_json(beams):
    return [{"text": b.text, "frames": [[w, int(f[0]), int(f[1])] for w, f in b.text_frames],
             "logit_score": float(b.logit_score), "lm_score": float(b.lm_score)} for b in beams]


def build_models(specs, toy):
    models = []
    for m in specs:
        if m["arpa_kind"] == "toy":
            path, words = toy, None
        else:
            wl = synth.make_workload(m["workload"])
            path, words = wl.arpa, wl.words
        unigrams = None
        if m.get("unigrams") is not None:
            unigrams = m["unigrams"]
        elif m.get("unigrams_first") is not None:
            unigrams = words[: m["unigrams_first"]]
        kw = {k: m[k] for k in ("alpha", "beta", "unk_score_offset", "score_boundary") if k in m}
        models.append(LanguageModel(kenlm.Model(path), unigrams, **kw))
    return models


def main():
    base = goldens.load_arrays(OUT)
    toy = os.path.join(REF_TESTS, "sample_data", "bugs_bunny_kenlm.arpa")
    SAMPLE_LABELS = [" ", "b", "g", "n", "s", "u", "y", ""]
    arrays, cases = {}, []

    def add(name, labels, specs, arr_name, x, split=None, stream=None, **dkw):
        dec = BeamSearchDecoderCTC(Alphabet.build_alphabet(labels), MultiLanguageModel(build_models(specs, toy)))
        case = {"name": name, "labels": labels, "models": specs, "array": arr_name, "decode": dkw}
        beams = dec.decode_beams(x, **dkw)
        case["beams"] = beams_json(beams)
        case["decode_text"] = dec.decode(x, **{k: v for k, v in dkw.items() if k != "prune_history"})
        if split is not None:      # carry the MultiLanguageModelState of the best beam into a second call
            first = dec.decode_beams(x[:split], **dkw)
            second = dec.decode_beams(x[split:], lm_start_state=first[0].last_lm_state, **dkw)
            case["split"] = split
            case["split_first"] = beams_json(first)
            case["split_second"] = beams_json(second)
        if stream is not None:     # chunked partial_decode_beams over the same models
            state_beams, cached_lm, cached_p = dec.get_starting_state()
            start, steps = 0, []
            kw = {k: v for k, v in dkw.items() if k in ("beam_width", "prune_history")}
            for i, end in enumerate(stream):
                out = dec.partial_decode_beams(x[start:end], cached_lm, cached_p, state_beams, start, is_end=(i == len(stream) - 1), **kw)
                steps.append({"start": start, "end": end, "beams": [
                    {"text": b.text, "partial_word": b.partial_word, "last_char": b.last_char,
                     "text_frames": [[int(s), int(e)] for s, e in b.text_frames],
                     "partial_frames": [int(b.partial_frames[0]), int(b.partial_frames[1])],
                     "logit_score": float(b.logit_score), "lm_score": float(b.lm_score)} for b in out]})
                state_beams, start = out, end
            case["stream"] = steps
        cases.append(case)

    # reference tests/test_decoder.py:386-401: twice the same model averages to the same result
    add("toy_twice", SAMPLE_LABELS, [dict(arpa_kind="toy"), dict(arpa_kind="toy")], "test_logits", base["test_logits"])
    add("toy_mixed_params", SAMPLE_LABELS, [dict(arpa_kind="toy", alpha=1.0, beta=0.5, unigrams=["bugs", "bunny"]),
                                           dict(arpa_kind="toy", alpha=0.2, unk_score_offset=-4.0, score_boundary=False)],
        "test_logits", base["test_logits"], split=4)
    w3 = dict(kind="char", vocab="B", n_words=300, lm_order=3)
    w2 = dict(kind="char", vocab="B", n_words=300, lm_order=2)
    w4 = dict(kind="char", vocab="B", n_words=300, lm_order=4)
    two = [dict(arpa_kind="synth", workload=w3, unigrams_first=300, alpha=0.5, beta=1.0),
           dict(arpa_kind="synth", workload=w2, unigrams_first=150, alpha=0.9, beta=0.3, unk_score_offset=-6.0)]
    three = two + [dict(arpa_kind="synth", workload=w4, alpha=0.3, beta=2.0, score_boundary=False)]
    wl = synth.make_workload(w3)
    for i, regime in enumerate(["peaky", "diffuse", "peaky", "diffuse"]):
        T = [90, 60, 120, 40][i]
        x = wl.utterance(7600 + i, T, regime)
        arrays["multi_%d" % i] = x
        dkw = dict(beam_width=[24, 100, 16, 50][i], prune_history=bool(i % 2))
        if i == 2:
            dkw.update(hotwords=[wl.words[3], wl.words[10]], hotword_weight=6.0)
        add("synth_two_%d" % i, wl.labels, two, "multi_%d" % i, x, split=(T // 2 if i < 2 else None),
            stream=([T // 3, T // 3 + 1, T] if i in (0, 3) else None), **dkw)
        if i < 2:
            add("synth_three_%d" % i, wl.labels, three, "multi_%d" % i, x, **dkw)

    np.savez_compressed(os.path.join(OUT, "multilm_arrays.npz"), **arrays)
    with open(os.path.join(OUT, "multilm_cases.json"), "w", encoding="utf-8") as fh:
        json.dump({"cases": cases, "generator": "oracle/gen_golden_multilm.py",
                   "reference": "pyctcdecode 0.6.0 MultiLanguageModel, numpy %s" % np.__version__}, fh, ensure_ascii=False, indent=0)
    print("wrote %d MultiLanguageModel cases" % len(cases))


if __name__ == "__main__":
    main()
