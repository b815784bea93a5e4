"""TEST INFRASTRUCTURE ONLY (build container only: needs /root/reference).

Generates tests/golden/{cases.json,arrays.npz,arrays_large.npz} by running the UNMODIFIED reference
(/root/reference/pyctcdecode, imported with the kenlm / pygtrie stand-ins of oracle/refshim)
on (a) the reference's own test fixtures (tests/test_decoder.py:186-223, sample_data/) and
(b) small seeded synthetic utterances (tests/synth.py).  The GPU box has no /root/reference,
so the parity tests read these committed vectors instead.

    python oracle/gen_golden.py
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
from pyctcdecode.alphabet import Alphabet  # noqa: E402

from tests import goldens, synth  # noqa: E402

REF_TESTS = "/root/reference/pyctcdecode/tests"
OUT = os.path.join(ROOT, "tests", "golden")


def beams_to_json(beams):
    return [{"text": b.text, "frames": [[w, int(f[0]), int(f[1])] for w, f in b.text_frames],
             "logit_score": float(b.logit_score), "lm_score": float(b.lm_score)} for b in beams]


def main():
    os.makedirs(OUT, exist_ok=True)
    arrays, cases = {}, []
    toy_arpa = open(os.path.join(REF_TESTS, "sample_data", "bugs_bunny_kenlm.arpa")).read()
    SAMPLE_LABELS = [" ", "b", "g", "n", "s", "u", "y", ""]
    vocab = {c: n for n, c in enumerate(SAMPLE_LABELS)}

    def onehot(chars, voc=vocab):
        m = np.zeros((len(chars), len(voc)))
        for i, c in enumerate(chars):
            m[i][voc[c]] = 1
        return m

    bugs, bunny = onehot("bugs"), onehot(["b", "u", "n", "", "n", "y"])
    blank, space = onehot([""]), onehot([" "])
    test_probs = np.vstack([np.vstack([bugs, blank, blank]) * 0.49 + bunny * 0.51, space, bunny])
    arrays["test_logits"] = np.log(np.clip(test_probs, 1e-15, 1))
    arrays["test_probs"] = test_probs
    arrays["bunny_bunny_probs"] = np.vstack([bugs, space, np.vstack([bugs, blank, blank]) * 0.51 + bunny * 0.49])
    arrays["history_logits"] = np.log(np.clip(np.vstack([test_probs] + [np.vstack([space, bunny])] * 5), 1e-15, 1))
    arrays["stretched"] = onehot([" ", "", "b", "u", "n", "", "n", "n", "y", "", " ", " "])
    with open(os.path.join(REF_TESTS, "sample_data", "libri_logits.json")) as fh:
        arrays["libri"] = np.array(json.load(fh))
    arrays["libri_f32"] = arrays["libri"].astype(np.float32)
    bpe_labels = ["▁bugs", "▁bun", "ny", ""]
    bvoc = {c: n for n, c in enumerate(bpe_labels)}
    arrays["bpe_frames"] = onehot(["", "▁bugs", "▁bun", "ny", "ny", ""], bvoc)
    libri_bpe_labels = ["▁⁇▁", "▁"] + ["##" + c for c in synth.LIBRI_LABELS[1:]]
    arrays["libri_bpe"] = np.hstack([np.full((arrays["libri"].shape[0], 1), -100.0), arrays["libri"]])
    arrays["empty29"] = np.zeros((0, 29))

    def add(name, labels, arr, lm=None, **dkw):
        kw = {}
        if lm is not None:
            kw = {k: v for k, v in lm.items() if k not in ("arpa_kind",)}
            if lm["arpa_kind"] == "toy":
                kw["kenlm_model_path"] = os.path.join(REF_TESTS, "sample_data", "bugs_bunny_kenlm.arpa")
        if kw.get("unigrams") == []:
            # build_ctcdecoder divides by zero in verify_alphabet_coverage for an empty list
            # (alphabet.py:169); the reference test builds the pieces by hand (tests/test_decoder.py:266)
            import kenlm
            from pyctcdecode import BeamSearchDecoderCTC, LanguageModel
            lm_obj = LanguageModel(kenlm.Model(kw["kenlm_model_path"]), [], alpha=kw.get("alpha", 0.5),
                                   beta=kw.get("beta", 1.5), unk_score_offset=kw.get("unk_score_offset", -10.0),
                                   score_boundary=kw.get("lm_score_boundary", True))
            dec = BeamSearchDecoderCTC(Alphabet.build_alphabet(labels), lm_obj)
        else:
            dec = build_ctcdecoder(labels, **kw)
        beams = dec.decode_beams(arrays[arr], **dkw)
        top = dec.decode(arrays[arr], **{k: v for k, v in dkw.items() if k != "prune_history"})
        lm_json = None
        if lm is not None:
            lm_json = {k: (list(v) if k == "unigrams" and v is not None else v) for k, v in lm.items() if k != "kenlm_model_path"}
        cases.append({"name": name, "labels": labels, "array": arr, "lm": lm_json, "decode": dkw,
                      "beams": beams_to_json(beams), "decode_text": top})

    toy = dict(arpa_kind="toy")
    # reference tests/test_decoder.py:245-300 (test_decoder, test_build_ctcdecoder)
    add("nolm", SAMPLE_LABELS, "test_logits")
    add("lm_default", SAMPLE_LABELS, "test_logits", dict(toy))
    add("lm_alpha0", SAMPLE_LABELS, "test_logits", dict(toy, alpha=0.0))
    add("lm_alpha1", SAMPLE_LABELS, "test_logits", dict(toy, alpha=1.0))
    add("lm_alpha1_emptyuni", SAMPLE_LABELS, "test_logits", dict(toy, alpha=1.0, unigrams=[]))
    add("lm_uni_bunny_unk0", SAMPLE_LABELS, "test_logits", dict(toy, alpha=1.0, unigrams=["bunny"], unk_score_offset=0.0))
    add("lm_uni_bunny_unk10", SAMPLE_LABELS, "test_logits", dict(toy, alpha=1.0, unigrams=["bunny"], unk_score_offset=-10.0))
    add("lm_unigrams", SAMPLE_LABELS, "test_logits", dict(toy, unigrams=["bugs", "bunny"]))  # :324-384 exact scores
    add("lm_noboundary", SAMPLE_LABELS, "test_logits", dict(toy, lm_score_boundary=False))
    add("lm_unk0_prune20", SAMPLE_LABELS, "test_logits", dict(toy, unk_score_offset=0.0), beam_prune_logp=-20.0)  # :505-513
    add("token_min0", SAMPLE_LABELS, "test_logits", dict(toy), token_min_logp=0.0)  # :409-411
    add("probs_input", SAMPLE_LABELS, "test_probs", dict(toy, unigrams=["bugs", "bunny"]))
    add("stateful_nolm", SAMPLE_LABELS, "bunny_bunny_probs")  # :426-456
    add("stateful_lm", SAMPLE_LABELS, "bunny_bunny_probs", dict(toy, unigrams=["bugs", "bunny"]))
    add("history_off", SAMPLE_LABELS, "history_logits", prune_history=False)  # :413-424
    add("history_on", SAMPLE_LABELS, "history_logits", prune_history=True)
    add("hot_bunny", SAMPLE_LABELS, "test_logits", dict(toy), hotwords=["bunny"], hotword_weight=20)  # :458-480
    add("hot_both", SAMPLE_LABELS, "test_logits", dict(toy), hotwords=["bugs", "bunny"], hotword_weight=20)
    add("hot_phrase", SAMPLE_LABELS, "test_logits", dict(toy), hotwords=["bugs bunny"], hotword_weight=20)
    add("hot_nolm", SAMPLE_LABELS, "test_logits", hotwords=["bugs"])
    add("hot_nolm_w25", SAMPLE_LABELS, "test_logits", hotwords=["bugs"], hotword_weight=25.0)
    add("stretched", SAMPLE_LABELS, "stretched")  # :721-730
    add("bpe_frames", bpe_labels, "bpe_frames")  # :732-744
    add("libri", synth.LIBRI_LABELS, "libri")  # :746-756
    add("libri_f32", synth.LIBRI_LABELS, "libri_f32")
    add("libri_history", synth.LIBRI_LABELS, "libri", prune_history=True)
    add("libri_beam5", synth.LIBRI_LABELS, "libri", beam_width=5)
    add("libri_bpe", libri_bpe_labels, "libri_bpe")  # :758-770
    add("libri_hot", synth.LIBRI_LABELS, "libri", hotwords=["goodeal", "set my"], hotword_weight=8.0)
    add("empty", synth.LIBRI_LABELS, "empty29")  # T=0 (:772-777)

    # ---- seeded synthetic, small ----------------------------------------------------
    fams = {
        "B_nolm": (dict(kind="char", vocab="B", n_words=300, lm_order=0), {}),
        "B_3gram": (dict(kind="char", vocab="B", n_words=300, lm_order=3), dict(alpha=0.5, beta=1.0)),
        "A_2gram": (dict(kind="char", vocab="A", n_words=300, lm_order=2), dict()),
        "C_bpe": (dict(kind="bpe", n_words=300, lm_order=0), {}),
        "C_bpe_4gram": (dict(kind="bpe", n_words=300, lm_order=4), dict(alpha=0.7, beta=2.0)),
    }
    rng = np.random.default_rng(2024)
    for fam, (wkw, lmkw) in fams.items():
        wl = synth.make_workload(wkw)
        for i in range(8):
            T = int(rng.integers(1, 90 if wl.V <= 64 else 36))
            regime = ["peaky", "diffuse", "flat"][i % 3] if wl.V <= 64 else ["peaky", "diffuse"][i % 2]
            seed = 5000 + i
            x = wl.utterance(seed, T, regime)
            if i == 5:
                x = x.astype(np.float64)
            if i == 6:
                e = np.exp(x - x.max(1, keepdims=True))
                x = (e / e.sum(1, keepdims=True)).astype(np.float32)
            name = "syn_%s_%d" % (fam, i)
            arrays[name] = x
            dkw = dict(beam_width=[100, 6, 20][i % 3], prune_history=bool(i % 2))
            if i % 4 == 3:
                dkw.update(hotwords=[wl.words[3], wl.words[10] + " " + wl.words[11]], hotword_weight=6.0)
            kw = dict(lmkw)
            if wl.arpa:
                kw.update(kenlm_model_path=wl.arpa, unigrams=wl.words)
            dec = build_ctcdecoder(wl.labels, **kw)
            beams = dec.decode_beams(x, **dkw)
            top = dec.decode(x, **{k: v for k, v in dkw.items() if k != "prune_history"})
            cases.append({"name": name, "labels": wl.labels, "array": name,
                          "lm": (dict(lmkw, arpa_kind="synth", workload=wkw) if wl.arpa else None),
                          "workload": wkw, "decode": dkw, "beams": beams_to_json(beams), "decode_text": top})

    # alphabet normalisation known answers (reference tests/test_alphabet.py + probes)
    alpha_cases = []
    for labels in [SAMPLE_LABELS, synth.LIBRI_LABELS, synth.W2V2_LABELS, bpe_labels, libri_bpe_labels,
                   ["<pad>", "<unk>", "a", "b", "|"], ["[PAD]", "[UNK]", "##a", "b", "c"], ["_", "a", " "],
                   ["<unk>", "▁a", "b", "▁"], ["a", "b", "c"]]:
        al = Alphabet.build_alphabet(labels)
        alpha_cases.append({"labels": labels, "normalized": al.labels, "is_bpe": al.is_bpe})

    goldens.save_arrays(OUT, arrays)
    with open(os.path.join(OUT, "cases.json"), "w", encoding="utf-8") as fh:
        json.dump({"toy_arpa": toy_arpa, "cases": cases, "alphabet": alpha_cases,
                   "generator": "oracle/gen_golden.py", "reference": "pyctcdecode 0.6.0 @ afecb676, numpy %s" % np.__version__},
                  fh, ensure_ascii=False, indent=0)
    print("wrote %d cases, %d arrays" % (len(cases), len(arrays)))


if __name__ == "__main__":
    main()
