"""Loader for tests/golden (vectors produced by oracle/gen_golden.py from the unmodified reference)."""
import json
import os

import numpy as np

from tests import synth

HERE = os.path.dirname(os.path.abspath(__file__))
_cache = {}

# The arrays of cases.json are stored in two files, so that neither is above 1 MB: the largest logits in the second.
ARRAY_FILES = ("arrays.npz", "arrays_large.npz")
LARGE_ARRAYS = ("syn_C_bpe_0", "syn_C_bpe_4gram_1", "syn_C_bpe_4gram_3")


def load_arrays(directory=os.path.join(HERE, "golden")):
    arrays = {}
    for name in ARRAY_FILES:
        arrays.update(np.load(os.path.join(directory, name)))
    return arrays


def save_arrays(directory, arrays):
    large = {k: v for k, v in arrays.items() if k in LARGE_ARRAYS}
    np.savez_compressed(os.path.join(directory, ARRAY_FILES[0]), **{k: v for k, v in arrays.items() if k not in large})
    np.savez_compressed(os.path.join(directory, ARRAY_FILES[1]), **large)


def load():
    if "g" not in _cache:
        with open(os.path.join(HERE, "golden", "cases.json"), encoding="utf-8") as fh:
            meta = json.load(fh)
        arrays = load_arrays()
        toy = os.path.join(synth.cache_dir(), "bugs_bunny_kenlm.arpa")
        with open(toy, "w", encoding="utf-8") as fh:
            fh.write(meta["toy_arpa"])
        _cache["g"] = {"meta": meta, "arrays": arrays, "toy_arpa": toy, "workloads": {}}
    return _cache["g"]


def lm_kwargs(g, case):
    """build_ctcdecoder keyword arguments (kenlm_model_path, unigrams, alpha, ...) for a golden case."""
    lm = case["lm"]
    if lm is None:
        return {}
    kw = {k: v for k, v in lm.items() if k not in ("arpa_kind", "workload")}
    if lm["arpa_kind"] == "toy":
        kw["kenlm_model_path"] = g["toy_arpa"]
    else:
        key = json.dumps(lm["workload"], sort_keys=True)
        if key not in g["workloads"]:
            g["workloads"][key] = synth.make_workload(lm["workload"])
        wl = g["workloads"][key]
        kw["kenlm_model_path"] = wl.arpa
        kw["unigrams"] = wl.words
    return kw


def beams_match(expected, got, tol=2e-4, exact_order=True):
    """got: list of (text, [(word,(s,e))...], logit, lm). Returns '' or a description of the first difference."""
    if len(expected) != len(got):
        return "beam count %d != %d" % (len(got), len(expected))
    for i, (e, g) in enumerate(zip(expected, got)):
        if e["text"] != g[0]:
            return "beam %d text %r != %r" % (i, g[0], e["text"])
        ef = [(w, (s, t)) for w, s, t in e["frames"]]
        gf = [(w, (int(f[0]), int(f[1]))) for w, f in g[1]]
        if ef != gf:
            return "beam %d frames %r != %r" % (i, gf, ef)
        if abs(e["logit_score"] - g[2]) > tol + 1e-6 * abs(e["logit_score"]):
            return "beam %d logit %r != %r" % (i, g[2], e["logit_score"])
        if abs(e["lm_score"] - g[3]) > tol + 1e-6 * abs(e["lm_score"]):
            return "beam %d lm %r != %r" % (i, g[3], e["lm_score"])
    return ""


def beams_match_tie_aware(expected, got, tol=2e-4, tie=1e-9):
    """Like beams_match, but beams the REFERENCE separates by at most `tie` in lm_score may come in any order:
    where integer-valued logits make several beams' scores agree to the last bits, the reference's order among
    them is decided by numpy's float32 rounding of the log-softmax, which the shared definition (DESIGN.md
    section 2, "Precision") does not reproduce bit for bit.  Everything else must be identical: the same beams
    (text AND word frames) with scores within `tol`, and the same order between beams that are not tied.
    Returns '' or a description of the first difference."""
    if len(expected) != len(got):
        return "beam count %d != %d" % (len(got), len(expected))

    def ident_e(e):
        return (e["text"], tuple((w, int(s), int(t)) for w, s, t in e["frames"]))

    def ident_g(g):
        return (g[0], tuple((w, int(f[0]), int(f[1])) for w, f in g[1]))

    slots = {}
    for j, g in enumerate(got):
        slots.setdefault(ident_g(g), []).append(j)
    pos = []
    for i, e in enumerate(expected):
        cands = slots.get(ident_e(e))
        if not cands:
            return "reference beam %d %r is missing" % (i, e["text"])
        # several beams may share text and frames (different last_char): take the closest score first
        cands.sort(key=lambda j: abs(got[j][3] - e["lm_score"]))
        j = cands.pop(0)
        g = got[j]
        if abs(e["logit_score"] - g[2]) > tol + 1e-6 * abs(e["logit_score"]):
            return "beam %d logit %r != %r" % (i, g[2], e["logit_score"])
        if abs(e["lm_score"] - g[3]) > tol + 1e-6 * abs(e["lm_score"]):
            return "beam %d lm %r != %r" % (i, g[3], e["lm_score"])
        pos.append(j)
    for a in range(len(expected)):
        for b in range(a + 1, len(expected)):
            if expected[a]["lm_score"] - expected[b]["lm_score"] > tie and pos[a] > pos[b]:
                return "beams %d and %d swapped (reference scores %r, %r)" % (a, b, expected[a]["lm_score"], expected[b]["lm_score"])
    return ""


def build_product_decoder(pkg, labels, **kw):
    """build_ctcdecoder, except for unigrams == [] where the reference itself divides by zero in
    verify_alphabet_coverage and its test assembles the pieces by hand (tests/test_decoder.py:266)."""
    if kw.get("unigrams") == []:
        lm = pkg.LanguageModel(pkg.NgramModel(kw["kenlm_model_path"]), [], alpha=kw.get("alpha", 0.5),
                               beta=kw.get("beta", 1.5), unk_score_offset=kw.get("unk_score_offset", -10.0),
                               score_boundary=kw.get("lm_score_boundary", True))
        return pkg.BeamSearchDecoderCTC(pkg.Alphabet.build_alphabet(labels), lm)
    return pkg.build_ctcdecoder(labels, **kw)


def load_stream():
    """tests/golden/stream_cases.json (oracle/gen_golden_stream.py: the reference's partial_decode_beams, call by call)."""
    if "s" not in _cache:
        with open(os.path.join(HERE, "golden", "stream_cases.json"), encoding="utf-8") as fh:
            meta = json.load(fh)
        arrays = dict(np.load(os.path.join(HERE, "golden", "stream_arrays.npz")))
        _cache["s"] = {"meta": meta, "arrays": arrays}
    return _cache["s"]


def stream_case_names():
    return [c["name"] for c in load_stream()["meta"]["cases"]]


def run_stream_case(pkg, name, tol=2e-4):
    """Drive the product's get_starting_state / partial_decode_beams through one recorded streaming case and
    compare every call's LMBeam list with what the unmodified reference returned.  Returns '' or the first
    difference.  Strings, frames and last_char must be identical; scores within `tol` (numpy's float32
    log-softmax differs from the shared definition in the last bits, DESIGN.md)."""
    g, s = load(), load_stream()
    case = next(c for c in s["meta"]["cases"] if c["name"] == name)
    x = s["arrays"][case["array"]] if case["array"] in s["arrays"] else g["arrays"][case["array"]]
    dec = build_product_decoder(pkg, case["labels"], **lm_kwargs(g, case))
    beams, cached_lm, cached_p = dec.get_starting_state()
    for i, step in enumerate(case["steps"]):
        call = step["call"]
        scorer = None
        if call.get("hotwords") is not None:
            scorer = pkg.HotwordScorer.build_scorer(call["hotwords"], weight=call.get("hotword_weight", 10.0))
        out = dec.partial_decode_beams(x[step["start"]:step["end"]], cached_lm, cached_p, beams, step["start"],
                                       hotword_scorer=scorer, force_next_word=bool(call.get("force_next_word", False)),
                                       is_end=step["is_end"], **case["common"])
        exp = step["beams"]
        if len(out) != len(exp):
            return "call %d: %d beams != %d" % (i, len(out), len(exp))
        # identical beams (strings, frames, last_char) with scores within tol; the ORDER must agree except between
        # beams the reference itself separates by less than 1e-9 (last-bit rounding of float32 numpy log-softmax
        # vs the shared definition decides such near-ties; DESIGN.md, "near-tie class")
        def ident(text, nw, pw, lc, tf, pf):
            return (text, nw, pw, lc, tuple(tuple(f) for f in tf), tuple(pf))
        got = {}
        for j, o in enumerate(out):
            got[ident(o.text, o.next_word, o.partial_word, o.last_char, o.text_frames, o.partial_frames)] = (j, o)
        pos = []
        for j, e in enumerate(exp):
            k = ident(e["text"], e["next_word"], e["partial_word"], e["last_char"], e["text_frames"], e["partial_frames"])
            if k not in got:
                return "call %d: reference beam %d %r missing (got rank %d: %r)" % (i, j, k[:4], j, (out[j].text, out[j].partial_word, out[j].last_char))
            gj, o = got[k]
            if abs(o.logit_score - e["logit_score"]) > tol + 1e-6 * abs(e["logit_score"]):
                return "call %d beam %d logit %r != %r" % (i, j, o.logit_score, e["logit_score"])
            if abs(o.lm_score - e["lm_score"]) > tol + 1e-6 * abs(e["lm_score"]):
                return "call %d beam %d lm %r != %r" % (i, j, o.lm_score, e["lm_score"])
            pos.append(gj)
        for a in range(len(exp)):
            for b in range(a + 1, len(exp)):
                if exp[a]["lm_score"] - exp[b]["lm_score"] > 1e-9 and pos[a] > pos[b]:
                    return "call %d: beams %d and %d swapped (scores %r, %r)" % (i, a, b, exp[a]["lm_score"], exp[b]["lm_score"])
        beams = out
    return ""


def load_unstable():
    """tests/golden/unstable_cases.json (oracle/gen_golden_unstable.py: cases the reference itself decides by
    rounding noise, recorded as what is common to its outcomes under a 1e-13 input perturbation)."""
    if "u" not in _cache:
        with open(os.path.join(HERE, "golden", "unstable_cases.json"), encoding="utf-8") as fh:
            _cache["u"] = json.load(fh)
    return _cache["u"]


def unstable_case_names(gpu=False):
    """`gpu`: the cases the GPU tests run (cases marked cpu_only are pinned on the oracle and the kernel logic only)"""
    return [c["name"] for c in load_unstable()["cases"] if not (gpu and c.get("cpu_only"))]


def run_unstable_case(decode_beams, name, tol=2e-4, tie=1e-9):
    """decode_beams(labels, x, **kw) -> [(text, [(word, (s, e))...], logit, lm)].  The beam SET (text + word frames)
    must equal the reference's; every beam's scores must be one of the pairs the reference family attaches to that
    beam; the list must be sorted by lm_score (exact ties in any order).  Returns '' or the first difference."""
    g = load()
    case = next(c for c in load_unstable()["cases"] if c["name"] == name)
    got = decode_beams(case["labels"], g["arrays"][case["array"]], **case["decode"])
    exp = {(b["text"], tuple((w, int(s), int(t)) for w, s, t in b["frames"])): b["scores"] for b in case["beams"]}
    if len(got) != len(exp):
        return "beam count %d != %d" % (len(got), len(exp))
    seen = set()
    for i, b in enumerate(got):
        key = (b[0], tuple((w, int(f[0]), int(f[1])) for w, f in b[1]))
        if key not in exp or key in seen:
            return "beam %d %r is not a beam of the reference (or appears twice)" % (i, b[0])
        seen.add(key)
        if not any(abs(p[0] - b[2]) <= tol + 1e-6 * abs(p[0]) and abs(p[1] - b[3]) <= tol + 1e-6 * abs(p[1]) for p in exp[key]):
            return "beam %d scores (%r, %r) not among the reference's %r" % (i, b[2], b[3], exp[key])
        if i and got[i - 1][3] < b[3] - tie:
            return "beams %d and %d are not in score order" % (i - 1, i)
    if got and got[0][0] != case["beams"][0]["text"]:
        return "top beam %r != %r" % (got[0][0], case["beams"][0]["text"])
    return ""


def load_multilm():
    """tests/golden/multilm_cases.json (oracle/gen_golden_multilm.py: the reference's MultiLanguageModel)."""
    if "m" not in _cache:
        with open(os.path.join(HERE, "golden", "multilm_cases.json"), encoding="utf-8") as fh:
            meta = json.load(fh)
        _cache["m"] = {"meta": meta, "arrays": dict(np.load(os.path.join(HERE, "golden", "multilm_arrays.npz")))}
    return _cache["m"]


def multilm_case_names():
    return [c["name"] for c in load_multilm()["meta"]["cases"]]


def build_multilm_decoder(pkg, case):
    g = load()
    models = []
    for m in case["models"]:
        if m["arpa_kind"] == "toy":
            path, words = g["toy_arpa"], None
        else:
            key = json.dumps(m["workload"], sort_keys=True)
            if key not in g["workloads"]:
                g["workloads"][key] = synth.make_workload(m["workload"])
            path, words = g["workloads"][key].arpa, g["workloads"][key].words
        unigrams = m.get("unigrams")
        if unigrams is None and m.get("unigrams_first") is not None:
            unigrams = words[: m["unigrams_first"]]
        kw = {k: m[k] for k in ("alpha", "beta", "unk_score_offset", "score_boundary") if k in m}
        models.append(pkg.LanguageModel(pkg.NgramModel(path), unigrams, **kw))
    return pkg.BeamSearchDecoderCTC(pkg.Alphabet.build_alphabet(case["labels"]), pkg.MultiLanguageModel(models))


def run_multilm_case(pkg, name, tol=2e-4):
    """The product's decoder over a MultiLanguageModel against what the unmodified reference returned: all beams
    (text, word frames, both scores), decode(), a second call started from the best beam's MultiLanguageModelState,
    and chunked partial_decode_beams.  Returns '' or the first difference."""
    g, m = load(), load_multilm()
    case = next(c for c in m["meta"]["cases"] if c["name"] == name)
    x = m["arrays"][case["array"]] if case["array"] in m["arrays"] else g["arrays"][case["array"]]
    dec = build_multilm_decoder(pkg, case)
    dkw = case["decode"]

    def as_tuples(beams):
        return [(b.text, b.text_frames, b.logit_score, b.lm_score) for b in beams]

    out = dec.decode_beams(x, **dkw)
    diff = beams_match(case["beams"], as_tuples(out), tol=tol)
    if diff:
        return "decode_beams: " + diff
    if dec.decode(x, **{k: v for k, v in dkw.items() if k != "prune_history"}) != case["decode_text"]:
        return "decode() text differs"
    if "split" in case:
        first = dec.decode_beams(x[:case["split"]], **dkw)
        diff = beams_match(case["split_first"], as_tuples(first), tol=tol)
        if diff:
            return "first half: " + diff
        state = first[0].last_lm_state
        if state is None or len(state.states) != len(case["models"]):
            return "last_lm_state is not a MultiLanguageModelState with %d states" % len(case["models"])
        second = dec.decode_beams(x[case["split"]:], lm_start_state=state, **dkw)
        diff = beams_match(case["split_second"], as_tuples(second), tol=tol)
        if diff:
            return "second half (from the carried state): " + diff
    if "stream" in case:
        beams, cached_lm, cached_p = dec.get_starting_state()
        kw = {k: v for k, v in dkw.items() if k in ("beam_width", "prune_history")}
        for i, step in enumerate(case["stream"]):
            got = dec.partial_decode_beams(x[step["start"]:step["end"]], cached_lm, cached_p, beams, step["start"],
                                           is_end=(i == len(case["stream"]) - 1), **kw)
            exp = step["beams"]
            if len(got) != len(exp):
                return "stream call %d: %d beams != %d" % (i, len(got), len(exp))
            for j, (o, e) in enumerate(zip(got, exp)):
                a = (o.text, o.partial_word, o.last_char, [list(f) for f in o.text_frames], list(o.partial_frames))
                b = (e["text"], e["partial_word"], e["last_char"], e["text_frames"], e["partial_frames"])
                if a != b:
                    return "stream call %d beam %d: %r != %r" % (i, j, a, b)
                if abs(o.lm_score - e["lm_score"]) > tol + 1e-6 * abs(e["lm_score"]) or abs(o.logit_score - e["logit_score"]) > tol + 1e-6 * abs(e["logit_score"]):
                    return "stream call %d beam %d scores (%r, %r) != (%r, %r)" % (i, j, o.logit_score, o.lm_score, e["logit_score"], e["lm_score"])
            beams = got
    return ""
