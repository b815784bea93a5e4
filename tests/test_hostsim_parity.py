"""CPU tests of the KERNEL LOGIC: the product host code (pyctcdecode_b200) is pointed at the
tests/hostsim simulation build of the very same kernel sources (see tests/hostsim/cuda_shim.h)
and compared with the oracle and with the golden vectors of the unmodified reference.
This does not replace the `-m gpu` parity tests; it is how kernel logic is kept testable in a
container without a GPU."""
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle as orc
from tests import goldens, synth

HOSTSIM = os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostsim")


@pytest.fixture(scope="module")
def sim():
    subprocess.check_call(["make", "-s", "-C", HOSTSIM])
    import pyctcdecode_b200
    from pyctcdecode_b200 import _lib
    _lib.use_library(os.path.join(HOSTSIM, "libb200ctc_hostsim.so"))
    yield pyctcdecode_b200
    _lib._lib = None


def _beams(out):
    return [(b.text, b.text_frames, b.logit_score, b.lm_score) for b in out]


def _names():
    return [c["name"] for c in goldens.load()["meta"]["cases"]]


@pytest.mark.parametrize("name", _names())
def test_hostsim_matches_reference_golden(sim, golden, name):
    case = next(c for c in golden["meta"]["cases"] if c["name"] == name)
    dec = goldens.build_product_decoder(sim, case["labels"], **goldens.lm_kwargs(golden, case))
    x = golden["arrays"][case["array"]]
    got = _beams(dec.decode_beams(x, **case["decode"]))
    assert goldens.beams_match(case["beams"], got) == ""
    kw = {k: v for k, v in case["decode"].items() if k != "prune_history"}
    assert dec.decode(x, **kw) == case["decode_text"]


FAMILIES = {
    "B_nolm": (dict(kind="char", vocab="B", n_words=400, lm_order=0), {}),
    "B_3gram": (dict(kind="char", vocab="B", n_words=400, lm_order=3), dict(alpha=0.5, beta=1.0)),
    "A_2gram": (dict(kind="char", vocab="A", n_words=400, lm_order=2), dict()),
    "B_5gram": (dict(kind="char", vocab="B", n_words=150, lm_order=5), dict(alpha=0.9, beta=0.3, unk_score_offset=-4.0)),
    "C_bpe": (dict(kind="bpe", n_words=400, lm_order=0), {}),
    "C_bpe_4gram": (dict(kind="bpe", n_words=400, lm_order=4), dict(alpha=0.7, beta=2.0)),
}


def _compare(ref, got, tol=1e-9):
    assert len(ref) == len(got)
    for r, g in zip(ref, got):
        assert r[0] == g[0]
        assert [(w, tuple(f)) for w, f in r[1]] == [(w, tuple(f)) for w, f in g[1]]
        assert abs(r[2] - g[2]) <= tol * max(1.0, abs(r[2]))
        assert abs(r[3] - g[3]) <= tol * max(1.0, abs(r[3]))


@pytest.mark.parametrize("fam", sorted(FAMILIES))
def test_hostsim_vs_oracle_random(sim, fam):
    wkw, lmkw = FAMILIES[fam]
    wl = synth.make_workload(wkw)
    kw = dict(lmkw)
    if wl.arpa:
        kw.update(kenlm_model_path=wl.arpa, unigrams=wl.words)
    dec = sim.build_ctcdecoder(wl.labels, **kw)
    ora = orc.OracleDecoder(wl.labels, **kw)
    rng = np.random.default_rng(99)
    n_cases = 18 if wl.V <= 64 else 8
    for i in range(n_cases):
        T = int(rng.integers(0, 140 if wl.V <= 64 else 50))
        regime = ["peaky", "diffuse", "flat"][i % 3] if wl.V <= 64 else ["peaky", "diffuse"][i % 2]
        x = wl.utterance(700 + i, T, regime) if T else np.zeros((0, wl.V), np.float32)
        if i % 5 == 4:
            x = x.astype(np.float64)
        if i % 7 == 6 and T:
            e = np.exp(x - x.max(1, keepdims=True))
            x = (e / e.sum(1, keepdims=True)).astype(x.dtype)
        dkw = dict(beam_width=[100, 3, 17, 1][i % 4], prune_history=bool(i % 2), beam_prune_logp=[-10.0, -4.0, -25.0][i % 3],
                   token_min_logp=[-5.0, -8.0][i % 2])
        if i % 4 == 2:
            dkw.update(hotwords=[wl.words[2], wl.words[7] + " " + wl.words[9]], hotword_weight=7.5)
        _compare(ora.decode_beams(x, **dkw), _beams(dec.decode_beams(x, **dkw)))


def test_hostsim_ragged_batch_matches_single(sim):
    wl = synth.make_workload(FAMILIES["B_3gram"][0])
    kw = dict(FAMILIES["B_3gram"][1], kenlm_model_path=wl.arpa, unigrams=wl.words)
    dec = sim.build_ctcdecoder(wl.labels, **kw)
    ora = orc.OracleDecoder(wl.labels, **kw)
    Ts = [40, 0, 77, 5, 120, 1, 33]
    xs = [wl.utterance(900 + i, T, "diffuse" if i % 2 else "peaky") if T else np.zeros((0, wl.V), np.float32) for i, T in enumerate(Ts)]
    texts = dec.decode_batch(None, xs, beam_width=25)
    assert texts == ora.decode_batch(xs, beam_width=25)
    beams = dec.decode_beams_batch(None, xs, beam_width=25)
    for x, b in zip(xs, beams):
        _compare(ora.decode_beams(x, beam_width=25), _beams(b))
        assert all(o.last_lm_state is None for o in b)


def test_hostsim_duplicate_blank_labels_and_state(sim):
    # two pad-like labels normalise to the same blank string; they must behave as one token
    labels = ["<pad>", "[PAD]", "a", "b", " "]
    dec = sim.build_ctcdecoder(labels)
    ora = orc.OracleDecoder(labels)
    rng = np.random.default_rng(5)
    x = rng.standard_normal((40, 5)).astype(np.float32) * 2
    _compare(ora.decode_beams(x, beam_width=12), _beams(dec.decode_beams(x, beam_width=12)))


def test_hostsim_lm_start_state_roundtrip(sim, golden):
    case = next(c for c in golden["meta"]["cases"] if c["name"] == "stateful_lm")
    dec = goldens.build_product_decoder(sim, case["labels"], **goldens.lm_kwargs(golden, case))
    probs = golden["arrays"]["bunny_bunny_probs"]
    # reference tests/test_decoder.py:447-456
    assert dec.decode(probs[:4]) + " " + dec.decode(probs[4:]) == "bugs bugs"
    top = dec.decode_beams(probs[:4])[0]
    assert top.last_lm_state is not None
    text = top.text + " " + dec.decode_beams(probs[4:], lm_start_state=top.last_lm_state)[0].text
    assert text == "bugs bunny"


def test_hostsim_errors(sim):
    dec = sim.build_ctcdecoder(synth.LIBRI_LABELS)
    with pytest.raises(ValueError):
        dec.decode(np.zeros((4, 7), np.float32))
    with pytest.raises(ValueError):
        dec.decode(np.zeros((4,), np.float32))
    assert dec.decode(np.zeros((0, 29))) == ""


def test_hostsim_special_single_token_steps(sim):
    """The in-place single-token frames and the merge-free sorted frames of the latency-first kernel
    (b2c_fast_cheap_step / b2c_fast_sorted_step) against the oracle, incl. exact ties and tiny beams."""
    wl = synth.make_workload(FAMILIES["B_nolm"][0])
    dec = sim.build_ctcdecoder(wl.labels)
    ora = orc.OracleDecoder(wl.labels)
    inplace = ranked = 0
    for x, kw in synth.special_step_cases(wl):
        got = _beams(dec.decode_beams(x, **kw))
        tm = dec.last_timings()
        inplace += tm["inplace_frames"]
        ranked += tm["sorted_frames"]
        _compare(ora.decode_beams(x, **kw), got)
    assert inplace > 1000 and ranked > 100      # the special steps really ran
    # with an LM only the branch-(i) in-place frames apply; hotwords and BPE likewise
    for fam in ("B_3gram", "C_bpe"):
        wkw, lmkw = FAMILIES[fam]
        wl2 = synth.make_workload(wkw)
        kw2 = dict(lmkw)
        if wl2.arpa:
            kw2.update(kenlm_model_path=wl2.arpa, unigrams=wl2.words)
        dec2 = sim.build_ctcdecoder(wl2.labels, **kw2)
        ora2 = orc.OracleDecoder(wl2.labels, **kw2)
        n = 0
        for i in range(4):
            x = wl2.utterance(5000 + i, 200 if wl2.V <= 64 else 80, "peaky")
            for hot in (None, [wl2.words[3], wl2.words[10]]):
                for prune in (True, False):
                    _compare(ora2.decode_beams(x, prune_history=prune, hotwords=hot), _beams(dec2.decode_beams(x, prune_history=prune, hotwords=hot)))
                    n += dec2.last_timings()["inplace_frames"]
        assert n > 0


@pytest.mark.parametrize("name", goldens.stream_case_names())
def test_hostsim_streaming_matches_reference_golden(sim, name):
    """get_starting_state / partial_decode_beams, call by call, against the unmodified reference's outputs."""
    assert goldens.run_stream_case(sim, name) == ""


def test_hostsim_streaming_chunks_equal_whole(sim):
    """Chunked partial_decode_beams (several streams per launch) ends in the beams decode_beams gives for the
    whole utterance (reference tests/test_decoder.py:515-563 states this property for its own decoder)."""
    for fam in ("B_nolm", "B_3gram", "C_bpe_4gram"):
        wkw, lmkw = FAMILIES[fam]
        wl = synth.make_workload(wkw)
        kw = dict(lmkw)
        if wl.arpa:
            kw.update(kenlm_model_path=wl.arpa, unigrams=wl.words)
        dec = sim.build_ctcdecoder(wl.labels, **kw)
        T = 90 if wl.V <= 64 else 40
        xs = [wl.utterance(8200 + i, T, ["peaky", "diffuse"][i % 2]) for i in range(3)]
        whole = [dec.decode_beams(x, beam_width=16) for x in xs]
        states = [dec.get_starting_state() for _ in xs]
        beams = [s[0] for s in states]
        caches = [s[1] for s in states]
        bounds = [0, 17, 18, 50, T]
        for a, b in zip(bounds[:-1], bounds[1:]):
            beams = dec.partial_decode_beams_batch([x[a:b] for x in xs], caches, beams, [a] * len(xs), beam_width=16, is_end=(b == T))
        for w, got in zip(whole, beams):
            assert [o.text for o in w] == [g.text for g in got]
            assert [[f for _, f in o.text_frames] for o in w] == [[tuple(f) for f in g.text_frames] for g in got]
            for o, g in zip(w, got):
                assert abs(o.logit_score - g.logit_score) <= 1e-9 * max(1.0, abs(o.logit_score))
                assert abs(o.lm_score - g.lm_score) <= 1e-9 * max(1.0, abs(o.lm_score))


def test_hostsim_streaming_host_caches_are_transparent(sim):
    """The streaming host path keeps word hashes per word and per returned text (decoder.py, _stream_states): the
    results must not depend on what the caches hold -- two streams interleaved on one decoder, beams re-wrapped as new
    Beam objects, and a decoder that receives another decoder's beams mid-stream (every text misses its cache) all
    give the beams of an undisturbed run, call by call."""
    from pyctcdecode_b200.decoder import Beam
    for fam in ("B_nolm", "B_3gram", "C_bpe_4gram"):
        wkw, lmkw = FAMILIES[fam]
        wl = synth.make_workload(wkw)
        kw = dict(lmkw)
        if wl.arpa:
            kw.update(kenlm_model_path=wl.arpa, unigrams=wl.words)
        T = 120 if wl.V <= 64 else 60
        bounds = list(range(0, T, 20)) + [T]
        xs = [wl.utterance(9300 + i, T, "peaky") for i in range(2)]

        def run(dec_for_call, rewrap):
            outs = []
            for i, x in enumerate(xs):
                beams, cache, pcache = dec_for_call(0, i).get_starting_state()
                calls = []
                for c, (a, b) in enumerate(zip(bounds[:-1], bounds[1:])):
                    got = dec_for_call(c, i).partial_decode_beams(x[a:b], cache, pcache, beams, a, beam_width=24, is_end=(b == T))
                    calls.append(got)
                    beams = [Beam.from_lm_beam(g) for g in got] if rewrap else got
                outs.append(calls)
            return outs

        plain = sim.build_ctcdecoder(wl.labels, **kw)
        want = run(lambda c, i: plain, False)
        # (a) re-wrapped beams, (b) a different decoder every other call: its caches have never seen the texts
        a, b = sim.build_ctcdecoder(wl.labels, **kw), sim.build_ctcdecoder(wl.labels, **kw)
        assert run(lambda c, i: a, True) == want
        assert run(lambda c, i: (a, b)[c % 2], False) == want
        # (c) the two streams interleaved call by call on ONE decoder (each call evicts half of the other stream's texts)
        dec = sim.build_ctcdecoder(wl.labels, **kw)
        st = [dec.get_starting_state() for _ in xs]
        beams = [s_[0] for s_ in st]
        got = [[] for _ in xs]
        for a_, b_ in zip(bounds[:-1], bounds[1:]):
            for i, x in enumerate(xs):
                beams[i] = dec.partial_decode_beams(x[a_:b_], st[i][1], st[i][2], beams[i], a_, beam_width=24, is_end=(b_ == T))
                got[i].append(beams[i])
        assert got == want


def test_hostsim_lm_blob_file_roundtrip(sim, tmp_path):
    """NgramModel.save_blob / build_ctcdecoder(kenlm_model_path="*.b2clm") (SURVEY 8f-3: cached flattened LM):
    the decoder built from the blob file decodes exactly like the one built from the ARPA file."""
    wkw, lmkw = FAMILIES["B_3gram"]
    wl = synth.make_workload(wkw)
    dec = sim.build_ctcdecoder(wl.labels, kenlm_model_path=wl.arpa, unigrams=wl.words, **lmkw)
    path = str(tmp_path / "lm.b2clm")
    dec._language_model.ngram_model.save_blob(path)
    dec2 = sim.build_ctcdecoder(wl.labels, kenlm_model_path=path, **lmkw)
    for i in range(4):
        x = wl.utterance(8400 + i, 80, ["peaky", "diffuse"][i % 2])
        assert _beams(dec.decode_beams(x, beam_width=20, hotwords=[wl.words[5]])) == _beams(dec2.decode_beams(x, beam_width=20, hotwords=[wl.words[5]]))
    with open(path, "r+b") as fh:       # a damaged file is rejected, not decoded with
        fh.write(b"\x00\x00\x00\x00")
    with pytest.raises(ValueError):
        sim.build_ctcdecoder(wl.labels, kenlm_model_path=path)


@pytest.mark.parametrize("name", goldens.multilm_case_names())
def test_hostsim_multi_language_model_matches_reference_golden(sim, name):
    """MultiLanguageModel (mean of 2-3 n-gram models with their own parameters and unigram lists) against the
    unmodified reference: all beams, decode(), carried MultiLanguageModelState, chunked streaming."""
    assert goldens.run_multilm_case(sim, name) == ""


@pytest.mark.parametrize("order", ["1", "3"])
def test_hostsim_results_do_not_depend_on_work_item_order(order):
    """hostsim replays the work items of every phase in another order (B200CTC_HOSTSIM_ORDER: 1 reverse, 3 odd items
    first; csrc/b2c_cta.h).  Any order is a legal interleaving of the CUDA execution, so the parity tests must pass
    unchanged -- this catches code that silently relies on thread order inside a phase."""
    import sys
    env = dict(os.environ, B200CTC_HOSTSIM_ORDER=order, B200CTC_FORCE_V5="1")
    here = os.path.abspath(__file__)
    r = subprocess.run([sys.executable, "-m", "pytest", here, "-x", "-q", "-k", "special or random or ragged or streaming_chunks"],
                       env=env, cwd=os.path.dirname(os.path.dirname(here)), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout[-3000:]


def test_hostsim_text_only_results_equal_full_results(sim):
    """decode_batch() asks the library for texts only (no frames, no word vectors: assemble_text); the texts must be
    the top beams' texts of the full result path, for character and BPE alphabets."""
    for fam in ("B_nolm", "B_3gram", "C_bpe", "C_bpe_4gram"):
        wkw, lmkw = FAMILIES[fam]
        wl = synth.make_workload(wkw)
        kw = dict(lmkw)
        if wl.arpa:
            kw.update(kenlm_model_path=wl.arpa, unigrams=wl.words)
        dec = sim.build_ctcdecoder(wl.labels, **kw)
        T = 120 if wl.V <= 64 else 50
        xs = [wl.utterance(8600 + i, T - 7 * i, ["peaky", "diffuse"][i % 2]) for i in range(6)] + [np.zeros((0, wl.V), np.float32)]
        texts = dec.decode_batch(None, xs, beam_width=20)
        full = [dec.decode_beams(x, beam_width=20, prune_history=True)[0].text for x in xs]
        assert texts == full


def test_hostsim_general_kernel_in_place_frames():
    """b2c_inplace_step (general kernel: beam_width > 128, streaming, MultiLanguageModel) against the oracle; run in
    a subprocess with the latency-first kernel disabled so that beams <= 128 take the general kernels too."""
    import sys
    code = r'''
import os, sys
sys.path.insert(0, %r)
import numpy as np
from tests import synth
from oracle import oracle as orc
import pyctcdecode_b200 as sim
from pyctcdecode_b200 import _lib
_lib.use_library(%r)
total = 0
for wkw, lmkw in [(dict(kind="char", vocab="B", n_words=400, lm_order=0), {}), (dict(kind="char", vocab="B", n_words=400, lm_order=3), dict(alpha=0.5, beta=1.0))]:
    wl = synth.make_workload(wkw)
    kw = dict(lmkw)
    if wl.arpa:
        kw.update(kenlm_model_path=wl.arpa, unigrams=wl.words)
    dec = sim.build_ctcdecoder(wl.labels, **kw)
    ora = orc.OracleDecoder(wl.labels, **kw)
    for i, (x, dkw) in enumerate(synth.special_step_cases(wl, n_cases=18)):
        if i %% 3 == 0:
            dkw = dict(dkw, beam_width=300)
        got = dec.decode_beams(x, **dkw)
        total += dec.last_timings()["inplace_frames"]
        ref = ora.decode_beams(x, **dkw)
        assert len(got) == len(ref)
        for g, r in zip(got, ref):
            assert g.text == r[0] and g.text_frames == r[1]
            assert abs(g.logit_score - r[2]) <= 1e-9 * max(1.0, abs(r[2])) and abs(g.lm_score - r[3]) <= 1e-9 * max(1.0, abs(r[3]))
assert total > 500, total
''' % (os.path.dirname(HOSTSIM.rstrip("/")).rsplit("/tests", 1)[0], os.path.join(HOSTSIM, "libb200ctc_hostsim.so"))
    subprocess.check_call(["make", "-s", "-C", HOSTSIM])
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, B200CTC_NO_V5="1"), stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout[-3000:]


def test_hostsim_half_precision_inputs(sim):
    """float16 / bfloat16 logits travel as 2-byte elements (dtype codes 2 / 3) and are widened to float32 on the
    device: the result must equal decoding the float32-widened matrix, for lists, one [B, T, V] array and torch
    tensors; a mixed list falls back to float64 on the host."""
    import torch
    wl = synth.make_workload(FAMILIES["B_3gram"][0])
    kw = dict(FAMILIES["B_3gram"][1], kenlm_model_path=wl.arpa, unigrams=wl.words)
    dec = sim.build_ctcdecoder(wl.labels, **kw)
    xs = [wl.utterance(8700 + i, 60, ["peaky", "diffuse"][i % 2]) for i in range(4)]
    h16 = [x.astype(np.float16) for x in xs]
    want16 = [_beams(dec.decode_beams(h.astype(np.float32), beam_width=16)) for h in h16]
    assert [_beams(b) for b in dec.decode_beams_batch(None, h16, beam_width=16)] == want16
    assert [_beams(b) for b in dec.decode_beams_batch(None, np.stack(h16), beam_width=16)] == want16
    assert [_beams(b) for b in dec.decode_beams_batch(None, torch.from_numpy(np.stack(h16)), beam_width=16)] == want16
    bf = [torch.from_numpy(x).to(torch.bfloat16) for x in xs]
    wantbf = [_beams(dec.decode_beams(t.float().numpy(), beam_width=16)) for t in bf]
    assert [_beams(b) for b in dec.decode_beams_batch(None, bf, beam_width=16)] == wantbf
    assert [_beams(b) for b in dec.decode_beams_batch(None, torch.stack(bf), beam_width=16)] == wantbf
    mixed = dec.decode_batch(None, [bf[0], xs[1]], beam_width=16)
    assert mixed[1] == dec.decode(xs[1], beam_width=16)
    # subnormal, zero, inf and NaN bit patterns convert like numpy does
    special = np.array([[0.0, -0.0, 6e-8, -6.1e-5, 65504.0, np.inf, -np.inf, 1.0]] * 2, dtype=np.float16)
    lab = ["a", "b", "c", "d", "e", "f", "g", ""]
    d2 = sim.build_ctcdecoder(lab)
    assert _beams(d2.decode_beams(special)) == _beams(d2.decode_beams(special.astype(np.float32)))


@pytest.mark.parametrize("fam", ["B_3gram", "B_5gram", "A_2gram"])
def test_hostsim_scored_in_place_frames_with_lm(sim, fam):
    """b2c_fast_scored_step: one ordinary character after a one-token frame WITH an LM / hotwords (new partial-word
    scores per beam; in place only if the new lm_scores keep slot order and threshold) against the oracle."""
    wkw, lmkw = FAMILIES[fam]
    wl = synth.make_workload(wkw)
    kw = dict(lmkw, kenlm_model_path=wl.arpa, unigrams=wl.words)
    dec = sim.build_ctcdecoder(wl.labels, **kw)
    ora = orc.OracleDecoder(wl.labels, **kw)
    inplace = frames = 0
    for i, (x, dkw) in enumerate(synth.special_step_cases(wl, n_cases=24, seed=11)):
        if i % 4 == 1:
            dkw = dict(dkw, hotwords=[wl.words[2], wl.words[7] + " " + wl.words[9]], hotword_weight=7.5)
        got = _beams(dec.decode_beams(x, **dkw))
        tm = dec.last_timings()
        inplace += tm["inplace_frames"]
        frames += tm["frames"]
        _compare(ora.decode_beams(x, **dkw), got)
    assert inplace > 0.4 * frames, (inplace, frames)


def test_hostsim_quickstart_example_runs(sim, capsys):
    """examples/quickstart.py (the reference README's usage patterns) runs end to end on the simulated kernels."""
    import runpy
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples", "quickstart.py")
    mod = runpy.run_path(path)
    assert isinstance(mod["main"](), str)
    out = capsys.readouterr().out
    assert "decode_batch" in out and "after frame" in out


def test_hostsim_decoder_is_thread_safe(sim):
    """One decoder object called from 8 threads at once (the reference decoder can be; ADVICE r1): the handle
    serialises the calls, every thread gets the results a lone call gets."""
    import threading

    wkw, lmkw = FAMILIES["B_3gram"]
    wl = synth.make_workload(wkw)
    dec = sim.build_ctcdecoder(wl.labels, kenlm_model_path=wl.arpa, unigrams=wl.words, **lmkw)
    xs = [wl.utterance(8600 + i, 40 + 7 * i, ["peaky", "diffuse"][i % 2]) for i in range(8)]
    want = [(dec.decode(x, beam_width=16), _beams(dec.decode_beams(x, beam_width=16))) for x in xs]
    got, errors = [None] * len(xs), []

    def work(i):
        try:
            for _ in range(5):
                got[i] = (dec.decode(xs[i], beam_width=16), _beams(dec.decode_beams(xs[i], beam_width=16)))
        except Exception as exc:  # pragma: no cover
            errors.append(exc)

    threads = [threading.Thread(target=work, args=(i,)) for i in range(len(xs))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors
    assert got == want


def test_hostsim_blob_decoder_save_load_roundtrip(sim, tmp_path):
    """save_to_dir / load_from_dir of a decoder built from a *.b2clm blob (ADVICE r1: the round trip was broken)."""
    wkw, lmkw = FAMILIES["B_3gram"]
    wl = synth.make_workload(wkw)
    dec = sim.build_ctcdecoder(wl.labels, kenlm_model_path=wl.arpa, unigrams=wl.words, **lmkw)
    path = str(tmp_path / "lm.b2clm")
    dec._language_model.ngram_model.save_blob(path)
    dec2 = sim.build_ctcdecoder(wl.labels, kenlm_model_path=path, **lmkw)
    out = tmp_path / "saved"
    out.mkdir()
    dec2.save_to_dir(str(out))
    dec3 = sim.BeamSearchDecoderCTC.load_from_dir(str(out))
    lm2, lm3 = dec2._language_model, dec3._language_model
    assert (lm3.alpha, lm3.beta) == (lm2.alpha, lm2.beta)
    for tok in ("", wl.words[3][:2], "zzzzqqq"):     # host mirror of the partial-word score agrees with the ARPA-built model
        assert lm3.score_partial_token(tok) == dec._language_model.score_partial_token(tok)
    for i in range(3):
        x = wl.utterance(8700 + i, 60, "peaky")
        assert _beams(dec3.decode_beams(x, beam_width=20)) == _beams(dec.decode_beams(x, beam_width=20))


def test_hostsim_corrupt_blob_fields_are_rejected(sim, tmp_path):
    """b2c_lm_from_blob checks offsets, masks and ids against the blob size (ADVICE r1), not just the magic."""
    import struct

    wkw, lmkw = FAMILIES["B_3gram"]
    wl = synth.make_workload(wkw)
    dec = sim.build_ctcdecoder(wl.labels, kenlm_model_path=wl.arpa, unigrams=wl.words, **lmkw)
    path = str(tmp_path / "lm.b2clm")
    dec._language_model.ngram_model.save_blob(path)
    good = open(path, "rb").read()
    # header: magic u64, total u64, order i32, bos u32, eos u32, n_vocab u32, have i32, n_uni i32, key scheme i32,
    # reserved i32, then u64 off_uni, off_ngrams, ngram_mask, ...
    for off, fmt, bad in ((16, "<i", 99), (20, "<I", 0x7FFFFFFF), (40, "<i", 7), (48, "<Q", len(good) + 4096), (64, "<Q", 12345),
                          (56, "<Q", len(good) - 8)):
        data = bytearray(good)
        struct.pack_into(fmt, data, off, bad)
        bad_path = str(tmp_path / ("bad_%d.b2clm" % off))
        with open(bad_path, "wb") as fh:
            fh.write(bytes(data))
        with pytest.raises(ValueError):
            sim.build_ctcdecoder(wl.labels, kenlm_model_path=bad_path)
    with open(str(tmp_path / "short.b2clm"), "wb") as fh:
        fh.write(good[: len(good) // 2])
    with pytest.raises(ValueError):
        sim.build_ctcdecoder(wl.labels, kenlm_model_path=str(tmp_path / "short.b2clm"))


@pytest.mark.parametrize("name", goldens.unstable_case_names())
def test_hostsim_on_reference_unstable_goldens(sim, name):
    """Kernel logic on the cases the reference itself decides by rounding noise (tests/goldens.py run_unstable_case)."""
    def run(labels, x, **kw):
        return _beams(sim.build_ctcdecoder(labels).decode_beams(x, **kw))

    assert goldens.run_unstable_case(run, name) == ""


@pytest.mark.parametrize("fam", ["B_3gram", "B_5gram", "C_bpe_4gram"])
def test_hostsim_kenlm_binary_equals_arpa(sim, tmp_path, fam):
    """KenLM binary files of the probing model type (SURVEY 8f-3; reference decoder.py:1074 takes what kenlm.Model takes).
    The same model as ARPA text and in the binary layout (written by tests/kenlm_binary.py, an independent Python
    restatement of the published layout -- no kenlm-built file exists here, see csrc/b2c_lm_host.h) must give identical
    host queries and identical decodes; the binary's tables keep KenLM's own n-gram keys."""
    from tests import kenlm_binary

    wkw, lmkw = FAMILIES[fam]
    wl = synth.make_workload(wkw)
    path = str(tmp_path / "model.binary")
    info = kenlm_binary.write_probing_binary(wl.arpa, path)
    assert info["order"] == wkw["lm_order"]
    a = sim.NgramModel(wl.arpa, wl.words)
    b = sim.NgramModel(path, wl.words)
    assert b.order == a.order
    from pyctcdecode_b200.language_model import B200LMState as LMS
    rng = np.random.default_rng(5)
    st_a, st_b = LMS(), LMS()
    a.BeginSentenceWrite(st_a)
    b.BeginSentenceWrite(st_b)
    for i in range(300):
        w = wl.words[int(rng.integers(len(wl.words)))] if i % 7 else "zzzunknown"
        assert (w in a) == (w in b)
        na, nb = LMS(), LMS()
        assert a.BaseScore(st_a, w, na) == b.BaseScore(st_b, w, nb)
        assert na.backoffs == nb.backoffs and len(na.words) == len(nb.words)
        st_a, st_b = (na, nb) if i % 11 else (LMS(), LMS())
    dec_a = sim.build_ctcdecoder(wl.labels, kenlm_model_path=wl.arpa, unigrams=wl.words, **lmkw)
    dec_b = sim.build_ctcdecoder(wl.labels, kenlm_model_path=path, unigrams=wl.words, **lmkw)
    for i in range(4):
        x = wl.utterance(8800 + i, 70 if wl.V <= 64 else 30, ["peaky", "diffuse"][i % 2])
        assert _beams(dec_a.decode_beams(x, beam_width=24, hotwords=[wl.words[4]])) == _beams(dec_b.decode_beams(x, beam_width=24, hotwords=[wl.words[4]]))


def test_hostsim_kenlm_binary_rejects_what_it_cannot_read(sim, tmp_path):
    from tests import kenlm_binary

    wl = synth.make_workload(FAMILIES["B_3gram"][0])
    path = str(tmp_path / "model.bin")
    kenlm_binary.write_probing_binary(wl.arpa, path)
    good = bytearray(open(path, "rb").read())
    cases = {"trie.bin": (88 + 8, b"\x02\x00\x00\x00"),           # model_type = TRIE
             "novocab.bin": (88 + 12, b"\x00"),                  # has_vocabulary = false
             "counts.bin": (88 + 20, b"\x07\x00\x00\x00"),       # unigram count changed: the sections no longer line up
             "version.bin": (49, b"4")}                          # format version 4
    for name, (off, patch) in cases.items():
        data = bytearray(good)
        data[off:off + len(patch)] = patch
        p = str(tmp_path / name)
        open(p, "wb").write(bytes(data))
        with pytest.raises((ValueError, OSError, RuntimeError)):
            sim.NgramModel(p, wl.words).order          # the file is parsed when the model is first used
    open(str(tmp_path / "cut.bin"), "wb").write(bytes(good[: len(good) * 2 // 3]))
    with pytest.raises((ValueError, OSError, RuntimeError)):
        sim.NgramModel(str(tmp_path / "cut.bin"), wl.words).order


@pytest.mark.parametrize("chunks", ["2", "5"])
def test_hostsim_chunked_launches_give_the_same_results(chunks):
    """Chunked launches of the latency-first kernel (frames [t0, t1) per launch, state parked in HBM in between -- what
    the pipelined host path runs) forced for every call (B200CTC_FORCE_CHUNKS): the parity tests must pass unchanged."""
    import sys
    env = dict(os.environ, B200CTC_FORCE_CHUNKS=chunks, B200CTC_FORCE_V5="1")
    here = os.path.abspath(__file__)
    r = subprocess.run([sys.executable, "-m", "pytest", here, "-x", "-q", "-k", "golden or special or random or ragged or text_only"],
                       env=env, cwd=os.path.dirname(os.path.dirname(here)), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout[-3000:]


@pytest.mark.parametrize("fam,dtype", [("B_3gram", np.float32), ("C_bpe_4gram", np.float32), ("B_nolm", np.float64)])
def test_hostsim_pipelined_host_batches(sim, fam, dtype, monkeypatch):
    monkeypatch.setenv("B200CTC_PIPELINE_ALL", "1")        # also compute-bound calls (by default only copy-bound ones)
    """The pipelined call (one [B, T, V] host block, second call of a configuration onwards): chunks along T are
    copied / prepared / decoded in turn.  Same transcripts and beams as the plain call; probability input -- found
    out only after the last chunk -- makes the call redo itself as a plain call."""
    wkw, lmkw = FAMILIES[fam]
    wl = synth.make_workload(wkw)
    kw = dict(lmkw)
    if wl.arpa:
        kw.update(kenlm_model_path=wl.arpa, unigrams=wl.words)
    dec = sim.build_ctcdecoder(wl.labels, **kw)
    ora = orc.OracleDecoder(wl.labels, **kw)
    T = 300
    xs = np.stack([wl.utterance(9100 + i, T, ["peaky", "diffuse"][i % 2] if wl.V <= 64 else "peaky") for i in range(5)]).astype(dtype)
    want = ora.decode_batch(list(xs), beam_width=24)
    assert dec.decode_batch(None, xs, beam_width=24) == want            # first call: plain (no hint yet)
    launches_plain = dec.last_timings()["launches"]
    assert dec.decode_batch(None, xs, beam_width=24) == want            # second call: pipelined
    assert dec.last_timings()["launches"] > launches_plain               # one streaming + one beam launch per chunk
    got = dec.decode_beams_batch(None, xs, beam_width=24)
    ref = ora.decode_beams_batch(list(xs), beam_width=24)
    for w, g in zip(ref, got):
        _compare(w, _beams(g))
    # probabilities in one utterance of the block: the pipelined attempt notices at the end and the call is redone
    e = np.exp(xs - xs.max(2, keepdims=True))
    probs = (e / e.sum(2, keepdims=True)).astype(dtype)
    want_p = ora.decode_batch(list(probs), beam_width=24)
    assert dec.decode_batch(None, probs, beam_width=24) == want_p
    assert dec.decode_batch(None, probs, beam_width=24) == want_p


def test_hostsim_gated_launch_gives_up_cleanly(sim, monkeypatch):
    """A gated launch whose later chunks never become ready (here: hostsim launches the beam kernel right after the
    first chunk) must give up with B2C_ERR_GATE -- no hang, no garbage -- and the call is redone as a plain call."""
    monkeypatch.setenv("B200CTC_PIPELINE_ALL", "1")
    monkeypatch.setenv("B200CTC_HOSTSIM_GATE_EARLY", "1")
    wkw, lmkw = FAMILIES["B_3gram"]
    wl = synth.make_workload(wkw)
    kw = dict(lmkw, kenlm_model_path=wl.arpa, unigrams=wl.words)
    dec = sim.build_ctcdecoder(wl.labels, **kw)
    ora = orc.OracleDecoder(wl.labels, **kw)
    xs = np.stack([wl.utterance(9300 + i, 300, "peaky") for i in range(4)])
    want = ora.decode_batch(list(xs), beam_width=24)
    for _ in range(3):
        assert dec.decode_batch(None, xs, beam_width=24) == want


def test_hostsim_hinted_plain_calls(sim):
    """Hinted plain calls (any input that is not pipelined: lists of arrays, device tensors): from the second call of
    a configuration the beam kernel is planned from the previous call's statistics and launched without waiting for
    this call's -- the same results; a batch whose statistics ask for another plan (here: diffuse posteriors after
    peaky ones) is found out (hint-only plan != last statistics-based plan, or the refresh every 32nd call) and is
    planned from its statistics."""
    wkw, lmkw = FAMILIES["B_nolm"]
    wl = synth.make_workload(wkw)
    dec = sim.build_ctcdecoder(wl.labels)
    ora = orc.OracleDecoder(wl.labels)
    peaky = [wl.utterance(9500 + i, 200 + 10 * i, "peaky") for i in range(4)]
    want = ora.decode_batch(peaky, beam_width=32)
    flags = []
    for _ in range(3):
        assert dec.decode_batch(None, peaky, beam_width=32) == want
        flags.append(dec.last_timings()["hinted"])
    assert flags == [0, 1, 1]
    # another beam width is another configuration: its first call plans from the statistics
    want16 = ora.decode_batch(peaky, beam_width=16)
    assert dec.decode_batch(None, peaky, beam_width=16) == want16
    assert dec.last_timings()["hinted"] == 0
    assert dec.decode_batch(None, peaky, beam_width=16) == want16
    assert dec.last_timings()["hinted"] == 1
    # full beams (decode_beams_batch) through hinted calls
    ref = ora.decode_beams_batch(peaky, beam_width=16)
    for w, g in zip(ref, dec.decode_beams_batch(None, peaky, beam_width=16)):
        _compare(w, _beams(g))
    # diffuse posteriors behind the same configuration: correct whichever way each call was planned, over a refresh
    diffuse = [wl.utterance(9600 + i, 120, "diffuse") for i in range(3)]
    want_d = ora.decode_batch(diffuse, beam_width=16)
    for _ in range(40):
        assert dec.decode_batch(None, diffuse, beam_width=16) == want_d
    assert dec.decode_batch(None, peaky, beam_width=16) == want16
