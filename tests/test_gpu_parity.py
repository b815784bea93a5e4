"""GPU parity tests (`pytest -m gpu`, run on the B200 box): the CUDA path through the C ABI
against (a) the golden vectors generated from the unmodified reference, (b) the CPU oracle on
seeded inputs at sizes the oracle finishes in seconds, (c) size-independent properties at
BASELINE.json's full sizes.  Nothing here reads /root/reference.

Tolerances: transcripts and word frames must be identical; beam scores within 1e-9 relative of
the oracle (same float64 operation order; only CUDA's vs glibc's exp/log can differ in the
last bit) and within 2e-4 absolute of the numpy-evaluated reference goldens (numpy computes
the float32 log-softmax with its own SIMD exp/log, see DESIGN.md)."""
import os

import numpy as np
import pytest

from tests import goldens, synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    g.build()
    import pyctcdecode_b200
    from pyctcdecode_b200 import _lib
    _lib._lib = None  # make sure the real CUDA library is bound, not a test build
    L = _lib.lib()
    assert _lib.library_path() == _lib.DEFAULT_LIBRARY
    if L.b2c_device_count() < 1:
        pytest.skip("no CUDA device on this machine (the GPU parity tests run on the B200 box)")
    return pyctcdecode_b200


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    oracle.build()
    return oracle


def _beams(out):
    return [(b.text, b.text_frames, b.logit_score, b.lm_score) for b in out]


def _compare(ref, got, tol=1e-9):
    assert len(ref) == len(got)
    for r, g in zip(ref, got):
        assert r[0] == g[0]
        assert [(w, tuple(f)) for w, f in r[1]] == [(w, tuple(f)) for w, f in g[1]]
        assert abs(r[2] - g[2]) <= tol * max(1.0, abs(r[2]))
        assert abs(r[3] - g[3]) <= tol * max(1.0, abs(r[3]))


def _names():
    return [c["name"] for c in goldens.load()["meta"]["cases"]]


@pytest.mark.parametrize("name", goldens.unstable_case_names(gpu=True))
def test_gpu_on_reference_unstable_goldens(pkg, name):
    """Cases the unmodified reference decides by rounding noise (oracle/gen_golden_unstable.py): the CUDA path must
    lie inside the family of reference outcomes (same beam set, per-beam scores among the family's, sorted)."""
    def run(labels, x, **kw):
        return _beams(pkg.build_ctcdecoder(labels).decode_beams(x, **kw))

    assert goldens.run_unstable_case(run, name) == ""


@pytest.mark.parametrize("name", _names())
def test_gpu_matches_reference_golden(pkg, golden, name):
    case = next(c for c in golden["meta"]["cases"] if c["name"] == name)
    dec = goldens.build_product_decoder(pkg, case["labels"], **goldens.lm_kwargs(golden, case))
    x = golden["arrays"][case["array"]]
    assert goldens.beams_match(case["beams"], _beams(dec.decode_beams(x, **case["decode"]))) == ""
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


@pytest.mark.parametrize("fam", sorted(FAMILIES))
def test_gpu_vs_oracle_random(pkg, orc, fam):
    wkw, lmkw = FAMILIES[fam]
    wl = synth.make_workload(wkw)
    kw = dict(lmkw)
    if wl.arpa:
        kw.update(kenlm_model_path=wl.arpa, unigrams=wl.words)
    dec = pkg.build_ctcdecoder(wl.labels, **kw)
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


@pytest.mark.parametrize("regime,lm_order,B", [("peaky", 0, 48), ("diffuse", 0, 12), ("peaky", 3, 48), ("diffuse", 3, 16)])
def test_gpu_vs_oracle_headline_shape(pkg, orc, regime, lm_order, B):
    """Wav2Vec2-shaped utterances (T=1000, V=32, beam=100): decode_batch() transcripts identical to
    the oracle's decode(), decode_beams_batch() beams identical incl. frames and scores."""
    wl = synth.CharWorkload("B", n_words=5000, lm_order=lm_order)
    kw = dict(kenlm_model_path=wl.arpa, unigrams=wl.words, alpha=0.5, beta=1.0) if lm_order else {}
    dec = pkg.build_ctcdecoder(wl.labels, **kw)
    ora = orc.OracleDecoder(wl.labels, **kw)
    xs = wl.batch(10_000, B, 1000, regime)
    threads = os.cpu_count() or 1
    assert dec.decode_batch(None, xs, beam_width=100) == ora.decode_batch(xs, n_threads=threads, beam_width=100)
    got = dec.decode_beams_batch(None, xs[:8], beam_width=100)
    want = ora.decode_beams_batch(xs[:8], n_threads=threads, beam_width=100)
    for w, g in zip(want, got):
        _compare(w, _beams(g))


def test_gpu_bpe_hotwords_batch(pkg, orc):
    """Conformer-like BPE vocabulary (V=1024, T=500) with a 4-gram model and hotwords."""
    wl = synth.BpeWorkload(n_words=3000, lm_order=4)
    kw = dict(kenlm_model_path=wl.arpa, unigrams=wl.words, alpha=0.5, beta=1.0)
    dec = pkg.build_ctcdecoder(wl.labels, **kw)
    ora = orc.OracleDecoder(wl.labels, **kw)
    xs = wl.batch(20_000, 24, 500, "peaky") + wl.batch(21_000, 4, 300, "diffuse")
    hot = wl.hotwords()
    threads = os.cpu_count() or 1
    assert dec.decode_batch(None, xs, beam_width=100, hotwords=hot) == ora.decode_batch(xs, n_threads=threads, beam_width=100, hotwords=hot)


def test_gpu_full_size_properties(pkg):
    """BASELINE config C2 (B=256, T=1000, V=32, beam=100): size-independent properties --
    batch decode equals per-utterance decode (shards are independent), repeat calls are
    bit-identical, device-resident input equals host input, any permutation of the batch gives
    the permuted result."""
    import torch

    wl = synth.CharWorkload("B", n_words=20000, lm_order=0)
    dec = pkg.build_ctcdecoder(wl.labels)
    xs = wl.batch(1, 256, 1000, "peaky")
    full = dec.decode_batch(None, xs, beam_width=100)
    assert full == dec.decode_batch(None, xs, beam_width=100)
    for i in (0, 17, 101, 255):
        assert dec.decode(xs[i], beam_width=100) == full[i]
    perm = np.random.default_rng(0).permutation(256)
    assert dec.decode_batch(None, [xs[i] for i in perm], beam_width=100) == [full[i] for i in perm]
    dev = torch.from_numpy(np.stack(xs)).cuda()
    assert dec.decode_batch(None, [dev[i] for i in range(256)], beam_width=100) == full
    assert all(len(t) > 0 for t in full)


def test_gpu_beam_width_sweep(pkg, orc):
    wl = synth.CharWorkload("B", n_words=5000, lm_order=0)
    dec = pkg.build_ctcdecoder(wl.labels)
    ora = orc.OracleDecoder(wl.labels)
    xs = wl.batch(30_000, 6, 400, "peaky")
    for bw in (10, 50, 500, 2000):
        assert dec.decode_batch(None, xs, beam_width=bw) == ora.decode_batch(xs, n_threads=os.cpu_count() or 1, beam_width=bw)


def test_gpu_ragged_and_empty(pkg, orc):
    wl = synth.CharWorkload("A", n_words=400, lm_order=2)
    kw = dict(kenlm_model_path=wl.arpa, unigrams=wl.words)
    dec = pkg.build_ctcdecoder(wl.labels, **kw)
    ora = orc.OracleDecoder(wl.labels, **kw)
    Ts = [40, 0, 77, 5, 120, 1, 33, 0]
    xs = [wl.utterance(900 + i, T, "diffuse" if i % 2 else "peaky") if T else np.zeros((0, wl.V), np.float32) for i, T in enumerate(Ts)]
    assert dec.decode_batch(None, xs, beam_width=25) == ora.decode_batch(xs, beam_width=25)
    assert dec.decode_batch(None, [], beam_width=25) == []
    with pytest.raises(ValueError):
        dec.decode(np.zeros((4, 7), np.float32))


@pytest.mark.parametrize("variant", ["0", "1", "2", "general"])
def test_gpu_kernel_variants_agree(pkg, orc, variant, monkeypatch):
    """Every beam-kernel variant (latency-first 1024x2 / 512x3 / 256x4 CTAs per SM, and the general kernel with
    the latency-first one disabled) must give the oracle's beams, including on frames that overflow the
    shared-memory candidate tier (diffuse utterances force the out-of-line HBM-tier step)."""
    if variant == "general":
        monkeypatch.setenv("B200CTC_NO_V5", "1")
    else:
        monkeypatch.setenv("B200CTC_V5_VARIANT", variant)
        monkeypatch.setenv("B200CTC_FORCE_V5", "1")
    wl = synth.CharWorkload("B", n_words=2000, lm_order=3)
    kw = dict(kenlm_model_path=wl.arpa, unigrams=wl.words, alpha=0.5, beta=1.0)
    dec = pkg.build_ctcdecoder(wl.labels, **kw)
    ora = orc.OracleDecoder(wl.labels, **kw)
    xs = wl.batch(40_000, 10, 300, "peaky") + wl.batch(41_000, 6, 200, "diffuse")
    threads = os.cpu_count() or 1
    got = dec.decode_beams_batch(None, xs, beam_width=100, prune_history=True)
    tm = dec.last_timings()
    assert tm["kernel_variant"] == (2 if variant != "general" else tm["kernel_variant"])
    want = ora.decode_beams_batch(xs, n_threads=threads, beam_width=100, prune_history=True)
    for w, g in zip(want, got):
        _compare(w, _beams(g))
    dec2 = pkg.build_ctcdecoder(wl.labels)          # no LM: the text arena is bypassed in the latency-first kernel
    ora2 = orc.OracleDecoder(wl.labels)
    assert dec2.decode_batch(None, xs, beam_width=100) == ora2.decode_batch(xs, n_threads=threads, beam_width=100)


def test_gpu_padded_batch_lengths_and_half_precision(pkg):
    """SURVEY 8f-4: one padded [B, T, V] CUDA tensor + lengths (the padding rows are never read), and
    fp16 / bf16 tensors (widened to float32 on the device) decode like the per-utterance float32 arrays."""
    import torch

    wl = synth.CharWorkload("B", n_words=2000, lm_order=0)
    dec = pkg.build_ctcdecoder(wl.labels)
    Ts = [300, 120, 1, 0, 257, 300, 33, 64, 299]
    xs = [wl.utterance(50_000 + i, T, "peaky") if T else np.zeros((0, wl.V), np.float32) for i, T in enumerate(Ts)]
    want = dec.decode_batch(None, xs, beam_width=50)
    pad = np.full((len(Ts), 300, wl.V), np.nan, np.float32)      # NaN padding: reading it would poison the result
    for i, x in enumerate(xs):
        pad[i, :len(x)] = x
    dev = torch.from_numpy(pad).cuda()
    assert dec.decode_batch(None, dev, beam_width=50, lengths=Ts) == want
    assert dec.decode_batch(None, pad, beam_width=50, lengths=Ts) == want
    beams = dec.decode_beams_batch(None, dev, beam_width=50, lengths=Ts)
    assert [b[0].text for b in beams] == want
    with pytest.raises(ValueError):
        dec.decode_batch(None, dev, beam_width=50, lengths=Ts[:-1])
    # half precision: the values are rounded by the caller; decoding the widened values must match
    full = torch.from_numpy(np.stack([wl.utterance(51_000 + i, 200, "peaky") for i in range(6)]))
    for dt in (torch.float16, torch.bfloat16):
        h = full.to(dt).cuda()
        ref = dec.decode_batch(None, h.float().cpu().numpy(), beam_width=50)
        assert dec.decode_batch(None, h, beam_width=50) == ref
        assert dec.decode(h[2], beam_width=50) == ref[2]
        assert dec.decode_batch(None, h, beam_width=50, lengths=[200, 150, 1, 0, 77, 200]) == \
            dec.decode_batch(None, h.float(), beam_width=50, lengths=[200, 150, 1, 0, 77, 200])
        assert dec.decode_batch(None, [t for t in h.cpu()], beam_width=50) == ref         # host tensors: 2-byte H2D
    h16 = full.numpy().astype(np.float16)
    assert dec.decode_batch(None, [x for x in h16], beam_width=50) == dec.decode_batch(None, h16.astype(np.float32), beam_width=50)


@pytest.mark.parametrize("variant", ["0", "1", "2"])
def test_gpu_special_single_token_steps(pkg, orc, variant, monkeypatch):
    """In-place single-token frames and merge-free sorted frames (b2c_fast_cheap_step / b2c_fast_sorted_step)
    on the device against the oracle: varying sharpness, exact ties (integer logits), beams from 2 to 128, in
    every capacity variant of the latency-first kernel."""
    monkeypatch.setenv("B200CTC_V5_VARIANT", variant)
    monkeypatch.setenv("B200CTC_FORCE_V5", "1")
    wl = synth.make_workload(dict(kind="char", vocab="B", n_words=400, lm_order=0))
    dec = pkg.build_ctcdecoder(wl.labels)
    ora = orc.OracleDecoder(wl.labels)
    inplace = ranked = 0
    for n, (x, kw) in enumerate(synth.special_step_cases(wl)):
        got = _beams(dec.decode_beams(x, **kw))
        tm = dec.last_timings()
        inplace += tm["inplace_frames"]
        ranked += tm["sorted_frames"]
        want = ora.decode_beams(x, **kw)
        try:
            _compare(want, got)
        except AssertionError as e:
            first = next((j for j, (w, g) in enumerate(zip(want, got)) if w[0] != g[0] or abs(w[3] - g[3]) > 1e-9 * max(1.0, abs(w[3]))), -1)
            raise AssertionError("case %d T=%d %r: %d vs %d beams, first difference at beam %d: want %r got %r; timings %r"
                                 % (n, x.shape[0], kw, len(want), len(got), first, want[first] if first >= 0 else None,
                                    got[first] if 0 <= first < len(got) else None,
                                    {k: tm[k] for k in ("kernel_variant", "cap_candidates", "oversize_frames", "inplace_frames", "sorted_frames")})) from e
    assert inplace > 1000 and ranked > 100, (inplace, ranked)


@pytest.mark.parametrize("name", goldens.stream_case_names())
def test_gpu_streaming_matches_reference_golden(pkg, name):
    """get_starting_state / partial_decode_beams on the device, call by call, against the outputs of the
    unmodified reference (tests/golden/stream_cases.json, oracle/gen_golden_stream.py)."""
    assert goldens.run_stream_case(pkg, name) == ""


def test_gpu_streaming_batch_equals_whole(pkg):
    wl = synth.make_workload(dict(kind="char", vocab="B", n_words=400, lm_order=3))
    dec = pkg.build_ctcdecoder(wl.labels, kenlm_model_path=wl.arpa, unigrams=wl.words, alpha=0.5, beta=1.0)
    T = 300
    xs = [wl.utterance(8300 + i, T, ["peaky", "diffuse"][i % 2]) for i in range(12)]
    whole = dec.decode_beams_batch(None, xs, beam_width=32)
    states = [dec.get_starting_state() for _ in xs]
    beams, caches = [s[0] for s in states], [s[1] for s in states]
    for a in range(0, T, 64):
        b = min(T, a + 64)
        beams = dec.partial_decode_beams_batch([x[a:b] for x in xs], caches, beams, [a] * len(xs), beam_width=32, is_end=(b == T))
    for w, got in zip(whole, beams):
        assert [o.text for o in w] == [g.text for g in got]
        assert [[f for _, f in o.text_frames] for o in w] == [[tuple(f) for f in g.text_frames] for g in got]
        for o, g in zip(w, got):
            assert abs(o.logit_score - g.logit_score) <= 1e-9 * max(1.0, abs(o.logit_score))
            assert abs(o.lm_score - g.lm_score) <= 1e-9 * max(1.0, abs(o.lm_score))


@pytest.mark.parametrize("name", goldens.multilm_case_names())
def test_gpu_multi_language_model_matches_reference_golden(pkg, name):
    """MultiLanguageModel on the device against the unmodified reference (tests/golden/multilm_cases.json)."""
    assert goldens.run_multilm_case(pkg, name) == ""


@pytest.mark.parametrize("fam", ["3gram", "5gram"])
def test_gpu_scored_in_place_frames_with_lm(pkg, orc, fam):
    """b2c_fast_scored_step / the scored form of b2c_inplace_step on the device against the oracle (LM + hotwords)."""
    wkw, lmkw = {"3gram": (dict(kind="char", vocab="B", n_words=400, lm_order=3), dict(alpha=0.5, beta=1.0)),
                 "5gram": (dict(kind="char", vocab="B", n_words=150, lm_order=5), dict(alpha=0.9, beta=0.3, unk_score_offset=-4.0))}[fam]
    wl = synth.make_workload(wkw)
    kw = dict(lmkw, kenlm_model_path=wl.arpa, unigrams=wl.words)
    dec = pkg.build_ctcdecoder(wl.labels, **kw)
    ora = orc.OracleDecoder(wl.labels, **kw)
    inplace = frames = 0
    for i, (x, dkw) in enumerate(synth.special_step_cases(wl, n_cases=40, seed=11)):
        if i % 4 == 1:
            dkw = dict(dkw, hotwords=[wl.words[2], wl.words[7] + " " + wl.words[9]], hotword_weight=7.5)
        if i % 5 == 3:
            dkw = dict(dkw, beam_width=300)          # general kernel
        got = _beams(dec.decode_beams(x, **dkw))
        tm = dec.last_timings()
        inplace += tm["inplace_frames"]
        frames += tm["frames"]
        _compare(ora.decode_beams(x, **dkw), got)
    assert inplace > 0.4 * frames, (inplace, frames)


# ---- BASELINE.json configurations at FULL size against the oracle (VERDICT r1, weak 2) -----------------------------
def _threads():
    import bench
    return bench.host_cores()


def test_gpu_full_size_c3_vs_oracle(pkg, orc):
    """C3: B=1024, T=1000, V=32, beam 100 + 3-gram (alpha 0.5, beta 1.0): every transcript identical to the oracle's."""
    import bench
    spec = bench.WORKLOADS["c3"]
    wl, kw, hot = bench.workload_objects(spec)
    dec = pkg.build_ctcdecoder(wl.labels, **kw)
    ora = orc.OracleDecoder(wl.labels, **kw)
    xs = wl.batch(1, spec["batch"], spec["T"], "peaky")
    got = dec.decode_batch(None, xs, beam_width=100)
    assert got == dec.decode_batch(None, np.stack(xs), beam_width=100)       # second call: the residency variant chosen from the hint
    want = ora.decode_batch(xs, n_threads=_threads(), beam_width=100)
    bad = [i for i, (a, b) in enumerate(zip(want, got)) if a != b]
    assert not bad, "%d of %d transcripts differ, first: %r vs %r" % (len(bad), len(xs), want[bad[0]], got[bad[0]])


@pytest.mark.parametrize("dtype", ["f32", "f16"])
def test_gpu_full_size_c4_shape_vs_oracle(pkg, orc, dtype):
    """C4 shape on one GPU: B=512, T=500, V=1024 BPE, beam 100 + 4-gram + 16 hotwords, float32 and float16 logits."""
    import bench
    spec = bench.WORKLOADS["c4"]
    wl, kw, hot = bench.workload_objects(spec)
    dec = pkg.build_ctcdecoder(wl.labels, **kw)
    ora = orc.OracleDecoder(wl.labels, **kw)
    xs = wl.batch(1, spec["batch"], spec["T"], "peaky")
    if dtype == "f16":
        xs16 = [x.astype(np.float16) for x in xs]
        xs = [x.astype(np.float32) for x in xs16]
        got = dec.decode_batch(None, np.stack(xs16), beam_width=100, hotwords=hot)
    else:
        got = dec.decode_batch(None, xs, beam_width=100, hotwords=hot)
    want = ora.decode_batch(xs, n_threads=_threads(), beam_width=100, hotwords=hot)
    bad = [i for i, (a, b) in enumerate(zip(want, got)) if a != b]
    assert not bad, "%d of %d transcripts differ, first: %r vs %r" % (len(bad), len(xs), want[bad[0]], got[bad[0]])


@pytest.mark.parametrize("beam,B", [(10, 256), (50, 256), (500, 64), (2000, 24)])
def test_gpu_full_T_beam_sweep_vs_oracle(pkg, orc, beam, B):
    """C5 shape (T=1000, V=32): the beam sweep against the oracle; the wide beams on as many utterances as the oracle
    finishes in seconds on the box's host cores."""
    wl = synth.CharWorkload("B", n_words=20000, lm_order=0)
    dec = pkg.build_ctcdecoder(wl.labels)
    ora = orc.OracleDecoder(wl.labels)
    xs = wl.batch(1, B, 1000, "peaky")
    got = dec.decode_batch(None, xs, beam_width=beam)
    want = ora.decode_batch(xs, n_threads=_threads(), beam_width=beam)
    bad = [i for i, (a, b) in enumerate(zip(want, got)) if a != b]
    assert not bad, "%d of %d transcripts differ" % (len(bad), len(xs))
    g = dec.decode_beams_batch(None, xs[:2], beam_width=beam)
    w = ora.decode_beams_batch(xs[:2], n_threads=2, beam_width=beam)
    for a, b in zip(w, g):
        _compare(a, _beams(b))


def test_gpu_differential_fuzz(pkg):
    """tools/fuzz_hostsim.py through the CUDA library (VERDICT r1: 'differential fuzzing never runs on the device'):
    random vocabulary family / LM / hotwords / prune settings / beams 1-300 / sharpness / exact ties / chunked streaming."""
    from tools import fuzz_hostsim
    assert fuzz_hostsim.fuzz(220, 2027) == 0


def test_gpu_decoder_is_thread_safe(pkg):
    """8 threads on one decoder object: calls are serialised inside the handle, every thread gets the lone-call result."""
    import threading

    wl = synth.make_workload(dict(kind="char", vocab="B", n_words=400, lm_order=3))
    dec = pkg.build_ctcdecoder(wl.labels, kenlm_model_path=wl.arpa, unigrams=wl.words, alpha=0.5, beta=1.0)
    xs = [wl.utterance(8600 + i, 80 + 11 * i, ["peaky", "diffuse"][i % 2]) for i in range(8)]
    want = [(dec.decode(x, beam_width=32), _beams(dec.decode_beams(x, beam_width=32))) for x in xs]
    got, errors = [None] * len(xs), []

    def work(i):
        try:
            for _ in range(10):
                got[i] = (dec.decode(xs[i], beam_width=32), _beams(dec.decode_beams(xs[i], beam_width=32)))
        except Exception as exc:  # pragma: no cover
            errors.append(exc)

    threads = [threading.Thread(target=work, args=(i,)) for i in range(len(xs))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors
    assert got == want


def test_gpu_tensor_device_and_stream_order(pkg):
    """CUDA tensors: the decoder of the tensors' device runs (a decoder bound to another device raises), and logits
    still being written on a side stream are waited for (the decoder's stream waits on torch's current stream)."""
    import torch

    wl = synth.CharWorkload("B", n_words=2000, lm_order=0)
    dec = pkg.build_ctcdecoder(wl.labels)
    x = torch.from_numpy(np.stack(wl.batch(61_000, 16, 400, "peaky")))
    want = dec.decode_batch(None, x.numpy(), beam_width=50)
    side = torch.cuda.Stream()
    for _ in range(3):
        with torch.cuda.stream(side):
            big = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
            for _ in range(20):
                big.fill_(1)                                  # ~ms of queued work ahead of the producer of the logits
            dev = torch.zeros_like(x, device="cuda")
            dev.copy_(x.pin_memory(), non_blocking=True)
            assert dec.decode_batch(None, dev, beam_width=50) == want
    bound = pkg.build_ctcdecoder(wl.labels, device=0)
    assert bound.decode_batch(None, dev, beam_width=50) == want
    if torch.cuda.device_count() > 1:
        other = x.to("cuda:1")
        with pytest.raises(ValueError):
            bound.decode_batch(None, other, beam_width=50)
        assert dec.decode_batch(None, other, beam_width=50) == want          # unbound decoder: follows the tensor
        with pytest.raises(ValueError):
            dec.decode_batch(None, [dev[0], other[1]], beam_width=50)


def test_gpu_kenlm_binary_equals_arpa(pkg, tmp_path):
    """A KenLM binary (probing layout, written by tests/kenlm_binary.py) decodes on the device exactly like the ARPA
    text of the same model: the device tables keep KenLM's own n-gram keys (csrc/b2c_lm.h key_scheme)."""
    from tests import kenlm_binary

    wl = synth.make_workload(dict(kind="char", vocab="B", n_words=2000, lm_order=4))
    path = str(tmp_path / "model.binary")
    kenlm_binary.write_probing_binary(wl.arpa, path)
    kw = dict(unigrams=wl.words, alpha=0.6, beta=1.2)
    dec_a = pkg.build_ctcdecoder(wl.labels, kenlm_model_path=wl.arpa, **kw)
    dec_b = pkg.build_ctcdecoder(wl.labels, kenlm_model_path=path, **kw)
    xs = wl.batch(70_000, 24, 300, "peaky") + wl.batch(71_000, 8, 200, "diffuse")
    assert dec_a.decode_batch(None, xs, beam_width=100) == dec_b.decode_batch(None, xs, beam_width=100)
    a = dec_a.decode_beams_batch(None, xs[:6], beam_width=50, hotwords=[wl.words[3]])
    b = dec_b.decode_beams_batch(None, xs[:6], beam_width=50, hotwords=[wl.words[3]])
    assert [_beams(x) for x in a] == [_beams(x) for x in b]


def test_gpu_pipelined_host_batches(pkg, orc, monkeypatch):
    monkeypatch.setenv("B200CTC_PIPELINE_ALL", "1")        # also compute-bound calls (by default only copy-bound ones)
    """Pipelined calls on the device: a [B, T, V] float32 host block is cut into chunks along T, chunk c+1 crosses PCIe
    while chunk c runs through the lane-per-row streaming kernel and a chunked launch of the beam kernel (state parked
    in HBM between launches).  Second call of a configuration onwards; same results as the plain call (first call),
    with and without an LM; probability input falls back to a plain call."""
    for lm_order in (0, 3):
        wl = synth.CharWorkload("B", n_words=5000, lm_order=lm_order)
        kw = dict(kenlm_model_path=wl.arpa, unigrams=wl.words, alpha=0.5, beta=1.0) if lm_order else {}
        dec = pkg.build_ctcdecoder(wl.labels, **kw)
        ora = orc.OracleDecoder(wl.labels, **kw)
        xs = np.stack(wl.batch(81_000, 40, 1000, "peaky"))
        want = ora.decode_batch(list(xs), n_threads=_threads(), beam_width=100)
        assert dec.decode_batch(None, xs, beam_width=100) == want
        plain = dec.last_timings()["launches"]
        for _ in range(3):
            assert dec.decode_batch(None, xs, beam_width=100) == want
        assert dec.last_timings()["launches"] > plain
        got = dec.decode_beams_batch(None, xs[:6], beam_width=100)
        got = dec.decode_beams_batch(None, xs[:6], beam_width=100)
        ref = ora.decode_beams_batch(list(xs[:6]), n_threads=6, beam_width=100)
        for w, g in zip(ref, got):
            _compare(w, _beams(g))
    e = np.exp(xs[:8] - xs[:8].max(2, keepdims=True))
    probs = (e / e.sum(2, keepdims=True)).astype(np.float32)
    want_p = ora.decode_batch(list(probs), n_threads=8, beam_width=100)
    assert dec.decode_batch(None, probs, beam_width=100) == want_p
    assert dec.decode_batch(None, probs, beam_width=100) == want_p


@pytest.mark.parametrize("chunks", ["3"])
def test_gpu_chunked_launches_give_the_same_results(chunks):
    """B200CTC_FORCE_CHUNKS on the device: chunked launches of the latency-first kernel for every call of a child
    pytest run over the special-step and ragged cases."""
    import subprocess
    import sys
    env = dict(os.environ, B200CTC_FORCE_CHUNKS=chunks, B200CTC_FORCE_V5="1")
    here = os.path.abspath(__file__)
    r = subprocess.run([sys.executable, "-m", "pytest", here, "-x", "-q", "-m", "gpu", "-k", "special_single or ragged or headline_shape"],
                       env=env, cwd=os.path.dirname(os.path.dirname(here)), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout[-3000:]


@pytest.mark.gpu
def test_gpu_hinted_plain_calls(pkg, orc):
    """From the second call of a configuration the beam kernel is planned from the previous call's statistics and
    launched without waiting for this call's (device tensors and lists of arrays; b2c_timings_t.hinted): same results;
    another beam width is another configuration; diffuse posteriors behind a peaky hint are decoded correctly whichever
    way each call was planned (over a refresh call)."""
    import torch
    wl = synth.make_workload(dict(kind="char", vocab="B", n_words=400, lm_order=0))
    dec = pkg.build_ctcdecoder(wl.labels)
    ora = orc.OracleDecoder(wl.labels)
    peaky = np.stack([wl.utterance(9500 + i, 400, "peaky") for i in range(24)])
    want = ora.decode_batch(list(peaky), beam_width=32)
    dev = torch.from_numpy(peaky).cuda()
    flags = []
    for _ in range(3):
        assert dec.decode_batch(None, dev, beam_width=32) == want
        flags.append(dec.last_timings()["hinted"])
    assert flags == [0, 1, 1]
    # a ragged list of host arrays (not one [B, T, V] block, so not a pipelined call): hinted as well
    ragged = [wl.utterance(9550 + i, 300 + 7 * i, "peaky") for i in range(12)]
    want16 = ora.decode_batch(ragged, beam_width=16)
    assert dec.decode_batch(None, ragged, beam_width=16) == want16
    assert dec.last_timings()["hinted"] == 0
    assert dec.decode_batch(None, ragged, beam_width=16) == want16
    assert dec.last_timings()["hinted"] == 1
    diffuse = [wl.utterance(9600 + i, 150 + i, "diffuse") for i in range(6)]
    want_d = ora.decode_batch(diffuse, beam_width=16)
    for _ in range(36):
        assert dec.decode_batch(None, diffuse, beam_width=16) == want_d
    assert dec.decode_batch(None, ragged, beam_width=16) == want16


@pytest.mark.gpu
def test_gpu_wide_alphabet_rows_with_special_values(pkg, orc):
    """The warp-per-row streaming kernel (V > 32, float32) takes its branch-free path only for rows without NaN /
    infinity; rows with -inf (masked vocabulary entries), +inf or NaN go through the general routine.  Same tokens and
    scores as the oracle either way (masked entries; the other special values in a few rows of every utterance)."""
    wl = synth.make_workload(dict(kind="bpe", n_words=400, lm_order=0))
    dec = pkg.build_ctcdecoder(wl.labels)
    ora = orc.OracleDecoder(wl.labels)
    rng = np.random.default_rng(5)
    xs = []
    for i in range(6):
        x = wl.utterance(9700 + i, 120, "peaky").astype(np.float32)
        rows = rng.choice(len(x), size=12, replace=False)
        for j, r in enumerate(rows):
            cols = rng.choice(x.shape[1], size=40, replace=False)
            low = cols[x[r, cols] < x[r].max() - 3.0]          # never the frame's best token
            x[r, low] = -np.inf if j % 3 else np.float32(-3.0e38)
        xs.append(x)
    got = dec.decode_beams_batch(None, xs, beam_width=24)
    ref = ora.decode_beams_batch(xs, beam_width=24)
    for w, g in zip(ref, got):
        _compare(w, _beams(g))
