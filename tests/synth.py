"""Deterministic synthetic workloads for the CTC beam-search path (SURVEY.md section 8d).

Test / bench infrastructure, not part of the product package.  Everything is seeded with
``numpy.random.default_rng`` so that the container, the GPU box and every rank generate the
same tensors.

Vocabularies
  A  LibriSpeech characters (reference tests/test_decoder.py:155-184), V=29 after the blank
     is appended by the alphabet normaliser.
  B  Wav2Vec2-base, 32 labels in HF order (tutorials/02_pipeline_huggingface.ipynb:87);
     after normalisation blank=0, unk=3, space=4.
  C  synthetic sentencepiece-style BPE, V=1024 after normalisation; the lone BPE marker
     U+2581 is NOT included (it would trigger the force_next_break quirk on every use).

Utterance logits: a word sequence is sampled from the synthetic n-gram model, spelled into a
CTC alignment (each symbol held 1-3 frames, 0-3 blanks between symbols, a mandatory blank
between doubled symbols), cut / blank-padded to T; x = N(0,1) float32 noise, x[t, target]
+= margin and with probability ``conf`` one random competitor gets margin-1.
Regimes: "peaky" (margin 8, conf 0.10) is the headline, "diffuse" (margin 6, conf 0.15) the
stress case.
"""
import hashlib
import os
import tempfile

import numpy as np

BPE = "▁"

LIBRI_LABELS = [" "] + [chr(ord("a") + i) for i in range(26)] + ["'"]
W2V2_LABELS = ["<pad>", "<s>", "</s>", "<unk>", "|", "E", "T", "A", "O", "N", "I", "H", "S", "R", "D", "L", "U",
               "M", "W", "C", "F", "G", "Y", "P", "B", "V", "K", "'", "X", "J", "Q", "Z"]

REGIMES = {"peaky": (8.0, 0.10), "diffuse": (6.0, 0.15), "flat": (0.0, 0.0)}


def make_word_list(n_words, letters, seed=1, min_len=1, max_len=10):
    """Pseudo-words with Zipfian probabilities. Returns (words, probs)."""
    rng = np.random.default_rng(seed)
    letters = list(letters)
    # letter frequencies roughly geometric so that words look non-uniform
    lp = np.array([0.9 ** i for i in range(len(letters))])
    lp /= lp.sum()
    words, seen = [], set()
    while len(words) < n_words:
        n = int(rng.integers(min_len, max_len + 1))
        w = "".join(letters[i] for i in rng.choice(len(letters), size=n, p=lp))
        if w not in seen:
            seen.add(w)
            words.append(w)
    ranks = np.arange(1, n_words + 1, dtype=np.float64)
    probs = 1.0 / ranks
    probs /= probs.sum()
    return words, probs


def write_synthetic_arpa(path, words, probs, order=3, seed=2, succ_lo=4, succ_hi=8, hi_succ=(2, 4)):
    """Write a suffix- and prefix-closed ARPA model. Returns the successor tables used for sampling."""
    rng = np.random.default_rng(seed)
    n = len(words)
    vocab = ["<unk>", "<s>", "</s>"] + list(words)
    widx = {w: i for i, w in enumerate(vocab)}

    def rnd_p(k):
        return rng.uniform(-5.0, -0.3, size=k)

    def rnd_b(k):
        return rng.uniform(-1.5, 0.0, size=k)

    # level[k] maps context tuple (k words) -> list of successor word ids
    levels = [None] * (order + 1)
    # bigram successors: for <s> and every word
    succ1 = {}
    ctx_ids = [widx["<s>"]] + [widx[w] for w in words]
    cum = np.cumsum(probs)
    for c in ctx_ids:
        k = int(rng.integers(succ_lo, succ_hi + 1))
        # Zipf-biased successors, plus </s> sometimes
        picks = np.unique(np.searchsorted(cum, rng.random(k)))
        s = [widx[words[min(i, n - 1)]] for i in picks]
        if c != widx["<s>"] and rng.random() < 0.3:
            s.append(widx["</s>"])
        succ1[(c,)] = s
    levels[1] = succ1
    for lvl in range(2, order):
        prev = levels[lvl - 1]
        cur = {}
        for ctx, succs in prev.items():
            for b in succs:
                if b == widx["</s>"]:
                    continue
                new_ctx = ctx + (b,)
                # successors must keep the model suffix closed: new_ctx[1:] + (c,) has to exist
                lower = prev.get(new_ctx[1:])
                if not lower:
                    continue
                k = int(rng.integers(hi_succ[0], hi_succ[1] + 1))
                if k >= len(lower):
                    chosen = list(lower)
                else:
                    chosen = [lower[i] for i in sorted(rng.choice(len(lower), size=k, replace=False))]
                cur[new_ctx] = chosen
        levels[lvl] = cur

    grams = [None, [], [], [], [], [], []]
    # unigrams
    uni_lp = np.log10(np.maximum(probs, 1e-12))
    has_ext1 = set(k[0] for k in levels[1].keys())
    grams[1].append((-8.0, ("<unk>",), None))
    grams[1].append((-99.0, ("<s>",), float(rnd_b(1)[0])))
    grams[1].append((-1.5, ("</s>",), None))
    bo = rnd_b(n)
    for i, w in enumerate(words):
        grams[1].append((float(uni_lp[i]) - 0.3, (w,), float(bo[i]) if widx[w] in has_ext1 else None))
    for lvl in range(1, order):
        table = levels[lvl]
        nxt = levels[lvl + 1] if lvl + 1 < order else None
        for ctx, succs in table.items():
            ps = rnd_p(len(succs))
            bs = rnd_b(len(succs))
            for j, s in enumerate(succs):
                gram = ctx + (s,)
                is_ctx = nxt is not None and gram in nxt
                backoff = float(bs[j]) if (is_ctx and lvl + 1 < order) else None
                grams[lvl + 1].append((float(ps[j]), tuple(vocab[g] for g in gram), backoff))
    with open(path, "w", encoding="utf-8") as fh:
        fh.write("\\data\\\n")
        for o in range(1, order + 1):
            fh.write("ngram %d=%d\n" % (o, len(grams[o])))
        for o in range(1, order + 1):
            fh.write("\n\\%d-grams:\n" % o)
            for p, ws, b in grams[o]:
                if b is None:
                    fh.write("%.6f\t%s\n" % (p, " ".join(ws)))
                else:
                    fh.write("%.6f\t%s\t%.6f\n" % (p, " ".join(ws), b))
        fh.write("\n\\end\\\n")
    return {"vocab": vocab, "levels": levels, "widx": widx}


def cache_dir():
    """Per-user directory under the system temp dir: on a shared machine another user's directory is not writable."""
    d = os.path.join(tempfile.gettempdir(), "b200ctc_synth-%d" % os.getuid())
    os.makedirs(d, exist_ok=True)
    return d


def cached_arpa(n_words, letters, order, seed=1, tag=""):
    """Create (or reuse) a synthetic ARPA under cache_dir(). Returns (path, words, probs, tables)."""
    key = hashlib.sha1(("%d|%s|%d|%d|%s|v3" % (n_words, "".join(letters), order, seed, tag)).encode()).hexdigest()[:12]
    d = cache_dir()
    path = os.path.join(d, "lm_%s.arpa" % key)
    words, probs = make_word_list(n_words, letters, seed=seed)
    tmp = path + ".tmp%d" % os.getpid()
    tables = write_synthetic_arpa(tmp, words, probs, order=order, seed=seed + 1)
    os.replace(tmp, path)
    return path, words, probs, tables


def sample_sentence(rng, words, probs, tables, max_words):
    """Follow the model's successor tables; fall back to the Zipf unigram distribution."""
    out = []
    cum = np.cumsum(probs)
    if tables is None:
        for _ in range(max_words):
            out.append(words[min(int(np.searchsorted(cum, rng.random())), len(words) - 1)])
        return out
    vocab, levels, widx = tables["vocab"], tables["levels"], tables["widx"]
    hist = [widx["<s>"]]
    eos = widx["</s>"]
    for _ in range(max_words):
        nxt = None
        for lvl in range(len(levels) - 1, 0, -1):
            tab = levels[lvl]
            if tab is None or len(hist) < lvl:
                continue
            succs = tab.get(tuple(hist[-lvl:]))
            if succs:
                nxt = succs[int(rng.integers(0, len(succs)))]
                break
        if nxt is None or nxt == eos or rng.random() < 0.15:
            nxt = widx[words[min(int(np.searchsorted(cum, rng.random())), len(words) - 1)]]
        out.append(vocab[nxt])
        hist.append(nxt)
    return out


def ctc_alignment(rng, symbol_ids, blank_id, T):
    """Spell symbol ids into a length-T CTC frame alignment."""
    frames = []
    prev = None
    for s in symbol_ids:
        nb = int(rng.integers(0, 4))
        if prev is not None and s == prev and nb == 0:
            nb = 1
        frames.extend([blank_id] * nb)
        frames.extend([s] * int(rng.integers(1, 4)))
        prev = s
        if len(frames) >= T:
            break
    frames = frames[:T]
    frames.extend([blank_id] * (T - len(frames)))
    return np.asarray(frames, dtype=np.int64)


def collapse_alignment(align, norm_labels, blank_id):
    """CTC collapse of a frame alignment (repeats, then blanks) -> text with single spaces."""
    out, prev = [], None
    for a in align:
        a = int(a)
        if a != prev and a != blank_id:
            out.append(norm_labels[a])
        prev = a
    return " ".join("".join(out).replace("\u2581", " ").split())


def word_errors(ref, hyp):
    """(word-level edit distance, reference length)"""
    r, h = ref.split(), hyp.split()
    row = list(range(len(h) + 1))
    for i in range(1, len(r) + 1):
        prev, row[0] = row[0], i
        for j in range(1, len(h) + 1):
            cur = min(row[j] + 1, row[j - 1] + 1, prev + (r[i - 1] != h[j - 1]))
            prev, row[j] = row[j], cur
    return row[len(h)], len(r)


def logits_from_alignment(rng, align, V, margin, conf):
    T = len(align)
    x = rng.standard_normal((T, V), dtype=np.float32)
    x[np.arange(T), align] += np.float32(margin)
    if conf > 0:
        mask = rng.random(T) < conf
        comp = rng.integers(0, V, size=T)
        x[np.arange(T)[mask], comp[mask]] += np.float32(margin - 1.0)
    return x


class CharWorkload:
    """Vocab A or B with optional synthetic n-gram model."""

    def __init__(self, vocab="B", n_words=20000, lm_order=0, seed=1):
        if vocab == "A":
            self.labels = list(LIBRI_LABELS)
            self.norm_labels = self.labels + [""]
            letters = self.labels[1:]
            self.space_id, self.blank_id = 0, len(self.labels)
        else:
            self.labels = list(W2V2_LABELS)
            self.norm_labels = ["", "<s>", "</s>", "⁇", " "] + self.labels[5:]
            letters = self.labels[5:]
            self.space_id, self.blank_id = 4, 0
        self.V = len(self.norm_labels)
        self.char_id = {c: i for i, c in enumerate(self.norm_labels) if len(c) == 1 and c != " "}
        if lm_order > 0:
            self.arpa, self.words, self.probs, self.tables = cached_arpa(n_words, letters, lm_order, seed=seed, tag=vocab)
        else:
            self.arpa, self.tables = None, None
            self.words, self.probs = make_word_list(n_words, letters, seed=seed)

    def utterance(self, seed, T, regime="peaky"):
        margin, conf = REGIMES[regime]
        rng = np.random.default_rng(seed)
        sent = sample_sentence(rng, self.words, self.probs, self.tables, max_words=max(2, T // 8))
        syms = []
        for wi, w in enumerate(sent):
            if wi:
                syms.append(self.space_id)
            syms.extend(self.char_id[c] for c in w)
        align = ctc_alignment(rng, syms, self.blank_id, T)
        return logits_from_alignment(rng, align, self.V, margin, conf)

    def batch(self, seed0, B, T, regime="peaky"):
        return [self.utterance(seed0 + i, T, regime) for i in range(B)]

    def truth(self, seed, T):
        """The text the alignment of utterance(seed, T, .) spells (ground truth for WER; the last word may be cut)."""
        rng = np.random.default_rng(seed)
        sent = sample_sentence(rng, self.words, self.probs, self.tables, max_words=max(2, T // 8))
        syms = []
        for wi, w in enumerate(sent):
            if wi:
                syms.append(self.space_id)
            syms.extend(self.char_id[c] for c in w)
        return collapse_alignment(ctc_alignment(rng, syms, self.blank_id, T), self.norm_labels, self.blank_id)


class BpeWorkload:
    """Vocab C: synthetic BPE pieces over lower-case letters."""

    def __init__(self, n_words=50000, lm_order=0, seed=1, V=1024):
        letters = [chr(ord("a") + i) for i in range(26)]
        if lm_order > 0:
            self.arpa, self.words, self.probs, self.tables = cached_arpa(n_words, letters, lm_order, seed=seed, tag="C")
        else:
            self.arpa, self.tables = None, None
            self.words, self.probs = make_word_list(n_words, letters, seed=seed)
        # piece inventory: single letters in both forms, then most frequent word prefixes /
        # inner substrings weighted by word probability
        start_cnt, cont_cnt = {}, {}
        for w, p in zip(self.words[:5000], self.probs[:5000]):
            for L in (2, 3, 4):
                if len(w) >= L:
                    start_cnt[w[:L]] = start_cnt.get(w[:L], 0.0) + p
                for i in range(1, len(w) - L + 1):
                    cont_cnt[w[i:i + L]] = cont_cnt.get(w[i:i + L], 0.0) + p
        n_special = 2  # <unk>, <pad>
        n_start = 400 - 26
        n_cont = V - n_special - 400 - 26
        starts = [s for s, _ in sorted(start_cnt.items(), key=lambda kv: (-kv[1], kv[0]))[:n_start]]
        conts = [s for s, _ in sorted(cont_cnt.items(), key=lambda kv: (-kv[1], kv[0]))[:n_cont]]
        self.labels = ["<unk>", "<pad>"] + [BPE + c for c in letters] + [BPE + s for s in starts] + letters + conts
        assert len(self.labels) == len(set(self.labels))
        self.norm_labels = [BPE + "⁇" + BPE, ""] + self.labels[2:]
        self.V = len(self.norm_labels)
        self.blank_id = 1
        self.start_id = {p[1:]: i for i, p in enumerate(self.norm_labels) if p.startswith(BPE) and i >= 2}
        self.cont_id = {p: i for i, p in enumerate(self.norm_labels) if i >= 2 and not p.startswith(BPE)}

    def segment(self, w):
        ids = []
        L = min(4, len(w))
        while L > 1 and w[:L] not in self.start_id:
            L -= 1
        ids.append(self.start_id[w[:L]])
        i = L
        while i < len(w):
            L = min(4, len(w) - i)
            while L > 1 and w[i:i + L] not in self.cont_id:
                L -= 1
            ids.append(self.cont_id[w[i:i + L]])
            i += L
        return ids

    def utterance(self, seed, T, regime="peaky"):
        margin, conf = REGIMES[regime]
        rng = np.random.default_rng(seed)
        sent = sample_sentence(rng, self.words, self.probs, self.tables, max_words=max(2, T // 5))
        syms = []
        for w in sent:
            syms.extend(self.segment(w))
        align = ctc_alignment(rng, syms, self.blank_id, T)
        return logits_from_alignment(rng, align, self.V, margin, conf)

    def batch(self, seed0, B, T, regime="peaky"):
        return [self.utterance(seed0 + i, T, regime) for i in range(B)]

    def truth(self, seed, T):
        rng = np.random.default_rng(seed)
        sent = sample_sentence(rng, self.words, self.probs, self.tables, max_words=max(2, T // 5))
        syms = []
        for w in sent:
            syms.extend(self.segment(w))
        return collapse_alignment(ctc_alignment(rng, syms, self.blank_id, T), self.norm_labels, self.blank_id)

    def hotwords(self, n=16, seed=7):
        rng = np.random.default_rng(seed)
        return [self.words[i] for i in sorted(rng.choice(2000, size=n, replace=False))]


def make_workload(spec):
    """Build a workload from the dict stored in tests/golden/cases.json."""
    kw = dict(spec)
    kind = kw.pop("kind")
    return CharWorkload(**kw) if kind == "char" else BpeWorkload(**kw)


def special_step_cases(wl, n_cases=60, seed=7):
    """Seeded (logits, decode kwargs) pairs that drive the kernel's single-token special steps (in-place frames,
    binary-search ranking of merge-free frames): peaky logits of varying sharpness, integer-valued logits (exact
    score ties), small and large beams, all prune settings.  Shared by the hostsim and the GPU parity tests."""
    rng = np.random.default_rng(seed)
    for i in range(n_cases):
        T = int(rng.integers(20, 300))
        margin = float(rng.choice([5.0, 6.0, 7.0, 8.0, 10.0]))
        x = (wl.utterance(9000 + i, T, "peaky") * (margin / 8.0)).astype(np.float32)
        if i % 6 == 0:
            x = np.round(x).astype(np.float32)
        kw = dict(beam_width=int(rng.choice([2, 5, 17, 50, 100, 128])), prune_history=bool(i % 2),
                  beam_prune_logp=float(rng.choice([-10.0, -3.0, -20.0])), token_min_logp=float(rng.choice([-5.0, -3.0, -7.0])))
        yield x, kw
