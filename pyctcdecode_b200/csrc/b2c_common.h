// b200ctc -- shared host/device definitions for the CTC prefix beam-search path.
//
// Everything here is plain data layout + small pure functions usable from CUDA device code,
// from the host side of the library, and from the CPU "hostsim" build of the same kernel
// bodies that tests/ uses to exercise kernel logic on machines without a GPU
// (tests/hostsim; never part of the product path).
//
// String-free beam search: the reference keys beams on Python strings
// (text, partial_word, last_char; reference decoder.py:215-216).  Here every string is
// represented by a 61-bit polynomial hash of its UTF-8 bytes that can be extended token by
// token, texts by a chained 64-bit hash of their word hashes.  KenLM itself identifies words
// and n-grams by 64-bit hashes only, so this is the same class of approximation the
// reference already runs on.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define B2C_HD __host__ __device__ __forceinline__
#define B2C_D __device__ __forceinline__
#else
#define B2C_HD inline
#define B2C_D inline
#endif

typedef unsigned long long u64;
typedef unsigned int u32;
typedef unsigned short u16;
typedef unsigned char u8;

#define B2C_MAX_ORDER 6
#define B2C_MAX_HIST (B2C_MAX_ORDER - 1)
#define B2C_NONE_U32 0xFFFFFFFFu
#define B2C_NO_TOK 0xFFFFu

// ---------------------------------------------------------------------------------------
// hashing
// ---------------------------------------------------------------------------------------
#define B2C_P61 0x1FFFFFFFFFFFFFFFull
#define B2C_HASH_BASE 0x0A3B1C5D7E9F2461ull  // fixed "random" base < 2^61 - 1

B2C_HD u64 b2c_mod61(u64 lo, u64 hi) {
    // (hi * 2^64 + lo) mod (2^61 - 1), for products of two values < 2^61 (hi < 2^58)
    u64 r = (lo & B2C_P61) + ((lo >> 61) | (hi << 3));
    r = (r & B2C_P61) + (r >> 61);
    if (r >= B2C_P61) r -= B2C_P61;
    return r;
}
B2C_HD u64 b2c_mulmod61(u64 a, u64 b) {
#if defined(__CUDA_ARCH__)
    return b2c_mod61(a * b, __umul64hi(a, b));
#else
    unsigned __int128 p = static_cast<unsigned __int128>(a) * b;
    return b2c_mod61(static_cast<u64>(p), static_cast<u64>(p >> 64));
#endif
}
B2C_HD u64 b2c_addmod61(u64 a, u64 b) {
    u64 r = a + b;
    if (r >= B2C_P61) r -= B2C_P61;
    return r;
}
// hash(s + t) from hash(s), hash(t), BASE^len_bytes(t)
B2C_HD u64 b2c_hash_append(u64 hs, u64 ht, u64 pow_t) { return b2c_addmod61(b2c_mulmod61(hs, pow_t), ht); }

B2C_HD u64 b2c_mix64(u64 x) {  // splitmix64 finaliser
    x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull;
    x ^= x >> 27; x *= 0x94D049BB133111EBull;
    x ^= x >> 31;
    return x;
}
#define B2C_TEXT_SEED 0x6A09E667F3BCC908ull
// identity of "text + ' ' + word" from the identity of text and the word hash
B2C_HD u64 b2c_text_append(u64 text_hash, u64 word_hash) {
    return b2c_mix64(text_hash * 0x9E3779B97F4A7C15ull + word_hash + 0x632BE59BD9B4E019ull);
}
// merge key of a beam: (text, partial_word, last_char)  (reference decoder.py:215-216)
B2C_HD u64 b2c_beam_key(u64 text_hash, u64 part_hash, u32 part_len, u32 last_tok) {
    // three independent multiplies, one avalanche round (the key is on the critical path of a frame)
    u64 k = text_hash * 0xD6E8FEB86659FD93ull + part_hash * 0xA24BAED4963EE407ull +
            (static_cast<u64>(part_len) | ((static_cast<u64>(last_tok) + 1) << 20)) * 0x9FB21C651E98DF25ull;
    k = b2c_mix64(k);
    return k ? k : 1;
}
// n-gram chain: start from the predicted word, extend with context words (most recent first)
B2C_HD u64 b2c_ngram_start(u32 word) { return b2c_mix64(static_cast<u64>(word) + 0x51ED270B1ull); }
B2C_HD u64 b2c_ngram_extend(u64 h, u32 ctx_word) {
    u64 k = (h * 0x7C9B0F3D5A6E1B47ull) ^ ((static_cast<u64>(ctx_word) + 1) * 0xF858B9A5D3C17E2Bull);
    k = b2c_mix64(k);
    return k ? k : 1;
}
B2C_HD u64 b2c_hist_fold(u64 h, u64 word_hash) { return b2c_mix64(h * 0xC2B2AE3D27D4EB4Full + word_hash + 1); }
#define B2C_HIST_SEED 0x3C6EF372FE94F82Bull
// the same chain as KenLM's probing search computes it (lm/search_hashed.hh: the node of a unigram is its word index,
// detail::CombineWordHash extends it by one context word): tables read from a KenLM binary keep KenLM's own keys --
// they cannot be re-keyed, the file stores the combined hash only
B2C_HD u64 b2c_kenlm_start(u32 word) { return static_cast<u64>(word); }
B2C_HD u64 b2c_kenlm_extend(u64 h, u32 ctx_word) {
    return (h * 8978948897894561157ull) ^ ((static_cast<u64>(ctx_word) + 1) * 17894857484156487943ull);
}
enum { B2C_KEYS_B2C = 0, B2C_KEYS_KENLM = 1 };

// order-preserving map double -> u64 (larger double -> larger key); NaN sorts above +inf
B2C_HD u64 b2c_f64_key(double d) {
    union { double d; u64 u; } c;
    c.d = d;
    return (c.u & 0x8000000000000000ull) ? ~c.u : (c.u | 0x8000000000000000ull);
}
B2C_HD double b2c_key_f64(u64 k) {
    union { double d; u64 u; } c;
    c.u = (k & 0x8000000000000000ull) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k;
    return c.d;
}

// ---------------------------------------------------------------------------------------
// vocabulary (the normalised alphabet, reference alphabet.py:139-148 / decoder.py:287-288)
// ---------------------------------------------------------------------------------------
enum { B2C_TF_BLANK = 1, B2C_TF_SPACE = 2, B2C_TF_BPE_LEAD = 4, B2C_TF_BPE_TRAIL = 8 };

struct B2cTok {          // 32 bytes, one per label
    u64 raw_hash;        // hash of the full label (branch iv appends the full label)
    u64 raw_pow;         // BASE^len_bytes(label)
    u64 clean_hash;      // hash of the label without leading/trailing U+2581 (branch ii)
    u16 raw_nchars;      // python len(label)
    u16 clean_nchars;
    u16 canon;           // first token id with the same label string (string compare semantics)
    u16 flags;
};

// ---------------------------------------------------------------------------------------
// n-gram model, flattened (KenLM probing-model semantics: float32 log10 prob / backoff,
// backoff == -0.0f means "no extension" exactly like lm/model.hh kNoExtensionBackoff)
// ---------------------------------------------------------------------------------------
struct B2cNgram { u64 key; float prob; float backoff; };            // key 0 = empty slot
struct B2cVocab { u64 key; u32 id; u32 flags; };                     // flags bit0: in unigram set
struct B2cUni { float prob; float backoff; };

struct B2cLmView {
    int order;                 // 0: no language model
    u32 bos_id, eos_id;
    u32 n_vocab;
    int have_unigrams;         // unigrams were given (reference: char_trie is not None)
    int n_unigrams;            // size of the filtered unigram set
    int key_scheme;            // B2C_KEYS_*: how the keys of the n-gram table chain word ids
    int pad_view;
    const B2cUni* uni;
    const B2cNgram* ngrams; u64 ngram_mask;
    const B2cVocab* vocab; u64 vocab_mask;
    const u64* prefixes; u64 prefix_mask;   // hashes of every code-point prefix of every unigram
};

struct B2cLmState {            // kenlm::ngram::State
    u32 words[B2C_MAX_HIST];
    float backoff[B2C_MAX_HIST];
    u32 length;
};

struct B2cHot { u64 key; u32 min_len; u32 is_word; };                // hotword prefix table

// MultiLanguageModel (reference language_model.py:455-502): the mean of up to B2C_MAX_LMS n-gram models, each
// with its own tables, vocabulary, unigram set and alpha / beta / unk offset / boundary flag.  Model 0 lives
// in B2cParams::lm and the scalar parameters; models 1.. in lmx[].
#define B2C_MAX_LMS 4
struct B2cLmExtra {
    B2cLmView lm;
    double alpha, beta, unk_offset;
    int score_boundary;
    int pad;
};

// ---------------------------------------------------------------------------------------
// decode parameters (one block per decode call, passed by value to the kernels)
// ---------------------------------------------------------------------------------------
struct B2cParams {
    int V;
    int is_bpe;
    int has_dup_labels;        // two token ids share a label string (their candidates can merge across tokens)
    int beam_width;
    int prune_history;
    int hist_n;                // max(1, lm order - 1)   (reference decoder.py:244)
    int out_beams;             // beams returned per utterance (1 for decode_batch)
    int narrow_chain;          // text-only calls: 8-byte backtrack nodes (no word frames), b2c_chain_store / _load
    double prune_logp;
    double token_min_logp;
    double alpha, beta, unk_offset, log_base_change;
    int score_boundary;
    int n_hot;                 // number of hotword unigrams (0: none)
    int hot_min_len_all;       // shortest hotword (answer for the empty prefix)
    double hot_weight;
    double bucket_scale;       // score buckets per nat for the O(m) ranking (host computed)
    const B2cHot* hot; u64 hot_mask;
    const B2cTok* toks;
    B2cLmView lm;
    int n_lm;                  // 0: none, 1: one model, > 1: MultiLanguageModel (general kernel only)
    int pad_lm;
    const B2cLmExtra* lmx;     // [n_lm - 1] models 1.. (device memory; the parameter block stays small: it is copied
                               // into every out-of-line call of the hot kernels)
};

// ---------------------------------------------------------------------------------------
// per-utterance prefix structures kept in HBM arenas
// ---------------------------------------------------------------------------------------
enum { B2C_CK_CONT = 0, B2C_CK_SPACE = 1, B2C_CK_BPE = 2, B2C_CK_ROOT = 3 };   // ROOT: input beam `tok` of a streaming call
struct B2cChain {              // 16 bytes: one emitted (non-blank, non-repeat) token of a beam
    u32 parent;
    u16 tok;
    u8 kind;                   // B2C_CK_*
    u8 has_word;               // boundary kinds: a finished word was flushed, frames valid
    int ws, we;                // frames of the flushed word
};
// Text-only calls (decode / decode_batch) never read the word frames: their nodes are the first 8 bytes only, packed
// parent | tok << 32 | kind << 48 | has_word << 56, at index `id` of a u64 view of the same arena -- half the HBM
// write traffic of the beam kernel (one node per emitted token of every surviving beam).
B2C_HD void b2c_chain_store(B2cChain* arena, u32 id, const B2cChain& c, bool narrow) {
    if (narrow) {
        reinterpret_cast<u64*>(arena)[id] = static_cast<u64>(c.parent) | (static_cast<u64>(c.tok) << 32) |
                                            (static_cast<u64>(c.kind) << 48) | (static_cast<u64>(c.has_word) << 56);
    } else {
        arena[id] = c;
    }
}
B2C_HD B2cChain b2c_chain_load(const B2cChain* arena, u32 id, bool narrow) {
    if (!narrow) return arena[id];
    const u64 v = reinterpret_cast<const u64*>(arena)[id];
    B2cChain c;
    c.parent = static_cast<u32>(v);
    c.tok = static_cast<u16>(v >> 32);
    c.kind = static_cast<u8>(v >> 48);
    c.has_word = static_cast<u8>(v >> 56);
    c.ws = -1;
    c.we = -1;
    return c;
}
struct B2cText {               // one distinct "text" (sequence of finished words)
    u64 win[B2C_MAX_HIST];     // hashes of the last hist_n words, most recent first
    u64 hist_hash;
    double raw_lm;             // sum of word LM scores (reference raw_lm_score)
    B2cLmState st;
    u32 hw_count;              // hotword unigram matches in the text
    u32 n_win;
};

// streaming (reference partial_decode_beams, decoder.py:669-728): the beams a call starts from, string-free.
// The host hashes the words of every input beam; the kernel replays them through the LM / hotword scorer, which
// reproduces what the reference keeps in cached_lm_scores (raw LM score, LM state) without carrying a cache.
struct B2cStreamBeam {
    u64 part_hash;             // partial_word
    double logit;              // logit_score
    u32 word_off, n_words;     // finished words of `text`: word_hash / word_len [word_off, word_off + n_words)
    u32 part_len;              // python len(partial_word)
    u32 last_tok;              // canonical token id of last_char, B2C_NO_TOK for None
    int pf_s, pf_e;            // partial_frames
};
struct B2cStreamUtt { u32 beam_off, n_beams; int t0; u32 pad; };   // t0: processed_frames
// what _finalize_beams does at the end of a call (decoder.py:558-602); same values as include/b200ctc.h
#ifndef B2C_FIN_EOS
#define B2C_FIN_EOS 0          // force_next_word or is_end, scored with is_eos=True (decode_beams; is_end=True)
#define B2C_FIN_FLUSH 1        // force_next_word=True, is_end=False: partial words become words, no </s>
#define B2C_FIN_KEEP 2         // neither: beams keep their partial words (streaming continues)
#endif

#define B2C_LOG_MIN_CLIP (-0x1.144f69ff9ffc4p+5)   // np.log(1e-15)
#define B2C_AVG_TOKEN_LEN 6

// status codes written per utterance
enum { B2C_OK = 0, B2C_ERR_CHAIN_FULL = 1, B2C_ERR_TEXT_FULL = 2, B2C_ERR_CAND_FULL = 3,
       B2C_ERR_GATE = 8 };      // a gated launch waited too long for the streaming stage of its next chunk (host: plain call)
