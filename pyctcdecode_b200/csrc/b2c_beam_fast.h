// b200ctc -- latency-first variant of the per-utterance prefix beam search for beam_width <= B2C_FAST_W
// (same algorithm and the same results as b2c_beam.h, which stays the general path).
//
// A C2-shaped batch (256 utterances x 1000 frames on 148 SMs) keeps every utterance resident, so the
// batch takes exactly as long as ONE utterance: T dependent frames.  What bounds it is the latency
// of a frame, not throughput.  Compared with the general kernel this variant therefore
//   * uses a compile-time shared-memory layout (B2cFastSmem): every array address is
//     base + constant, no descriptor of generic pointers lives in registers or local memory;
//   * keeps the token lists of the next frames in shared-memory RINGS filled by asynchronous copies
//     (cp.async / LDGSTS, no register staging): 16-byte frame records (token count + first token inline) 18-32
//     frames ahead, token ids / log-probs up to 7 frames ahead, issued at the top of an iteration and waited for
//     just before its closing barrier -- no global load is on the critical path of a frame and no barrier has
//     a register-destined load in flight; for small alphabets (V <= 64) the per-label records live in shared
//     memory for the whole launch;
//   * handles RUNS of single-token frames (blank / held symbol / plain characters) in one step: the records of
//     the next frames are already in the ring, so R frames cost one round of bookkeeping, R dependent additions
//     per beam and one vote (b2c_fast_run_step);
//   * enumerates candidates as (token k outer, beam b = thread inner): no index division, the
//     token record is a warp-uniform shared-memory broadcast;
//   * stores each candidate's own logit sum and (beam, token) pair, so the fold / fusion / commit
//     phases never re-derive them;
//   * merge keys without an avalanche round (b2c_fast_key), probing the full grouping table with their
//     folded low bits (load <= 0.5 at capacity, ~0.06 typically);
//   * clears grouping / history-prune slots by their owners instead of sweeping the tables.
// Frames with more than CAP candidates (or more than B2C_FAST_KS tokens) are rare on ASR-like
// posteriors; they take the general out-of-line step on the HBM candidate tier (b2c_fast_slow_step).
//
// Four kinds of frame steps, chosen per frame from block-uniform facts (token count, the previous frame's
// token, mode flags):
//   b2c_fast_cheap_step   one token after a one-token frame (same token / blank / plain character without LM and
//                         hotwords): nothing can merge, reorder or be pruned -> the table is updated in place
//   b2c_fast_scored_step  the same with LM / hotwords and an ordinary character: new per-beam scores first, in place
//                         only if they keep slot order and threshold
//   b2c_fast_sorted_step  K >= 2 tokens after a one-token frame, no LM / hotwords / space: the candidates are K
//                         sorted lists that cannot merge -> ranks by search, one commit per thread
//   b2c_fast_step         everything else: expand + group | fold + fuse + bucket | threshold + rank + commit
// Every special step re-checks what float64 rounding could change and falls back to b2c_fast_step on the untouched
// state, so all three give the reference's result (tests: special_step_cases, hostsim work-item-order replay).
//
// Reference lines restated: decoder.py:443-554 (frame loop), :211-224 (merge), :346-424 (LM
// fusion), :545-554 (threshold, top-N, history prune).  Order-dependence notes: b2c_beam.h.
#pragma once
#include <cstddef>
#include "b2c_beam.h"

#define B2C_FAST_KS 32          // most tokens of a frame any variant stages (larger frames: out-of-line step)
#define B2C_FAST_HR 32          // frame-record ring (frames)
#define B2C_FAST_TR 8           // token ring (frames)
#define B2C_FAST_RMAX 6         // longest run of in-place frames handled by one step (<= B2C_FAST_TR - 2)
#define B2C_FAST_W 128          // threads per CTA = beam slots (one per thread)
#define B2C_FAST_NW (B2C_FAST_W / 32)   // warps per CTA (per-warp slot arrays have one entry each)

#if defined(__CUDA_ARCH__)
#define B2C_LAST_THREAD if (threadIdx.x == blockDim.x - 1)
// work for ONE warp -- the last one, which holds the slots >= 96 and has the fewest live beams -- so that the other
// warps walk straight into the frame step: items strided over its lanes
#define B2C_IN_LAST_WARP if ((threadIdx.x >> 5) == (blockDim.x >> 5) - 1)
#define B2C_FOR_LANES(i, n) for (int i = static_cast<int>(threadIdx.x & 31); i < static_cast<int>(n); i += 32)
#else
#define B2C_LAST_THREAD if (true)
#define B2C_IN_LAST_WARP if (true)
#define B2C_FOR_LANES(i, n) B2C_FOR(i, n)
#endif

constexpr u32 b2c_pt_cap_c(int W) {
    u32 p = 16;
    while (p < 2u * static_cast<u32>(W)) p <<= 1;
    return p;
}

struct B2cFastTab {          // one beam table (same fields as B2cBeamTab)
    double logit[B2C_FAST_W], lm_hw[B2C_FAST_W], pscore[B2C_FAST_W];
    u64 text_hash[B2C_FAST_W], part_hash[B2C_FAST_W], hist_hash[B2C_FAST_W];
    u32 text_node[B2C_FAST_W], chain[B2C_FAST_W];
    int pf_s[B2C_FAST_W], pf_e[B2C_FAST_W];
    u16 last_tok[B2C_FAST_W], part_len[B2C_FAST_W];
};

// asynchronous global -> shared copies (LDGSTS); hostsim: plain copies
B2C_HD void b2c_cp_async4(void* dst_smem, const void* src) {
#if defined(__CUDA_ARCH__)
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(static_cast<u32>(__cvta_generic_to_shared(dst_smem))), "l"(src) : "memory");
#else
    *static_cast<u32*>(dst_smem) = *static_cast<const u32*>(src);
#endif
}
B2C_HD void b2c_cp_async8(void* dst_smem, const void* src) {
#if defined(__CUDA_ARCH__)
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(static_cast<u32>(__cvta_generic_to_shared(dst_smem))), "l"(src) : "memory");
#else
    *static_cast<u64*>(dst_smem) = *static_cast<const u64*>(src);
#endif
}
B2C_HD void b2c_cp_async16(void* dst_smem, const void* src) {
#if defined(__CUDA_ARCH__)
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(static_cast<u32>(__cvta_generic_to_shared(dst_smem))), "l"(src) : "memory");
#else
    static_cast<u64*>(dst_smem)[0] = static_cast<const u64*>(src)[0];
    static_cast<u64*>(dst_smem)[1] = static_cast<const u64*>(src)[1];
#endif
}
B2C_HD void b2c_cp_async_wait_all() {
#if defined(__CUDA_ARCH__)
    asm volatile("cp.async.wait_all;" ::: "memory");
#endif
}

// LT: entries of the shared-memory label table (V <= LT: the table is resident, runs of in-place frames are
// enabled); 0: labels are staged per frame from global memory (large alphabets)
template <int CAP, int LT>
struct B2cFastSmem {
    static constexpr u32 HT = 2u * CAP;               // grouping table slots
    static constexpr u32 PT = b2c_pt_cap_c(B2C_FAST_W); // history-prune table slots
    static constexpr int KR = CAP >= 1024 ? 32 : 16;   // tokens per frame the rings hold (wider frames: out-of-line step)
    static constexpr int LTN = LT > 0 ? LT : 1;
    B2cScalars sc;
    u32 ticket;                                       // work-queue ticket of this CTA
    u32 holes;                                        // the current beam table has history-pruned slots (see b2c_fast_step)
    u32 cheap_bad;                                    // a thread's exactness check of b2c_fast_scored_step failed (rare)
    u32 run_fail;                                     // b2c_fast_run_step: first frame of the run whose exactness check failed
    u32 wmask[B2C_FAST_NW];                           // per warp: live slots of the current table (b2c_fast_sorted_step)
#if defined(B2C_PHASE_CLOCKS)
    u64 pclk[32];                                     // profiling builds: cycles between marks, thread 0
    long long pclk_last;
#endif
    u32 wtop[B2C_FAST_NW];                            // per warp: 1 + best rank selected this frame
    alignas(16) u64 wmax[B2C_FAST_NW];                // per warp: best score key of this frame
    alignas(16) B2cFastTab tab[2];
    // selection
    u64 phk[B2C_FAST_W];
    u32 ord[B2C_FAST_W], pslot[B2C_FAST_W];
    u32 pt_idx[PT], pt_min[PT];
    alignas(16) u32 bcnt[B2C_NBUCKET];
    alignas(16) u32 bhead[B2C_NBUCKET];
    alignas(16) u32 bpre[B2C_FAST_NW][B2C_NBUCKET];
    // candidates
    u64 ckey[CAP];           // merge key; after phase B: order-preserving score key of group leaders, 0 otherwise
    double cfold[CAP];       // phase A: own logit sum; after phase B (leaders): merged logit_score
    u64 cph[CAP];            // partial-word hash | branch type << 61
    u32 cmeta[CAP];          // partial length | canonical token << 16
    u32 cslot[CAP], cnext[CAP], clast[CAP];
    u32 cbk[CAP];            // beam | token index << 16
    u32 ht_idx[HT + 1], ht_min[HT + 1], ht_max[HT + 1], ht_cnt[HT + 1];   // slot HT: never claimed (candidates of dead beams)
    // token lists: label records of the current / next frame, rings of frame records and of (id, log-prob) lists
    alignas(16) B2cTok stok[2][LT > 0 ? 1 : KR];   // staged label records (large alphabets only)
    alignas(16) B2cFrameRec rh[B2C_FAST_HR];
    alignas(16) double rlp[B2C_FAST_TR][KR];
    alignas(16) u32 rid[B2C_FAST_TR][KR];
    alignas(16) B2cTok ltab[LTN];
    u32 ffirst[KR];              // BPE force_next_break side arrays
    u8 fall[KR];
};

B2C_HD void b2c_fast_tab_view(B2cFastTab& t, B2cBeamTab& v) {
    v.logit = t.logit; v.lm_hw = t.lm_hw; v.pscore = t.pscore;
    v.text_hash = t.text_hash; v.part_hash = t.part_hash; v.hist_hash = t.hist_hash;
    v.text_node = t.text_node; v.chain = t.chain;
    v.pf_s = t.pf_s; v.pf_e = t.pf_e;
    v.last_tok = t.last_tok; v.part_len = t.part_len;
}

// descriptor for the general helpers (b2c_utt_begin, b2c_finalize, the out-of-line slow step);
// `slow`: hide the shared-memory tier so that the general frame step works on the HBM tier
template <int CAP, int LT>
B2C_HD void b2c_fast_work(B2cFastSmem<CAP, LT>& S, const B2cLayout& L, u8* g, int par, bool slow, B2cWork& W) {
    W.sc = &S.sc;
    b2c_fast_tab_view(S.tab[par], W.cur);
    b2c_fast_tab_view(S.tab[par ^ 1], W.nxt);
    W.phk = S.phk; W.ord = S.ord; W.pslot = S.pslot;
    W.pt_cap = B2cFastSmem<CAP, LT>::PT;
    W.pt_idx = S.pt_idx; W.pt_min = S.pt_min;
    W.n_bucket = B2C_NBUCKET;
    W.bcnt = S.bcnt; W.bhead = S.bhead; W.bpre = &S.bpre[0][0];
    W.stok = nullptr; W.slp = nullptr; W.sid = nullptr;
    B2cCandTier& c = W.tier_s;
    c.cap = slow ? 0u : static_cast<u32>(CAP);
    c.ht_cap = B2cFastSmem<CAP, LT>::HT;
    c.ckey = S.ckey; c.cfold = S.cfold; c.cth = nullptr; c.cph = S.cph;
    c.cmeta = S.cmeta; c.cslot = S.cslot; c.cnext = S.cnext; c.clast = S.clast;
    c.ht_idx = S.ht_idx; c.ht_min = S.ht_min; c.ht_max = S.ht_max; c.ht_cnt = S.ht_cnt;
    if (L.cap_g) b2c_carve_tier(g + L.g_tier, L.cap_g, L.ht_g, W.tier_g);
    else W.tier_g = W.tier_s;
    {
        u8* p = g + L.g_tk;
        W.tk_ffirst = reinterpret_cast<u32*>(b2c_carve(p, 4ull * L.V));
        W.tk_fall = reinterpret_cast<u8*>(b2c_carve(p, static_cast<u64>(L.V)));
    }
    W.chain = reinterpret_cast<B2cChain*>(g + L.g_chain);
    W.chain_cap = L.chain_cap;
    W.text = reinterpret_cast<B2cText*>(g + L.g_text);
    W.text_cap = L.text_cap;
#if defined(B2C_PHASE_CLOCKS)
    for (int q = 0; q < 16; ++q) W.clk[q] = 0;
    W.clk_last = 0;
#endif
}

// label record of token k of the current frame: straight from the resident table (small alphabets: one more
// dependent shared-memory load, no per-frame staging), or from the staged copy (large alphabets)
template <int CAP, int LT>
B2C_HD const B2cTok& b2c_fast_tok(const B2cFastSmem<CAP, LT>& S, int sb, int slot, int k) {
    if (LT > 0) return S.ltab[S.rid[slot][k]];
    return S.stok[sb][k];
}

// per-warp maxima go to the warp's own slot (no atomics); readers combine the slots after the barrier
B2C_HD void b2c_warp_max_u64_slot(u64 v, u64* slots) {
#if defined(__CUDA_ARCH__)
    const u32 hi = static_cast<u32>(v >> 32), lo = static_cast<u32>(v);
    const u32 mhi = __reduce_max_sync(0xFFFFFFFFu, hi);
    const u32 mlo = __reduce_max_sync(0xFFFFFFFFu, hi == mhi ? lo : 0u);
    if ((threadIdx.x & 31) == 0) slots[threadIdx.x >> 5] = (static_cast<u64>(mhi) << 32) | mlo;
#else
    slots[0] = v;
#endif
}
B2C_HD void b2c_warp_max_u32_slot(u32 v, u32* slots) {
#if defined(__CUDA_ARCH__)
    const u32 m = __reduce_max_sync(0xFFFFFFFFu, v);
    if ((threadIdx.x & 31) == 0) slots[threadIdx.x >> 5] = m;
#else
    slots[0] = v;
#endif
}
template <class T>
B2C_HD T b2c_max_slots(const T* s) {
    T m = s[0];
#pragma unroll
    for (int c = 1; c < B2C_FAST_NW; ++c) m = s[c] > m ? s[c] : m;
    return m;
}

// merge key without the avalanche round of b2c_beam_key: a multiply-add combination of the (already
// well-mixed) hashes is collision-free unless a 64-bit linear relation holds; the high half is
// folded into the low half so that the low bits, which index the tables, depend on every input bit
B2C_HD u64 b2c_fast_key(u64 text_hash, u64 part_hash, u32 part_len, u32 last_tok) {
    u64 k = text_hash * 0xD6E8FEB86659FD93ull + part_hash * 0xA24BAED4963EE407ull +
            (static_cast<u64>(part_len) | ((static_cast<u64>(last_tok) + 1) << 20)) * 0x9FB21C651E98DF25ull;
    k ^= k >> 32;
    return k ? k : 1;
}

// conflict-free variant of b2c_bucket_scan_warp: every lane owns 8 consecutive buckets = two 16-byte words
B2C_HD void b2c_bucket_scan_warp_v(const u32* bcnt, u32* pre) {
#if defined(__CUDA_ARCH__)
    const u32 lane = threadIdx.x & 31;
    const uint4 a = reinterpret_cast<const uint4*>(bcnt)[2 * lane], b = reinterpret_cast<const uint4*>(bcnt)[2 * lane + 1];
    const u32 sum = a.x + a.y + a.z + a.w + b.x + b.y + b.z + b.w;
    u32 incl = sum;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const u32 o = __shfl_up_sync(0xFFFFFFFFu, incl, off);
        if (lane >= static_cast<u32>(off)) incl += o;
    }
    uint4 pa, pb;
    pa.x = incl - sum; pa.y = pa.x + a.x; pa.z = pa.y + a.y; pa.w = pa.z + a.z;
    pb.x = pa.w + a.w; pb.y = pb.x + b.x; pb.z = pb.y + b.y; pb.w = pb.z + b.z;
    reinterpret_cast<uint4*>(pre)[2 * lane] = pa;
    reinterpret_cast<uint4*>(pre)[2 * lane + 1] = pb;
    __syncwarp();
#else
    b2c_bucket_scan_warp(bcnt, pre);
#endif
}

#if defined(B2C_PHASE_CLOCKS) && defined(__CUDA_ARCH__)
#define B2C_FMARK(idx) do { if (threadIdx.x == 0) { const long long _c = clock64(); S.pclk[idx] += static_cast<u64>(_c - S.pclk_last); S.pclk_last = _c; } } while (0)
#else
#define B2C_FMARK(idx) ((void)0)
#endif

#define B2C_INVALID_TOK 0xFFFEu      // last_tok of a history-pruned slot (BPE force logic skips it)

// candidate i (a group leader) becomes beam j of the next frame (decoder.py:452-534 metadata); called by the
// thread that owns the candidate, inside the ranking loop
template <int CAP, int LT>
B2C_HD void b2c_fast_commit(const B2cParams& P, B2cFastSmem<CAP, LT>& S, const B2cFastTab& cur, B2cFastTab& nx,
                            B2cChain* chain_arena, B2cText* text_arena, u32 text_cap, int sb, int slot, int t, u32 j, u32 i,
                            u32 last, u32 flags) {
    const u32 bk = S.cbk[last];
    const u32 bl = bk & 0xFFFFu, k = bk >> 16;
    const u64 cph = S.cph[last];
    const u32 type = static_cast<u32>(cph >> 61);
    const u64 part_hash = cph & B2C_PH_MASK;
    const u32 meta = S.cmeta[last];
    const u32 part_len = meta & 0xFFFFu;
    const u32 word_len = (type == 1 || type == 2) ? static_cast<u32>(cur.part_len[bl]) : 0u;
    u64 th = cur.text_hash[bl];
    if (word_len > 0) th = b2c_text_append(th, cur.part_hash[bl]);
    nx.logit[j] = S.cfold[i];
    nx.text_hash[j] = th;
    nx.part_hash[j] = part_hash;
    nx.part_len[j] = static_cast<u16>(part_len);
    nx.last_tok[j] = static_cast<u16>(meta >> 16);
    // partial_frames (decoder.py:454-461,495,513,519-523)
    const int ps0 = cur.pf_s[bl], pe0 = cur.pf_e[bl];
    int pfs, pfe;
    if (type == 0) { pfs = ps0; pfe = (b2c_fast_tok<CAP, LT>(S, sb, slot, static_cast<int>(k)).flags & B2C_TF_BLANK) ? pe0 : t + 1; }
    else if (type == 1) { pfs = t; pfe = t + 1; }
    else if (type == 2) { pfs = -1; pfe = -1; }
    else { pfs = ps0 < 0 ? t : ps0; pfe = t + 1; }
    nx.pf_s[j] = pfs;
    nx.pf_e[j] = pfe;
    // backtrack chain: the node of (frame t, new slot j) has the fixed id t * B2C_FAST_W + j -- no allocation counter
    u32 chain = cur.chain[bl];
    if (type != 0) {
        const u32 id = static_cast<u32>(t) * B2C_FAST_W + j;
        B2cChain c;
        c.parent = chain;
        c.tok = static_cast<u16>(S.rid[slot][k]);
        c.kind = type == 3 ? B2C_CK_CONT : (type == 2 ? B2C_CK_SPACE : B2C_CK_BPE);
        c.has_word = word_len > 0 ? 1 : 0;
        c.ws = ps0;
        c.we = pe0;
        b2c_chain_store(chain_arena, id, c, P.narrow_chain != 0);
        chain = id;
    }
    nx.chain[j] = chain;
    // text level
    u32 tnode = cur.text_node[bl];
    double lm_hw = cur.lm_hw[bl];
    u64 hh = cur.hist_hash[bl];
    if (word_len > 0) {
        if (flags & B2C_FL_PSCORE) {
            B2cTextCommit tc;
            b2c_commit_text(P, text_arena, text_cap, &S.sc.text_used, &S.sc.status, tnode, cur.part_hash[bl], word_len, &tc);
            tnode = tc.node;
            lm_hw = tc.lm_hw;
            hh = tc.hist_hash;
        } else {
            // no LM, no hotwords: hist_n == 1, the text-level score stays hot_weight * 0 and nothing ever reads
            // a text node other than the root -> no arena traffic on word boundaries
            hh = b2c_hist_fold(B2C_HIST_SEED, cur.part_hash[bl]);
        }
    }
    nx.text_node[j] = tnode;
    nx.lm_hw[j] = lm_hw;
    nx.hist_hash[j] = hh;
    double ps = 0.0;
    if (type == 0) ps = cur.pscore[bl];
    else if (part_len > 0) ps = b2c_partial_score_of(P, (flags & B2C_FL_PSCORE) != 0, part_hash, part_len);
    nx.pscore[j] = ps;
}

// ---- helpers of the search-ranked step (b2c_fast_sorted_step) ---------------------------------------------------
#define B2C_SORTED_MAXK 8
B2C_HD u32 b2c_live_before(const u32* wm, u32 pos) {   // live slots with index < pos (pos <= 32 * B2C_FAST_NW)
    u32 c = 0;
#if defined(__CUDACC__)
#pragma unroll
#endif
    for (u32 w = 0; w < B2C_FAST_NW; ++w) {
        const u32 lo = w * 32;
        u32 m = wm[w];
        if (pos < lo + 32) m = pos > lo ? (m & ((1u << (pos - lo)) - 1u)) : 0u;
#if defined(__CUDA_ARCH__)
        c += static_cast<u32>(__popc(m));
#else
        c += static_cast<u32>(__builtin_popcount(m));
#endif
    }
    return c;
}

// The candidate scores of token k2 form the list cf[k2 * n + p] = (logit[p] + lp[k2]) + 0.0, p < n, non-increasing in p
// (written once per frame by the slots' owners, phase 1 of b2c_fast_sorted_step).  b2c_sorted_counts answers NS
// questions at once: how many leading entries of list q sort before the score s[q] -- entry >= s (ge) or > s.
// "> s" is asked as ">= the next double above s" (scores are finite and never -0.0: x + 0.0), so a probe is ONE
// shared-memory load and ONE comparison; the NS questions advance in lockstep so that their rounds overlap.
B2C_HD double b2c_next_up(double s) {        // smallest double > s, for finite s that is not -0.0
    union { double d; u64 u; } c;
    c.d = s;
    c.u = (c.u >> 63) ? c.u - 1 : c.u + 1;
    return c.d;
}
B2C_HD u32 b2c_list_probe(const double* list, u32 n, u32 p, double s) {
    // branch-free on purpose (a short-circuit && puts every probe into its own divergence region and serialises the
    // loads): the index is clamped, the load unconditional, the answer masked
    const u32 q = p < n ? p : n - 1;
    const double v = list[q];
    const u32 in_range = p < n ? 1u : 0u, hit = v >= s ? 1u : 0u;
    return in_range & hit;
}
template <int NS>
B2C_HD void b2c_sorted_counts(const double* const (&list)[NS], u32 n, const double (&s)[NS], u32 (&cnt)[NS]) {
    // branch-free binary search, the NS questions in lockstep: the count grows by `step` whenever entry count + step - 1
    // still sorts before s.  ~7 instructions per probe and question, log2(n) dependent rounds; the rounds of the NS
    // questions overlap (the frame is bound by instruction count x dependent-issue latency, not by the loads).
    u32 pos[NS];
#if defined(__CUDACC__)
#pragma unroll
#endif
    for (int q = 0; q < NS; ++q) pos[q] = 0;
    u32 step = 128;
    while (step > n) step >>= 1;            // n >= 1; block-uniform
#if defined(__CUDACC__)
#pragma unroll 1
#endif
    for (; step > 0; step >>= 1) {
#if defined(__CUDACC__)
#pragma unroll
#endif
        for (int q = 0; q < NS; ++q) pos[q] += step * b2c_list_probe(list[q], n, pos[q] + step - 1, s[q]);
    }
#if defined(__CUDACC__)
#pragma unroll
#endif
    for (int q = 0; q < NS; ++q) cnt[q] = pos[q];
}
// one question against the list logit[p] + lp2 computed on the fly, n <= N (unit test: tests/hostsim/t_sorted_count.cpp)
template <int N>
B2C_HD u32 b2c_sorted_count(const double* logit, u32 n, double lp2, double s, bool ge) {
    static_assert(N <= 128, "radix search covers 128 entries");
    double tmp[N];
    for (u32 p = 0; p < n; ++p) tmp[p] = (logit[p] + lp2) + 0.0;
    const double* const l1[1] = {tmp};
    const double s1[1] = {ge ? s : b2c_next_up(s)};
    u32 c1[1];
    b2c_sorted_counts<1>(l1, n, s1, c1);
    return c1[0];
}

// Ranks of the candidates of a frame whose K candidate lists cf[k * n + b] are non-increasing in b (b2c_fast_sorted_step).  Work items are the candidates i = k * n + b, strided over the threads -- NOT
// "a slot and its K candidates per thread": the candidates that can still land inside the beam width are the first few
// entries of every list (a candidate of the r-th best token has at least r + 1 lists in front of its own position), so
// per-slot work would leave the whole frame waiting for the threads of the first slots (K (K - 1) searches each).
// An item first looks at ENTRY b OF EVERY OTHER LIST: where that entry already sorts before the candidate, so do all
// entries above it -- a lower bound on the rank that needs no search and discards most items; the survivors run one
// binary search per other list (three lists in lockstep).
//   masks + mstride * k   eligible entries of list k (bit b; 4 words): live slots (sorted step, mstride 0) or unmerged
//                         live entries (list-ranked step, mstride 4)
//   mask_all              entries eligible in EVERY list (a subset of each list's mask: the lower bound counts it)
//   extra(s, i)           groups outside the lists that sort before score s / enumeration index i (merged groups)
//   place(i, k, b, rank)  called for every candidate with score >= thr whose rank is < width
template <class Extra, class Place>
B2C_HD void b2c_rank_list_items(const double* cf, u32 n, int K, const u32* masks, u32 mstride, const u32* mask_all, double thr,
                                u32 width, Extra extra, Place place) {
    const u32 M = n * static_cast<u32>(K);
    const float rcp_n = 1.0f / static_cast<float>(n);
    B2C_FOR(i, M) {
        u32 k, b;
        b2c_divmod(static_cast<u32>(i), n, rcp_n, k, b);
        const u32* const mk = masks + mstride * k;
        if (!((mk[b >> 5] >> (b & 31)) & 1u)) continue;
        const double s = cf[i] + 0.0;
        if (!(s >= thr)) continue;
        const double su = b2c_next_up(s);       // "> s" asked as ">= next_up(s)"
        // same list: the eligible entries above this one (equal scores keep slot order)
        u32 rank = b2c_live_before(mk, b) + extra(s, static_cast<u32>(i));
        if (K > 1) {
            // another list k2: its entries that sort before (k, b) -- score greater, or equal and enumerated earlier (k2 < k)
            u32 npass = 0;
            for (int k2 = 0; k2 < K; ++k2) {        // branch-free: the own list is probed too and masked
                const double v = cf[static_cast<u32>(k2) * n + b];
                const u32 other = static_cast<u32>(k2) != k ? 1u : 0u;
                const u32 hit = v >= (static_cast<u32>(k2) < k ? s : su) ? 1u : 0u;
                npass += other & hit;
            }
            if (npass > 0 && rank + npass * b2c_live_before(mask_all, b + 1) >= width) continue;
            for (int q0 = 0; q0 < K - 1 && rank < width; q0 += 3) {
                // the other lists in order, three at a time: list index q -> token q + (q >= k)
                const int left = K - 1 - q0;
                const u32 ka = static_cast<u32>(q0) + (static_cast<u32>(q0) >= k ? 1u : 0u);
                const u32 kb = static_cast<u32>(q0 + 1) + (static_cast<u32>(q0 + 1) >= k ? 1u : 0u);
                const u32 kc = static_cast<u32>(q0 + 2) + (static_cast<u32>(q0 + 2) >= k ? 1u : 0u);
                if (left >= 3) {
                    const double* const l3[3] = {cf + ka * n, cf + kb * n, cf + kc * n};
                    const double q3[3] = {ka < k ? s : su, kb < k ? s : su, kc < k ? s : su};
                    u32 c3[3];
                    b2c_sorted_counts<3>(l3, n, q3, c3);
                    rank += b2c_live_before(masks + mstride * ka, c3[0]) + b2c_live_before(masks + mstride * kb, c3[1]) +
                            b2c_live_before(masks + mstride * kc, c3[2]);
                } else if (left == 2) {
                    const double* const l2[2] = {cf + ka * n, cf + kb * n};
                    const double q2[2] = {ka < k ? s : su, kb < k ? s : su};
                    u32 c2[2];
                    b2c_sorted_counts<2>(l2, n, q2, c2);
                    rank += b2c_live_before(masks + mstride * ka, c2[0]) + b2c_live_before(masks + mstride * kb, c2[1]);
                } else {
                    const double* const l1[1] = {cf + ka * n};
                    const double q1[1] = {ka < k ? s : su};
                    u32 c1[1];
                    b2c_sorted_counts<1>(l1, n, q1, c1);
                    rank += b2c_live_before(masks + mstride * ka, c1[0]);
                }
            }
        }
        if (rank < width) place(static_cast<u32>(i), k, b, rank);
    }
}

// -----------------------------------------------------------------------------------------
// one frame with at most CAP candidates and at most B2C_FAST_KS tokens, all in shared memory: three phases,
// three block barriers (the third is issued by the caller after it has staged the next frame's tokens).
//
// Beam tables may have HOLES: the beam of rank r is written to slot r by the thread that ranked it, before the
// history prune (decoder.py:550-552) is known; a slot is live iff it holds the best rank of its history key
// (pt_min[pslot[r]] == r).  The next frame simply skips dead slots -- the relative order of the live beams,
// which is all the reference's order dependence needs, is the rank order either way -- so there is no
// compaction pass and no fourth phase.  S.holes says whether the current table is in that form; wtop / wmax
// hold the number of slots and the best score key of the previous frame (per-warp maxima).
// Invariants on entry: grouping table clear; prune table = entries pslot[0 .. n) iff S.holes.
// -----------------------------------------------------------------------------------------
template <int CAP, int LT>
B2C_HD void b2c_fast_step(const B2cParams& P, B2cFastSmem<CAP, LT>& S, B2cChain* chain_arena, B2cText* text_arena,
                          u32 text_cap, int par, int t, int sb, int slot, int K) {
    typedef B2cFastSmem<CAP, LT> SM;
    B2cFastTab& cur = S.tab[par];
    B2cFastTab& nx = S.tab[par ^ 1];
    const u32 n = b2c_max_slots(S.wtop);                       // slots of the current table (live + dead)
    const u32 M = n * static_cast<u32>(K);
    const u32 flags = S.sc.flags;
    const bool is_bpe = (flags & B2C_FL_BPE) != 0, prune = (flags & B2C_FL_PRUNE) != 0;
    const bool holes = S.holes != 0;
    const double ref = b2c_key_f64(b2c_max_slots(S.wmax));     // best score of the previous frame
    const double bscale = P.bucket_scale;
    constexpr u32 hmask = SM::HT - 1, ptmask = SM::PT - 1;
    B2C_FMARK(0);

    if (is_bpe) {
        if (holes) {   // the force_next_break scan reads last_tok of every beam: mark the dead slots first
            B2C_FOR(b, n) {
                if (S.pt_min[S.pslot[b]] != static_cast<u32>(b)) cur.last_tok[b] = B2C_INVALID_TOK;
            }
            B2C_SYNC();
        }
        if (LT > 0) b2c_bpe_force(S.ltab, S.rid[slot], K, cur.last_tok, n, S.ffirst, S.fall, &S.sc.force_break);
        else b2c_bpe_force(S.stok[sb], nullptr, K, cur.last_tok, n, S.ffirst, S.fall, &S.sc.force_break);
    }

    // ---- phase A: expand (decoder.py:447-534), merge key, grouping ---------------------------------
    B2C_FOR(s, B2C_NBUCKET) { S.bcnt[s] = 0; S.bhead[s] = B2C_NONE_U32; }
    B2C_FOR(b, n) {
        const bool live = !holes || S.pt_min[S.pslot[b]] == static_cast<u32>(b);
        const u32 plen = cur.part_len[b];
        const u64 ph = cur.part_hash[b];
        const u64 th0 = cur.text_hash[b];
        const u32 ltok = cur.last_tok[b];
        const double lg = cur.logit[b];
        for (int k = 0; k < K; ++k) {
            const u32 i = static_cast<u32>(k) * n + static_cast<u32>(b);
            // a dead beam's candidates sit in a grouping slot of their own that nobody claims: never a group leader
            // (phase B), key 0 in phase C, and never mistaken for a member of the group that owns slot 0
            if (!live) { S.cslot[i] = SM::HT; continue; }
            const B2cTok ti = b2c_fast_tok<CAP, LT>(S, sb, slot, k);
            u64 th = th0;
            u64 nph;
            u32 nplen, type;
            if ((ti.flags & B2C_TF_BLANK) || ltok == ti.canon) {                                                 // (i)
                type = 0; nph = ph; nplen = plen;
            } else if (is_bpe && ((ti.flags & B2C_TF_BPE_LEAD) || S.fall[k] || S.ffirst[k] == static_cast<u32>(b))) {   // (ii)
                type = 1; nph = ti.clean_hash; nplen = ti.clean_nchars;
                if (plen) th = b2c_text_append(th, ph);
            } else if (!is_bpe && (ti.flags & B2C_TF_SPACE)) {                                                   // (iii)
                type = 2; nph = 0; nplen = 0;
                if (plen) th = b2c_text_append(th, ph);
            } else {                                                                                             // (iv)
                type = 3; nph = b2c_hash_append(ph, ti.raw_hash, ti.raw_pow); nplen = plen + ti.raw_nchars;
            }
            S.cph[i] = nph | (static_cast<u64>(type) << 61);
            S.cmeta[i] = (nplen & 0xFFFFu) | (static_cast<u32>(ti.canon) << 16);
            S.cbk[i] = static_cast<u32>(b) | (static_cast<u32>(k) << 16);
            S.cfold[i] = lg + S.rlp[slot][k];
            const u64 key = b2c_fast_key(th, nph, nplen, ti.canon);
            S.ckey[i] = key;
            b2c_fence_block();
            // group equal keys: claim a slot or join the group that owns it
            u32 slot = static_cast<u32>(key) & hmask;
            bool claimed = false;
            while (true) {
                const u32 rep = b2c_atomic_cas_u32(&S.ht_idx[slot], B2C_NONE_U32, i);
                if (rep == B2C_NONE_U32) { claimed = true; break; }
                b2c_fence_block();
                if (S.ckey[rep] == key) break;
                slot = (slot + 1) & hmask;
            }
            S.cslot[i] = slot;
            if (!claimed) {      // the claimer is known from ht_idx: only joiners (merges) track the group's extent
                b2c_atomic_min_u32(&S.ht_min[slot], i);
                b2c_atomic_max_u32(&S.ht_max[slot], i);
                b2c_atomic_add_u32(&S.ht_cnt[slot], 1u);
            }
        }
    }
    B2C_SYNC();
    B2C_FMARK(1);

    // ---- phase B: fold each group (decoder.py:211-224), LM / hotword fusion (:346-424), bucket, max ---
    if (holes) {   // the validity tests of phase A are done: release the previous frame's prune entries
        B2C_FOR(r, n) {
            const u32 s = S.pslot[r];
            S.pt_idx[s] = B2C_NONE_U32;
            S.pt_min[s] = B2C_NONE_U32;
        }
    }
    {
        u64 tmax = 0;
        B2C_FOR(i, M) {
            const u32 slot = S.cslot[i];
            u32 first = S.ht_idx[slot], last = first;
            const u32 cnt = S.ht_cnt[slot] + 1;
            if (cnt > 1) {
                const u32 lo = S.ht_min[slot], hi = S.ht_max[slot];
                first = lo < first ? lo : first;
                last = hi > last ? hi : last;
            }
            if (first != static_cast<u32>(i)) { S.ckey[i] = 0; continue; }
            double s = S.cfold[i];
            for (u32 j = (cnt == 2) ? last : static_cast<u32>(i) + 1; cnt > 1 && j <= last; ++j) {
                if (S.cslot[j] != slot) continue;
                s = b2c_sum_log_scores_ool(s, S.cfold[j]);
            }
            S.cfold[i] = s;
            S.clast[i] = last;
            const u64 cph = S.cph[last];
            const u32 type = static_cast<u32>(cph >> 61);
            const u32 part_len = S.cmeta[last] & 0xFFFFu;
            const u32 bl = S.cbk[last] & 0xFFFFu;
            double lm_hw = cur.lm_hw[bl];
            // without LM and hotwords the text-level score is the constant hot_weight * 0: no text node is read
            if ((flags & B2C_FL_PSCORE) && (type == 1 || type == 2) && cur.part_len[bl] > 0) {
                B2cTextNew tn;
                b2c_text_extend(P, text_arena, text_cap, cur.text_node[bl], cur.part_hash[bl], cur.part_len[bl], 0, &tn, nullptr);
                lm_hw = tn.lm_hw;
            }
            double ps = 0.0;
            if (type == 0) ps = cur.pscore[bl];
            else if (part_len > 0) ps = b2c_partial_score_of(P, (flags & B2C_FL_PSCORE) != 0, cph & B2C_PH_MASK, part_len);
            const double sco = b2c_combine_score((flags & B2C_FL_LM) != 0, s, lm_hw, ps, part_len);
            const u64 key = b2c_f64_key(sco);
            S.ckey[i] = key;
            const u32 bkt = b2c_bucket(ref, sco, bscale);
            b2c_atomic_add_u32(&S.bcnt[bkt], 1u);
#if defined(__CUDA_ARCH__)
            S.cnext[i] = atomicExch(&S.bhead[bkt], static_cast<u32>(i));
#else
            S.cnext[i] = S.bhead[bkt];
            S.bhead[bkt] = static_cast<u32>(i);
#endif
            if (key > tmax) tmax = key;
        }
        b2c_warp_max_u64_slot(tmax, S.wmax);
    }
    B2C_SYNC();
    B2C_FMARK(2);

    // ---- phase C: threshold (:545-546), stable top-N (:548): rank = bucket prefix + order inside the
    //      bucket; the owner of a selected candidate commits it as beam `rank` of the next frame and enters
    //      its history key into the prune table (:550-552); grouping slots are released -------------------
    u32* const bpre = S.bpre[b2c_warp_id()];
    b2c_bucket_scan_warp_v(S.bcnt, bpre);
    const double max_score = b2c_key_f64(b2c_max_slots(S.wmax));
    const double thr = max_score + P.prune_logp;
    const u32 width = static_cast<u32>(P.beam_width);
    {
        u32 my_top = 0;
        B2C_FOR(i, M) {
            const u64 key = S.ckey[i];
            {
                const u32 slot = S.cslot[i];
                S.ht_idx[slot] = B2C_NONE_U32;
                S.ht_min[slot] = B2C_NONE_U32;
                S.ht_max[slot] = 0;
                S.ht_cnt[slot] = 0;
            }
            if (key == 0) continue;
            const double sco = b2c_key_f64(key);
            if (!(sco >= thr)) continue;
            const u32 bkt = b2c_bucket(ref, sco, bscale);
            u32 rank = bpre[bkt];
            if (rank >= width) continue;          // every candidate of a better bucket outranks it: no need to walk its own
            for (u32 j = S.bhead[bkt]; j != B2C_NONE_U32;) {      // the candidate itself adds 0; both loads of a step are independent
                const u64 kj = S.ckey[j];
                const u32 jn = S.cnext[j];
                const u32 gt = kj > key ? 1u : 0u, eq_before = (kj == key ? 1u : 0u) & (j < static_cast<u32>(i) ? 1u : 0u);
                rank += gt | eq_before;
                j = jn;
            }
            if (rank >= width) continue;
            if (rank + 1 > my_top) my_top = rank + 1;
            const u32 last = S.clast[i];
            if (prune) {
                const u32 bl = S.cbk[last] & 0xFFFFu;
                const u64 cph = S.cph[last];
                const u32 type = static_cast<u32>(cph >> 61);
                const u32 meta = S.cmeta[last];
                u64 hh = cur.hist_hash[bl];
                if ((type == 1 || type == 2) && cur.part_len[bl] > 0)       // a one-word history does not depend on the parent
                    hh = P.hist_n == 1 ? b2c_hist_fold(B2C_HIST_SEED, cur.part_hash[bl])
                                       : b2c_hist_extend(text_arena + cur.text_node[bl], P.hist_n, cur.part_hash[bl]);
                const u64 hk = b2c_fast_key(hh, cph & B2C_PH_MASK, meta & 0xFFFFu, meta >> 16);
                S.phk[rank] = hk;
                b2c_fence_block();
                u32 slot = static_cast<u32>(hk) & ptmask;
                while (true) {
                    const u32 rep = b2c_atomic_cas_u32(&S.pt_idx[slot], B2C_NONE_U32, rank);
                    if (rep == B2C_NONE_U32) break;
                    b2c_fence_block();
                    if (S.phk[rep] == hk) break;
                    slot = (slot + 1) & ptmask;
                }
                S.pslot[rank] = slot;
                b2c_atomic_min_u32(&S.pt_min[slot], rank);
            }
            b2c_fast_commit(P, S, cur, nx, chain_arena, text_arena, text_cap, sb, slot, t, rank, static_cast<u32>(i), last, flags);
        }
        b2c_warp_max_u32_slot(my_top, S.wtop);         // the selected ranks are exactly 0 .. max(wtop)-1
    }
    B2C_LAST_THREAD { S.holes = prune ? 1u : 0u; }
    B2C_FMARK(3);
    B2C_FMARK(4);
}

// -----------------------------------------------------------------------------------------
// single-token frames that cannot reorder, merge or prune anything.
//
// After a frame with ONE selected token c' every beam has last_char == c' (all four branches of
// decoder.py:452-534 set last_char = char), and the beams' (text, partial_word) pairs are pairwise distinct.
// If the next frame also selects one token c, every beam produces exactly one candidate and
//   * c == c' or c is the blank: branch (i) for every beam -- nothing changes but logit_score += p, last_char
//     and the end of partial_frames (decoder.py:454-461);
//   * c is an ordinary character (not the space, regular alphabet) and there is neither an LM nor hotwords:
//     branch (iv) for every beam -- the partial words grow by the same suffix, so keys (merge and history
//     prune) stay pairwise distinct exactly as before, and lm_score == logit_score + 0.
// In both cases the candidates are the old beams in the old order with the same number added to every
// logit_score: no merge (decoder.py:211-224), the same history-prune survivors (:227-258), and -- unless
// float64 rounding interferes -- the same order and the same threshold outcome (:545-548).  The rounding
// caveat is CHECKED, not assumed: every slot recomputes its lm_score and the frame takes this path only if
// the scores are still non-increasing in slot (= rank) order and all above max + beam_prune_logp; otherwise
// the general step runs on the untouched state.  One vote barrier, no table swap, no grouping, no ranking.
// -----------------------------------------------------------------------------------------
enum { B2C_CHEAP_NO = 0, B2C_CHEAP_T0 = 1, B2C_CHEAP_T3 = 2, B2C_CHEAP_T3P = 3 };
B2C_HD int b2c_fast_cheap_kind(u32 flags, u32 prev_single, const B2cTok& ti) {
    if (prev_single == B2C_NONE_U32) return B2C_CHEAP_NO;
    if ((ti.flags & B2C_TF_BLANK) || prev_single == ti.canon) return B2C_CHEAP_T0;
    if ((flags & B2C_FL_BPE) || (ti.flags & B2C_TF_SPACE)) return B2C_CHEAP_NO;
    // an ordinary character: without LM and hotwords the scores move together (T3); with them every beam's
    // partial-word score changes, so the new scores are computed and the frame is in place only if they
    // still come out in slot order and above the threshold (T3P, b2c_fast_scored_step)
    return (flags & B2C_FL_PSCORE) ? B2C_CHEAP_T3P : B2C_CHEAP_T3;
}

// label record of the first token of frame f (a frame whose record is in the ring): the resident table for small
// alphabets; with per-frame staging (LT == 0) only the CURRENT frame's record is available (stok[sb][0])
template <int CAP, int LT>
B2C_HD const B2cTok& b2c_fast_tok0(const B2cParams& P, const B2cFastSmem<CAP, LT>& S, int f, int sb) {
    (void)P;
    if (LT > 0) return S.ltab[S.rh[f & (B2C_FAST_HR - 1)].id0];
    return S.stok[sb][0];
}

// A RUN of R >= 1 consecutive in-place frames t .. t+R-1 (each selects one token, kinds T0 / T3 as above; the caller
// has established R from the frame records in the ring).  Per slot: R dependent additions, the exactness check of
// every frame (threshold; with LM / hotwords also the order against the next slot), ONE vote, then the R updates
// applied from registers.  Returns the number of frames done: R, or fewer when a check failed at frame t + r (the
// frames before it are applied, frame t + r is left to the general step), 0 = state untouched.
// With LM / hotwords only T0 frames are in a run: the text-level and partial-word scores of a slot are constants.
template <int CAP, int LT>
B2C_HD int b2c_fast_run_step(const B2cParams& P, B2cFastSmem<CAP, LT>& S, B2cChain* chain_arena, int par, int t, int sb, int R) {
    constexpr int HM = B2C_FAST_HR - 1;
    B2cFastTab& cur = S.tab[par];
    const u32 n = b2c_max_slots(S.wtop);
    const u32 flags = S.sc.flags;
    const bool has_lm = (flags & B2C_FL_LM) != 0;
    const bool holes = S.holes != 0;
    const bool plain = (flags & B2C_FL_PSCORE) == 0;
    const double prune = P.prune_logp;
    // slot 0 holds rank 0 = the best score of the previous frame, and it is always live.  Without LM and hotwords
    // lm_score is logit_score + (+-0) + 0: adding the same p to every beam keeps the order (rounding is monotone,
    // equal results keep their slot order), so only the threshold has to be re-checked.
    const double lmhw0 = cur.lm_hw[0], ps0s = cur.pscore[0];
    const u32 plen0 = cur.part_len[0];
    B2C_FOR(b, n) {
        double l = cur.logit[b], l0 = cur.logit[0];
        int fail = R;
        if (plain) {
#if defined(__CUDACC__)
#pragma unroll 1
#endif
            for (int j = 0; j < R; ++j) {
                const double p = S.rh[(t + j) & HM].lp0;
                l = l + p;
                l0 = l0 + p;
                const double thr = (l0 + 0.0) + prune;
                if (!((l + 0.0) >= thr) && j < fail) fail = j;
            }
        } else {
            const bool has_next = static_cast<u32>(b) + 1 < n;
            const u32 bn = has_next ? static_cast<u32>(b) + 1 : static_cast<u32>(b);
            double ln = cur.logit[bn];
            const double lmhw = cur.lm_hw[b], ps = cur.pscore[b], lmhwn = cur.lm_hw[bn], psn = cur.pscore[bn];
            const u32 plen = cur.part_len[b], plenn = cur.part_len[bn];
#if defined(__CUDACC__)
#pragma unroll 1
#endif
            for (int j = 0; j < R; ++j) {
                const double p = S.rh[(t + j) & HM].lp0;
                l = l + p;
                l0 = l0 + p;
                ln = ln + p;
                const double top = b2c_combine_score(has_lm, l0, lmhw0, ps0s, plen0);
                const double mine = b2c_combine_score(has_lm, l, lmhw, ps, plen);
                bool ok = mine >= top + prune;
                if (has_next) ok = ok && mine >= b2c_combine_score(has_lm, ln, lmhwn, psn, plenn);
                if (!ok && j < fail) fail = j;
            }
        }
        if (fail < R) b2c_atomic_min_u32(&S.run_fail, static_cast<u32>(fail));
    }
    B2C_FMARK(17);
    B2C_SYNC();
    B2C_FMARK(18);
    int Rok = R;
    if (S.run_fail != B2C_NONE_U32) {      // block-uniform, rare
        Rok = static_cast<int>(S.run_fail);
        B2C_SYNC();
        B2C_LEADER { S.run_fail = B2C_NONE_U32; }
        if (Rok == 0) return 0;
    }
    double top = 0.0;
    B2C_FOR(b, n) {
        // dead (history-pruned) slots keep their place in the score order: only their logit follows
        double l = cur.logit[b];
        const bool live = !holes || S.pt_min[S.pslot[b]] == static_cast<u32>(b);
        u64 ph = cur.part_hash[b];
        u32 plen = cur.part_len[b], chain = cur.chain[b], canon = cur.last_tok[b];
        int pfs = cur.pf_s[b], pfe = cur.pf_e[b];
        u32 prev = canon;                                  // every live beam ends in the previous frame's single token
#if defined(__CUDACC__)
#pragma unroll 1
#endif
        for (int j = 0; j < Rok; ++j) {
            const B2cFrameRec h = S.rh[(t + j) & HM];
            l = l + h.lp0;
            if (!live) continue;
            const B2cTok& ti = b2c_fast_tok0<CAP, LT>(P, S, t + j, sb);
            const bool blank = (ti.flags & B2C_TF_BLANK) != 0;
            if (blank || prev == ti.canon) {               // branch (i)
                if (!blank) pfe = t + j + 1;
            } else {                                       // branch (iv): a plain character
                const u32 id = static_cast<u32>(t + j) * B2C_FAST_W + static_cast<u32>(b);
                B2cChain c;
                c.parent = chain;
                c.tok = h.id0;
                c.kind = B2C_CK_CONT;
                c.has_word = 0;
                c.ws = pfs;
                c.we = pfe;
                b2c_chain_store(chain_arena, id, c, P.narrow_chain != 0);
                chain = id;
                ph = b2c_hash_append(ph, ti.raw_hash, ti.raw_pow);
                plen += ti.raw_nchars;
                if (pfs < 0) pfs = t + j;
                pfe = t + j + 1;
            }
            prev = ti.canon;
        }
        cur.logit[b] = l;
        if (b == 0) top = plain ? l + 0.0 : b2c_combine_score(has_lm, l, lmhw0, ps0s, plen0);
        if (!live) continue;
        cur.last_tok[b] = static_cast<u16>(prev);
        cur.part_hash[b] = ph;
        cur.part_len[b] = static_cast<u16>(plen);
        cur.chain[b] = chain;
        cur.pf_s[b] = pfs;
        cur.pf_e[b] = pfe;
        // best score of the last frame = reference point of the next frame's score buckets (slot 0's thread)
        if (b == 0) {
            S.wmax[0] = b2c_f64_key(top);
            for (int w = 1; w < B2C_FAST_NW; ++w) S.wmax[w] = 0ull;
        }
    }
    return Rok;
}

// -----------------------------------------------------------------------------------------
// One ordinary character after a one-token frame WITH a language model and / or hotwords: still no merge (same
// argument as above) and the same history-prune survivors, but lm_score = logit_score + lm_hw(text) +
// score(partial_word + c) changes per beam (decoder.py:397-420).  Every slot computes its new partial-word score
// and lm_score; if the scores are still non-increasing in slot order (equal scores keep their order, as the stable
// nlargest of decoder.py:548 would) and all reach max + beam_prune_logp, the reference's result is the old beams in
// the old order with the new fields -> in-place update.  Otherwise the state is untouched and the general step runs.
// Scratch: S.cfold[slot] (new lm_score), S.ckey[slot] (new partial score, as bits).
// -----------------------------------------------------------------------------------------
template <int CAP, int LT>
B2C_HD bool b2c_fast_scored_step(const B2cParams& P, B2cFastSmem<CAP, LT>& S, B2cChain* chain_arena, int par, int t,
                                 int sb, int slot) {
    B2cFastTab& cur = S.tab[par];
    const u32 n = b2c_max_slots(S.wtop);
    const u32 flags = S.sc.flags;
    const bool has_lm = (flags & B2C_FL_LM) != 0;
    const bool holes = S.holes != 0;
    const B2cTok ti = b2c_fast_tok<CAP, LT>(S, sb, slot, 0);
    const double p = S.rlp[slot][0];
    B2C_FOR(b, n) {
        const u64 nph = b2c_hash_append(cur.part_hash[b], ti.raw_hash, ti.raw_pow);
        const u32 nplen = static_cast<u32>(cur.part_len[b]) + ti.raw_nchars;
        const double ps = b2c_partial_score_of(P, true, nph, nplen & 0xFFFFu);
        union { double d; u64 u; } c;
        c.d = ps;
        S.ckey[b] = c.u;
        S.cfold[b] = b2c_combine_score(has_lm, cur.logit[b] + p, cur.lm_hw[b], ps, nplen & 0xFFFFu);
    }
    B2C_SYNC();
    const double top = S.cfold[0];
    const double thr = top + P.prune_logp;
    B2C_FOR(b, n) {
        const double mine = S.cfold[b];
        bool ok = mine >= thr;
        if (static_cast<u32>(b) + 1 < n) ok = ok && mine >= S.cfold[b + 1];
        if (!ok) S.cheap_bad = 1;
    }
    B2C_SYNC();
    if (S.cheap_bad) {      // block-uniform
        B2C_SYNC();
        B2C_LEADER { S.cheap_bad = 0; }
        return false;
    }
    B2C_FOR(b, n) {
        cur.logit[b] = cur.logit[b] + p;
        union { double d; u64 u; } c;
        c.u = S.ckey[b];
        // dead slots keep their place in the score order: logit and partial-word fields follow, no backtrack node
        const int ps0 = cur.pf_s[b], pe0 = cur.pf_e[b];
        cur.part_hash[b] = b2c_hash_append(cur.part_hash[b], ti.raw_hash, ti.raw_pow);
        cur.part_len[b] = static_cast<u16>(cur.part_len[b] + ti.raw_nchars);
        cur.pscore[b] = c.d;
        cur.last_tok[b] = ti.canon;
        if (ps0 < 0) cur.pf_s[b] = t;
        cur.pf_e[b] = t + 1;
        const bool live = !holes || S.pt_min[S.pslot[b]] == static_cast<u32>(b);
        if (!live) continue;
        const u32 id = static_cast<u32>(t) * B2C_FAST_W + static_cast<u32>(b);
        B2cChain cn;
        cn.parent = cur.chain[b];
        cn.tok = static_cast<u16>(S.rid[slot][0]);
        cn.kind = B2C_CK_CONT;
        cn.has_word = 0;
        cn.ws = ps0;
        cn.we = pe0;
        b2c_chain_store(chain_arena, id, cn, P.narrow_chain != 0);
        cur.chain[b] = id;
    }
    B2C_FOR(w, B2C_FAST_NW) { S.wmax[w] = w == 0 ? b2c_f64_key(top) : 0ull; }
    return true;
}

// -----------------------------------------------------------------------------------------
// multi-token frames that cannot merge: ranking by binary search instead of grouping + buckets.
//
// Same precondition as b2c_fast_cheap_step: the previous frame selected ONE token c', so every beam ends in c'
// and the (text, partial_word) pairs are pairwise distinct.  If now K >= 2 tokens with pairwise different label
// strings are selected, none of them the space (regular alphabet) and there is neither an LM nor hotwords, then
//   * a candidate's key is (text, partial_word [+ c], c): different tokens give different last_char, one token
//     maps distinct beams to distinct keys -> no two candidates merge (decoder.py:211-224 is the identity);
//   * lm_score == logit_score + 0, and inside one token the candidates are in beam (= score) order.
// So the candidate scores form K non-increasing lists, and the position of a candidate in the stable sort of
// decoder.py:548 is a sum of K - 1 binary searches plus its position in its own list.  No grouping table, no
// fold, no score buckets.  Phases: liveness masks (and release of the previous prune entries) | ranks | commit
// (one new beam per thread) -- the third barrier is the caller's.
// -----------------------------------------------------------------------------------------
template <int CAP, int LT>
B2C_HD bool b2c_fast_sorted_ok(const B2cParams& P, const B2cFastSmem<CAP, LT>& S, int sb, int slot, int K, u32 prev_single) {
    if (prev_single == B2C_NONE_U32 || K < 2 || K > B2C_SORTED_MAXK || P.has_dup_labels) return false;
    if (S.sc.flags & (B2C_FL_PSCORE | B2C_FL_BPE)) return false;
    u32 fl = 0;
    for (int k = 0; k < K; ++k) fl |= b2c_fast_tok<CAP, LT>(S, sb, slot, k).flags;
    return (fl & B2C_TF_SPACE) == 0;
}

// returns false (state untouched) when the best score is not finite
template <int CAP, int LT>
B2C_HD bool b2c_fast_sorted_step(const B2cParams& P, B2cFastSmem<CAP, LT>& S, B2cChain* chain_arena, int par, int t,
                                 int sb, int slot, int K, u32 prev_single) {
    typedef B2cFastSmem<CAP, LT> SM;
    B2cFastTab& cur = S.tab[par];
    B2cFastTab& nx = S.tab[par ^ 1];
    const u32 n = b2c_max_slots(S.wtop);
    const bool prune = (S.sc.flags & B2C_FL_PRUNE) != 0;
    const bool holes = S.holes != 0;
    constexpr u32 ptmask = SM::PT - 1;
    // best score of the frame (block-uniform): rank-0 beam + best token
    const double* const slp = S.rlp[slot];
    double top = (cur.logit[0] + slp[0]) + 0.0;
    for (int k = 1; k < K; ++k) {
        const double v = (cur.logit[0] + slp[k]) + 0.0;
        if (v > top || v != v) top = v;
    }
    if (!(top >= -1.7976931348623157e308)) return false;      // NaN / -inf (only from such input): general step
    const double thr = top + P.prune_logp;
    const u32 width = static_cast<u32>(P.beam_width);

    // ---- phase 1: which slots are live; the live owner of a prune entry releases it ----------------
#if !defined(__CUDA_ARCH__)
    for (int w = 0; w < B2C_FAST_NW; ++w) S.wmask[w] = 0;
#endif
    B2C_FOR(b, B2C_FAST_W) {
        bool live = static_cast<u32>(b) < n;
        if (live && holes) {
            const u32 ps = S.pslot[b];
            live = S.pt_min[ps] == static_cast<u32>(b);
            if (live) { S.pt_idx[ps] = B2C_NONE_U32; S.pt_min[ps] = B2C_NONE_U32; }
        }
#if defined(__CUDA_ARCH__)
        const u32 m = __ballot_sync(0xFFFFFFFFu, live);
        if ((threadIdx.x & 31) == 0) S.wmask[threadIdx.x >> 5] = m;
#else
        if (live) S.wmask[b >> 5] |= 1u << (b & 31);
#endif
        // the K candidate lists (dead slots keep their place in the score order): cf[k * n + b]
        if (static_cast<u32>(b) < n) {
            const double lg = cur.logit[b];
            for (int k = 0; k < K; ++k) S.cfold[static_cast<u32>(k) * n + static_cast<u32>(b)] = (lg + slp[k]) + 0.0;
        }
    }
    B2C_SYNC();
    B2C_FMARK(20);

    // ---- phase 2: threshold (:545-546) and rank (:548) of every candidate ---------------------------
    {
        u32 my_top = 0;
        // candidate (b, k) takes rank `rank` (if it is inside the beam width)
        auto place = [&](u32 b, u32 k, u32 rank) {
            if (rank >= width) return;
            S.ord[rank] = b | (k << 16);
            if (rank + 1 > my_top) my_top = rank + 1;
        };
        if (K <= 3) {
            // two or three tokens (84 % of these frames): a slot and its candidates per thread, all its questions in
            // lockstep.  Same token: the live beams before this one (equal scores keep beam order); another token k2:
            // its candidates that sort before (k, b) -- score greater, or equal and enumerated earlier (k2 < k).
            u32 wm[B2C_FAST_NW];
            for (int w = 0; w < B2C_FAST_NW; ++w) wm[w] = S.wmask[w];
            const double* const cf = S.cfold;
            B2C_FOR(b, n) {
                if (!((S.wmask[b >> 5] >> (b & 31)) & 1u)) continue;
                const u32 ub = static_cast<u32>(b);
                const u32 lb = b2c_live_before(wm, ub);
                if (K == 2) {
                    const double s0 = cf[ub], s1 = cf[n + ub];
                    const double* const l2[2] = {cf + n, cf};
                    const double q2[2] = {b2c_next_up(s0), s1};
                    u32 c2[2];
                    b2c_sorted_counts<2>(l2, n, q2, c2);
                    if (s0 >= thr) place(ub, 0u, lb + b2c_live_before(wm, c2[0]));
                    if (s1 >= thr) place(ub, 1u, lb + b2c_live_before(wm, c2[1]));
                } else {
                    const double s0 = cf[ub], s1 = cf[n + ub], s2 = cf[2 * n + ub];
                    const double u0 = b2c_next_up(s0), u1 = b2c_next_up(s1);
                    const double* const l6[6] = {cf + n, cf + 2 * n, cf, cf + 2 * n, cf, cf + n};
                    const double q6[6] = {u0, u0, s1, u1, s2, s2};
                    u32 c6[6];
                    b2c_sorted_counts<6>(l6, n, q6, c6);
                    if (s0 >= thr) place(ub, 0u, lb + b2c_live_before(wm, c6[0]) + b2c_live_before(wm, c6[1]));
                    if (s1 >= thr) place(ub, 1u, lb + b2c_live_before(wm, c6[2]) + b2c_live_before(wm, c6[3]));
                    if (s2 >= thr) place(ub, 2u, lb + b2c_live_before(wm, c6[4]) + b2c_live_before(wm, c6[5]));
                }
            }
        } else {
            // four to eight tokens: K (K - 1) questions per slot would leave the frame waiting for the first slots --
            // candidates strided over the threads, most of them discarded by a bound that needs no search
            b2c_rank_list_items(S.cfold, n, K, S.wmask, 0u, S.wmask, thr, width, [](double, u32) { return 0u; },
                                [&](u32, u32 k, u32 b, u32 rank) { place(b, k, rank); });
        }
        b2c_warp_max_u32_slot(my_top, S.wtop);         // the selected ranks are exactly 0 .. max(wtop)-1
    }
    B2C_FMARK(21);
    B2C_SYNC();
    B2C_FMARK(22);

    // ---- phase 3: rank r becomes beam r (decoder.py:452-534 metadata), history key into the prune table ---
    const u32 n_new = b2c_max_slots(S.wtop);
    B2C_FOR(r, n_new) {
        const u32 e = S.ord[r];
        const u32 b = e & 0xFFFFu, k = e >> 16;
        const B2cTok ti = b2c_fast_tok<CAP, LT>(S, sb, slot, static_cast<int>(k));
        const bool blank = (ti.flags & B2C_TF_BLANK) != 0;
        const bool same = blank || ti.canon == prev_single;                      // branch (i), else branch (iv)
        const u64 ph = cur.part_hash[b];
        const u32 plen = cur.part_len[b];
        const int ps0 = cur.pf_s[b], pe0 = cur.pf_e[b];
        u64 nph = ph;
        u32 nplen = plen;
        u32 chain = cur.chain[b];
        int pfs = ps0, pfe = blank ? pe0 : t + 1;
        if (!same) {
            nph = b2c_hash_append(ph, ti.raw_hash, ti.raw_pow);
            nplen = plen + ti.raw_nchars;
            pfs = ps0 < 0 ? t : ps0;
            const u32 id = static_cast<u32>(t) * B2C_FAST_W + static_cast<u32>(r);
            B2cChain c;
            c.parent = chain;
            c.tok = static_cast<u16>(S.rid[slot][k]);
            c.kind = B2C_CK_CONT;
            c.has_word = 0;
            c.ws = ps0;
            c.we = pe0;
            b2c_chain_store(chain_arena, id, c, P.narrow_chain != 0);
            chain = id;
        }
        const u64 hh = cur.hist_hash[b];
        nx.logit[r] = cur.logit[b] + slp[k];
        nx.lm_hw[r] = cur.lm_hw[b];
        nx.pscore[r] = same ? cur.pscore[b] : 0.0;
        nx.text_hash[r] = cur.text_hash[b];
        nx.part_hash[r] = nph;
        nx.hist_hash[r] = hh;
        nx.text_node[r] = cur.text_node[b];
        nx.chain[r] = chain;
        nx.pf_s[r] = pfs;
        nx.pf_e[r] = pfe;
        nx.last_tok[r] = ti.canon;
        nx.part_len[r] = static_cast<u16>(nplen);
        if (prune) {
            const u64 hk = b2c_fast_key(hh, nph, nplen & 0xFFFFu, ti.canon);
            S.phk[r] = hk;
            b2c_fence_block();
            u32 slot = static_cast<u32>(hk) & ptmask;
            while (true) {
                const u32 rep = b2c_atomic_cas_u32(&S.pt_idx[slot], B2C_NONE_U32, static_cast<u32>(r));
                if (rep == B2C_NONE_U32) break;
                b2c_fence_block();
                if (S.phk[rep] == hk) break;
                slot = (slot + 1) & ptmask;
            }
            S.pslot[r] = slot;
            b2c_atomic_min_u32(&S.pt_min[slot], static_cast<u32>(r));
        }
    }
    B2C_FOR(w, B2C_FAST_NW) { S.wmax[w] = w == 0 ? b2c_f64_key(top) : 0ull; }
    B2C_LAST_THREAD { S.holes = prune ? 1u : 0u; }
    return true;
}

// squeeze the dead slots out of the current table (into the other one: the caller flips its parity) and
// leave the state the general helpers expect: sc.n_beams / sc.prev_max set, prune table clear
template <int CAP, int LT>
B2C_HDN void b2c_fast_compact(B2cFastSmem<CAP, LT>* Sp, int par) {
    B2cFastSmem<CAP, LT>& S = *Sp;
    const B2cFastTab& cur = S.tab[par];
    B2cFastTab& nx = S.tab[par ^ 1];
    const u32 n = b2c_max_slots(S.wtop);
    const bool holes = S.holes != 0;
    const double prev_max = b2c_key_f64(b2c_max_slots(S.wmax));
    B2C_FOR(b, n) { S.ord[b] = (!holes || S.pt_min[S.pslot[b]] == static_cast<u32>(b)) ? 1u : 0u; }
    B2C_SYNC();
    B2C_FOR(b, n) {
        if (!S.ord[b]) continue;
        u32 j = 0;
        for (int q = 0; q < b; ++q) j += S.ord[q];
        nx.logit[j] = cur.logit[b]; nx.lm_hw[j] = cur.lm_hw[b]; nx.pscore[j] = cur.pscore[b];
        nx.text_hash[j] = cur.text_hash[b]; nx.part_hash[j] = cur.part_hash[b]; nx.hist_hash[j] = cur.hist_hash[b];
        nx.text_node[j] = cur.text_node[b]; nx.chain[j] = cur.chain[b];
        nx.pf_s[j] = cur.pf_s[b]; nx.pf_e[j] = cur.pf_e[b];
        nx.last_tok[j] = cur.last_tok[b]; nx.part_len[j] = cur.part_len[b];
    }
    B2C_SYNC();
    if (holes) {
        B2C_FOR(r, n) {
            const u32 s = S.pslot[r];
            S.pt_idx[s] = B2C_NONE_U32;
            S.pt_min[s] = B2C_NONE_U32;
        }
    }
    B2C_LEADER {
        u32 live = 0;
        for (u32 q = 0; q < n; ++q) live += S.ord[q];
        S.sc.n_beams = live;
        S.sc.n_sel = 0;
        S.sc.prev_max = prev_max;
        S.holes = 0;
        S.wtop[0] = live;
        for (int c = 1; c < B2C_FAST_NW; ++c) S.wtop[c] = 0;
    }
    B2C_SYNC();
}

// A frame that does not fit the shared-memory tier (or the token stage): the general step on the
// HBM tier, out of line, with its own descriptor.  Restores the invariants of b2c_fast_step.
template <int CAP, int LT>
B2C_HDN void b2c_fast_slow_step(B2cParams P, B2cLayout L, u8* smem, u8* g, int par, int t, const u32* tk_id, const double* tk_lp,
                                int K, int K_next) {
    B2cFastSmem<CAP, LT>& S = *reinterpret_cast<B2cFastSmem<CAP, LT>*>(smem);
    B2cWork W;
    b2c_fast_work(S, L, g, par, true, W);
    const u32 M = S.sc.n_beams * static_cast<u32>(K);
    const B2cCandTier C = W.tier_g;
    u32 H = b2c_ht_size(M);
    if (H > C.ht_cap) H = C.ht_cap;
    b2c_clear_tables(W, C, H);
    B2C_SYNC();
    b2c_frame_step<false>(P, W, t, tk_id, tk_lp, K, K_next);      // ends with a block barrier
    // the general step compacts its survivors and leaves their prune entries pslot[0 .. n_sel) behind
    if (S.sc.flags & B2C_FL_PRUNE) {
        B2C_FOR(r, S.sc.n_sel) {
            const u32 s = S.pslot[r];
            S.pt_idx[s] = B2C_NONE_U32;
            S.pt_min[s] = B2C_NONE_U32;
        }
    }
    B2C_LEADER {
        S.holes = 0;
        S.wtop[0] = S.sc.n_beams;
        S.wmax[0] = b2c_f64_key(S.sc.prev_max);
        for (int c = 1; c < B2C_FAST_NW; ++c) { S.wtop[c] = 0; S.wmax[c] = 0; }
    }
}

// -----------------------------------------------------------------------------------------
// one CTA: utterances from the work queue, all frames, finalisation
//
// Token staging (per utterance).  K1 left, per frame, a 16-byte record {offset, count, first token id, its
// log-prob} and compact (id, log-prob) lists.  Three shared-memory structures are kept ahead of the frame loop by
// cp.async copies issued at the TOP of an iteration and completed (wait_all + the closing barrier) at its end:
//   rh[32]       frame records; frames < hv are visible, hv - t >= 18 at the top of every iteration
//   rid/rlp[8]   token lists of frames < tv (tv <= t + 8; a frame's slot is frame & 7)
//   stok[2]      label records of the current frame's tokens (copied from the resident table, or loaded from the
//                global table one frame ahead for large alphabets: register staged, stored before the barrier)
// An iteration handles frame t, or a run of R in-place frames t .. t+R-1 with t + R < tv (the label records of
// frame t + R are staged during the iteration, which needs its ids in the ring).
// -----------------------------------------------------------------------------------------
template <int CAP, int LT>
B2C_HD void b2c_beam_block_fast(const B2cBeamArgs& A, int slot_cta, u8* smem) {
    typedef B2cFastSmem<CAP, LT> SM;
    constexpr int KR = SM::KR;
    constexpr int HM = B2C_FAST_HR - 1, TM = B2C_FAST_TR - 1;
    SM& S = *reinterpret_cast<SM*>(smem);
    const B2cLayout& L = A.L;
    u8* g = A.gws + static_cast<u64>(slot_cta) * L.gws_bytes;
    B2cChain* const chain_arena = reinterpret_cast<B2cChain*>(g + L.g_chain);
    B2cText* const text_arena = reinterpret_cast<B2cText*>(g + L.g_text);
    const u32 text_cap = L.text_cap;
    const int V = A.P.V;
    u32 st_over[6] = {0, 0, 0, 0, 0, 0};    // candidate-count histogram of the fast frames (last thread's copy counts)
    u32 st_frames = 0, st_inplace = 0, st_sorted = 0;
    B2C_LEADER {
        for (int q = 0; q < 6; ++q) S.sc.m_over[q] = 0;
        S.sc.m_frames = 0;
    }
    if (LT > 0) {       // the label table stays resident for the whole launch
        B2C_FOR(c, V < LT ? V : LT) { S.ltab[c] = A.P.toks[c]; }
    }
#if defined(B2C_PHASE_CLOCKS) && defined(__CUDA_ARCH__)
    if (threadIdx.x == 0) {
        for (int q = 0; q < 32; ++q) S.pclk[q] = 0;
        S.pclk_last = clock64();
    }
#endif

    // Chunked launches (A.chunk_t1 > 0; the host pipelines copy / streaming stage / beam search along T): CTA i keeps
    // utterance order[i] over all launches of a call, processes frames [chunk_t0, chunk_t1) and parks its state --
    // everything in front of the per-frame candidate scratch -- in HBM between two launches.
    const bool chunked = A.chunk_t1 > 0;
    constexpr u32 SAVE_WORDS = static_cast<u32>(offsetof(SM, ckey) / 4);
    u32* const parked = chunked ? reinterpret_cast<u32*>(A.state + static_cast<u64>(slot_cta) * A.state_stride) : nullptr;
    bool chunk_done = false;
    while (true) {
        u32 q;
        if (chunked) {
            if (chunk_done || slot_cta >= A.n_utts) break;
            chunk_done = true;
            q = static_cast<u32>(slot_cta);
        } else {
            B2C_LEADER { S.ticket = b2c_atomic_add_u32(A.next, 1u); }
            B2C_SYNC();
            q = S.ticket;
            if (q >= static_cast<u32>(A.n_utts)) break;
        }
        const int u = A.order[q];
        const int Tn = A.T[u];
        const u64 f0 = A.frame_off[u];
        const B2cFrameRec* recs = A.tok_rec + f0;
        const int ts = chunked ? A.chunk_t0 : 0;                                     // first frame of this launch
        int te = (chunked && !A.chunk_last && A.chunk_t1 < Tn) ? A.chunk_t1 : Tn;   // one past its last frame
        // gated launch: frames up to the first boundary are ready when the kernel starts; the later chunks are waited for
        const bool gated = !chunked && A.gate != nullptr && A.gate_n > 1;
        int gate_c = 0;
        if (gated && A.gate_bounds[1] < Tn) te = A.gate_bounds[1];
        const bool resume = chunked && ts > 0;
        if (resume && Tn <= ts) continue;                        // finished (and finalised) in an earlier launch
        // ---- fill the rings: records of the first frames, then the token lists of the first frames ----------------
        int hv = te - ts < B2C_FAST_HR ? te : ts + B2C_FAST_HR;  // records of frames < hv are (being) fetched
        B2C_FOR(c, hv - ts) { b2c_cp_async16(&S.rh[(ts + c) & HM], recs + ts + c); }
        b2c_cp_async_wait_all();
        int par = 0, sb = 0;
        u32 prev_single = B2C_NONE_U32;   // canonical token of the previous frame if it selected exactly one
        if (resume) {
            u32* const sw = reinterpret_cast<u32*>(smem);
            // the frame records just fetched live behind the parked region, the label table in front of ckey is
            // reloaded by every launch: only [0, ckey) is state
            B2C_FOR(i, SAVE_WORDS) {
                sw[i] = parked[i];
            }
            par = static_cast<int>(parked[SAVE_WORDS]);
            sb = static_cast<int>(parked[SAVE_WORDS + 1]);
            prev_single = parked[SAVE_WORDS + 2];
        } else {
            B2cWork W;
            b2c_fast_work(S, L, g, 0, false, W);
            b2c_utt_begin(A.P, W, A.start_states ? A.start_states + u : nullptr, 1, B2cStreamIn{nullptr, 0u, nullptr, nullptr});
        }
        B2C_FOR(s, SM::HT + 1) {
            S.ht_idx[s] = B2C_NONE_U32;
            S.ht_min[s] = B2C_NONE_U32;
            S.ht_max[s] = 0;
            S.ht_cnt[s] = 0;
        }
        if (!resume) {
        B2C_FOR(s, SM::PT) { S.pt_idx[s] = B2C_NONE_U32; S.pt_min[s] = B2C_NONE_U32; }
        B2C_FOR(s, B2C_NBUCKET) { S.bcnt[s] = 0; S.bhead[s] = B2C_NONE_U32; }
        B2C_LEADER {      // EMPTY_START_BEAM in the form b2c_fast_step expects: one slot, no holes, best score 0
            S.sc.n_sel = 0;
            S.holes = 0;
            S.cheap_bad = 0;
            S.run_fail = B2C_NONE_U32;
            for (int c = 0; c < B2C_FAST_NW; ++c) { S.wmax[c] = 0; S.wtop[c] = 0; S.wmask[c] = 0; }
            S.wtop[0] = 1;
            S.wmax[0] = b2c_f64_key(0.0);
            // backtrack nodes of the frame steps have fixed ids below B2C_FAST_W * T; the out-of-line step allocates above
            S.sc.chain_used = B2C_FAST_W * static_cast<u32>(Tn);
        }
        }
        B2C_SYNC();                                             // records visible
        int tv = te - ts < B2C_FAST_TR ? te : ts + B2C_FAST_TR;  // token lists of frames < tv are (being) fetched
        for (int f = ts; f < tv; ++f) {
            const B2cFrameRec hf = S.rh[f & HM];
            const u64 base = (f0 + static_cast<u64>(f & ~(B2C_RUN - 1))) * static_cast<u64>(V) + hf.off;
            const u32 kf = hf.cnt < static_cast<u32>(KR) ? hf.cnt : static_cast<u32>(KR);
            B2C_FOR(c, kf) {
                b2c_cp_async4(&S.rid[f & TM][c], A.tok_ids + base + c);
                b2c_cp_async8(&S.rlp[f & TM][c], A.tok_lp + base + c);
            }
        }
        b2c_cp_async_wait_all();
        B2C_SYNC();
        if (te > ts) {      // label records of the first frame (once per launch, latency exposed)
            const u32 c0 = S.rh[ts & HM].cnt;
            const u32 k0 = c0 < static_cast<u32>(KR) ? c0 : static_cast<u32>(KR);
            if (LT == 0) { B2C_FOR(c, k0) { S.stok[sb][c] = A.P.toks[S.rid[ts & TM][c]]; } }
        }
        B2C_SYNC();
        int t = ts;
#if defined(__CUDACC__)
#pragma unroll 1
#endif
        while (t < te) {
            const B2cFrameRec h = S.rh[t & HM];
            const int K = static_cast<int>(h.cnt);
            const int slot = t & TM;
            const u32 flags = S.sc.flags;
            // ---- what kind of step, and how many frames it covers ------------------------------------------
            const u32 Mq = b2c_max_slots(S.wtop) * static_cast<u32>(K);
            const bool oversize = Mq > static_cast<u32>(CAP) || K > KR;
            int kind = B2C_CHEAP_NO;
            int R = 1;
            if (!oversize && K == 1 && prev_single != B2C_NONE_U32) {
                kind = b2c_fast_cheap_kind(flags, prev_single, b2c_fast_tok0<CAP, LT>(A.P, S, t, sb));
                if (LT > 0 && (kind == B2C_CHEAP_T0 || kind == B2C_CHEAP_T3)) {
                    // extend the run while the next frames are in-place frames too; frame t + R must have its token
                    // list in the ring (its label records are staged during this iteration)
                    int lim = te - t < B2C_FAST_RMAX ? te - t : B2C_FAST_RMAX;
                    if (tv < te && tv - 1 - t < lim) lim = tv - 1 - t;
                    u32 pc = b2c_fast_tok0<CAP, LT>(A.P, S, t, sb).canon;
                    while (R < lim) {
                        const B2cFrameRec hn = S.rh[(t + R) & HM];
                        if (hn.cnt != 1) break;
                        const B2cTok& tn = S.ltab[hn.id0];
                        const int kn = b2c_fast_cheap_kind(flags, pc, tn);
                        if (kn != B2C_CHEAP_T0 && kn != B2C_CHEAP_T3) break;
                        pc = tn.canon;
                        ++R;
                    }
                }
            }
            // ---- prefetch: frame records, token lists (visible at the next iteration) -----------------------
            {
                const bool more_recs = hv < te && hv - t <= B2C_FAST_HR - 8;
                const int tv_new = t + B2C_FAST_TR < te ? t + B2C_FAST_TR : te;
                B2C_IN_LAST_WARP {
                    if (more_recs) {
                        B2C_FOR_LANES(c, 8) {
                            if (hv + c < te) b2c_cp_async16(&S.rh[(hv + c) & HM], recs + hv + c);
                        }
                    }
                    for (int f = tv; f < tv_new; ++f) {
                        const B2cFrameRec hf = S.rh[f & HM];
                        const u64 base = (f0 + static_cast<u64>(f & ~(B2C_RUN - 1))) * static_cast<u64>(V) + hf.off;
                        const u32 kf = hf.cnt < static_cast<u32>(KR) ? hf.cnt : static_cast<u32>(KR);
                        B2C_FOR_LANES(c, kf) {
                            b2c_cp_async4(&S.rid[f & TM][c], A.tok_ids + base + c);
                            b2c_cp_async8(&S.rlp[f & TM][c], A.tok_lp + base + c);
                        }
                    }
                }
                if (more_recs) hv = hv + 8 < te ? hv + 8 : te;
                if (tv_new > tv) tv = tv_new;
            }
#if defined(__CUDA_ARCH__)
            // large alphabets (no resident label table): the label records of frame t + 1 come from global memory --
            // loaded here into a register, stored to shared memory just before the closing barrier
            B2cTok ptk;
            bool has_ptk = false;
            if (LT == 0 && t + 1 < te) {
                const u32 cn1 = S.rh[(t + 1) & HM].cnt;
                has_ptk = threadIdx.x < (cn1 < static_cast<u32>(KR) ? cn1 : static_cast<u32>(KR));
                if (has_ptk) ptk = A.P.toks[S.rid[(t + 1) & TM][threadIdx.x]];
            }
#endif
            B2C_FMARK(16);
            bool in_place = false;      // the frame(s) updated the current table in place (no table swap)
            int done_frames = 0;
            if (oversize) {
                const u64 base_a = (f0 + static_cast<u64>(t & ~(B2C_RUN - 1))) * static_cast<u64>(V) + h.off;
                const int K_next = t + 1 < te ? static_cast<int>(S.rh[(t + 1) & HM].cnt) : 1;
                // the general step wants a dense table: squeeze first (the squeezed table is the other one)
                b2c_fast_compact<CAP, LT>(&S, par);
                par ^= 1;
                b2c_fast_slow_step<CAP, LT>(A.P, L, smem, g, par, t, A.tok_ids + base_a, A.tok_lp + base_a, K, K_next);
                done_frames = 1;
            } else {
                B2C_LAST_THREAD {
                    for (int c = 0; c < 6; ++c) st_over[c] += (Mq > (128u << c)) ? 1u : 0u;
                }
                if (kind == B2C_CHEAP_T3P) {
                    in_place = b2c_fast_scored_step<CAP, LT>(A.P, S, chain_arena, par, t, sb, slot);
                    done_frames = in_place ? 1 : 0;
                } else if (kind != B2C_CHEAP_NO) {
                    done_frames = b2c_fast_run_step<CAP, LT>(A.P, S, chain_arena, par, t, sb, R);
                    in_place = done_frames > 0;
                }
                if (in_place) {
                    B2C_LAST_THREAD { st_inplace += static_cast<u32>(done_frames); }
                    B2C_FMARK(5);
                } else if (kind == B2C_CHEAP_NO && b2c_fast_sorted_ok<CAP, LT>(A.P, S, sb, slot, K, prev_single)) {
                    if (b2c_fast_sorted_step<CAP, LT>(A.P, S, chain_arena, par, t, sb, slot, K, prev_single)) {
                        done_frames = 1;
                        B2C_LAST_THREAD { ++st_sorted; }
                        B2C_FMARK(7);
                    }
                }
                if (done_frames == 0) {
#if defined(B2C_PHASE_CLOCKS) && defined(__CUDA_ARCH__)
                    const long long c0 = clock64();
#endif
                    b2c_fast_step<CAP, LT>(A.P, S, chain_arena, text_arena, text_cap, par, t, sb, slot, K);
#if defined(B2C_PHASE_CLOCKS) && defined(__CUDA_ARCH__)
                    if (threadIdx.x == 0) {      // general frames by token count: cycles in 9..11, frames in 12..14
                        const int cls = K == 1 ? 0 : (K == 2 ? 1 : 2);
                        S.pclk[9 + cls] += static_cast<u64>(clock64() - c0);
                        S.pclk[12 + cls] += 1;
                    }
#endif
                    done_frames = 1;
                }
                B2C_LAST_THREAD { st_frames += static_cast<u32>(done_frames); }
            }
            // after a single-token frame every beam ends in that token (precondition of the in-place steps)
            const int t_last = t + done_frames - 1;
            if (done_frames == 1) prev_single = (K == 1) ? static_cast<u32>(b2c_fast_tok0<CAP, LT>(A.P, S, t, sb).canon) : B2C_NONE_U32;
            else prev_single = static_cast<u32>(S.ltab[S.rh[t_last & HM].id0].canon);
            // ---- label records of the next frame's tokens (its ids are in the ring: t + done_frames < tv) ------
            const int tn = t + done_frames;
#if defined(__CUDA_ARCH__)
            if (LT == 0) {
                if (has_ptk) S.stok[sb ^ 1][threadIdx.x] = ptk;        // tn == t + 1: without the table every step covers one frame
            }
#else
            if (LT == 0 && tn < te) {
                const u32 cn = S.rh[tn & HM].cnt;
                const u32 kb = cn < static_cast<u32>(KR) ? cn : static_cast<u32>(KR);
                B2C_FOR(c, kb) { S.stok[sb ^ 1][c] = A.P.toks[S.rid[tn & TM][c]]; }
            }
#endif
            B2C_FMARK(19);
            b2c_cp_async_wait_all();
            B2C_SYNC();
            B2C_FMARK(6);
            if (!in_place) par ^= 1;
            sb ^= 1;
            t = tn;
            if (gated && t >= te && te < Tn) {
                // ---- the next chunk of frames: wait until the streaming stage has written its token lists ------------
                B2C_LEADER {
#if defined(__CUDA_ARCH__)
                    const volatile u32* flag = A.gate + gate_c + 1;
                    const long long c0 = clock64();
                    while (*flag == 0u) {
                        __nanosleep(200);
                        if (clock64() - c0 > 80000000ll) { S.sc.status |= B2C_ERR_GATE; break; }      // ~40 ms: give up
                    }
                    __threadfence();
#else
                    if (A.gate[gate_c + 1] == 0u) S.sc.status |= B2C_ERR_GATE;
#endif
                }
                B2C_SYNC();
                if (S.sc.status & B2C_ERR_GATE) break;           // block-uniform
                ++gate_c;
                te = (gate_c + 1 < A.gate_n && A.gate_bounds[gate_c + 1] < Tn) ? A.gate_bounds[gate_c + 1] : Tn;
                // refill the rings from frame t
                hv = te - t < B2C_FAST_HR ? te : t + B2C_FAST_HR;
                B2C_FOR(c, hv - t) { b2c_cp_async16(&S.rh[(t + c) & HM], recs + t + c); }
                b2c_cp_async_wait_all();
                B2C_SYNC();
                tv = te - t < B2C_FAST_TR ? te : t + B2C_FAST_TR;
                for (int f = t; f < tv; ++f) {
                    const B2cFrameRec hf = S.rh[f & HM];
                    const u64 base = (f0 + static_cast<u64>(f & ~(B2C_RUN - 1))) * static_cast<u64>(V) + hf.off;
                    const u32 kf = hf.cnt < static_cast<u32>(KR) ? hf.cnt : static_cast<u32>(KR);
                    B2C_FOR(c, kf) {
                        b2c_cp_async4(&S.rid[f & TM][c], A.tok_ids + base + c);
                        b2c_cp_async8(&S.rlp[f & TM][c], A.tok_lp + base + c);
                    }
                }
                b2c_cp_async_wait_all();
                B2C_SYNC();
                if (LT == 0) {
                    const u32 c0n = S.rh[t & HM].cnt;
                    const u32 k0 = c0n < static_cast<u32>(KR) ? c0n : static_cast<u32>(KR);
                    B2C_FOR(c, k0) { S.stok[sb][c] = A.P.toks[S.rid[t & TM][c]]; }
                    B2C_SYNC();
                }
            }
        }
        if (chunked && te < Tn) {      // more frames in a later launch: park the state
            const u32* const sw = reinterpret_cast<const u32*>(smem);
            B2C_FOR(i, SAVE_WORDS) { parked[i] = sw[i]; }
            B2C_LEADER {
                parked[SAVE_WORDS] = static_cast<u32>(par);
                parked[SAVE_WORDS + 1] = static_cast<u32>(sb);
                parked[SAVE_WORDS + 2] = prev_single;
            }
            continue;
        }
        B2cOut O;
        const u64 ob = static_cast<u64>(A.P.out_beams);
        O.n_beams = A.out_nbeams + u;
        O.status = A.out_status + u;
        O.scores = A.out_scores + static_cast<u64>(u) * ob * 2;
        O.n_tok = A.out_ntok + static_cast<u64>(u) * ob;
        O.n_words = A.out_nwords + static_cast<u64>(u) * ob;
        O.stride = static_cast<u32>(Tn) + 1;
        O.toks = A.out_toks + ob * (f0 + static_cast<u64>(u));
        O.frames = A.out_frames + 2 * ob * (f0 + static_cast<u64>(u));
        O.states = A.out_states + static_cast<u64>(u) * ob;
        O.aux = nullptr;
        O.states_x = nullptr;
        b2c_fast_compact<CAP, LT>(&S, par);
        par ^= 1;
        {
            B2cWork W;
            b2c_fast_work(S, L, g, par, false, W);
            b2c_finalize(A.P, W, O, B2C_FIN_EOS);
        }
        B2C_FMARK(8);
    }
    if (A.m_stats) {
        B2C_LAST_THREAD {
            for (int c = 0; c < 6; ++c)
                if (st_over[c]) b2c_atomic_add_u32(A.m_stats + c, st_over[c]);
            if (st_frames) b2c_atomic_add_u32(A.m_stats + 6, st_frames);
            if (st_inplace) b2c_atomic_add_u32(A.m_stats + 7, st_inplace);
            if (st_sorted) b2c_atomic_add_u32(A.m_stats + 8, st_sorted);
        }
        B2C_LEADER {   // frames that took the general step counted themselves in shared memory
            for (int c = 0; c < 6; ++c)
                if (S.sc.m_over[c]) b2c_atomic_add_u32(A.m_stats + c, S.sc.m_over[c]);
            if (S.sc.m_frames) b2c_atomic_add_u32(A.m_stats + 6, S.sc.m_frames);
        }
    }
#if defined(B2C_PHASE_CLOCKS) && defined(__CUDA_ARCH__)
    if (threadIdx.x == 0 && A.phase_clk)
        for (int c = 0; c < 32; ++c) atomicAdd(A.phase_clk + c, S.pclk[c]);
#endif
}
