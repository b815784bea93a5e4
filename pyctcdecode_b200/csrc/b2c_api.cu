// b200ctc -- C ABI implementation (include/b200ctc.h): kernels, workspace layout, batch
// orchestration, result assembly.  Compiled by nvcc for sm_100a into libb200ctc.so.
// With -DB2C_HOSTSIM (tests/hostsim only) the same file is compiled by g++ against a stub of
// the CUDA runtime and runs the kernel bodies block by block on the CPU so that kernel logic
// can be tested where there is no GPU; that build is never loaded by the product package.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <numeric>
#include <string>
#include <thread>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <vector>

#ifdef B2C_HOSTSIM
#include "cuda_shim.h"
#else
#include <cuda_runtime.h>
#endif

#include "../../include/b200ctc.h"
#include "b2c_beam.h"
#include "b2c_common.h"
#include "b2c_lm_host.h"
#include "b2c_prepare.h"

#define B2C_VERSION 100
#define B2C_BEAM_THREADS 128
#define B2C_PREP_THREADS (B2C_PREP_WARPS * 32)

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
#define CUDA_OK(expr)                                                                         \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess)                                                                \
            return fail(B2C_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));     \
    } while (0)

// =========================================================================================
// workspace layout (shared memory + per-slot HBM workspace), computed on the host and
// interpreted by the kernel
// =========================================================================================
static inline u64 al16(u64 x) { return (x + 15) & ~15ull; }
static inline u64 tab_bytes(int W) { return 6 * al16(8ull * W) + 4 * al16(4ull * W) + 2 * al16(2ull * W) + 64; }
static inline u64 sel_bytes(int W, int n_warps, int nb) { return al16(8ull * W) + 2 * al16(4ull * W) + 2 * al16(4ull * pt_cap_for(W)) + 2 * al16(4ull * nb) +
           (nb == B2C_NBUCKET ? al16(4ull * B2C_NBUCKET * n_warps) : al16(4ull * (nb + 32))) +
           al16(sizeof(B2cTok) * B2C_STAGE_K) + al16(8ull * B2C_STAGE_K) + al16(4ull * B2C_STAGE_K) + 64; }
static inline u64 tier_bytes(u32 cap, u32 ht) { return al16(8ull * cap) * 4 + al16(4ull * cap) * 4 + al16(4ull * ht) * 4 + 64; }

static u32 pow2_ge(u32 x) {
    u32 p = 16;
    while (p < x) p <<= 1;
    return p;
}

// cap_request > 0: "fast" layout -- shared-memory candidate tier of exactly cap_request entries, no
// HBM tier, beam tables in shared memory (the caller checks smem_bytes against the budget).
// cap_request == 0: general layout -- what fits in shared memory plus an HBM tier sized for the
// worst case beam_width * V.
static B2cLayout make_layout(int W, int V, int T_max, bool full_caps, u32 smem_budget, u32 cap_request, u64 worst_m = 0, int n_warps = 4,
                             u64 extra_chain = 0, u64 extra_text = 0, int n_lm = 1, int n_bucket = B2C_NBUCKET, u32 cap_max = 512) {
    B2cLayout L;
    std::memset(&L, 0, sizeof(L));
    L.W = W;
    L.V = V;
    L.n_warps = n_warps;
    L.n_bucket = n_bucket;
    const u64 worst = static_cast<u64>(W) * static_cast<u64>(V);
    u64 fixed = 128 + sel_bytes(W, n_warps, n_bucket);
    if (cap_request) {
        L.beams_in_smem = 1;
        fixed += 2 * tab_bytes(W);
        L.cap_s = cap_request;
        L.ht_s = pow2_ge(2 * cap_request);
        if (worst_m > cap_request) {   // rare oversize frames of a fast-class utterance use the HBM tier
            L.cap_g = static_cast<u32>(std::min<u64>(worst_m, 0x7FFFFFFFull));
            L.ht_g = pow2_ge(2 * L.cap_g);
        }
    } else {
        L.beams_in_smem = (fixed + 2 * tab_bytes(W) + tier_bytes(256, 512) <= smem_budget) ? 1 : 0;
        if (L.beams_in_smem) fixed += 2 * tab_bytes(W);
        u32 cap = cap_max;
        while (cap > 64 && fixed + tier_bytes(cap, pow2_ge(2 * cap)) > smem_budget) cap >>= 1;
        L.cap_s = cap;
        L.ht_s = pow2_ge(2 * cap);
        if (worst > cap) {
            L.cap_g = static_cast<u32>(std::min<u64>(worst, 0x7FFFFFFFull));
            L.ht_g = pow2_ge(2 * L.cap_g);
        }
    }
    const u64 wt = static_cast<u64>(W) * static_cast<u64>(std::max(T_max, 1));
    L.chain_cap = static_cast<u32>(std::min<u64>(wt + 16 + extra_chain, 0x7FFFFFF0ull));
    L.text_cap = static_cast<u32>(std::min<u64>((full_caps ? wt + 16 : wt / 4 + 4096) + extra_text, 0x7FFFFFF0ull));
    u64 s = 0;
    L.s_sc = static_cast<u32>(s); s += 128;
    if (L.beams_in_smem) {
        L.s_tab[0] = static_cast<u32>(s); s += tab_bytes(W);
        L.s_tab[1] = static_cast<u32>(s); s += tab_bytes(W);
    }
    L.s_sel = static_cast<u32>(s); s += sel_bytes(W, n_warps, n_bucket);
    L.s_tier = static_cast<u32>(s); s += tier_bytes(L.cap_s, L.ht_s);
    L.smem_bytes = static_cast<u32>(s);
    u64 g = 0;
    if (!L.beams_in_smem) {
        L.g_tab[0] = g; g += tab_bytes(W);
        L.g_tab[1] = g; g += tab_bytes(W);
    }
    L.g_tier = g; if (L.cap_g) g += tier_bytes(L.cap_g, L.ht_g);
    L.g_tk = g; g += al16(4ull * V) + al16(static_cast<u64>(V)) + 64;
    L.g_chain = g; g += al16(sizeof(B2cChain) * static_cast<u64>(L.chain_cap));
    L.g_text = g; g += al16(sizeof(B2cText) * static_cast<u64>(L.text_cap)) +
                      al16(sizeof(B2cLmState) * static_cast<u64>(L.text_cap) * static_cast<u64>(n_lm > 1 ? n_lm - 1 : 0));
    L.gws_bytes = (g + 255) & ~255ull;
    return L;
}

// =========================================================================================
// kernels
// =========================================================================================
struct B2cBeamArgs {
    B2cParams P;
    B2cLayout L;
    int n_utts;
    const int* order;          // utterance ids, longest first
    u32* next;                 // work queue head
    const u64* frame_off;
    const int* T;
    const B2cFrameRec* tok_rec;
    const u32* tok_ids;
    const double* tok_lp;
    u8* gws;                   // [slots][L.gws_bytes]
    const B2cLmState* start_states;  // optional [n_utts]
    // streaming calls (general kernel only): input beams per utterance, what to do at the end of the call
    const B2cStreamUtt* s_utts;      // optional [n_utts]
    const B2cStreamBeam* s_beams;
    const u64* s_word_hash;
    const u32* s_word_len;
    int fin_mode;                    // B2C_FIN_*
    int* out_aux;                    // [n_utts][out_beams][4], streaming calls only
    B2cLmState* out_states_x;        // [n_utts][out_beams][n_lm - 1], MultiLanguageModel only
    // outputs
    int* out_nbeams;
    int* out_status;
    double* out_scores;
    int* out_ntok;
    int* out_nwords;
    u32* out_toks;
    int* out_frames;
    B2cLmState* out_states;
    // chunked launches of the latency-first kernel (chunk_t1 > 0): frames [chunk_t0, chunk_t1) of every utterance, CTA i
    // bound to utterance order[i], state parked in `state` between launches
    int chunk_t0, chunk_t1, chunk_last, pad_chunk;
    u8* state;
    u64 state_stride;
    // gated launch (gate != nullptr): ONE launch whose CTAs wait, at the boundaries gate_bounds[1..gate_n-1], for the
    // flag gate[c] that the host sets (stream-ordered) once the streaming stage has written chunk c's token lists
    const u32* gate;
    int gate_n;
    int gate_bounds[5];
    u64* phase_clk;            // [16] profiling builds only (-DB2C_PHASE_CLOCKS)
    u32* m_stats;              // [8] frames over 128..4096 candidates, total frames (adaptive sizing), in-place frames, sorted (no-merge) frames
};

// kFast: every frame of every utterance handed to this launch fits the shared-memory candidate
// tier (the host guarantees beam_width * max tokens-per-frame <= cap_s) and the beam tables are in
// shared memory; the general variant works through generic pointers and may use the HBM tier.
template <bool kFast>
B2C_HD void b2c_beam_block(const B2cBeamArgs& A, int slot, u8* smem) {
    const B2cLayout& L = A.L;
    u8* g = A.gws + static_cast<u64>(slot) * L.gws_bytes;
    B2cWork W;
    b2c_make_work(L, smem, g, 0, kFast || L.beams_in_smem, W);
    int parity = 0;      // which beam table is current (the out-of-line step rebuilds its descriptor from it)
    u32* s_cur = reinterpret_cast<u32*>(smem + L.s_sc + 120);  // queue ticket of this CTA
    B2C_LEADER {
        for (int q = 0; q < 6; ++q) W.sc->m_over[q] = 0;
        W.sc->m_frames = 0;
        W.sc->m_inplace = 0;
    }
#if defined(B2C_PHASE_CLOCKS) && defined(__CUDA_ARCH__)
    for (int q = 0; q < 16; ++q) W.clk[q] = 0;
    W.clk_last = clock64();
#endif

    while (true) {
        B2C_LEADER { *s_cur = b2c_atomic_add_u32(A.next, 1u); }
        B2C_SYNC();
        const u32 q = *s_cur;
        if (q >= static_cast<u32>(A.n_utts)) break;
        const int u = A.order[q];
        const int Tn = A.T[u];
        const u64 f0 = A.frame_off[u];
        const B2cFrameRec* recs = A.tok_rec + f0;
        B2cFrameRec rec;
        rec.off = 0;
        rec.cnt = 1;
        if (Tn > 0) rec = recs[0];
        B2cStreamIn sin{nullptr, 0u, nullptr, nullptr};
        int t0_frames = 0;
        if (A.s_utts) {
            const B2cStreamUtt su = A.s_utts[u];
            sin.beams = A.s_beams + su.beam_off;
            sin.n_beams = su.n_beams;
            sin.word_hash = A.s_word_hash;
            sin.word_len = A.s_word_len;
            t0_frames = su.t0;
        }
        b2c_utt_begin(A.P, W, A.start_states ? A.start_states + static_cast<u64>(u) * (A.P.n_lm > 1 ? A.P.n_lm : 1) : nullptr,
                      static_cast<int>(rec.cnt), sin);
#if defined(__CUDACC__)
#pragma unroll 1
#endif
        u32 prev_single = B2C_NONE_U32;   // canonical token of the previous frame if it selected exactly one token
        for (int t = 0; t < Tn; ++t) {
            B2cFrameRec nxt;
            nxt.off = 0;
            nxt.cnt = 1;
            if (t + 1 < Tn) nxt = recs[t + 1];      // one frame ahead: hides the load latency
            const u64 base = (f0 + static_cast<u64>(t & ~(B2C_RUN - 1))) * static_cast<u64>(A.P.V) + rec.off;
            bool in_place = false;
            u32 single = B2C_NONE_U32;
            if (rec.cnt == 1) {
                const u16 id0 = rec.id0;
                const B2cTok t0 = A.P.toks[id0];
                single = t0.canon;
                const int kind = b2c_inplace_kind(W.sc->flags, prev_single, t0.flags, t0.canon);
                if (kind != B2C_INPLACE_NO)
                    in_place = b2c_inplace_step(A.P, W, t + t0_frames, kind, id0, t0, rec.lp0, static_cast<int>(nxt.cnt));
                B2C_MARK(5);
            }
            prev_single = single;
            if (in_place) {
                // no table swap, no parity flip
            } else if (kFast && W.sc->n_beams * rec.cnt > L.cap_s) {
                b2c_frame_step_slow(A.P, L, smem, g, parity, t + t0_frames, A.tok_ids + base, A.tok_lp + base, static_cast<int>(rec.cnt), static_cast<int>(nxt.cnt));
                b2c_swap_tabs(W.cur, W.nxt);   // the out-of-line step swapped its private descriptor
                parity ^= 1;
            } else {
                b2c_frame_step<kFast>(A.P, W, t + t0_frames, A.tok_ids + base, A.tok_lp + base, static_cast<int>(rec.cnt), static_cast<int>(nxt.cnt));
                parity ^= 1;
            }
            rec = nxt;
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
        O.aux = A.out_aux ? A.out_aux + 4 * static_cast<u64>(u) * ob : nullptr;
        O.states_x = A.out_states_x ? A.out_states_x + static_cast<u64>(u) * ob * (A.P.n_lm - 1) : nullptr;
        b2c_finalize(A.P, W, O, A.fin_mode);
        B2C_MARK(8);
    }
    B2C_LEADER {
        if (A.m_stats) {
            for (int q = 0; q < 6; ++q)
                if (W.sc->m_over[q]) b2c_atomic_add_u32(A.m_stats + q, W.sc->m_over[q]);
            b2c_atomic_add_u32(A.m_stats + 6, W.sc->m_frames);
            if (W.sc->m_inplace) b2c_atomic_add_u32(A.m_stats + 7, W.sc->m_inplace);
        }
    }
#if defined(B2C_PHASE_CLOCKS) && defined(__CUDA_ARCH__)
    if (threadIdx.x == 0 && A.phase_clk)
        for (int q = 0; q < 16; ++q) atomicAdd(A.phase_clk + q, W.clk[q]);
#endif
}

#include "b2c_beam_fast.h"
// latency-first kernel variants (beam_width <= 128): candidate capacity x resident CTAs per SM.  A is the
// latency choice (batch resident at once); B and C trade capacity for residency when the batch is larger
// than the resident set and the candidate histogram of the previous call says the frames fit.
// Each variant exists with the label table resident in shared memory (alphabets of up to B2C_FAST_LT labels: runs of
// in-place frames enabled) and with per-frame label staging (larger alphabets).
#define B2C_FAST_LT 64
typedef B2cFastSmem<1024, B2C_FAST_LT> B2cFastSmemA;      // 2 CTAs per SM
typedef B2cFastSmem<512, B2C_FAST_LT> B2cFastSmemB;       // 3 CTAs per SM
typedef B2cFastSmem<256, B2C_FAST_LT> B2cFastSmemC;       // 4 CTAs per SM
static const u32 kV5Cap[3] = {1024, 512, 256};
static const int kV5Occ[3] = {2, 3, 4};
// [variant][0: staged labels, 1: resident table]
static const size_t kV5Smem[3][2] = {{sizeof(B2cFastSmem<1024, 0>), sizeof(B2cFastSmemA)},
                                     {sizeof(B2cFastSmem<512, 0>), sizeof(B2cFastSmemB)},
                                     {sizeof(B2cFastSmem<256, 0>), sizeof(B2cFastSmemC)}};
// bytes a CTA parks between two chunked launches: everything in front of the per-frame candidate scratch
typedef B2cFastSmem<1024, 0> B2cFastSmemA0;
typedef B2cFastSmem<512, 0> B2cFastSmemB0;
typedef B2cFastSmem<256, 0> B2cFastSmemC0;
static const size_t kV5Save[3][2] = {{offsetof(B2cFastSmemA0, ckey), offsetof(B2cFastSmemA, ckey)},
                                     {offsetof(B2cFastSmemB0, ckey), offsetof(B2cFastSmemB, ckey)},
                                     {offsetof(B2cFastSmemC0, ckey), offsetof(B2cFastSmemC, ckey)}};
#define B2C_PIPE_CHUNKS 4
#define B2C_E_RETRY_PLAIN (-1000)     // internal: the pipelined attempt must be redone as a plain call
static_assert(2 * (sizeof(B2cFastSmemA) + 1024) <= 228 * 1024, "variant A: 2 CTAs per SM");
static_assert(3 * (sizeof(B2cFastSmemB) + 1024) <= 228 * 1024, "variant B: 3 CTAs per SM");
static_assert(4 * (sizeof(B2cFastSmemC) + 1024) <= 228 * 1024, "variant C: 4 CTAs per SM");

// half-precision logits (B2C_DTYPE_F16 / B2C_DTYPE_BF16) travel over PCIe as they are and are widened to float32 on the
// device, exactly (every half / bfloat16 value is a float32 value); the path then computes as for float32 input
B2C_HD float b2c_f16_bits_to_float(u16 h) {
    const u32 sign = static_cast<u32>(h & 0x8000u) << 16;
    u32 exp = (h >> 10) & 0x1Fu, man = h & 0x3FFu, out;
    if (exp == 0) {
        if (man == 0) {
            out = sign;
        } else {                                   // subnormal: normalise
            int e = -1;
            do { ++e; man <<= 1; } while (!(man & 0x400u));
            out = sign | (static_cast<u32>(127 - 15 - e) << 23) | ((man & 0x3FFu) << 13);
        }
    } else if (exp == 31) {
        out = sign | 0x7F800000u | (man << 13);
    } else {
        out = sign | ((exp + 127 - 15) << 23) | (man << 13);
    }
    union { u32 u; float f; } c;
    c.u = out;
    return c.f;
}
B2C_HD float b2c_bf16_bits_to_float(u16 h) {
    union { u32 u; float f; } c;
    c.u = static_cast<u32>(h) << 16;
    return c.f;
}
B2C_HD void b2c_widen_range(const u16* src, float* dst, u64 begin, u64 end, u64 step, int bf16) {
    for (u64 i = begin; i < end; i += step) dst[i] = bf16 ? b2c_bf16_bits_to_float(src[i]) : b2c_f16_bits_to_float(src[i]);
}

#ifndef B2C_HOSTSIM
__global__ void __launch_bounds__(256) b2c_widen_kernel(const u16* src, float* dst, u64 n, int bf16) {
    b2c_widen_range(src, dst, static_cast<u64>(blockIdx.x) * blockDim.x + threadIdx.x, n, static_cast<u64>(gridDim.x) * blockDim.x, bf16);
}
template <int CAP, int OCC, int LT>
__global__ void __launch_bounds__(B2C_FAST_W, OCC) b2c_beam_fast_kernel(const B2cBeamArgs A) {
    extern __shared__ __align__(16) u8 b2c_smem[];
    b2c_beam_block_fast<CAP, LT>(A, static_cast<int>(blockIdx.x), b2c_smem);
}
// device-resident utterances that are not adjacent in memory (a padded [B, T, V] batch with lengths, a list
// of separate tensors): ONE launch packs their valid rows, instead of one cudaMemcpyAsync per utterance
__global__ void __launch_bounds__(256) b2c_gather_kernel(const void* const* src, const u64* frame_off, const int* T, u64 row_words,
                                                         u32* dst, int n_utts, int chunks) {
    const int u = static_cast<int>(blockIdx.x) / chunks, c = static_cast<int>(blockIdx.x) % chunks;
    if (u >= n_utts) return;
    const u64 words = static_cast<u64>(T[u]) * row_words;
    const u32* s = static_cast<const u32*>(src[u]);
    u32* o = dst + frame_off[u] * row_words;
    for (u64 i = static_cast<u64>(c) * blockDim.x + threadIdx.x; i < words; i += static_cast<u64>(chunks) * blockDim.x) o[i] = s[i];
}
// float32, V <= 32: one lane per row, tiles of 32 rows brought in by bulk asynchronous copies (b2c_prepare.h)
__global__ void __launch_bounds__(B2C_TILE_WARPS * 32) b2c_tokens_tile_kernel(const B2cPrepArgs A) {
    __shared__ B2cTileShared sh;
    b2c_tokens_tiles_v32(A, static_cast<int>(blockIdx.x), static_cast<int>(gridDim.x), &sh);
}
template <class T>
__global__ void __launch_bounds__(128) b2c_decide_kernel(const B2cPrepArgs A) {
    __shared__ B2cDecideShared sh;
    b2c_decide_block<T>(A, static_cast<int>(blockIdx.x), &sh);
}
template <class T>
__global__ void __launch_bounds__(B2C_PREP_THREADS, 4) b2c_tokens_kernel(const B2cPrepArgs A) {
    __shared__ B2cPrepShared sh;
    b2c_tokens_block<T>(A, static_cast<int>(blockIdx.x), static_cast<int>(gridDim.x), &sh);
}
// kThreads x kOcc bound the register allocation: (128,4) and (256,2) -> <= 128 registers, (128,2) -> <= 255
template <bool kFast, int kThreads, int kOcc>
__global__ void __launch_bounds__(kThreads, kOcc) b2c_beam_kernel(const B2cBeamArgs A) {
    extern __shared__ __align__(16) u8 b2c_smem[];
    b2c_beam_block<kFast>(A, static_cast<int>(blockIdx.x), b2c_smem);
}
#endif

// =========================================================================================
// objects
// =========================================================================================
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return 0;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            e = cudaMalloc(&p, bytes);
            want = bytes;
        }
        if (e != cudaSuccess) { p = nullptr; return fail(B2C_E_NOMEM, std::string("cudaMalloc: ") + cudaGetErrorString(e)); }
        cap = want;
        return 0;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class U> U* as() const { return static_cast<U*>(p); }
};
struct PinBuf {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return 0;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMallocHost(&p, want);
        if (e != cudaSuccess) { p = nullptr; return fail(B2C_E_NOMEM, std::string("cudaMallocHost: ") + cudaGetErrorString(e)); }
        cap = want;
        return 0;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
    template <class U> U* as() const { return static_cast<U*>(p); }
};

struct b2c_lm {
    B2cLmHost host;
    std::map<int, const void*> dev;       // device -> blob address
    std::map<int, void*> owned;           // device -> memory we allocated
    std::mutex mu;
};

// a few persistent host threads for the per-utterance string building (spawning threads per call costs
// tens of microseconds each and occasionally milliseconds)
struct HostPool {
    std::vector<std::thread> workers;
    std::mutex mu;
    std::condition_variable cv_work, cv_done;
    const std::function<void(int)>* fn = nullptr;
    int n_tasks = 0, generation = 0, active = 0;
    std::atomic<int> next{0}, done{0};
    bool stop = false;
    void start(int n) {
        for (int i = 0; i < n; ++i) workers.emplace_back([this]() { loop(); });
    }
    void drain(const std::function<void(int)>& f, int n) {
        while (true) {
            const int i = next.fetch_add(1);
            if (i >= n) break;
            f(i);
            done.fetch_add(1);
        }
    }
    void loop() {
        int seen = 0;
        while (true) {
            const std::function<void(int)>* f;
            int n;
            {
                std::unique_lock<std::mutex> lk(mu);
                cv_work.wait(lk, [&]() { return stop || generation != seen; });
                if (stop) return;
                seen = generation;
                f = fn;
                n = n_tasks;
                ++active;
            }
            drain(*f, n);
            {
                std::lock_guard<std::mutex> lk(mu);
                --active;
            }
            cv_done.notify_all();
        }
    }
    // runs f(0..tasks-1) on the workers and the calling thread; returns when every task has finished and no
    // worker is still inside this generation (f may live on the caller's stack)
    void run(int tasks, const std::function<void(int)>& f) {
        if (workers.empty() || tasks <= 1) {
            for (int i = 0; i < tasks; ++i) f(i);
            return;
        }
        {
            std::lock_guard<std::mutex> lk(mu);
            fn = &f;
            n_tasks = tasks;
            next.store(0);
            done.store(0);
            ++generation;
        }
        cv_work.notify_all();
        drain(f, tasks);
        std::unique_lock<std::mutex> lk(mu);
        cv_done.wait(lk, [&]() { return done.load() >= tasks && active == 0; });
        n_tasks = 0;          // a worker that wakes up late for this generation finds nothing to do
    }
    ~HostPool() {
        {
            std::lock_guard<std::mutex> lk(mu);
            stop = true;
        }
        cv_work.notify_all();
        for (auto& t : workers) t.join();
    }
};

struct b2c_decoder {
    std::unique_ptr<HostPool> pool;
    int device = 0;
    cudaStream_t stream = nullptr;
    int V = 0, is_bpe = 0, has_dup_labels = 0;
    std::vector<std::string> labels, clean;
    std::vector<B2cTok> toks;
    b2c_lm* lm = nullptr;
    double alpha = 0.5, beta = 1.5, unk = -10.0;
    int score_boundary = 1;
    // MultiLanguageModel: models 1.. (model 0 is `lm` with the scalars above)
    struct ExtraLm { b2c_lm* lm; double alpha, beta, unk; int score_boundary; };
    std::vector<ExtraLm> lmx;
    int n_sm = 1;
    size_t smem_optin = 48 * 1024;
    DevBuf d_raw, d_lmx, d_stream, d_mstats, d_sumk, d_clk, d_maxk, d_toks, d_logits, d_meta, d_tok_start, d_tok_ids, d_tok_lp, d_rowsum, d_set, d_isprob, d_approx, d_ws, d_hot, d_states,
        d_out_small, d_out_toks, d_out_frames;
    PinBuf h_sumk, h_maxk, h_meta, h_out_small, h_out_toks, h_out_frames, h_mstats;
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaStream_t cls_stream[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};   // one per capacity class
    cudaEvent_t cls_done[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t fork_ev = nullptr;
    cudaEvent_t caller_ev = nullptr;      // b2c_decoder_wait_stream: the caller's stream at the time of the call
    // pipelined calls (host input): chunks along T are copied on copy_stream while earlier chunks are decoded
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t copied[B2C_PIPE_CHUNKS] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t chunk_ev[3 * B2C_PIPE_CHUNKS] = {};
    DevBuf d_state, d_gate;
    cudaStream_t prep_stream = nullptr;   // gated pipelined calls: streaming stage of the later chunks, concurrent with the beam kernel
    cudaEvent_t prep_ev[3] = {nullptr, nullptr, nullptr};    // inputs ready / first chunk streamed / all streamed and decided
    bool pipe_refused = false;            // the last pipelined attempt of this configuration could not be planned
    double last_device_ms = 0.0;          // streaming stage + beam kernel of the previous call (chunk sizing of pipelined calls)
    int plain_v5 = -2, plain_cap = 0;     // kernel variant / capacity class of the last PLAIN call (pipelined calls must plan the same)
    // hinted plain calls: the beam kernel is planned from the hint alone and launched right behind the streaming stage
    // (no wait for this call's token statistics in the middle of the call) when that plan is the one the last
    // statistics-based call of the configuration ran
    bool hinted_refused = false;          // the hint-only plan differed: plan from the statistics until the next refresh
    u32 hinted_calls = 0;                 // every 32nd call of a configuration plans from its statistics again (data may drift)
    std::mutex call_mu;                   // b2c_decode_batch is serialised per handle (scratch buffers are per handle)
    b2c_timings_t tm;
    // adaptive sizing: candidate-count histogram of the previous call with the same configuration
    bool hint_valid = false;
    int hint_beam = 0, hint_lm = 0, hint_hot = 0, hint_prune = 0;
    u32 hint_over[6] = {0, 0, 0, 0, 0, 0};
    u32 hint_frames = 0;
};

struct BeamRes {
    std::string text;
    std::vector<std::string> words;
    std::vector<int32_t> frames;
    double logit = 0, lm = 0;
    B2cLmState st;
    std::vector<B2cLmState> stx;   // MultiLanguageModel: states of models 1..
    std::vector<u32> raw;      // streaming calls: emitted tokens since the input beam, oldest first
    std::string s_first, s_mid, s_last;   // ... and replayed into strings (b2c_packed_t.stream_pieces)
    bool s_boundary = false;
    int aux[4] = {-1, -1, -1, -1};
};
struct b2c_result {
    std::vector<std::vector<BeamRes>> utts;
    bool has_lm = false;
    std::string joined;        // b2c_result_top_texts: top-1 texts, each followed by '\0'
    bool joined_built = false;
    // b2c_result_packed
    bool packed_built = false;
    int n_models = 1;
    std::vector<int32_t> pk_nb, pk_nw, pk_frames;
    std::vector<double> pk_scores;
    std::vector<b2c_lm_state_t> pk_states;
    std::string pk_texts;
    bool streaming = false;
    std::vector<int32_t> pk_aux, pk_ntok, pk_boundary;
    std::vector<u32> pk_toks;
    std::string pk_pieces;
};

// hotword table (language_model.py:152-189): every code-point prefix of every hotword unigram
static void build_hot(const b2c_decode_opts_t* o, std::vector<B2cHot>& tab, int& n_hot, int& min_len_all) {
    std::map<u64, std::pair<u32, u32>> pref;  // key -> (min_len, is_word)
    n_hot = 0;
    min_len_all = 0;
    for (int i = 0; i < o->n_hotwords; ++i) {
        const char* s = o->hotwords[i];
        if (!s) continue;
        const size_t L = std::strlen(s);
        size_t p = 0;
        while (p < L) {
            while (p < L && std::isspace(static_cast<unsigned char>(s[p]))) ++p;
            size_t q = p;
            while (q < L && !std::isspace(static_cast<unsigned char>(s[q]))) ++q;
            if (q > p) {
                ++n_hot;
                const u32 nchars = b2c_utf8_len(s + p, q - p);
                if (min_len_all == 0 || static_cast<int>(nchars) < min_len_all) min_len_all = static_cast<int>(nchars);
                u64 h = 0;
                for (size_t k = p; k < q; ++k) {
                    h = b2c_addmod61(b2c_mulmod61(h, B2C_HASH_BASE), static_cast<u64>(static_cast<unsigned char>(s[k])) + 1);
                    const bool boundary = (k + 1 == q) || ((static_cast<unsigned char>(s[k + 1]) & 0xC0) != 0x80);
                    if (!boundary) continue;
                    auto it = pref.find(h + 1);
                    const u32 is_word = (k + 1 == q) ? 1u : 0u;
                    if (it == pref.end()) pref[h + 1] = {nchars, is_word};
                    else {
                        if (nchars < it->second.first) it->second.first = nchars;
                        it->second.second |= is_word;
                    }
                }
            }
            p = q;
        }
    }
    u64 size = 16;
    while (size < pref.size() * 2 + 2) size <<= 1;
    tab.assign(size, B2cHot{0, 0, 0});
    for (auto& kv : pref) {
        u64 slot = b2c_mix64(kv.first) & (size - 1);
        while (tab[slot].key != 0) slot = (slot + 1) & (size - 1);
        tab[slot] = B2cHot{kv.first, kv.second.first, kv.second.second};
    }
}

// decode() / decode_batch() want the text only: no word vector, no frames
static void assemble_text(const b2c_decoder* d, const u32* toks, int nt, BeamRes& br) {
    br.text.clear();
    br.text.reserve(static_cast<size_t>(nt > 0 ? nt : 0) + 16);      // one allocation (most tokens are one byte)
    br.words.clear();
    br.frames.clear();
    bool open_word = false;      // the current word has at least one character
    bool need_space = false;     // a finished word precedes
    for (int i = nt - 1; i >= 0; --i) {
        const u32 tok = toks[i] & 0xFFFFu, kind = toks[i] >> 16;
        if (kind != B2C_CK_CONT) {       // word boundary: space, or a BPE piece that starts the next word
            if (open_word) need_space = true;
            open_word = false;
            if (kind != B2C_CK_BPE) continue;
        }
        const std::string& piece = kind == B2C_CK_CONT ? d->labels[tok] : d->clean[tok];
        if (piece.empty()) continue;
        if (!open_word && need_space) br.text += ' ';
        br.text += piece;
        open_word = true;
    }
}
static void assemble_beam(const b2c_decoder* d, const u32* toks, int nt, const int* frames, int nw, BeamRes& br) {
    std::string word;
    br.words.clear();
    for (int i = nt - 1; i >= 0; --i) {
        const u32 tok = toks[i] & 0xFFFFu, kind = toks[i] >> 16;
        if (kind == B2C_CK_CONT) {
            word += d->labels[tok];
        } else {
            if (!word.empty()) br.words.push_back(word);
            word = (kind == B2C_CK_BPE) ? d->clean[tok] : std::string();
        }
    }
    if (!word.empty()) br.words.push_back(word);
    br.text.clear();
    for (size_t i = 0; i < br.words.size(); ++i) {
        if (i) br.text += ' ';
        br.text += br.words[i];
    }
    br.frames.resize(static_cast<size_t>(nw) * 2);
    for (int w = 0; w < nw; ++w) {
        br.frames[2 * w] = frames[2 * (nw - 1 - w)];
        br.frames[2 * w + 1] = frames[2 * (nw - 1 - w) + 1];
    }
    // zip(text.split(), text_frames) (decoder.py:661) truncates to the shorter list
    const size_t n = std::min(br.words.size(), static_cast<size_t>(nw));
    br.words.resize(n);
    br.frames.resize(n * 2);
}

struct MetaHost {   // one pinned staging block -> one H2D copy
    std::vector<u64> frame_off;
    std::vector<int> T, order;
};

// streaming pass (every utterance as logits) -> decide (exact only where the approximate mean row sum is near 1) ->
// second pass over the utterances that turned out to be probabilities (returns at once when there is none)
template <class T>
static int launch_prepare(b2c_decoder* d, const B2cPrepArgs& A0, int n_utts, int grid_tile, int grid_tok) {
    B2cPrepArgs A = A0, A1 = A0;
    A.mode = 0;
    A1.mode = 1;
#ifdef B2C_HOSTSIM
    (void)d;
    (void)grid_tile;
    std::unique_ptr<B2cPrepShared> sh(new B2cPrepShared());
    for (int b = 0; b < grid_tok; ++b) b2c_tokens_block<T>(A, b, grid_tok, sh.get());
    std::unique_ptr<B2cDecideShared> dsh(new B2cDecideShared());
    for (int u = 0; u < n_utts; ++u) b2c_decide_block<T>(A, u, dsh.get());
    for (int b = 0; b < grid_tok; ++b) b2c_tokens_block<T>(A1, b, grid_tok, sh.get());
#else
    if (sizeof(T) == 4 && A.V <= 32) b2c_tokens_tile_kernel<<<grid_tile, B2C_TILE_WARPS * 32, 0, d->stream>>>(A);
    else b2c_tokens_kernel<T><<<grid_tok, B2C_PREP_THREADS, 0, d->stream>>>(A);
    b2c_decide_kernel<T><<<n_utts, 128, 0, d->stream>>>(A);
    b2c_tokens_kernel<T><<<grid_tok, B2C_PREP_THREADS, 0, d->stream>>>(A1);
    CUDA_OK(cudaGetLastError());
#endif
    return 0;
}

// v5 >= 0: variant of the latency-first kernel (b2c_beam_fast.h); A.L.smem_bytes is kV5Smem[v5] then
static int launch_beam(b2c_decoder* d, const B2cBeamArgs& A, int slots, bool fast, int per_sm, int threads, cudaStream_t stream,
                       int v5 = -1) {
#ifdef B2C_HOSTSIM
    (void)d;
    (void)stream;
    (void)per_sm;
    (void)threads;
    std::vector<u8> smem(A.L.smem_bytes + 64);
    const bool table = A.P.V <= B2C_FAST_LT;
    for (int s = 0; s < slots; ++s) {
        if (v5 == 0 && table) b2c_beam_block_fast<1024, B2C_FAST_LT>(A, s, smem.data());
        else if (v5 == 0) b2c_beam_block_fast<1024, 0>(A, s, smem.data());
        else if (v5 == 1 && table) b2c_beam_block_fast<512, B2C_FAST_LT>(A, s, smem.data());
        else if (v5 == 1) b2c_beam_block_fast<512, 0>(A, s, smem.data());
        else if (v5 == 2 && table) b2c_beam_block_fast<256, B2C_FAST_LT>(A, s, smem.data());
        else if (v5 == 2) b2c_beam_block_fast<256, 0>(A, s, smem.data());
        else if (fast) b2c_beam_block<true>(A, s, smem.data());
        else b2c_beam_block<false>(A, s, smem.data());
    }
#else
    const int smem = static_cast<int>(A.L.smem_bytes);
#define B2C_LAUNCH_V5(CAP, OCC, LT)                                                                                     \
    do {                                                                                                               \
        CUDA_OK(cudaFuncSetAttribute(b2c_beam_fast_kernel<CAP, OCC, LT>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); \
        b2c_beam_fast_kernel<CAP, OCC, LT><<<slots, B2C_FAST_W, A.L.smem_bytes, stream>>>(A);                         \
    } while (0)
    if (v5 >= 0) {
        const bool table = A.P.V <= B2C_FAST_LT;
        if (v5 == 0 && table) B2C_LAUNCH_V5(1024, 2, B2C_FAST_LT);
        else if (v5 == 0) B2C_LAUNCH_V5(1024, 2, 0);
        else if (v5 == 1 && table) B2C_LAUNCH_V5(512, 3, B2C_FAST_LT);
        else if (v5 == 1) B2C_LAUNCH_V5(512, 3, 0);
        else if (table) B2C_LAUNCH_V5(256, 4, B2C_FAST_LT);
        else B2C_LAUNCH_V5(256, 4, 0);
        CUDA_OK(cudaGetLastError());
        return 0;
    }
#undef B2C_LAUNCH_V5
#define B2C_LAUNCH_BEAM(FAST, THREADS, OCC)                                                                            \
    do {                                                                                                               \
        if (smem > 48 * 1024)                                                                                          \
            CUDA_OK(cudaFuncSetAttribute(b2c_beam_kernel<FAST, THREADS, OCC>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); \
        b2c_beam_kernel<FAST, THREADS, OCC><<<slots, THREADS, A.L.smem_bytes, stream>>>(A);                           \
    } while (0)
    (void)per_sm;
    if (fast && threads == 32) B2C_LAUNCH_BEAM(true, 32, 8);           // 255 registers x 32 threads: 8 one-warp CTAs per SM
    else if (fast && threads == 256) B2C_LAUNCH_BEAM(true, 256, 1);    // 255 registers x 256 threads: the whole register file
    else if (fast && threads == 64) B2C_LAUNCH_BEAM(true, 64, 4);     // 255 registers x 64 threads: 4 CTAs per SM
    else if (fast) B2C_LAUNCH_BEAM(true, 128, 2);                 // 255 registers x 128 threads: 2 CTAs per SM
    else if (threads == 512) B2C_LAUNCH_BEAM(false, 512, 1);      // 128 registers x 512 threads (beam tables in HBM: latency-bound)
    else if (threads == 256) B2C_LAUNCH_BEAM(false, 256, 1);
    else B2C_LAUNCH_BEAM(false, 128, 2);
#undef B2C_LAUNCH_BEAM
    CUDA_OK(cudaGetLastError());
#endif
    return 0;
}


// =========================================================================================
// C ABI
// =========================================================================================
extern "C" {

const char* b2c_last_error(void) { return g_err.c_str(); }
int b2c_version(void) { return B2C_VERSION; }
int b2c_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

// ---- language model -----------------------------------------------------------------------
int b2c_lm_build_from_arpa(const char* arpa_path, const char* const* unigrams, long n_unigrams, b2c_lm_t** out) {
    if (!arpa_path || !out) return fail(B2C_E_ARG, "null argument");
    std::unique_ptr<b2c_lm> lm(new b2c_lm());
    if (!b2c_lm_build(lm->host, arpa_path, unigrams, n_unigrams)) return fail(B2C_E_IO, lm->host.error);
    *out = lm.release();
    return 0;
}
// ARPA text or a KenLM binary (probing model type), told apart by the file's first bytes
int b2c_lm_build_from_file(const char* path, const char* const* unigrams, long n_unigrams, b2c_lm_t** out) {
    if (!path || !out) return fail(B2C_E_ARG, "null argument");
    if (!b2c_is_kenlm_binary(path)) return b2c_lm_build_from_arpa(path, unigrams, n_unigrams, out);
    std::unique_ptr<b2c_lm> lm(new b2c_lm());
    if (!b2c_lm_build_kenlm_binary(lm->host, path, unigrams, n_unigrams)) return fail(B2C_E_IO, lm->host.error);
    *out = lm.release();
    return 0;
}
int b2c_lm_blob(const b2c_lm_t* lm, const void** data, size_t* size) {
    if (!lm || !data || !size) return fail(B2C_E_ARG, "null argument");
    *data = lm->host.blob.data();
    *size = lm->host.blob.size();
    return 0;
}
// every offset, mask and id of a blob is checked before anything dereferences it: blobs come from files and from
// other ranks
static const char* blob_defect(const B2cLmHeader* h, size_t size) {
    if (h->magic != B2C_LM_MAGIC) return "bad magic";
    if (h->total_bytes != size) return "size does not match the header";
    if (h->order < 1 || h->order > B2C_MAX_ORDER) return "n-gram order out of range";
    if (h->n_vocab < 1 || h->bos_id >= h->n_vocab || h->eos_id >= h->n_vocab) return "vocabulary ids out of range";
    auto pow2m1 = [](u64 m) { return m >= 15 && ((m + 1) & m) == 0; };
    if (!pow2m1(h->ngram_mask) || !pow2m1(h->vocab_mask) || !pow2m1(h->prefix_mask)) return "table mask is not 2^k - 1";
    auto inside = [&](u64 off, u64 count, u64 elem) {
        return off >= sizeof(B2cLmHeader) && (off & 7) == 0 && off <= size && count <= (size - off) / elem;
    };
    if (!inside(h->off_uni, h->n_vocab, sizeof(B2cUni))) return "unigram array outside the blob";
    if (!inside(h->off_ngrams, h->ngram_mask + 1, sizeof(B2cNgram))) return "n-gram table outside the blob";
    if (!inside(h->off_vocab, h->vocab_mask + 1, sizeof(B2cVocab))) return "vocabulary table outside the blob";
    if (!inside(h->off_prefix, h->prefix_mask + 1, sizeof(u64))) return "prefix table outside the blob";
    if (h->have_unigrams != 0 && h->have_unigrams != 1) return "bad unigram flag";
    if (h->key_scheme != B2C_KEYS_B2C && h->key_scheme != B2C_KEYS_KENLM) return "unknown key scheme";
    if (h->n_unigrams < 0 || static_cast<u64>(h->n_unigrams) > h->n_vocab) return "bad unigram count";
    return nullptr;
}
int b2c_lm_from_blob(const void* data, size_t size, b2c_lm_t** out) {
    if (!data || !out || size < sizeof(B2cLmHeader)) return fail(B2C_E_ARG, "bad blob");
    B2cLmHeader h;
    std::memcpy(&h, data, sizeof(h));
    if (const char* why = blob_defect(&h, size)) return fail(B2C_E_ARG, std::string("not a valid b200ctc LM blob: ") + why);
    std::unique_ptr<b2c_lm> lm(new b2c_lm());
    lm->host.blob.assign(static_cast<const unsigned char*>(data), static_cast<const unsigned char*>(data) + size);
    // vocabulary ids stored in the table must index the unigram array
    const B2cLmView v = lm->host.view(lm->host.blob.data());
    for (u64 s = 0; s <= v.vocab_mask; ++s)
        if (v.vocab[s].key != 0 && v.vocab[s].id >= v.n_vocab) return fail(B2C_E_ARG, "not a valid b200ctc LM blob: vocabulary id out of range");
    *out = lm.release();
    return 0;
}
int b2c_lm_have_unigrams(const b2c_lm_t* lm) { return lm ? lm->host.header()->have_unigrams : 0; }
int b2c_lm_upload(b2c_lm_t* lm, int device) {
    if (!lm) return fail(B2C_E_ARG, "null lm");
    std::lock_guard<std::mutex> lk(lm->mu);
    if (lm->dev.count(device)) return 0;
    CUDA_OK(cudaSetDevice(device));
    void* p = nullptr;
    CUDA_OK(cudaMalloc(&p, lm->host.blob.size()));
    CUDA_OK(cudaMemcpy(p, lm->host.blob.data(), lm->host.blob.size(), cudaMemcpyHostToDevice));
    lm->dev[device] = p;
    lm->owned[device] = p;
    return 0;
}
int b2c_lm_adopt_device_blob(b2c_lm_t* lm, int device, const void* device_ptr, size_t size) {
    if (!lm || !device_ptr) return fail(B2C_E_ARG, "null argument");
    if (size != lm->host.blob.size()) return fail(B2C_E_ARG, "device blob size mismatch");
    std::lock_guard<std::mutex> lk(lm->mu);
    lm->dev[device] = device_ptr;
    return 0;
}
void b2c_lm_destroy(b2c_lm_t* lm) {
    if (!lm) return;
    for (auto& kv : lm->owned) {
        cudaSetDevice(kv.first);
        cudaFree(kv.second);
    }
    delete lm;
}
int b2c_lm_order(const b2c_lm_t* lm) { return lm ? lm->host.header()->order : 0; }
static B2cLmView host_view(const b2c_lm_t* lm) { return lm->host.view(lm->host.blob.data()); }
int b2c_lm_contains(const b2c_lm_t* lm, const char* word) {
    if (!lm || !word) return 0;
    B2cLmView v = host_view(lm);
    size_t n = std::strlen(word);
    if (n == 0) return 0;
    return b2c_vocab_find(v, b2c_hash_bytes(word, n)) ? 1 : 0;
}
int b2c_lm_in_unigrams(const b2c_lm_t* lm, const char* word) {
    if (!lm || !word) return 0;
    B2cLmView v = host_view(lm);
    size_t n = std::strlen(word);
    if (n == 0) return 0;
    const B2cVocab* e = b2c_vocab_find(v, b2c_hash_bytes(word, n));
    return (e && (e->flags & 1u)) ? 1 : 0;
}
int b2c_lm_has_prefix(const b2c_lm_t* lm, const char* prefix) {
    if (!lm || !prefix) return 0;
    B2cLmView v = host_view(lm);
    size_t n = std::strlen(prefix);
    if (n == 0) return v.n_unigrams > 0 ? 1 : 0;
    return b2c_prefix_contains(v, b2c_hash_bytes(prefix, n)) ? 1 : 0;
}
static void to_internal(const b2c_lm_state_t* s, B2cLmState& o) {
    o.length = s->length;
    for (int i = 0; i < B2C_MAX_HIST; ++i) { o.words[i] = s->words[i]; o.backoff[i] = s->backoff[i]; }
}
static void from_internal(const B2cLmState& s, b2c_lm_state_t* o) {
    o->length = s.length;
    for (int i = 0; i < B2C_MAX_HIST; ++i) {
        o->words[i] = i < static_cast<int>(s.length) ? s.words[i] : 0;
        o->backoff[i] = i < static_cast<int>(s.length) ? s.backoff[i] : 0.0f;
    }
}
void b2c_lm_begin_sentence(const b2c_lm_t* lm, b2c_lm_state_t* st) {
    std::memset(st, 0, sizeof(*st));
    if (!lm) return;
    B2cLmView v = host_view(lm);
    st->length = 1;
    st->words[0] = v.bos_id;
    st->backoff[0] = v.uni[v.bos_id].backoff;
}
void b2c_lm_null_context(const b2c_lm_t*, b2c_lm_state_t* st) { std::memset(st, 0, sizeof(*st)); }
float b2c_lm_base_score(const b2c_lm_t* lm, const b2c_lm_state_t* in, const char* word, b2c_lm_state_t* out) {
    B2cLmView v = host_view(lm);
    B2cLmState a, b;
    to_internal(in, a);
    u32 wid = 0;
    size_t n = std::strlen(word);
    if (n) {
        const B2cVocab* e = b2c_vocab_find(v, b2c_hash_bytes(word, n));
        if (e) wid = e->id;
    }
    std::memset(&b, 0, sizeof(b));
    float r = b2c_lm_base_score(v, a, wid, b);
    from_internal(b, out);
    return r;
}

// ---- decoder ------------------------------------------------------------------------------
static const char* BPE_MARK = "\xE2\x96\x81";

int b2c_decoder_create(const char* const* labels, int n_labels, int is_bpe, b2c_lm_t* lm, int device, b2c_decoder_t** out) {
    if (!labels || n_labels <= 0 || n_labels > 65534 || !out) return fail(B2C_E_ARG, "bad labels");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
        return fail(B2C_E_CUDA, "no CUDA device: libb200ctc has no CPU path");
    if (device < 0 || device >= ndev) return fail(B2C_E_ARG, "bad device index");
    std::unique_ptr<b2c_decoder> d(new b2c_decoder());
    d->device = device;
    d->V = n_labels;
    d->is_bpe = is_bpe ? 1 : 0;
    d->lm = lm;
    std::memset(&d->tm, 0, sizeof(d->tm));
    bool have_blank = false;
    for (int i = 0; i < n_labels; ++i) {
        std::string s = labels[i] ? labels[i] : "";
        if (s.find(' ') != std::string::npos && s != " ")
            return fail(B2C_E_ARG, "labels containing a space inside a longer string are not supported");
        B2cTok t;
        std::memset(&t, 0, sizeof(t));
        std::string clean = s;
        if (s.empty()) { t.flags |= B2C_TF_BLANK; have_blank = true; }
        if (!d->is_bpe && s == " ") t.flags |= B2C_TF_SPACE;
        if (d->is_bpe) {
            if (s.size() >= 3 && s.compare(0, 3, BPE_MARK) == 0) { t.flags |= B2C_TF_BPE_LEAD; clean = clean.substr(3); }
            if (s.size() >= 3 && s.compare(s.size() - 3, 3, BPE_MARK) == 0) {
                t.flags |= B2C_TF_BPE_TRAIL;
                clean = clean.size() >= 3 ? clean.substr(0, clean.size() - 3) : std::string();
            }
        }
        t.raw_hash = b2c_hash_bytes(s.data(), s.size());
        t.raw_pow = b2c_pow_bytes(s.size());
        t.clean_hash = b2c_hash_bytes(clean.data(), clean.size());
        t.raw_nchars = static_cast<u16>(b2c_utf8_len(s.data(), s.size()));
        t.clean_nchars = static_cast<u16>(b2c_utf8_len(clean.data(), clean.size()));
        t.canon = static_cast<u16>(i);
        for (int j = 0; j < i; ++j)
            if (d->labels[j] == s) { t.canon = static_cast<u16>(j); d->has_dup_labels = 1; break; }
        d->labels.push_back(s);
        d->clean.push_back(clean);
        d->toks.push_back(t);
    }
    if (!have_blank) return fail(B2C_E_ARG, "labels must contain the CTC blank \"\" (pass Alphabet.labels)");
    CUDA_OK(cudaSetDevice(device));
    CUDA_OK(cudaStreamCreate(&d->stream));
    for (int i = 0; i < 6; ++i) CUDA_OK(cudaEventCreate(&d->ev[i]));
    for (int i = 0; i < 5; ++i) {
        CUDA_OK(cudaStreamCreate(&d->cls_stream[i]));
        CUDA_OK(cudaEventCreate(&d->cls_done[i]));
    }
    CUDA_OK(cudaEventCreate(&d->fork_ev));
    CUDA_OK(cudaEventCreateWithFlags(&d->caller_ev, cudaEventDisableTiming));
    CUDA_OK(cudaStreamCreate(&d->copy_stream));
    CUDA_OK(cudaStreamCreate(&d->prep_stream));
    for (int i = 0; i < 3; ++i) CUDA_OK(cudaEventCreateWithFlags(&d->prep_ev[i], cudaEventDisableTiming));
    for (int i = 0; i < B2C_PIPE_CHUNKS; ++i) CUDA_OK(cudaEventCreateWithFlags(&d->copied[i], cudaEventDisableTiming));
    for (int i = 0; i < 3 * B2C_PIPE_CHUNKS; ++i) CUDA_OK(cudaEventCreate(&d->chunk_ev[i]));
    int v = 0;
    CUDA_OK(cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device));
    d->n_sm = v;
    CUDA_OK(cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    d->smem_optin = static_cast<size_t>(v);
    if (d->d_toks.ensure(sizeof(B2cTok) * n_labels)) return B2C_E_NOMEM;
    CUDA_OK(cudaMemcpy(d->d_toks.p, d->toks.data(), sizeof(B2cTok) * n_labels, cudaMemcpyHostToDevice));
    if (lm) {
        int rc = b2c_lm_upload(lm, device);
        if (rc) return rc;
    }
    *out = d.release();
    return 0;
}

int b2c_decoder_add_lm(b2c_decoder_t* d, b2c_lm_t* lm) {
    if (!d || !lm) return fail(B2C_E_ARG, "null argument");
    if (!d->lm) return fail(B2C_E_ARG, "the decoder was created without a language model");
    if (d->lmx.size() + 2 > B2C_MAX_LMS) return fail(B2C_E_ARG, "at most 4 language models");
    if (lm->dev.find(d->device) == lm->dev.end()) {
        const int rc = b2c_lm_upload(lm, d->device);
        if (rc) return rc;
    }
    d->lmx.push_back(b2c_decoder::ExtraLm{lm, 0.5, 1.5, -10.0, 1});
    return 0;
}
int b2c_decoder_set_params_lm(b2c_decoder_t* d, int index, double alpha, double beta, double unk, int boundary) {
    if (!d) return fail(B2C_E_ARG, "null decoder");
    if (index == 0) return b2c_decoder_set_params(d, alpha, beta, unk, boundary);
    if (index < 0 || index > static_cast<int>(d->lmx.size())) return fail(B2C_E_ARG, "no such language model");
    b2c_decoder::ExtraLm& x = d->lmx[index - 1];
    x.alpha = alpha;
    x.beta = beta;
    x.unk = unk;
    x.score_boundary = boundary ? 1 : 0;
    return 0;
}
void b2c_decoder_destroy(b2c_decoder_t* d) {
    if (!d) return;
    cudaSetDevice(d->device);
    if (d->stream) cudaStreamSynchronize(d->stream);
    DevBuf* bufs[] = {&d->d_raw, &d->d_lmx, &d->d_stream, &d->d_mstats, &d->d_sumk, &d->d_clk, &d->d_maxk, &d->d_toks, &d->d_logits, &d->d_meta, &d->d_tok_start, &d->d_tok_ids, &d->d_tok_lp, &d->d_rowsum, &d->d_set,
                      &d->d_isprob, &d->d_approx, &d->d_ws, &d->d_hot, &d->d_states, &d->d_out_small, &d->d_out_toks, &d->d_out_frames};
    for (DevBuf* b : bufs) b->release();
    PinBuf* pins[] = {&d->h_sumk, &d->h_maxk, &d->h_meta, &d->h_out_small, &d->h_out_toks, &d->h_out_frames, &d->h_mstats};
    for (PinBuf* b : pins) b->release();
    for (int i = 0; i < 6; ++i) if (d->ev[i]) cudaEventDestroy(d->ev[i]);
    for (int i = 0; i < 5; ++i) {
        if (d->cls_stream[i]) cudaStreamDestroy(d->cls_stream[i]);
        if (d->cls_done[i]) cudaEventDestroy(d->cls_done[i]);
    }
    if (d->fork_ev) cudaEventDestroy(d->fork_ev);
    if (d->caller_ev) cudaEventDestroy(d->caller_ev);
    if (d->copy_stream) cudaStreamDestroy(d->copy_stream);
    if (d->prep_stream) cudaStreamDestroy(d->prep_stream);
    for (int i = 0; i < 3; ++i) if (d->prep_ev[i]) cudaEventDestroy(d->prep_ev[i]);
    d->d_gate.release();
    for (int i = 0; i < B2C_PIPE_CHUNKS; ++i) if (d->copied[i]) cudaEventDestroy(d->copied[i]);
    for (int i = 0; i < 3 * B2C_PIPE_CHUNKS; ++i) if (d->chunk_ev[i]) cudaEventDestroy(d->chunk_ev[i]);
    d->d_state.release();
    if (d->stream) cudaStreamDestroy(d->stream);
    delete d;
}

int b2c_decoder_device(const b2c_decoder_t* d) { return d ? d->device : -1; }

// Device-resident logits produced on another stream (e.g. torch's current stream): everything the decoder enqueues
// from now on waits for what that stream holds at this moment.
int b2c_decoder_wait_stream(b2c_decoder_t* d, void* cuda_stream) {
    if (!d) return fail(B2C_E_ARG, "null decoder");
    std::lock_guard<std::mutex> lk(d->call_mu);
    CUDA_OK(cudaSetDevice(d->device));
    CUDA_OK(cudaEventRecord(d->caller_ev, static_cast<cudaStream_t>(cuda_stream)));
    CUDA_OK(cudaStreamWaitEvent(d->stream, d->caller_ev, 0));
    return 0;
}

int b2c_decoder_set_params(b2c_decoder_t* d, double alpha, double beta, double unk, int boundary) {
    if (!d) return fail(B2C_E_ARG, "null decoder");
    d->alpha = alpha;
    d->beta = beta;
    d->unk = unk;
    d->score_boundary = boundary ? 1 : 0;
    return 0;
}

void b2c_decode_opts_default(b2c_decode_opts_t* o) {
    std::memset(o, 0, sizeof(*o));
    o->beam_width = 100;
    o->beam_prune_logp = -10.0;
    o->token_min_logp = -5.0;
    o->prune_history = 0;
    o->hotword_weight = 10.0;
    o->max_out_beams = 1;
}

static int decode_batch_locked(b2c_decoder_t* d, const void* const* logits, const int32_t* T, int n_utts, int dtype, int is_device,
                               const b2c_decode_opts_t* opts, b2c_result_t** out, bool allow_pipe);

int b2c_decode_batch(b2c_decoder_t* d, const void* const* logits, const int32_t* T, int n_utts, int dtype, int is_device,
                     const b2c_decode_opts_t* opts, b2c_result_t** out) {
    if (!d || !opts || !out || n_utts < 0 || (n_utts > 0 && (!logits || !T))) return fail(B2C_E_ARG, "null argument");
    std::lock_guard<std::mutex> call_lock(d->call_mu);      // one call at a time per handle (any number of threads may call)
    int rc = decode_batch_locked(d, logits, T, n_utts, dtype, is_device, opts, out, true);
    // a pipelined attempt that could not be planned, or that met probability input (decided after the fact): plain call
    if (rc == B2C_E_RETRY_PLAIN) rc = decode_batch_locked(d, logits, T, n_utts, dtype, is_device, opts, out, false);
    return rc;
}

static int decode_batch_locked(b2c_decoder_t* d, const void* const* logits, const int32_t* T, int n_utts, int dtype, int is_device,
                               const b2c_decode_opts_t* opts, b2c_result_t** out, bool allow_pipe) {
    if (dtype < B2C_DTYPE_F32 || dtype > B2C_DTYPE_BF16) return fail(B2C_E_ARG, "dtype must be one of B2C_DTYPE_F32 / F64 / F16 / BF16");
    // half-precision input: copied as 2-byte elements, widened on the device, then the float32 path
    const int dtype_in = dtype;
    const bool half_in = dtype_in == B2C_DTYPE_F16 || dtype_in == B2C_DTYPE_BF16;
    if (half_in) dtype = B2C_DTYPE_F32;
    if (opts->beam_width < 1) return fail(B2C_E_ARG, "beam_width must be >= 1");
    if (opts->beam_width > 65535) return fail(B2C_E_ARG, "beam_width above 65535 is not supported");
    std::unique_ptr<b2c_result> res(new b2c_result());
    res->utts.resize(n_utts);
    res->has_lm = d->lm != nullptr;
    // opt-in host-side section timing (B200CTC_HOST_PROFILE=1, stderr)
    static const bool host_prof = std::getenv("B200CTC_HOST_PROFILE") != nullptr;
    auto hp_t0 = std::chrono::steady_clock::now();
    double hp_ms[6] = {0, 0, 0, 0, 0, 0};
    auto hp_mark = [&](int k) {
        const auto now = std::chrono::steady_clock::now();
        hp_ms[k] += std::chrono::duration<double, std::milli>(now - hp_t0).count();
        hp_t0 = now;
    };
    if (n_utts == 0) { *out = res.release(); return 0; }
    CUDA_OK(cudaSetDevice(d->device));
    const int V = d->V;
    const size_t esz = dtype == B2C_DTYPE_F32 ? 4 : 8;
    const size_t esz_in = half_in ? 2 : esz;         // element size of the caller's matrices
    std::memset(&d->tm, 0, sizeof(d->tm));

    // ---- batch geometry -------------------------------------------------------------------
    std::vector<u64> frame_off(n_utts);
    u64 total_frames = 0;
    int T_max = 0;
    for (int i = 0; i < n_utts; ++i) {
        if (T[i] < 0) return fail(B2C_E_ARG, "negative T");
        if (T[i] > 0 && !logits[i]) return fail(B2C_E_ARG, "null logits pointer");
        frame_off[i] = total_frames;
        total_frames += static_cast<u64>(T[i]);
        T_max = std::max(T_max, static_cast<int>(T[i]));
    }
    std::vector<int> order(n_utts);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return T[a] > T[b]; });
    const int OB = std::max(1, std::min(opts->max_out_beams, opts->beam_width));
    // ---- streaming input (partial_decode_beams): flatten the per-utterance beam / word lists -----------
    if (opts->finalize_mode < B2C_FIN_EOS || opts->finalize_mode > B2C_FIN_KEEP) return fail(B2C_E_ARG, "bad finalize_mode");
    const bool streaming = opts->stream_states != nullptr || opts->finalize_mode != B2C_FIN_EOS;
    std::vector<B2cStreamUtt> s_utts;
    std::vector<B2cStreamBeam> s_beams;
    std::vector<u64> s_wh;
    std::vector<u32> s_wl;
    int s_max_beams = 0;
    u64 s_max_words = 0;
    if (opts->stream_states) {
        s_utts.resize(n_utts);
        for (int i = 0; i < n_utts; ++i) {
            const b2c_stream_state_t& ss = opts->stream_states[i];
            if (ss.n_beams < 0 || ss.n_beams > 65535 || (ss.n_beams > 0 && !ss.beams)) return fail(B2C_E_ARG, "bad stream state");
            B2cStreamUtt su;
            su.beam_off = static_cast<u32>(s_beams.size());
            su.n_beams = static_cast<u32>(ss.n_beams);
            su.t0 = ss.processed_frames;
            su.pad = 0;
            const u32 wbase = static_cast<u32>(s_wh.size());
            u64 words = 0;
            for (int b = 0; b < ss.n_beams; ++b) {
                const b2c_stream_beam_t& ib = ss.beams[b];
                if (static_cast<u64>(ib.word_off) + ib.n_words > static_cast<u64>(std::max(ss.n_words, 0)))
                    return fail(B2C_E_ARG, "stream beam word range outside the state's word list");
                if (ib.last_tok != B2C_NO_TOK && ib.last_tok >= static_cast<u32>(V)) return fail(B2C_E_ARG, "stream beam last_tok out of range");
                B2cStreamBeam sb;
                sb.part_hash = ib.part_hash;
                sb.logit = ib.logit_score;
                sb.word_off = wbase + ib.word_off;
                sb.n_words = ib.n_words;
                sb.part_len = ib.part_len;
                sb.last_tok = ib.last_tok == B2C_NO_TOK ? B2C_NO_TOK : d->toks[ib.last_tok].canon;
                sb.pf_s = ib.pf_s;
                sb.pf_e = ib.pf_e;
                s_beams.push_back(sb);
                words += ib.n_words;
            }
            for (int w = 0; w < ss.n_words; ++w) { s_wh.push_back(ss.word_hashes[w]); s_wl.push_back(ss.word_lens[w]); }
            s_utts[i] = su;
            s_max_beams = std::max(s_max_beams, ss.n_beams);
            s_max_words = std::max(s_max_words, words);
        }
    }
    const int W_tab = std::max(opts->beam_width, s_max_beams);     // capacity of the beam tables

    // ---- parameters -----------------------------------------------------------------------
    B2cParams P;
    std::memset(&P, 0, sizeof(P));
    P.V = V;
    P.is_bpe = d->is_bpe;
    P.has_dup_labels = d->has_dup_labels;
    P.beam_width = opts->beam_width;
    P.prune_history = opts->prune_history ? 1 : 0;
    P.out_beams = OB;
    P.narrow_chain = (opts->text_only != 0 && !streaming) ? 1 : 0;
    P.prune_logp = opts->beam_prune_logp;
    P.token_min_logp = opts->token_min_logp;
    P.alpha = d->alpha; P.beta = d->beta; P.unk_offset = d->unk;
    P.log_base_change = 0x1.26bb1bbb55516p+1;  // 1.0 / math.log10(math.e) (constants.py:18)
    P.score_boundary = d->score_boundary;
    P.hot_weight = opts->hotword_weight;
    P.bucket_scale = b2c_bucket_scale(opts->beam_prune_logp);
    P.toks = d->d_toks.as<B2cTok>();
    if (d->lm) {
        auto it = d->lm->dev.find(d->device);
        if (it == d->lm->dev.end()) return fail(B2C_E_INTERNAL, "language model is not resident on this device");
        P.lm = d->lm->host.view(it->second);
        if (P.lm.order > B2C_MAX_ORDER) return fail(B2C_E_ARG, "n-gram order too large");
        P.n_lm = 1 + static_cast<int>(d->lmx.size());
    }
    int max_order = P.lm.order;     // MultiLanguageModel.order is the maximum (language_model.py:468-470)
    std::vector<B2cLmExtra> lmx_host(d->lmx.size());
    for (size_t j = 0; j < d->lmx.size(); ++j) {
        const b2c_decoder::ExtraLm& x = d->lmx[j];
        auto it = x.lm->dev.find(d->device);
        if (it == x.lm->dev.end()) return fail(B2C_E_INTERNAL, "language model is not resident on this device");
        B2cLmExtra& X = lmx_host[j];
        std::memset(&X, 0, sizeof(X));
        X.lm = x.lm->host.view(it->second);
        if (X.lm.order > B2C_MAX_ORDER) return fail(B2C_E_ARG, "n-gram order too large");
        X.alpha = x.alpha;
        X.beta = x.beta;
        X.unk_offset = x.unk;
        X.score_boundary = x.score_boundary;
        max_order = std::max(max_order, X.lm.order);
    }
    if (!lmx_host.empty()) {
        if (d->d_lmx.ensure(sizeof(B2cLmExtra) * lmx_host.size())) return B2C_E_NOMEM;
        CUDA_OK(cudaMemcpy(d->d_lmx.p, lmx_host.data(), sizeof(B2cLmExtra) * lmx_host.size(), cudaMemcpyHostToDevice));
        P.lmx = d->d_lmx.as<B2cLmExtra>();
    }
    const int n_lm = std::max(1, P.n_lm);
    res->n_models = n_lm;
    res->streaming = streaming;
    P.hist_n = std::max(1, max_order - 1);
    std::vector<B2cHot> hot;
    build_hot(opts, hot, P.n_hot, P.hot_min_len_all);
    if (d->d_hot.ensure(hot.size() * sizeof(B2cHot))) return B2C_E_NOMEM;
    P.hot = d->d_hot.as<B2cHot>();
    P.hot_mask = hot.size() - 1;

    // ---- buffers --------------------------------------------------------------------------
    const u64 n_entries = std::max<u64>(total_frames * static_cast<u64>(V), 1);
    const bool contiguous_dev = [&]() {
        if (!is_device) return false;
        for (int i = 0; i + 1 < n_utts; ++i) {
            if (T[i + 1] == 0) continue;
            const char* expect = static_cast<const char*>(logits[0]) + frame_off[i + 1] * V * esz_in;
            if (static_cast<const char*>(logits[i + 1]) != expect) return false;
        }
        return T[0] > 0 || n_utts == 1;
    }();
    if ((half_in || !contiguous_dev) && d->d_logits.ensure(std::max<u64>(total_frames * V * esz, 16))) return B2C_E_NOMEM;
    if (half_in && !contiguous_dev && d->d_raw.ensure(std::max<u64>(total_frames * V * esz_in, 16))) return B2C_E_NOMEM;
    const size_t meta_bytes = al16(8ull * n_utts) + 3 * al16(4ull * n_utts) + 64 + al16(8ull * (n_utts + 1)) + al16(8ull * n_utts);
    if (d->d_meta.ensure(meta_bytes) || d->h_meta.ensure(meta_bytes)) return B2C_E_NOMEM;
    if (d->d_tok_start.ensure(sizeof(B2cFrameRec) * (total_frames + 1)) || d->d_tok_ids.ensure(4 * n_entries) ||
        d->d_tok_lp.ensure(8 * n_entries) || d->d_rowsum.ensure(std::max<u64>(8 * total_frames, 16)) ||
        d->d_isprob.ensure(4ull * n_utts) || d->d_approx.ensure(16ull * n_utts + 16))
        return B2C_E_NOMEM;
    u32 set_cap = 16;
    while (set_cap < 8u * (static_cast<u32>(V) + 1)) set_cap <<= 1;
    std::vector<u64> run_off(n_utts + 1, 0);
    for (int i = 0; i < n_utts; ++i) run_off[i + 1] = run_off[i] + (static_cast<u64>(T[i]) + B2C_RUN - 1) / B2C_RUN;
    const int runs_per_utt = std::max(1, (T_max + B2C_RUN - 1) / B2C_RUN);
    const u64 total_runs = static_cast<u64>(n_utts) * runs_per_utt;
    const int tiles_per_utt = std::max(1, (T_max + B2C_TILE_ROWS - 1) / B2C_TILE_ROWS);
    const int grid_tile = static_cast<int>(std::max<u64>(1, std::min<u64>((static_cast<u64>(n_utts) * tiles_per_utt + B2C_TILE_WARPS - 1) / B2C_TILE_WARPS, static_cast<u64>(d->n_sm) * 8)));
    const int grid_tok = static_cast<int>(std::max<u64>(1, std::min<u64>((total_runs + B2C_PREP_WARPS - 1) / B2C_PREP_WARPS, static_cast<u64>(d->n_sm) * 8)));
    if (V > 32) {
        if (d->d_set.ensure(2ull * set_cap * 2 * B2C_PREP_WARPS * grid_tok)) return B2C_E_NOMEM;
    }
    if (d->d_maxk.ensure(4ull * n_utts) || d->h_maxk.ensure(4ull * n_utts) || d->d_sumk.ensure(4ull * n_utts) ||
        d->h_sumk.ensure(4ull * n_utts))
        return B2C_E_NOMEM;
    const u32 smem_budget = static_cast<u32>(std::min<size_t>(d->smem_optin, 200 * 1024));
    // outputs
    const u64 off_nb = 0, off_st = al16(4ull * n_utts), off_sc = off_st + al16(4ull * n_utts),
              off_nt = off_sc + al16(16ull * OB * n_utts), off_nw = off_nt + al16(4ull * OB * n_utts),
              off_ls = off_nw + al16(4ull * OB * n_utts), off_ax = off_ls + al16(sizeof(B2cLmState) * static_cast<u64>(OB) * n_utts),
              off_lx = off_ax + (streaming ? al16(16ull * OB * n_utts) : 0),
              small_bytes = off_lx + al16(sizeof(B2cLmState) * static_cast<u64>(OB) * n_utts * static_cast<u64>(n_lm - 1));
    const u64 tok_bytes = 4ull * OB * (total_frames + n_utts), frm_bytes = 2 * tok_bytes;
    if (d->d_out_small.ensure(small_bytes) || d->h_out_small.ensure(small_bytes) || d->d_out_toks.ensure(tok_bytes) ||
        d->h_out_toks.ensure(tok_bytes) || d->d_out_frames.ensure(frm_bytes) || d->h_out_frames.ensure(frm_bytes))
        return B2C_E_NOMEM;
    if (opts->lm_start_states) {
        if (d->d_states.ensure(sizeof(B2cLmState) * static_cast<u64>(n_utts) * n_lm)) return B2C_E_NOMEM;
    }

    // ---- pipelined call? ---------------------------------------------------------------------
    // Host input in one [B, T, V] float32 block, alphabet of the lane-per-row streaming kernel, every utterance
    // resident in the latency-first beam kernel (known from the previous call of the same configuration): the batch
    // is cut into chunks along T; chunk c+1 crosses PCIe while chunk c goes through the streaming stage and the beam
    // kernel (chunked launches, state parked in HBM in between).  The launch plan cannot wait for this call's token
    // statistics then: it is made from the hint alone.  Probabilities-vs-logits is decided after the last chunk; a
    // call that turns out to hold probabilities is redone as a plain call (B2C_E_RETRY_PLAIN).
    const bool hint_ok = d->hint_valid && d->hint_beam == opts->beam_width && d->hint_lm == (P.lm.order > 0 ? 1 : 0) &&
                         d->hint_hot == (P.n_hot > 0 ? 1 : 0) && d->hint_prune == P.prune_history && d->hint_frames > 0;
    const bool no_pipe = std::getenv("B200CTC_NO_PIPELINE") != nullptr;
    bool pipe_candidate = allow_pipe && !no_pipe && !is_device && !half_in && T_max >= 8 * B2C_TILE_ROWS &&
                          !streaming && n_lm == 1 && opts->beam_width <= 128 && hint_ok && !d->pipe_refused;
    for (int i = 0; i < n_utts && pipe_candidate; ++i)
        pipe_candidate = T[i] == T_max && static_cast<const char*>(logits[i]) == static_cast<const char*>(logits[0]) + static_cast<u64>(i) * T_max * V * esz_in;
    if (!hint_ok) d->pipe_refused = false;                       // another configuration: a new attempt may be planned
    if (!hint_ok) { d->hinted_refused = false; d->hinted_calls = 0; }
    static const bool no_hinted = std::getenv("B200CTC_NO_HINTED") != nullptr;
    if (pipe_candidate && d->d_logits.ensure(std::max<u64>(total_frames * V * esz, 16))) return B2C_E_NOMEM;
    const int chunk_len = ((T_max + B2C_PIPE_CHUNKS * B2C_TILE_ROWS - 1) / (B2C_PIPE_CHUNKS * B2C_TILE_ROWS)) * B2C_TILE_ROWS;

    // ---- host -> device -------------------------------------------------------------------
    cudaStream_t st = d->stream;
    CUDA_OK(cudaEventRecord(d->ev[0], st));
    u8* hm = d->h_meta.as<u8>();
    u64* h_fo = reinterpret_cast<u64*>(hm);
    int* h_T = reinterpret_cast<int*>(hm + al16(8ull * n_utts));
    const size_t off_run = al16(8ull * n_utts) + al16(4ull * n_utts);
    const size_t off_ord = off_run + al16(8ull * (n_utts + 1));
    const size_t off_next = off_ord + 2 * al16(4ull * n_utts);
    const size_t off_ptr = off_next + 64;                        // [n_utts] source pointers (gather launch only)
    u64* h_run = reinterpret_cast<u64*>(hm + off_run);
    for (int i = 0; i <= n_utts; ++i) h_run[i] = run_off[i];
    int* h_ord = reinterpret_cast<int*>(hm + off_ord);           // [2 * n_utts]: class lists, then retry list
    u32* h_next = reinterpret_cast<u32*>(hm + off_next);         // [16] one queue head per launch
    for (int i = 0; i < n_utts; ++i) { h_fo[i] = frame_off[i]; h_T[i] = T[i]; }
    CUDA_OK(cudaMemcpyAsync(d->d_meta.p, hm, off_ord, cudaMemcpyHostToDevice, st));
    u8* dm = d->d_meta.as<u8>();
    const u64* d_fo = reinterpret_cast<const u64*>(dm);
    const int* d_T = reinterpret_cast<const int*>(dm + al16(8ull * n_utts));
    int* d_ord = reinterpret_cast<int*>(dm + off_ord);
    u32* d_next = reinterpret_cast<u32*>(dm + off_next);
    d->tm.h2d_bytes += static_cast<long long>(meta_bytes);
    const void* d_logits = nullptr;
    if (pipe_candidate) {
        d_logits = d->d_logits.p;                    // copied chunk by chunk further down
    } else if (contiguous_dev && !half_in) {
        d_logits = logits[0];
#ifndef B2C_HOSTSIM
    } else if (is_device && n_utts > 4 && !half_in) {
        d_logits = d->d_logits.p;
        const void** h_ptr = reinterpret_cast<const void**>(hm + off_ptr);
        for (int i = 0; i < n_utts; ++i) h_ptr[i] = logits[i];
        CUDA_OK(cudaMemcpyAsync(dm + off_ptr, h_ptr, 8ull * n_utts, cudaMemcpyHostToDevice, st));
        const int chunks = std::max(1, std::min(64, (d->n_sm * 8 + n_utts - 1) / n_utts));
        b2c_gather_kernel<<<n_utts * chunks, 256, 0, st>>>(reinterpret_cast<const void* const*>(dm + off_ptr), d_fo, d_T,
                                                         static_cast<u64>(V) * (esz / 4), d->d_logits.as<u32>(), n_utts, chunks);
        CUDA_OK(cudaGetLastError());
        d->tm.launches += 1;
#endif
    } else {
        d_logits = d->d_logits.p;
        const void* packed_half = contiguous_dev ? logits[0] : d->d_raw.p;      // half input only
        char* dst = half_in ? d->d_raw.as<char>() : d->d_logits.as<char>();
        // coalesce runs of utterances that are adjacent in the source into one copy
        int i = 0;
        while (i < n_utts && !(half_in && contiguous_dev)) {
            if (T[i] == 0) { ++i; continue; }
            int j = i;
            u64 bytes = static_cast<u64>(T[i]) * V * esz_in;
            while (j + 1 < n_utts && T[j + 1] > 0 &&
                   static_cast<const char*>(logits[j + 1]) == static_cast<const char*>(logits[i]) + bytes) {
                ++j;
                bytes += static_cast<u64>(T[j]) * V * esz_in;
            }
            CUDA_OK(cudaMemcpyAsync(dst + frame_off[i] * V * esz_in, logits[i], bytes,
                                    is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
            if (!is_device) d->tm.h2d_bytes += static_cast<long long>(bytes);
            i = j + 1;
        }
        if (half_in && total_frames > 0) {
            const u64 n_el = total_frames * static_cast<u64>(V);
#ifndef B2C_HOSTSIM
            const int blocks = static_cast<int>(std::min<u64>((n_el + 255) / 256, static_cast<u64>(d->n_sm) * 16));
            b2c_widen_kernel<<<blocks, 256, 0, st>>>(static_cast<const u16*>(packed_half), d->d_logits.as<float>(), n_el,
                                                     dtype_in == B2C_DTYPE_BF16 ? 1 : 0);
            CUDA_OK(cudaGetLastError());
#else
            b2c_widen_range(static_cast<const u16*>(packed_half), d->d_logits.as<float>(), 0, n_el, 1, dtype_in == B2C_DTYPE_BF16 ? 1 : 0);
#endif
            d->tm.launches += 1;
        }
    }
    CUDA_OK(cudaMemcpyAsync(d->d_hot.p, hot.data(), hot.size() * sizeof(B2cHot), cudaMemcpyHostToDevice, st));
    const B2cLmState* d_start = nullptr;
    std::vector<B2cLmState> start_host;
    if (opts->lm_start_states) {
        // with a MultiLanguageModel: n_lm consecutive states per utterance (MultiLanguageModelState.states)
        start_host.resize(static_cast<size_t>(n_utts) * n_lm);
        for (size_t i = 0; i < start_host.size(); ++i) to_internal(opts->lm_start_states + i, start_host[i]);
        CUDA_OK(cudaMemcpyAsync(d->d_states.p, start_host.data(), sizeof(B2cLmState) * start_host.size(), cudaMemcpyHostToDevice, st));
        d_start = d->d_states.as<B2cLmState>();
    }

    const B2cStreamUtt* d_sutt = nullptr;
    const B2cStreamBeam* d_sbeam = nullptr;
    const u64* d_swh = nullptr;
    const u32* d_swl = nullptr;
    if (!s_utts.empty()) {
        const size_t b0 = al16(sizeof(B2cStreamUtt) * s_utts.size()), b1 = al16(sizeof(B2cStreamBeam) * std::max<size_t>(s_beams.size(), 1)),
                     b2 = al16(8 * std::max<size_t>(s_wh.size(), 1)), b3 = al16(4 * std::max<size_t>(s_wl.size(), 1));
        if (d->d_stream.ensure(b0 + b1 + b2 + b3)) return B2C_E_NOMEM;
        u8* base = d->d_stream.as<u8>();
        CUDA_OK(cudaMemcpyAsync(base, s_utts.data(), sizeof(B2cStreamUtt) * s_utts.size(), cudaMemcpyHostToDevice, st));
        if (!s_beams.empty()) CUDA_OK(cudaMemcpyAsync(base + b0, s_beams.data(), sizeof(B2cStreamBeam) * s_beams.size(), cudaMemcpyHostToDevice, st));
        if (!s_wh.empty()) {
            CUDA_OK(cudaMemcpyAsync(base + b0 + b1, s_wh.data(), 8 * s_wh.size(), cudaMemcpyHostToDevice, st));
            CUDA_OK(cudaMemcpyAsync(base + b0 + b1 + b2, s_wl.data(), 4 * s_wl.size(), cudaMemcpyHostToDevice, st));
        }
        d_sutt = reinterpret_cast<const B2cStreamUtt*>(base);
        d_sbeam = reinterpret_cast<const B2cStreamBeam*>(base + b0);
        d_swh = reinterpret_cast<const u64*>(base + b0 + b1);
        d_swl = reinterpret_cast<const u32*>(base + b0 + b1 + b2);
        d->tm.h2d_bytes += static_cast<long long>(b0 + b1 + b2 + b3);
    }

    // ---- prepare kernel ---------------------------------------------------------------------
    B2cPrepArgs PA;
    std::memset(&PA, 0, sizeof(PA));
    PA.logits = d_logits;
    PA.frame_off = d_fo;
    PA.T = d_T;
    PA.V = V;
    PA.token_min_logp = opts->token_min_logp;
    PA.run_off = reinterpret_cast<const u64*>(dm + off_run);
    PA.n_utts = n_utts;
    PA.total_frames = total_frames;
    PA.tok_rec = d->d_tok_start.as<B2cFrameRec>();
    PA.tok_ids = d->d_tok_ids.as<u32>();
    PA.tok_lp = d->d_tok_lp.as<double>();
    PA.rowsum = d->d_rowsum.p;
    PA.set_scratch = d->d_set.as<u16>();
    PA.set_cap = set_cap;
    PA.is_prob = d->d_isprob.as<int>();
    PA.tile_lo = 0;
    PA.tile_hi = tiles_per_utt;
    PA.run_lo = 0;
    PA.run_hi = runs_per_utt;
    PA.approx = d->d_approx.as<double>();
    CUDA_OK(cudaMemsetAsync(d->d_approx.p, 0, 16ull * n_utts + 16, st));
    PA.max_k = d->d_maxk.as<u32>();
    PA.sum_k = d->d_sumk.as<u32>();
    CUDA_OK(cudaMemsetAsync(d->d_maxk.p, 0, 4ull * n_utts, st));
    CUDA_OK(cudaMemsetAsync(d->d_sumk.p, 0, 4ull * n_utts, st));
    int rc = 0;
    bool hinted = false;
    if (!pipe_candidate) {
        CUDA_OK(cudaEventRecord(d->ev[1], st));
        rc = dtype == B2C_DTYPE_F32 ? launch_prepare<float>(d, PA, n_utts, grid_tile, grid_tok)
                                    : launch_prepare<double>(d, PA, n_utts, grid_tile, grid_tok);
        if (rc) return rc;
        CUDA_OK(cudaEventRecord(d->ev[2], st));
        d->tm.launches += 3;

        // ---- size the beam kernel from the token statistics of this batch ---------------------------
        CUDA_OK(cudaMemcpyAsync(d->h_maxk.p, d->d_maxk.p, 4ull * n_utts, cudaMemcpyDeviceToHost, st));
        CUDA_OK(cudaMemcpyAsync(d->h_sumk.p, d->d_sumk.p, 4ull * n_utts, cudaMemcpyDeviceToHost, st));
        hp_mark(0);                                   // argument checks, buffers, enqueue of H2D + prepare kernels
        // hinted plain call: plan now, from the hint alone, and launch the beam kernel right behind the streaming stage;
        // if the plan is not the one the last statistics-based call ran, wait for the statistics after all (below)
        hinted = allow_pipe && !no_hinted && hint_ok && !streaming && n_lm == 1 && opts->beam_width <= 128 && d->plain_v5 >= 0 &&
                 (d->hinted_calls++ % 32u) != 31u && !d->hinted_refused;
        if ((d->hinted_calls % 32u) == 0u) d->hinted_refused = false;       // the refresh call ran: try the hint again
        if (!hinted) {
            CUDA_OK(cudaStreamSynchronize(st));
            hp_mark(1);                               // wait: H2D + prepare kernels
        }
    }
    // without this call's statistics (pipelined and hinted calls): the worst case (V tokens in a frame) sizes the
    // workspace; the capacity class comes from the hint (one token per frame "on average" keeps the statistics-based
    // bound out of its way)
    std::vector<u32> nostat_maxk, nostat_sumk;
    if (pipe_candidate || hinted) {
        nostat_maxk.assign(n_utts, static_cast<u32>(V));
        nostat_sumk.resize(n_utts);
        for (int i = 0; i < n_utts; ++i) nostat_sumk[i] = static_cast<u32>(T[i]);
    }
    const u32* h_maxk = nullptr;
    const u32* h_sumk = nullptr;
    // ---- capacity class of the shared-memory candidate tier (ONE fast class per call) -------------
    // upper bound: sized for the TYPICAL frame of an utterance if all beam_width beams were alive
    // (2.5 x its mean tokens per frame, at least 4); with a hint from the previous call of the same
    // configuration (histogram of the per-frame candidate counts actually seen -- with an LM far fewer
    // beams stay alive): the smallest class that covers all but 0.4% of the frames.  The few wider
    // frames take the out-of-line HBM-tier step inside the same kernel, so every choice is exact.
    // Small classes run 64-thread CTAs (255 registers x 64 threads: 4 CTAs per SM), the others 128.
    static const int kNumCaps = 6;
    static const u32 kCaps[kNumCaps] = {128, 256, 512, 1024, 2048, 4096};
    // big classes leave room for one CTA per SM only: give that CTA 256 threads (a diffuse frame has ~650 candidates)
    auto threads_of = [&](int c) { return kCaps[c] <= 128 ? 32 : (kCaps[c] <= 256 ? 64 : (kCaps[c] >= 2048 ? 256 : 128)); };
    auto layout_of = [&](int c, int tmax, bool full, u64 worst_m) {
        // the 2048 / 4096-candidate classes own an SM anyway: they rank over the wide bucket array
        return make_layout(opts->beam_width, V, tmax, full, smem_budget, kCaps[c], worst_m, threads_of(c) / 32, 0, 0, 1,
                           kCaps[c] >= 2048 ? B2C_NBUCKET_WIDE : B2C_NBUCKET);
    };
    auto per_sm_of = [&](u32 smem_bytes, int threads) {
        const int by_smem = static_cast<int>(std::max<u64>(1, (224 * 1024) / std::max<u32>(smem_bytes + 1024, 2048)));
        return std::min(by_smem, threads == 32 ? 8 : (threads == 64 ? 4 : (threads >= 256 ? 1 : 2)));
    };
    bool cap_ok[kNumCaps];
    for (int c = 0; c < kNumCaps; ++c) cap_ok[c] = layout_of(c, 1, false, 0).smem_bytes <= smem_budget;
    std::vector<std::vector<int>> classes;                 // fast classes (one used per call), last = general
    bool use_v5 = false;
    int v5_top = -1, v5_variant = 0;
    auto classify = [&]() {
        classes.assign(kNumCaps + 1, std::vector<int>());
        use_v5 = false;
        v5_top = -1; v5_variant = 0;
        std::vector<int> cls_of(n_utts, kNumCaps);
        int top = -1, n_fast = 0;
        for (int u = 0; u < n_utts; ++u) {
            const double mean_k = T[u] > 0 ? static_cast<double>(h_sumk[u]) / T[u] : 1.0;
            const u32 typ_k = std::min<u32>(std::max<u32>(h_maxk[u], 1u), std::max<u32>(4u, static_cast<u32>(std::ceil(2.5 * mean_k))));
            const u64 need = std::min<u64>(static_cast<u64>(opts->beam_width) * typ_k,
                                           static_cast<u64>(opts->beam_width) * static_cast<u64>(V));
            for (int c = 0; c < kNumCaps && !streaming && n_lm == 1; ++c)      // streaming / multi-LM calls take the general kernel
                if (cap_ok[c] && need <= kCaps[c]) { cls_of[u] = c; break; }
            if (cls_of[u] < kNumCaps) { top = std::max(top, cls_of[u]); ++n_fast; }
        }
        if (top >= 0 && hint_ok) {
            int c_hint = kNumCaps - 1;
            for (int c = 0; c < kNumCaps; ++c)
                if (static_cast<double>(d->hint_over[c]) <= 0.004 * d->hint_frames) { c_hint = c; break; }
            while (c_hint < top && !cap_ok[c_hint]) ++c_hint;
            top = std::min(top, c_hint);
        }
        v5_top = top;                            // the class the statistics ask for, before the residency upgrade
        // upgrade while every fast utterance stays resident (fewer frames need the out-of-line step)
        while (top >= 0 && top + 1 < kNumCaps && cap_ok[top + 1]) {
            const u32 sb = layout_of(top + 1, 1, false, 0).smem_bytes;
            if (static_cast<long long>(d->n_sm) * per_sm_of(sb, threads_of(top + 1)) < n_fast) break;
            ++top;
        }
        // beam_width <= 128 and a typical frame within 1024 candidates: the latency-first kernel (v5) takes
        // the whole fast list; wider frames inside it go through its out-of-line HBM-tier step
        const bool force_v5 = std::getenv("B200CTC_FORCE_V5") != nullptr;      // tests: exercise the out-of-line step
        use_v5 = top >= 0 && opts->beam_width <= 128 && (force_v5 || kCaps[v5_top >= 0 ? v5_top : top] <= 1024) &&
                 kV5Smem[0][1] + 1024 <= d->smem_optin && std::getenv("B200CTC_NO_V5") == nullptr;
        // more utterances than variant A keeps resident: trade capacity for residency if the previous call's
        // histogram says that all but 0.4% of the frames fit (hint_over[q] = frames with > 128 << q candidates)
        if (use_v5 && hint_ok && n_fast > d->n_sm * kV5Occ[0] && std::getenv("B200CTC_V5_VARIANT") == nullptr) {
            for (int v = 2; v >= 1; --v) {
                const int q = kV5Cap[v] == 256 ? 1 : 2;
                if (static_cast<double>(d->hint_over[q]) <= 0.004 * d->hint_frames) { v5_variant = v; break; }
            }
        }
        if (const char* e = std::getenv("B200CTC_V5_VARIANT")) v5_variant = std::max(0, std::min(2, std::atoi(e)));
        for (int q = 0; q < n_utts; ++q) {
            const int u = order[q];             // keeps longest-first order inside every class
            classes[cls_of[u] < kNumCaps ? top : kNumCaps].push_back(u);
        }
    };
    B2cBeamArgs BA;
    std::memset(&BA, 0, sizeof(BA));
    BA.P = P;
    BA.frame_off = d_fo;
    BA.T = d_T;
    BA.tok_rec = PA.tok_rec;
    BA.tok_ids = PA.tok_ids;
    BA.tok_lp = PA.tok_lp;
    BA.start_states = d_start;
    BA.s_utts = d_sutt;
    BA.s_beams = d_sbeam;
    BA.s_word_hash = d_swh;
    BA.s_word_len = d_swl;
    BA.fin_mode = opts->finalize_mode;
    u8* ds = d->d_out_small.as<u8>();
    BA.out_nbeams = reinterpret_cast<int*>(ds + off_nb);
    BA.out_status = reinterpret_cast<int*>(ds + off_st);
    BA.out_scores = reinterpret_cast<double*>(ds + off_sc);
    BA.out_ntok = reinterpret_cast<int*>(ds + off_nt);
    BA.out_nwords = reinterpret_cast<int*>(ds + off_nw);
    BA.out_states = reinterpret_cast<B2cLmState*>(ds + off_ls);
    BA.out_aux = streaming ? reinterpret_cast<int*>(ds + off_ax) : nullptr;
    BA.out_states_x = n_lm > 1 ? reinterpret_cast<B2cLmState*>(ds + off_lx) : nullptr;
    BA.out_toks = d->d_out_toks.as<u32>();
    BA.out_frames = d->d_out_frames.as<int>();
    if (d->d_mstats.ensure(64)) return B2C_E_NOMEM;
    CUDA_OK(cudaMemsetAsync(d->d_mstats.p, 0, 64, st));
    BA.m_stats = d->d_mstats.as<u32>();
#if defined(B2C_PHASE_CLOCKS)
    if (d->d_clk.ensure(32 * 8)) return B2C_E_NOMEM;
    CUDA_OK(cudaMemsetAsync(d->d_clk.p, 0, 32 * 8, st));
    BA.phase_clk = d->d_clk.as<u64>();
#endif

    struct Launch { int cls; size_t ord_off; int count; B2cLayout L; int slots; int per_sm; int threads; int v5; };
    auto plan = [&](const std::vector<int>& utts, int cls, bool full, size_t ord_off) {
        Launch ln;
        ln.cls = cls;
        ln.ord_off = ord_off;
        ln.count = static_cast<int>(utts.size());
        int tmax = 1;
        u32 kmax = 1;
        for (int u : utts) {
            tmax = std::max(tmax, static_cast<int>(T[u]));
            kmax = std::max(kmax, h_maxk[u]);
        }
        const u64 worst_m = static_cast<u64>(W_tab) * std::min<u32>(kmax, static_cast<u32>(V));
        ln.v5 = (use_v5 && cls < kNumCaps) ? v5_variant : -1;
        if (ln.v5 >= 0) {
            // beam tables of capacity B2C_FAST_W; the HBM tier always exists (frames with more tokens than the rings hold use it too)
            const u32 cap5 = kV5Cap[ln.v5];
            ln.threads = B2C_FAST_W;
            // backtrack arena: fixed node ids of the frame steps below B2C_FAST_W * T, the out-of-line step allocates above
            ln.L = make_layout(B2C_FAST_W, V, tmax, full, smem_budget, cap5, std::max<u64>(worst_m, cap5 + 1), B2C_FAST_NW,
                               static_cast<u64>(B2C_FAST_W) * static_cast<u64>(std::max(tmax, 1)));
            ln.L.smem_bytes = static_cast<u32>(kV5Smem[ln.v5][V <= B2C_FAST_LT ? 1 : 0]);
            ln.per_sm = kV5Occ[ln.v5];
        } else {
        ln.threads = cls < kNumCaps ? threads_of(cls) : 128;
        if (cls < kNumCaps) {
            ln.L = layout_of(cls, tmax, full, worst_m);
        } else {
            // general kernel: the largest shared-memory candidate tier that fits (frames beyond it work on the HBM tier at
            // L2 latency) -- unless the launch has more utterances than SMs and the small tier keeps two CTAs per SM
            auto general = [&](u32 cap_max) {
                return make_layout(W_tab, V, tmax, full, smem_budget, 0, worst_m, B2C_MAXWARPS, static_cast<u64>(s_max_beams),
                                   s_max_words + static_cast<u64>(s_max_beams), n_lm, B2C_NBUCKET_WIDE, cap_max);
            };
            ln.L = general(2048);
            if (per_sm_of(ln.L.smem_bytes, 128) == 1 && ln.count > d->n_sm) {
                const B2cLayout small = general(512);
                if (per_sm_of(small.smem_bytes, 128) >= 2) ln.L = small;
            }
        }
        // the general kernel with room for one CTA per SM only (wide beams): that CTA gets the whole register file --
        // its phases are loops over hundreds to thousands of candidates, each a chain of dependent memory accesses
        if (cls == kNumCaps && per_sm_of(ln.L.smem_bytes, 128) == 1) ln.threads = 256;
        // beam tables that do not fit shared memory (beam_width in the thousands) live in HBM: every phase is a chain of L2
        // round trips, and twice the threads at half the registers hide more of them (measured at beam 2000 on the C2
        // shape: 56 -> 49 ms; with the tables in shared memory, beam 500, the spills cost more than they hide: 19 -> 22 ms)
        if (cls == kNumCaps && ln.threads == 256 && !ln.L.beams_in_smem) ln.threads = 512;
        ln.per_sm = per_sm_of(ln.L.smem_bytes, ln.threads);
        }
        ln.slots = std::min(ln.count, d->n_sm * ln.per_sm);
        const u64 budget = 16ull << 30;            // keep the HBM workspace bounded
        if (static_cast<u64>(ln.slots) * ln.L.gws_bytes > budget)
            ln.slots = static_cast<int>(std::max<u64>(1, budget / ln.L.gws_bytes));
        return ln;
    };
    std::vector<Launch> launches;
    size_t ord_used = 0;
    auto plan_launches = [&](bool with_stats) {
        h_maxk = with_stats ? d->h_maxk.as<u32>() : nostat_maxk.data();
        h_sumk = with_stats ? d->h_sumk.as<u32>() : nostat_sumk.data();
        classify();
        launches.clear();
        ord_used = 0;
        for (int c = 0; c <= kNumCaps; ++c) {
            if (classes[c].empty()) continue;
            launches.push_back(plan(classes[c], c, false, ord_used));
            for (int u : classes[c]) h_ord[ord_used++] = u;
        }
    };
    plan_launches(!(pipe_candidate || hinted));
    if (hinted && !(launches.size() == 1 && launches[0].v5 == d->plain_v5 && static_cast<int>(launches[0].L.cap_s) == d->plain_cap &&
                    launches[0].slots == std::min(launches[0].count, d->n_sm * launches[0].per_sm))) {
        // not the plan the last statistics-based call ran -- or the worst-case workspace of a plan without statistics (V tokens
        // in a frame: large alphabets) would cost resident CTAs: wait for this call's statistics and plan from them
        hinted = false;
        d->hinted_refused = true;
        CUDA_OK(cudaStreamSynchronize(st));
        hp_mark(1);
        plan_launches(true);
    }
    d->tm.hinted = hinted ? 1 : 0;
    for (size_t i = 0; i < 16; ++i) h_next[i] = 0;
    CUDA_OK(cudaMemcpyAsync(d_ord, h_ord, 4 * ord_used, cudaMemcpyHostToDevice, st));
    CUDA_OK(cudaMemcpyAsync(d_next, h_next, 64, cudaMemcpyHostToDevice, st));
    // the classes run CONCURRENTLY (one stream each, forked from / joined to the decoder's stream):
    // each launch's makespan is about one utterance's latency, serialising them would multiply it
    u64 ws_need = 0;
    std::vector<u64> ws_off;
    for (const Launch& ln : launches) {
        if (ln.L.smem_bytes > d->smem_optin) return fail(B2C_E_ARG, "beam_width too large for the shared-memory selection arrays");
        ws_off.push_back(ws_need);
        ws_need += static_cast<u64>(ln.slots) * ln.L.gws_bytes;
    }
    if (d->d_ws.ensure(ws_need)) return B2C_E_NOMEM;
    // chunked launches need ONE launch of the latency-first kernel with every utterance resident
    const bool can_chunk = launches.size() == 1 && launches[0].v5 >= 0 && launches[0].count <= launches[0].slots && !streaming;
    if (pipe_candidate && !can_chunk) {
        d->pipe_refused = true;                       // until the configuration (hint) changes
        return B2C_E_RETRY_PLAIN;
    }
    static const int force_chunks = std::getenv("B200CTC_FORCE_CHUNKS") ? std::atoi(std::getenv("B200CTC_FORCE_CHUNKS")) : 0;   // tests
    // Chunk boundaries.  A chunked launch ends when its SLOWEST utterance has finished the chunk, so every boundary
    // costs the spread of the per-chunk times (measured: 4 equal chunks at C2 take 4.8 ms of beam kernel instead of
    // 3.75).  Compute-bound calls (the copy is shorter than the decode) therefore use TWO chunks: a short first one whose
    // decode covers the copy of the rest; copy-bound calls (large alphabets) use equal chunks.
    std::vector<int> bounds{0, std::max(T_max, 0)};
    // GATED launch (preferred for pipelined calls): ONE beam launch that starts after the first chunk and waits, on the
    // device, for the flag of each later chunk -- no launch boundary, so no chunk pays for its slowest utterance.  The
    // streaming stage of the later chunks runs CONCURRENTLY with the beam kernel on another stream, which needs free SM
    // resources: only taken when the beam kernel leaves at least n_sm/8 CTA slots empty; a CTA that waits longer than
    // ~40 ms gives up with B2C_ERR_GATE and the call is redone as a plain call.
    // Which form of pipelining (measured on B200, profiles/pipeline_r02.txt):
    //   compute-bound calls (copy < 0.6 x decode; C2: copy 0.6 ms, decode 3.9 ms) -> the gated launch: 5.05 -> 4.42 ms of
    //     device time; chunked launches gain nothing there -- a chunked launch ends when its slowest utterance has finished
    //     the chunk, so every boundary costs the spread of the per-chunk times;
    //   copy-bound calls (C4 shape: copy 20 ms, decode 7 ms) -> chunked launches, equal chunks: 25.9 -> 20.8 ms (the gated
    //     form is slower there, 22.8 ms: the streaming stage of a 1 GB batch crawls on the SM slots the beam kernel leaves free).
    // The plan of a pipelined call comes from the hint alone; it must be the plan the previous plain call of this
    // configuration ran (another kernel variant would change the speed, not the result: diffuse batches decode 35 % slower
    // on the latency-first kernel the hint-only plan picks than on the capacity-class kernel their statistics pick).
    const double copy_ms_est = static_cast<double>(total_frames) * V * esz / 50.0e6;            // ~50 GB/s pinned H2D
    const double pipe_r = copy_ms_est / std::max(d->last_device_ms > 0 ? d->last_device_ms : copy_ms_est, 1e-3);
    const bool pipe_all = std::getenv("B200CTC_PIPELINE_ALL") != nullptr;
    const bool gated = pipe_candidate && can_chunk && std::getenv("B200CTC_NO_GATE") == nullptr && (pipe_r < 0.6 || pipe_all) &&
                       launches[0].count + d->n_sm / 8 <= d->n_sm * launches[0].per_sm;
    if (pipe_candidate) {
        const double r = pipe_r;
        const bool same_plan = launches[0].v5 == d->plain_v5 && static_cast<int>(launches[0].L.cap_s) == d->plain_cap;
        if ((!gated && r < 0.6 && !pipe_all) || (!same_plan && !pipe_all)) {
            d->pipe_refused = true;
            return B2C_E_RETRY_PLAIN;
        }
        bounds.clear();
        bounds.push_back(0);
        if (!gated && r < 0.6) {
            int f = static_cast<int>(1.15 * T_max * r / (1.0 + r));
            f = std::max(2 * B2C_TILE_ROWS, ((f + B2C_TILE_ROWS - 1) / B2C_TILE_ROWS) * B2C_TILE_ROWS);
            if (f < T_max) bounds.push_back(f);
        } else {
            for (int c = 1; c < B2C_PIPE_CHUNKS; ++c) if (c * chunk_len < T_max) bounds.push_back(c * chunk_len);
        }
        bounds.push_back(T_max);
    } else if (can_chunk && force_chunks > 1 && T_max >= 2) {
        const int nc = std::min(force_chunks, T_max), cl = (T_max + nc - 1) / nc;
        bounds.clear();
        for (int t0 = 0; t0 < T_max; t0 += cl) bounds.push_back(t0);
        bounds.push_back(T_max);
    }
    const int n_chunks = static_cast<int>(bounds.size()) - 1;
    bool chunk_timing = false, gated_call = false;
    if (n_chunks > 1) {
        const Launch& ln = launches[0];
        const u64 stride = (kV5Save[ln.v5][V <= B2C_FAST_LT ? 1 : 0] + 16 + 255) & ~255ull;
        if (d->d_state.ensure(stride * static_cast<u64>(ln.slots))) return B2C_E_NOMEM;
        BA.L = ln.L;
        BA.n_utts = ln.count;
        BA.order = d_ord + ln.ord_off;
        BA.next = d_next;
        BA.gws = d->d_ws.as<u8>();
        BA.state = d->d_state.as<u8>();
        BA.state_stride = stride;
        chunk_timing = pipe_candidate && n_chunks <= B2C_PIPE_CHUNKS;
        cudaStream_t ps = gated ? d->prep_stream : st;
        if (gated) {
            if (d->d_gate.ensure(64)) return B2C_E_NOMEM;
            CUDA_OK(cudaMemsetAsync(d->d_gate.p, 0, 64, st));
            CUDA_OK(cudaEventRecord(d->prep_ev[0], st));              // meta, memsets, hot table, LM states: uploaded
            CUDA_OK(cudaStreamWaitEvent(ps, d->prep_ev[0], 0));
            BA.gate = d->d_gate.as<u32>();
            BA.gate_n = n_chunks;
            for (int c = 0; c <= n_chunks; ++c) BA.gate_bounds[c] = bounds[c];
        }
        if (pipe_candidate) {
            // every chunk's copy is queued at once on the copy stream; the compute stream waits chunk by chunk
            const size_t pitch = static_cast<size_t>(T_max) * V * esz;
            for (int c = 0; c < n_chunks; ++c) {
                const int t0 = bounds[c], t1 = bounds[c + 1];
                CUDA_OK(cudaMemcpy2DAsync(d->d_logits.as<char>() + static_cast<size_t>(t0) * V * esz, pitch,
                                          static_cast<const char*>(logits[0]) + static_cast<size_t>(t0) * V * esz, pitch,
                                          static_cast<size_t>(t1 - t0) * V * esz, static_cast<size_t>(n_utts), cudaMemcpyHostToDevice, d->copy_stream));
                CUDA_OK(cudaEventRecord(d->copied[c % B2C_PIPE_CHUNKS], d->copy_stream));
                d->tm.h2d_bytes += static_cast<long long>(t1 - t0) * V * static_cast<long long>(esz) * n_utts;
            }
        }
        if (!gated) CUDA_OK(cudaEventRecord(d->ev[5], st));
        for (int c = 0; c < n_chunks; ++c) {
            const int t0 = bounds[c], t1 = bounds[c + 1];
            if (pipe_candidate) {
                CUDA_OK(cudaStreamWaitEvent(ps, d->copied[c % B2C_PIPE_CHUNKS], 0));
                if (chunk_timing) CUDA_OK(cudaEventRecord(d->chunk_ev[3 * c], ps));
                B2cPrepArgs PC = PA;
                PC.mode = 0;
                PC.tile_lo = t0 / B2C_TILE_ROWS;
                PC.tile_hi = (t1 + B2C_TILE_ROWS - 1) / B2C_TILE_ROWS;
                PC.run_lo = t0 / B2C_RUN;
                PC.run_hi = (t1 + B2C_RUN - 1) / B2C_RUN;
                const u64 run_items = static_cast<u64>(n_utts) * static_cast<u64>(PC.run_hi - PC.run_lo);
                const int grid_runs = static_cast<int>(std::max<u64>(1, std::min<u64>((run_items + B2C_PREP_WARPS - 1) / B2C_PREP_WARPS, static_cast<u64>(grid_tok))));
#ifdef B2C_HOSTSIM
                {
                    std::unique_ptr<B2cPrepShared> sh(new B2cPrepShared());
                    for (int b = 0; b < grid_runs; ++b) {
                        if (dtype == B2C_DTYPE_F32) b2c_tokens_block<float>(PC, b, grid_runs, sh.get());
                        else b2c_tokens_block<double>(PC, b, grid_runs, sh.get());
                    }
                }
#else
                if (dtype == B2C_DTYPE_F32 && V <= 32) {
                    const u64 items = static_cast<u64>(n_utts) * static_cast<u64>(PC.tile_hi - PC.tile_lo);
                    const int grid = static_cast<int>(std::max<u64>(1, std::min<u64>((items + B2C_TILE_WARPS - 1) / B2C_TILE_WARPS, static_cast<u64>(d->n_sm) * 8)));
                    b2c_tokens_tile_kernel<<<grid, B2C_TILE_WARPS * 32, 0, ps>>>(PC);
                } else if (dtype == B2C_DTYPE_F32) {
                    b2c_tokens_kernel<float><<<grid_runs, B2C_PREP_THREADS, 0, ps>>>(PC);
                } else {
                    b2c_tokens_kernel<double><<<grid_runs, B2C_PREP_THREADS, 0, ps>>>(PC);
                }
                CUDA_OK(cudaGetLastError());
#endif
                d->tm.launches += 1;
                if (chunk_timing) CUDA_OK(cudaEventRecord(d->chunk_ev[3 * c + 1], ps));
            }
            if (gated) {
                CUDA_OK(cudaMemsetAsync(d->d_gate.as<u32>() + c, 1, 4, ps));       // chunk c's token lists are in HBM
#ifdef B2C_HOSTSIM
                // hostsim runs a launch to completion at once: after the last chunk -- or, to test the give-up path
                // (the later chunks "never arrive"), right after the first one
                if (c == (std::getenv("B200CTC_HOSTSIM_GATE_EARLY") ? 0 : n_chunks - 1)) {
#else
                if (c == 0) {
#endif
                    // the beam kernel: ONE launch, behind the first chunk only
                    CUDA_OK(cudaEventRecord(d->prep_ev[1], ps));
                    CUDA_OK(cudaStreamWaitEvent(st, d->prep_ev[1], 0));
                    CUDA_OK(cudaEventRecord(d->ev[5], st));
                    BA.chunk_t0 = 0;
                    BA.chunk_t1 = 0;
                    rc = launch_beam(d, BA, ln.slots, true, ln.per_sm, ln.threads, st, ln.v5);
                    if (rc) return rc;
                    d->tm.launches += 1;
                }
                continue;
            }
            BA.chunk_t0 = t0;
            BA.chunk_t1 = t1;
            BA.chunk_last = c == n_chunks - 1 ? 1 : 0;
            rc = launch_beam(d, BA, ln.slots, true, ln.per_sm, ln.threads, st, ln.v5);
            if (rc) return rc;
            d->tm.launches += 1;
            if (chunk_timing) CUDA_OK(cudaEventRecord(d->chunk_ev[3 * c + 2], st));
        }
        BA.chunk_t1 = 0;
        BA.gate = nullptr;
        if (pipe_candidate) {
            // probabilities or logits: decided now that every row has been seen; a probability utterance voids the call
#ifdef B2C_HOSTSIM
            {
                std::unique_ptr<B2cDecideShared> dsh(new B2cDecideShared());
                for (int u = 0; u < n_utts; ++u) {
                    if (dtype == B2C_DTYPE_F32) b2c_decide_block<float>(PA, u, dsh.get());
                    else b2c_decide_block<double>(PA, u, dsh.get());
                }
            }
#else
            if (dtype == B2C_DTYPE_F32) b2c_decide_kernel<float><<<n_utts, 128, 0, ps>>>(PA);
            else b2c_decide_kernel<double><<<n_utts, 128, 0, ps>>>(PA);
            CUDA_OK(cudaGetLastError());
#endif
            d->tm.launches += 1;
            if (gated) {
                CUDA_OK(cudaEventRecord(d->prep_ev[2], ps));
                CUDA_OK(cudaStreamWaitEvent(st, d->prep_ev[2], 0));
            }
            CUDA_OK(cudaMemcpyAsync(d->h_maxk.p, d->d_approx.as<double>() + 2 * n_utts, 4, cudaMemcpyDeviceToHost, st));
        }
        gated_call = gated;
        d->tm.cap_candidates = static_cast<int>(ln.L.cap_s);
        d->tm.cta_threads = ln.threads;
        d->tm.cta_slots = ln.slots;
        d->tm.kernel_variant = 2;
    }
    if (n_chunks == 1) CUDA_OK(cudaEventRecord(d->ev[5], st));
    CUDA_OK(cudaEventRecord(d->fork_ev, st));
    int qi = 0;
    for (const Launch& ln : launches) {
        if (n_chunks > 1) break;
        cudaStream_t cs = launches.size() > 1 ? d->cls_stream[ln.cls < kNumCaps ? 0 : 1] : st;
        if (cs != st) CUDA_OK(cudaStreamWaitEvent(cs, d->fork_ev, 0));
        BA.L = ln.L;
        BA.n_utts = ln.count;
        BA.order = d_ord + ln.ord_off;
        BA.next = d_next + qi;
        BA.gws = d->d_ws.as<u8>() + ws_off[qi];
        ++qi;
        rc = launch_beam(d, BA, ln.slots, ln.cls < kNumCaps, ln.per_sm, ln.threads, cs, ln.v5);
        if (rc) return rc;
        d->tm.launches += 1;
        if (ln.cls < kNumCaps || launches.size() == 1) {
            d->tm.cap_candidates = static_cast<int>(ln.L.cap_s);
            d->tm.cta_threads = ln.threads;
            d->tm.cta_slots = ln.slots;
            d->tm.kernel_variant = ln.v5 >= 0 ? 2 : (ln.cls < kNumCaps ? 1 : 0);
            if (!pipe_candidate && !hinted && launches.size() == 1) { d->plain_v5 = ln.v5; d->plain_cap = static_cast<int>(ln.L.cap_s); }
        }
        if (cs != st) {
            CUDA_OK(cudaEventRecord(d->cls_done[ln.cls < kNumCaps ? 0 : 1], cs));
            CUDA_OK(cudaStreamWaitEvent(st, d->cls_done[ln.cls < kNumCaps ? 0 : 1], 0));
        }
    }
    CUDA_OK(cudaEventRecord(d->ev[3], st));

    // ---- device -> host -------------------------------------------------------------------
    CUDA_OK(cudaMemcpyAsync(d->h_out_small.p, d->d_out_small.p, small_bytes, cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaMemcpyAsync(d->h_out_toks.p, d->d_out_toks.p, tok_bytes, cudaMemcpyDeviceToHost, st));
    const bool text_only = opts->text_only != 0 && !streaming;
    if (!text_only) CUDA_OK(cudaMemcpyAsync(d->h_out_frames.p, d->d_out_frames.p, frm_bytes, cudaMemcpyDeviceToHost, st));
    if (d->h_mstats.ensure(64)) return B2C_E_NOMEM;
    CUDA_OK(cudaMemcpyAsync(d->h_mstats.p, d->d_mstats.p, 64, cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaEventRecord(d->ev[4], st));
    hp_mark(2);                                   // launch planning + enqueue of the beam kernel and D2H
    CUDA_OK(cudaStreamSynchronize(st));
    hp_mark(3);                                   // wait: beam kernel + D2H
    if (pipe_candidate && d->h_maxk.as<u32>()[0] != 0) return B2C_E_RETRY_PLAIN;   // some utterance holds probabilities
    if (gated_call) {
        const int* hst = reinterpret_cast<const int*>(d->h_out_small.as<u8>() + off_st);
        for (int i = 0; i < n_utts; ++i)
            if (hst[i] & B2C_ERR_GATE) {           // the streaming stage of a later chunk never got to run beside the beam kernel
                d->pipe_refused = true;
                return B2C_E_RETRY_PLAIN;
            }
    }
    d->tm.d2h_bytes += static_cast<long long>(small_bytes + tok_bytes + (text_only ? 0 : frm_bytes) + 8ull * n_utts + 32);
    {
        const u32* ms = d->h_mstats.as<u32>();
        d->hint_valid = true;
        d->hint_beam = opts->beam_width;
        d->hint_lm = P.lm.order > 0 ? 1 : 0;
        d->hint_hot = P.n_hot > 0 ? 1 : 0;
        d->hint_prune = P.prune_history;
        for (int q = 0; q < 6; ++q) d->hint_over[q] = ms[q];
        d->hint_frames = ms[6];
        for (int q = 0; q < 7; ++q) d->tm.cand_hist[q] = ms[q];
        d->tm.inplace_frames = ms[7];
        d->tm.sorted_frames = ms[8];
        d->tm.oversize_frames = 0;
        for (int q = 0; q < 6; ++q)
            if (static_cast<int>(128u << q) == d->tm.cap_candidates) d->tm.oversize_frames = ms[q];
    }

    u8* hs = d->h_out_small.as<u8>();
    int* h_status = reinterpret_cast<int*>(hs + off_st);
    std::vector<int> failed;
    for (int i = 0; i < n_utts; ++i) if (h_status[i] != B2C_OK) failed.push_back(i);
    // utterances whose arenas overflowed: decoded again by the general kernel with worst-case arenas
    if (!failed.empty()) {
        const Launch ln = plan(failed, kNumCaps, true, static_cast<size_t>(n_utts));
        if (ln.L.smem_bytes > d->smem_optin) return fail(B2C_E_ARG, "beam_width too large for the shared-memory selection arrays");
        if (d->d_ws.ensure(static_cast<u64>(ln.slots) * ln.L.gws_bytes)) return B2C_E_NOMEM;
        for (size_t i = 0; i < failed.size(); ++i) h_ord[n_utts + i] = failed[i];
        CUDA_OK(cudaMemcpyAsync(d_ord + n_utts, h_ord + n_utts, 4 * failed.size(), cudaMemcpyHostToDevice, st));
        CUDA_OK(cudaMemsetAsync(d_next + 15, 0, 4, st));
        BA.L = ln.L;
        BA.n_utts = ln.count;
        BA.order = d_ord + n_utts;
        BA.next = d_next + 15;
        BA.gws = d->d_ws.as<u8>();
        BA.chunk_t1 = 0;
        rc = launch_beam(d, BA, ln.slots, ln.cls < kNumCaps, ln.per_sm, ln.threads, st, ln.v5);
        if (rc) return rc;
        d->tm.launches += 1;
        CUDA_OK(cudaMemcpyAsync(d->h_out_small.p, d->d_out_small.p, small_bytes, cudaMemcpyDeviceToHost, st));
        CUDA_OK(cudaMemcpyAsync(d->h_out_toks.p, d->d_out_toks.p, tok_bytes, cudaMemcpyDeviceToHost, st));
        CUDA_OK(cudaMemcpyAsync(d->h_out_frames.p, d->d_out_frames.p, frm_bytes, cudaMemcpyDeviceToHost, st));
        CUDA_OK(cudaStreamSynchronize(st));
    }
    for (int i : failed)
        if (h_status[i] != B2C_OK) return fail(B2C_E_INTERNAL, "beam kernel workspace overflow (status " + std::to_string(h_status[i]) + ")");
#if defined(B2C_PHASE_CLOCKS)
    {
        u64 hc[32];
        CUDA_OK(cudaMemcpy(hc, d->d_clk.p, sizeof(hc), cudaMemcpyDeviceToHost));
        std::fprintf(stderr, "[b2c phase clocks, summed over CTAs, Mcycles]");
        for (int q = 0; q < 24; ++q) std::fprintf(stderr, " p%d=%.3f", q, hc[q] / 1e6);
        std::fprintf(stderr, "  frames=%llu\n", static_cast<unsigned long long>(total_frames));
    }
#endif
    float ms = 0.f;
    if (chunk_timing) {        // pipelined: kernels of the chunks interleave with waits for the copies -- sum them up
        float mp = 0.f, mb = 0.f;
        for (int c = 0; c < n_chunks; ++c) {
            if (cudaEventElapsedTime(&ms, d->chunk_ev[3 * c], d->chunk_ev[3 * c + 1]) == cudaSuccess) mp += ms;
            if (!gated_call && cudaEventElapsedTime(&ms, d->chunk_ev[3 * c + 1], d->chunk_ev[3 * c + 2]) == cudaSuccess) mb += ms;
        }
        if (gated_call && cudaEventElapsedTime(&ms, d->ev[5], d->ev[3]) == cudaSuccess) mb = ms;     // one launch, waits included
        d->tm.ms_prepare = mp;
        d->tm.ms_beam = mb;
        if (host_prof) {
            std::fprintf(stderr, "[b2c pipeline, ms after the call's first event]");
            for (int c = 0; c < n_chunks; ++c) {
                float a0 = 0.f, a1 = 0.f, a2 = 0.f;
                cudaEventElapsedTime(&a0, d->ev[0], d->chunk_ev[3 * c]);
                cudaEventElapsedTime(&a1, d->ev[0], d->chunk_ev[3 * c + 1]);
                if (!gated_call) cudaEventElapsedTime(&a2, d->ev[0], d->chunk_ev[3 * c + 2]);
                std::fprintf(stderr, "  chunk %d: copied %.3f streamed %.3f decoded %.3f", c, a0, a1, a2);
            }
            float a4 = 0.f;
            cudaEventElapsedTime(&a4, d->ev[0], d->ev[4]);
            std::fprintf(stderr, "  d2h done %.3f\n", a4);
        }
    } else {
        if (!pipe_candidate && cudaEventElapsedTime(&ms, d->ev[1], d->ev[2]) == cudaSuccess) d->tm.ms_prepare = ms;
        if (cudaEventElapsedTime(&ms, d->ev[5], d->ev[3]) == cudaSuccess) d->tm.ms_beam = ms;
    }
    if (cudaEventElapsedTime(&ms, d->ev[0], d->ev[4]) == cudaSuccess) d->tm.ms_total = ms;
    d->tm.frames = static_cast<long long>(total_frames);
    d->last_device_ms = static_cast<double>(d->tm.ms_prepare) + static_cast<double>(d->tm.ms_beam);
    // total selected tokens = last tok_start of the last utterance ... summed per utterance is not
    // available without a reduction; report the last utterance's end offset only when B == 1
    d->tm.tokens = 0;

    // ---- assemble results -------------------------------------------------------------------
    const int* h_nb = reinterpret_cast<const int*>(hs + off_nb);
    const double* h_sc = reinterpret_cast<const double*>(hs + off_sc);
    const int* h_nt = reinterpret_cast<const int*>(hs + off_nt);
    const int* h_nw = reinterpret_cast<const int*>(hs + off_nw);
    const B2cLmState* h_ls = reinterpret_cast<const B2cLmState*>(hs + off_ls);
    const int* h_ax = streaming ? reinterpret_cast<const int*>(hs + off_ax) : nullptr;
    const B2cLmState* h_lx = n_lm > 1 ? reinterpret_cast<const B2cLmState*>(hs + off_lx) : nullptr;
    const u32* h_toks = d->h_out_toks.as<u32>();
    const int* h_frames = d->h_out_frames.as<int>();
    auto assemble_range = [&](int u0, int u1) {
        for (int u = u0; u < u1; ++u) {
            const int nb = h_nb[u];
            res->utts[u].resize(nb);
            const u64 base = static_cast<u64>(OB) * (frame_off[u] + static_cast<u64>(u));
            const u64 stride = static_cast<u64>(T[u]) + 1;
            for (int r = 0; r < nb; ++r) {
                BeamRes& br = res->utts[u][r];
                const u64 k = static_cast<u64>(u) * OB + r;
                br.logit = h_sc[2 * k];
                br.lm = h_sc[2 * k + 1];
                br.st = h_ls[k];
                if (h_lx) br.stx.assign(h_lx + k * (n_lm - 1), h_lx + (k + 1) * (n_lm - 1));
                if (text_only) assemble_text(d, h_toks + base + r * stride, h_nt[k], br);
                else assemble_beam(d, h_toks + base + r * stride, h_nt[k], h_frames + 2 * (base + r * stride), h_nw[k], br);
                if (h_ax) {
                    const u32* tk = h_toks + base + r * stride;
                    br.raw.resize(static_cast<size_t>(h_nt[k]));
                    for (int q = 0; q < h_nt[k]; ++q) br.raw[q] = tk[h_nt[k] - 1 - q];
                    for (int q = 0; q < 4; ++q) br.aux[q] = h_ax[4 * k + q];
                    {   // the chain as strings (the host replays it onto the input beam's text / partial word)
                        std::string cur;
                        br.s_boundary = false;
                        for (const u32 v : br.raw) {
                            const u32 tok = v & 0xFFFFu, kind = v >> 16;
                            if (kind == B2C_CK_CONT) { cur += d->labels[tok]; continue; }
                            if (!br.s_boundary) { br.s_first = cur; br.s_boundary = true; }
                            else if (!cur.empty()) { if (!br.s_mid.empty()) br.s_mid += ' '; br.s_mid += cur; }
                            cur = kind == B2C_CK_BPE ? d->clean[tok] : std::string();
                        }
                        if (br.s_boundary) br.s_last = cur; else br.s_first = cur;
                    }
                    // assemble_beam truncated the frame list to the words it could name; keep all of them here
                    br.frames.resize(static_cast<size_t>(h_nw[k]) * 2);
                    const int* fr = h_frames + 2 * (base + r * stride);
                    for (int w = 0; w < h_nw[k]; ++w) {
                        br.frames[2 * w] = fr[2 * (h_nw[k] - 1 - w)];
                        br.frames[2 * w + 1] = fr[2 * (h_nw[k] - 1 - w) + 1];
                    }
                }
            }
        }
    };
    {
        // string building is independent per utterance: a few persistent host threads for large batches
        const u64 work = (total_frames + static_cast<u64>(n_utts)) * static_cast<u64>(OB);
        int n_thr = static_cast<int>(std::min<u64>(std::min<u64>(8, std::max(1u, std::thread::hardware_concurrency())), work / 32768));
        n_thr = std::min(n_thr, n_utts);
        if (n_thr <= 1) {
            assemble_range(0, n_utts);
        } else {
            if (!d->pool) {
                d->pool.reset(new HostPool());
                d->pool->start(static_cast<int>(std::min<u64>(8, std::max(1u, std::thread::hardware_concurrency()))) - 1);
            }
            const int chunks = n_thr * 4;
            const int per = (n_utts + chunks - 1) / chunks;
            const std::function<void(int)> task = [&](int c) { assemble_range(std::min(n_utts, c * per), std::min(n_utts, (c + 1) * per)); };
            d->pool->run(chunks, task);
        }
    }
    hp_mark(4);                                   // statistics read-back, result assembly
    if (host_prof)
        std::fprintf(stderr, "[b2c host ms] enqueue=%.3f wait_prepare=%.3f plan=%.3f wait_beam=%.3f assemble=%.3f\n", hp_ms[0],
                     hp_ms[1], hp_ms[2], hp_ms[3], hp_ms[4]);
    *out = res.release();
    return 0;
}

// ---- results ------------------------------------------------------------------------------
void b2c_result_free(b2c_result_t* r) { delete r; }
int b2c_result_n_utts(const b2c_result_t* r) { return r ? static_cast<int>(r->utts.size()) : 0; }
int b2c_result_n_beams(const b2c_result_t* r, int u) { return static_cast<int>(r->utts[u].size()); }
const char* b2c_result_text(const b2c_result_t* r, int u, int b) { return r->utts[u][b].text.c_str(); }
int b2c_result_top_texts(b2c_result_t* r, const char** data, size_t* size) {
    if (!r || !data || !size) return fail(B2C_E_ARG, "null argument");
    if (!r->joined_built) {
        size_t total = 0;
        for (const auto& u : r->utts) total += (u.empty() ? 0 : u[0].text.size()) + 1;
        r->joined.reserve(total);
        for (const auto& u : r->utts) {
            if (!u.empty()) r->joined += u[0].text;
            r->joined.push_back('\0');
        }
        r->joined_built = true;
    }
    *data = r->joined.data();
    *size = r->joined.size();
    return 0;
}
int b2c_result_packed(b2c_result_t* r, b2c_packed_t* out) {
    if (!r || !out) return fail(B2C_E_ARG, "null argument");
    if (!r->packed_built) {
        size_t nb = 0, nw = 0, nt = 0;
        for (const auto& u : r->utts)
            for (const auto& b : u) { ++nb; nw += b.frames.size() / 2; nt += b.text.size() + 1; }
        const int nm = r->has_lm ? std::max(1, r->n_models) : 0;
        r->pk_nb.reserve(r->utts.size());
        r->pk_nw.reserve(nb);
        r->pk_scores.reserve(2 * nb);
        r->pk_frames.reserve(2 * nw);
        r->pk_texts.reserve(nt);
        r->pk_states.reserve(nb * static_cast<size_t>(nm));
        for (const auto& u : r->utts) {
            r->pk_nb.push_back(static_cast<int32_t>(u.size()));
            for (const auto& b : u) {
                r->pk_nw.push_back(static_cast<int32_t>(b.frames.size() / 2));
                r->pk_scores.push_back(b.logit);
                r->pk_scores.push_back(b.lm);
                r->pk_frames.insert(r->pk_frames.end(), b.frames.begin(), b.frames.end());
                r->pk_texts += b.text;
                r->pk_texts.push_back('\0');
                for (int j = 0; j < nm; ++j) {
                    b2c_lm_state_t st;
                    from_internal(j == 0 ? b.st : b.stx[static_cast<size_t>(j) - 1], &st);
                    r->pk_states.push_back(st);
                }
                if (r->streaming) {
                    r->pk_aux.insert(r->pk_aux.end(), b.aux, b.aux + 4);
                    r->pk_ntok.push_back(static_cast<int32_t>(b.raw.size()));
                    r->pk_toks.insert(r->pk_toks.end(), b.raw.begin(), b.raw.end());
                    r->pk_boundary.push_back(b.s_boundary ? 1 : 0);
                    r->pk_pieces += b.s_first; r->pk_pieces.push_back('\0');
                    r->pk_pieces += b.s_mid; r->pk_pieces.push_back('\0');
                    r->pk_pieces += b.s_last; r->pk_pieces.push_back('\0');
                }
            }
        }
        r->packed_built = true;
    }
    out->n_utts = static_cast<int32_t>(r->utts.size());
    out->n_models = r->has_lm ? std::max(1, r->n_models) : 0;
    out->n_beams_total = static_cast<int64_t>(r->pk_nw.size());
    out->n_words_total = static_cast<int64_t>(r->pk_frames.size() / 2);
    out->n_beams = r->pk_nb.data();
    out->scores = r->pk_scores.data();
    out->n_words = r->pk_nw.data();
    out->frames = r->pk_frames.data();
    out->texts = r->pk_texts.data();
    out->texts_size = r->pk_texts.size();
    out->states = r->pk_states.empty() ? nullptr : r->pk_states.data();
    out->stream_aux = r->streaming ? r->pk_aux.data() : nullptr;
    out->n_stream_toks = r->streaming ? r->pk_ntok.data() : nullptr;
    out->stream_toks = r->streaming ? r->pk_toks.data() : nullptr;
    out->n_stream_toks_total = static_cast<int64_t>(r->pk_toks.size());
    out->stream_pieces = r->streaming ? r->pk_pieces.data() : nullptr;
    out->stream_pieces_size = r->pk_pieces.size();
    out->stream_boundary = r->streaming ? r->pk_boundary.data() : nullptr;
    return 0;
}
double b2c_result_logit_score(const b2c_result_t* r, int u, int b) { return r->utts[u][b].logit; }
double b2c_result_lm_score(const b2c_result_t* r, int u, int b) { return r->utts[u][b].lm; }
int b2c_result_n_words(const b2c_result_t* r, int u, int b) { return static_cast<int>(r->utts[u][b].words.size()); }
const char* b2c_result_word(const b2c_result_t* r, int u, int b, int w) { return r->utts[u][b].words[w].c_str(); }
const int32_t* b2c_result_frames(const b2c_result_t* r, int u, int b) { return r->utts[u][b].frames.data(); }
int b2c_result_lm_state(const b2c_result_t* r, int u, int b, b2c_lm_state_t* out) {
    if (!r->has_lm) return 0;
    from_internal(r->utts[u][b].st, out);
    return 1;
}
int b2c_result_lm_state_at(const b2c_result_t* r, int u, int b, int lm_index, b2c_lm_state_t* out) {
    if (!r->has_lm) return 0;
    const BeamRes& br = r->utts[u][b];
    if (lm_index == 0) { from_internal(br.st, out); return 1; }
    if (lm_index < 0 || lm_index > static_cast<int>(br.stx.size())) return 0;
    from_internal(br.stx[lm_index - 1], out);
    return 1;
}
int b2c_result_stream_beam(const b2c_result_t* r, int u, int b, int32_t aux[4], const uint32_t** toks, int* n_toks) {
    if (!r || u < 0 || u >= static_cast<int>(r->utts.size()) || b < 0 || b >= static_cast<int>(r->utts[u].size()))
        return fail(B2C_E_ARG, "no such beam");
    const BeamRes& br = r->utts[u][b];
    for (int q = 0; q < 4; ++q) aux[q] = br.aux[q];
    *toks = br.raw.data();
    *n_toks = static_cast<int>(br.raw.size());
    return 0;
}
int b2c_result_n_frames(const b2c_result_t* r, int u, int b) { return static_cast<int>(r->utts[u][b].frames.size() / 2); }
int b2c_hash_utf8(const char* s, uint64_t* hash, uint32_t* n_chars) {
    if (!s || !hash || !n_chars) return fail(B2C_E_ARG, "null argument");
    const size_t n = std::strlen(s);
    *hash = b2c_hash_bytes(s, n);
    *n_chars = b2c_utf8_len(s, n);
    return 0;
}
int b2c_hash_utf8_batch(const char* data, size_t size, int64_t count, uint64_t* hashes, uint32_t* n_chars) {
    if (count < 0 || (count > 0 && (!data || !hashes || !n_chars))) return fail(B2C_E_ARG, "null argument");
    size_t p = 0;
    for (int64_t i = 0; i < count; ++i) {
        size_t q = p;
        while (q < size && data[q] != '\0') ++q;
        if (q >= size) return fail(B2C_E_ARG, "b2c_hash_utf8_batch: fewer NUL-terminated strings than `count`");
        hashes[i] = b2c_hash_bytes(data + p, q - p);
        n_chars[i] = b2c_utf8_len(data + p, q - p);
        p = q + 1;
    }
    return 0;
}
int b2c_decoder_token_id(const b2c_decoder_t* d, const char* label) {
    if (!d || !label) return -1;
    for (size_t i = 0; i < d->labels.size(); ++i)
        if (d->labels[i] == label) return static_cast<int>(d->toks[i].canon);
    return -1;
}
int b2c_decoder_last_timings(const b2c_decoder_t* d, b2c_timings_t* out) {
    if (!d || !out) return fail(B2C_E_ARG, "null argument");
    *out = d->tm;
    return 0;
}

}  // extern "C"
