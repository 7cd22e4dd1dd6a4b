// dlz4_kernels.cuh -- sm_100a device code of the B200-native LZ4 block codec.
//
// One warp owns one chain of the reference's greedy single-probe match finder (src/block/blockCompress.js:31-233) and
// reproduces it bit for bit.  Parallelism inside a chain comes from the probe schedule: the next 32 probe positions are a
// pure function of (sIndex, searchMatchCount), so 32 lanes probe them at once (compress_block_warp: batch step; and the
// dense 32-position window of compress_span_warp).  Parallelism across chains comes from where the 32 KiB hash tables
// live: a few in shared memory, most in L2-resident global scratch (TabG16 / Tab12e / TabOv / TabG32).
//
//   compress    k_compress_fresh16h   fresh blocks <= 64 KiB (the headline kernel), 28 chains per SM
//               k_compress_overlay    blocks <= 4 KiB behind a shared prefix, one read-only initial table + per-warp overlay
//               k_compress_segments   linked chains and large blocks: speculative segments, k_seg_verify, k_seg_assemble
//               k_compress_generic32 / k_compress_chain   Int32 table in shared memory (prefix + table, short chains, compressRaw)
//   decompress  k_decompress_blocks   one warp per block, speculative lane-parallel token sizing, merged literal+match copy
//               k_jd_* / k_jdp_*      jump decoder for linked frames and large blocks: token scan, pointer doubling
//               k_decompress_chain    short linked frames, one warp
//   xxh32       k_xxh32_batch (per block), k_xxh32_stream (whole stream, stateful), frame packing kernels at the end
//
// No tensor cores: the work is byte-serial integer work bounded by latency and by the memory system, not FLOPs.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <limits.h>

namespace dlz4 {

// Phase timing (profiling build only: -DDLZ4_PHASE_TIMING): cycles per phase of the window path, summed over warps.
#ifdef DLZ4_PHASE_TIMING
__device__ unsigned long long g_phase[16];
#define PT_DECL unsigned long long pt_acc[16] = {0,0,0,0,0,0,0,0,0,0,0,0,0,0,0,0}; long long pt_t = clock64();
#define PT_MARK(i) { const long long pt_n = clock64(); pt_acc[i] += (unsigned long long)(pt_n - pt_t); pt_t = pt_n; }
#define PT_COUNT(i, v) { pt_acc[i] += (v); }
#define PT_FLUSH if (lane_id() == 0) { for (int pt_k = 0; pt_k < 16; ++pt_k) atomicAdd(&g_phase[pt_k], pt_acc[pt_k]); }
#define PT_USE(x) asm volatile("" ::"r"((uint32_t)(x)));
#else
#define PT_DECL
#define PT_MARK(i)
#define PT_COUNT(i, v)
#define PT_FLUSH
#define PT_USE(x)
#endif

#ifndef DLZ4_DEC_MINB
#define DLZ4_DEC_MINB 6                 // resident CTAs of the block decoder per SM the register allocation is held to
#endif
#ifndef DLZ4_DEC_PREFETCH
#define DLZ4_DEC_PREFETCH 1             // every real token of a window prefetches the line of its match source into L1
#endif
#ifndef DLZ4_DEC_Q
#define DLZ4_DEC_Q 2                    // sequences per step of the decoder's quick copy form
#endif
constexpr uint32_t FULL = 0xffffffffu;
constexpr int kHashEntries = 16384;

// per-block status, same numbering as DLZ4_E_* in include/dlz4_b200.h
enum : uint8_t { ST_OK = 0, ST_OUTPUT_TOO_SMALL = 1, ST_MALFORMED = 2, ST_OFFSET_ZERO = 3, ST_DICT_OOB = 4 };

__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31u; }

// Unaligned little-endian u32 built from aligned word loads.  Touches only words that contain one of
// the four requested bytes, so it can never leave an allocation that holds those bytes.
__device__ __forceinline__ uint32_t ld32u(const uint8_t *p) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const uint32_t *w = reinterpret_cast<const uint32_t *>(a & ~static_cast<uintptr_t>(3));
    const uint32_t sh = static_cast<uint32_t>(a & 3u) * 8u;
    const uint32_t lo = w[0];
    if (sh == 0) return lo;
    return __funnelshift_r(lo, w[1], sh);
}

__device__ __forceinline__ void st32u(uint8_t *p, uint32_t v) {
    if ((reinterpret_cast<uintptr_t>(p) & 3u) == 0) { *reinterpret_cast<uint32_t *>(p) = v; return; }
    p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); p[2] = (uint8_t)(v >> 16); p[3] = (uint8_t)(v >> 24);
}

// Warp-cooperative copy of n bytes, arbitrary alignment on both sides, non-overlapping.
// (No __restrict__: the decoder copies from bytes this kernel wrote; they must not become ld.global.nc.)
__device__ __forceinline__ void warp_copy(uint8_t *d, const uint8_t *s, uint32_t n, uint32_t lane) {
    if (n <= 64) {
        if (lane < n) d[lane] = s[lane];
        if (lane + 32 < n) d[lane + 32] = s[lane + 32];
        return;
    }
    const uint32_t head = static_cast<uint32_t>(-reinterpret_cast<intptr_t>(d)) & 3u;
    if (lane < head) d[lane] = s[lane];
    d += head; s += head; n -= head;
    const uint32_t nw = n >> 2;
    uint32_t *dw = reinterpret_cast<uint32_t *>(d);
    if ((reinterpret_cast<uintptr_t>(s) & 3u) == 0) {
        const uint32_t *sw = reinterpret_cast<const uint32_t *>(s);
        for (uint32_t i = lane; i < nw; i += 32) dw[i] = sw[i];
    } else {
        for (uint32_t i = lane; i < nw; i += 32) dw[i] = ld32u(s + 4 * i);
    }
    const uint32_t done = nw << 2;
    if (lane < n - done) d[done + lane] = s[done + lane];
}

// Sum_{u<x} (u >> 6): distance covered by x probes of the skip schedule sIndex += (count++ >> 6)
// (blockCompress.js:66-67), counted from count = 0.
__device__ __forceinline__ uint32_t skip_sum(uint32_t x) {
    const uint32_t q = x >> 6, r = x & 63u;
    return 32u * q * (q - 1u) + q * r;
}

// ------------------------------------------------------------------ source address spaces
// Virtual index v of the reference's `src` array -> byte.
struct SrcFlat {                          // src is one contiguous buffer
    const uint8_t *base;
    __device__ __forceinline__ uint32_t ld32(int32_t v) const { return ld32u(base + v); }
    __device__ __forceinline__ const uint8_t *lit_ptr(int32_t v) const { return base + v; }
};
struct SrcSplit {                         // src = prefix ++ block, stored apart (shared dictionary, config 4)
    const uint8_t *prefix; int32_t plen; const uint8_t *blk;
    __device__ __forceinline__ uint32_t byte(int32_t v) const { return v < plen ? prefix[v] : blk[v - plen]; }
    __device__ __forceinline__ uint32_t ld32(int32_t v) const {
        if (v >= plen) return ld32u(blk + (v - plen));
        if (v + 4 <= plen) return ld32u(prefix + v);
        return byte(v) | (byte(v + 1) << 8) | (byte(v + 2) << 16) | (byte(v + 3) << 24);
    }
    __device__ __forceinline__ const uint8_t *lit_ptr(int32_t v) const { return blk + (v - plen); }   // literals are never in the prefix
};

// ------------------------------------------------------------------ hash tables (shared memory)
// 16-bit table for a block of <= 65536 bytes that starts from an EMPTY table and has no history:
// stores (position - start); the value 0 doubles as "empty".  That is exact: position `start` is
// always the first probe, so the only slot where "candidate = start" could pass the 4-byte check is
// hash(seq@start), which really holds an entry from then on; in every other slot the check fails
// just as an empty slot would, and for the probe AT start the candidate equals the position and is
// rejected as in blockCompress.js:62.
struct Tab16 {
    uint16_t *t; int32_t start;
    __device__ __forceinline__ int32_t get(uint32_t h) const { return start + (int32_t)t[h]; }
    __device__ __forceinline__ void put(uint32_t h, int32_t p) { t[h] = (uint16_t)(p - start); }
};
// Same encoding as Tab16, but the 32 KiB live in global memory and are accessed with .cg loads / stores: L2-resident
// (126 MB of L2 hold ~2000 such tables next to the streamed data), never cached in L1.  Lets an SM run more block chains
// than its shared memory has room for tables; ordering between lanes of the owning warp comes from __syncwarp().
struct TabG16 {
    uint16_t *t; int32_t start;
    __device__ __forceinline__ int32_t get(uint32_t h) const { return start + (int32_t)__ldcg(t + h); }
    __device__ __forceinline__ void put(uint32_t h, int32_t p) { __stcg(t + h, (uint16_t)(p - start)); }
};
// Blocks of <= 4096 bytes (config 4: 4 KiB messages): zeroing a 32 KiB table per 4 KiB block costs more than the block.
// An entry is (epoch:4 | position:12) and counts only when its epoch is the current block's; the table is cleared once every
// 15 blocks.  Exact: an entry of another epoch is an entry the reference's fresh table does not have.
template <bool kGlobal>
struct Tab12e {
    uint16_t *t; int32_t start; uint32_t epoch;
    __device__ __forceinline__ uint32_t ld(uint32_t h) const { return kGlobal ? (uint32_t)__ldcg(t + h) : (uint32_t)t[h]; }
    __device__ __forceinline__ void st(uint32_t h, uint32_t v) { if (kGlobal) __stcg(t + h, (uint16_t)v); else t[h] = (uint16_t)v; }
    __device__ __forceinline__ int32_t dec(uint32_t v) const { return (v >> 12) == epoch ? start + (int32_t)(v & 4095u) : -1; }
    __device__ __forceinline__ int32_t get(uint32_t h) const { return dec(ld(h)); }
    __device__ __forceinline__ void put(uint32_t h, int32_t p) { st(h, (epoch << 12) | (uint32_t)(p - start)); }
};
// Small blocks that all start from the SAME initial table (config 4: a table warmed from / primed with a shared dictionary
// prefix): copying 64 KiB of table per 4 KiB message would cost 16x the message.  The initial table stays read-only in
// global memory (L1/L2-resident, shared by every warp); a per-warp 16-bit overlay holds the block's own inserts as
// (epoch:4 | position - start:12) and wins whenever its epoch is current.  Values are the reference's: position + 1, <= 0 empty.
template <bool kGlobal>
struct TabOv {
    uint16_t *ov; const int32_t *base; int32_t start; uint32_t epoch;
    __device__ __forceinline__ uint32_t raw(uint32_t h) const {
        const uint32_t v = kGlobal ? (uint32_t)__ldcg(ov + h) : (uint32_t)ov[h];
        return (v >> 12) == epoch ? (uint32_t)(start + (int32_t)(v & 4095u) + 1) : (uint32_t)__ldg(base + h);
    }
    __device__ __forceinline__ void st(uint32_t h, uint32_t v) { if (kGlobal) __stcg(ov + h, (uint16_t)v); else ov[h] = (uint16_t)v; }
    __device__ __forceinline__ int32_t get(uint32_t h) const { return (int32_t)raw(h) - 1; }
    __device__ __forceinline__ void put(uint32_t h, int32_t p) { st(h, (epoch << 12) | (uint32_t)(p - start)); }
};
// The reference's own representation: Int32, value = position + 1, <= 0 empty (blockCompress.js:54-55).
struct Tab32 {
    int32_t *t;
    __device__ __forceinline__ int32_t get(uint32_t h) const { return t[h] - 1; }
    __device__ __forceinline__ void put(uint32_t h, int32_t p) { t[h] = p + 1; }
};

// token + literal-length run + literals (blockCompress.js:75-140 / :179-230); returns new write pointer
template <class Src>
__device__ __forceinline__ uint8_t *emit_literals(uint8_t *d, const Src &S, int32_t anchor, uint32_t lit,
                                                   uint32_t token_low, uint32_t lane) {
    const uint32_t tok = ((lit < 15u ? lit : 15u) << 4) | token_low;
    if (lane == 0) d[0] = (uint8_t)tok;
    d += 1;
    if (lit >= 15u) {
        const uint32_t rest = lit - 15u, n255 = rest / 255u;
        for (uint32_t i = lane; i < n255; i += 32) d[i] = 255;
        if (lane == 0) d[n255] = (uint8_t)(rest - n255 * 255u);
        d += n255 + 1;
    }
    if (lit) warp_copy(d, S.lit_ptr(anchor), lit, lane);
    return d + lit;
}

// One LZ4 block by one warp.  All 32 lanes call this with identical arguments; returns bytes written.
template <class Tab, class Src>
__device__ uint32_t compress_block_warp(const Src &S, const int32_t start, const int32_t len, Tab &T, uint8_t *const out) {
    const uint32_t lane = lane_id();
    const uint32_t lt = (1u << lane) - 1u;
    const int32_t sEnd = start + len;
    const int32_t mflimit = sEnd - 12;          // blockCompress.js:34
    const int32_t matchLimit = sEnd - 5;        // :35
    int32_t sIndex = start, anchor = start;
    uint32_t smc = 67;                          // :40 searchMatchCount
    uint8_t *d = out;

    while (sIndex < mflimit) {                  // :48
        // lane k probes the k-th upcoming position of the skip schedule (:66-67)
        const uint32_t base_sum = skip_sum(smc);
        const int32_t p = sIndex + (int32_t)(skip_sum(smc + lane) - base_sum);
        const bool valid = p < mflimit;
        uint32_t seq = 0, h = 0x10000u + lane;  // invalid lanes get a unique pseudo-hash
        int32_t cand = -1;
        if (valid) {
            seq = S.ld32(p);                                    // :50
            h = (seq * 2654435761u) >> 18;                      // :53 (14 bits)
            cand = T.get(h);                                    // :54
        }
        // the serial loop would have seen the insert of an earlier probe of this batch in the same slot
        const uint32_t same = __match_any_sync(FULL, h);
        const uint32_t prev = same & lt;
        const int j = prev ? 31 - __clz(prev) : (int)lane;
        const int32_t pj = __shfl_sync(FULL, p, j);
        const uint32_t sj = __shfl_sync(FULL, seq, j);
        uint32_t cseq = sj;
        if (prev) cand = pj;
        const bool ok = valid && cand >= 0 && cand != p && (((uint32_t)(p - cand)) >> 16) == 0;   // :62
        if (ok && !prev) cseq = S.ld32(cand);                   // :63
        const bool hit = ok && cseq == seq;
        const uint32_t hits = __ballot_sync(FULL, hit);
        const uint32_t vmask = __ballot_sync(FULL, valid);
        const int hl = __ffs(hits) - 1;                          // first hit lane, -1 if none
        const uint32_t commit = hits ? ((2u << hl) - 1u) : vmask;  // probes the serial loop really executed
        // :55 table[hash] = sIndex+1 -- per slot the LAST executed probe wins
        if (((commit >> lane) & 1u) && ((same & commit) >> lane) == 1u) T.put(h, p);
        __syncwarp();
        if (!hits) {
            if (vmask != FULL) break;                            // ran into mflimit: loop ends
            sIndex += (int32_t)(skip_sum(smc + 32u) - base_sum);
            smc += 32u;
            continue;
        }
        const int32_t s0 = __shfl_sync(FULL, p, hl);
        const int32_t m0 = __shfl_sync(FULL, cand, hl);
        smc = 67;                                                // :71

        // :143-150 forward extension, 4 bytes per lane, 128 per round
        int32_t ml;
        for (int32_t base = 4;; base += 128) {
            const int32_t q = s0 + base + 4 * (int32_t)lane;
            int32_t nv = matchLimit - q;
            nv = nv > 4 ? 4 : nv;
            int32_t eq = 0;
            if (nv > 0) {
                const uint32_t x = S.ld32(q) ^ S.ld32(m0 + base + 4 * (int32_t)lane);
                eq = x ? ((__ffs(x) - 1) >> 3) : 4;
                eq = eq < nv ? eq : nv;
            }
            const uint32_t stop = __ballot_sync(FULL, eq < 4);
            if (stop) {
                const int l = __ffs(stop) - 1;
                ml = base + 4 * l + __shfl_sync(FULL, eq, l);
                break;
            }
        }

        const uint32_t code = (uint32_t)(ml - 4);               // :160
        d = emit_literals(d, S, anchor, (uint32_t)(s0 - anchor), code < 15u ? code : 15u, lane);
        const uint32_t offset = (uint32_t)(s0 - m0);             // :153
        if (lane == 0) { d[0] = (uint8_t)offset; d[1] = (uint8_t)(offset >> 8); }   // :156-157
        d += 2;
        if (code >= 15u) {                                       // :161-168
            const uint32_t rest = code - 15u, n255 = rest / 255u;
            for (uint32_t i = lane; i < n255; i += 32) d[i] = 255;
            if (lane == 0) d[n255] = (uint8_t)(rest - n255 * 255u);
            d += n255 + 1;
        }
        sIndex = anchor = s0 + ml;                               // :173-174
    }
    d = emit_literals(d, S, anchor, (uint32_t)(sEnd - anchor), 0u, lane);   // :179-230
    return (uint32_t)(d - out);
}

// The reference's Int32 representation in L2-resident global memory (large blocks and linked chains; see TabG16).
struct TabG32 {
    int32_t *t;
    __device__ __forceinline__ int32_t get(uint32_t h) const { return __ldcg(t + h) - 1; }
    __device__ __forceinline__ void put(uint32_t h, int32_t p) { __stcg(t + h, p + 1); }
};

// ------------------------------------------------------------------ v2: dense-window compressor
// Raw table access for the window path (write / read back / restore).
__device__ __forceinline__ uint32_t tab_raw(const Tab16 &T, uint32_t h) { return T.t[h]; }
__device__ __forceinline__ void tab_set_raw(Tab16 &T, uint32_t h, uint32_t v) { T.t[h] = (uint16_t)v; }
__device__ __forceinline__ uint32_t tab_enc(const Tab16 &T, int32_t p) { return (uint32_t)(p - T.start) & 0xFFFFu; }
__device__ __forceinline__ int32_t tab_dec(const Tab16 &T, uint32_t raw) { return T.start + (int32_t)raw; }
__device__ __forceinline__ uint32_t tab_raw(const TabG16 &T, uint32_t h) { return __ldcg(T.t + h); }
__device__ __forceinline__ void tab_set_raw(TabG16 &T, uint32_t h, uint32_t v) { __stcg(T.t + h, (uint16_t)v); }
__device__ __forceinline__ uint32_t tab_enc(const TabG16 &T, int32_t p) { return (uint32_t)(p - T.start) & 0xFFFFu; }
__device__ __forceinline__ int32_t tab_dec(const TabG16 &T, uint32_t raw) { return T.start + (int32_t)raw; }
template <bool G> __device__ __forceinline__ uint32_t tab_raw(const Tab12e<G> &T, uint32_t h) { return T.ld(h); }
template <bool G> __device__ __forceinline__ void tab_set_raw(Tab12e<G> &T, uint32_t h, uint32_t v) { T.st(h, v); }
template <bool G> __device__ __forceinline__ uint32_t tab_enc(const Tab12e<G> &T, int32_t p) { return (T.epoch << 12) | (uint32_t)(p - T.start); }
template <bool G> __device__ __forceinline__ int32_t tab_dec(const Tab12e<G> &T, uint32_t raw) { return T.dec(raw); }
template <bool G> __device__ __forceinline__ uint32_t tab_raw(const TabOv<G> &T, uint32_t h) { return T.raw(h); }
template <bool G> __device__ __forceinline__ void tab_set_raw(TabOv<G> &T, uint32_t h, uint32_t v) { T.st(h, v); }
template <bool G> __device__ __forceinline__ uint32_t tab_enc(const TabOv<G> &T, int32_t p) { return (T.epoch << 12) | (uint32_t)(p - T.start); }
template <bool G> __device__ __forceinline__ int32_t tab_dec(const TabOv<G> &, uint32_t raw) { return (int32_t)raw - 1; }
__device__ __forceinline__ uint32_t tab_raw(const TabG32 &T, uint32_t h) { return (uint32_t)__ldcg(T.t + h); }
__device__ __forceinline__ void tab_set_raw(TabG32 &T, uint32_t h, uint32_t v) { __stcg(T.t + h, (int32_t)v); }
__device__ __forceinline__ uint32_t tab_enc(const TabG32 &, int32_t p) { return (uint32_t)(p + 1); }
__device__ __forceinline__ int32_t tab_dec(const TabG32 &, uint32_t raw) { return (int32_t)raw - 1; }
__device__ __forceinline__ uint32_t tab_raw(const Tab32 &T, uint32_t h) { return (uint32_t)T.t[h]; }
__device__ __forceinline__ void tab_set_raw(Tab32 &T, uint32_t h, uint32_t v) { T.t[h] = (int32_t)v; }
__device__ __forceinline__ uint32_t tab_enc(const Tab32 &, int32_t p) { return (uint32_t)(p + 1); }
__device__ __forceinline__ int32_t tab_dec(const Tab32 &, uint32_t raw) { return (int32_t)raw - 1; }

// 4-byte cp.async (LDGSTS) into shared memory; src_size 0 zero-fills without touching global memory.
__device__ __forceinline__ void cp_async4(uint32_t smem_addr, const void *gptr, uint32_t src_size) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(smem_addr), "l"(gptr), "r"(src_size) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

constexpr int kRingLines = 3;                      // forward ring: three 128-byte lines per warp
constexpr int kRingBytes = kRingLines * 128;

// aligned word at byte index `idx` (multiple of 4 in address terms) of a read-only global buffer, 0 outside [lo, hi)
__device__ __forceinline__ uint32_t ldg_word_guard(const uint8_t *base, int32_t idx, int32_t lo, int32_t hi) {
    return (idx >= lo && idx < hi) ? __ldg(reinterpret_cast<const uint32_t *>(base + idx)) : 0u;
}

// One LZ4 block by one warp, contiguous read-only global source (`base` = virtual index 0).
//
// Dense path ("window"): while the skip schedule still steps by 1 (searchMatchCount <= 96 for all 32 probes) the next 32
// probe positions are the 32 consecutive bytes w..w+31.  One pass
//   (A) builds every lane's 32 source bytes from a register-resident copy of the forward 128-byte lines (shuffles only),
//       looks all 32 slots up and issues every candidate's 9 words in one go (one L2 round trip per window); in the shadow
//       of those loads it inserts all 32 positions and reads the slots back: if every lane reads its own position there is
//       no same-slot pair inside the window, hence every lane's candidate is the table state from before the window
//       whatever the parse does inside it; then verifies the candidates and pre-extends verified ones to 32 bytes,
//   (B) walks the window in registers only (first hit at or after `cur`, jump behind the match), handing every match head
//       its output offset,
//   (C) emits in parallel: a literal lane stores its own byte, a head lane its own token / length bytes / offset.  Literal
//       lanes behind the last match are written provisionally (their sequence is still open); only a run that reaches 15
//       literals needs them moved, which re-copies from memory (3 % of sequences on text),
//   (D) un-inserts the positions the serial loop would never have probed (inside matches).
// A window with a same-slot pair, the sparse schedule and the last bytes of a block fall back to the batch step of
// compress_block_warp (exact for every case).
// Parse state of one block (what the serial loop carries from probe to probe, plus the output cursor).
struct SpanState {
    int32_t sIndex, anchor;
    uint32_t smc;                // searchMatchCount
    uint32_t D;                  // output offset of the open sequence's token
    uint32_t pend;               // literals of the open sequence already stored provisionally at out[D+1 ..)
    int32_t head;                // out: position of the match that made the span stop (kSpanStopped)
};

// Runs the single-warp parse of the block [start, start + len) from state `st`.
//   limit >= start + len : parses to the end of the block, emits the final literals, returns the compressed size.
//   limit <  start + len : (segment-parallel compression) stops right after the first sequence whose match starts at a
//                          position >= limit -- a point defined by the serial parse alone, so it is the same however the
//                          probes were batched, and no literals are pending there -- leaves that state in `st`
//                          (st.D = bytes emitted, st.head = that match's position) and returns kSpanStopped.  If the block
//                          has no such sequence it is finished as above.
// kEmit == false runs the identical parse without writing output (warm-up of a speculative segment).
constexpr uint32_t kSpanStopped = 0xFFFFFFFFu;
// kSplit: the source is `pre[0, plen)` ++ block, stored apart (shared dictionary prefix of config 4); `base` is then the
// block's pointer minus plen, valid for indices >= plen only.
template <class Tab, bool kEmit, bool kSplit = false>
__device__ uint32_t compress_span_warp(const uint8_t *__restrict__ base, const int32_t start, const int32_t len, Tab &T,
                                       uint8_t *const out, uint32_t *const ring /* kRingBytes of shared memory */,
                                       SpanState &st, const int32_t limit, const uint8_t *__restrict__ pre = nullptr,
                                       const int32_t plen = 0) {
    const uint32_t lane = lane_id();
    const uint32_t lt = (1u << lane) - 1u;
    const int32_t sEnd = start + len;
    const int32_t mflimit = sEnd - 12;
    const int32_t matchLimit = sEnd - 5;
    int32_t sIndex = st.sIndex, anchor = st.anchor;
    uint32_t smc = st.smc;
    uint32_t D = st.D;
    uint32_t pend = st.pend;
    struct SrcSel {                              // unaligned 4-byte loads at virtual index v (match extension, batch step)
        const uint8_t *base, *pre; int32_t plen;
        __device__ __forceinline__ uint32_t ld32(int32_t v) const {
            if (!kSplit || v >= plen) return ld32u(base + v);
            if (v + 4 <= plen) return ld32u(pre + v);
            uint32_t r = 0;
            for (int k = 0; k < 4; ++k) r |= (uint32_t)(v + k < plen ? pre[v + k] : base[v + k]) << (8 * k);
            return r;
        }
        __device__ __forceinline__ const uint8_t *lit_ptr(int32_t v) const { return base + v; }
    } S{base, pre, plen};

    // forward ring: the 128-byte lines around the window live in a 3-line shared-memory ring filled by cp.async one line
    // ahead of use (no registers, no scoreboard dependency between the prefetch and the window's own loads)
    const uintptr_t gaddr = reinterpret_cast<uintptr_t>(base);
    const int32_t wlo = start - (int32_t)((gaddr + (uint32_t)start) & 3u);   // first word holding block bytes
    const int32_t whi = sEnd;                                                  // words starting below sEnd hold block bytes
    const uint32_t ring_s = (uint32_t)__cvta_generic_to_shared(ring);
    const uint64_t line0 = (gaddr + (uint32_t)wlo) >> 7;                        // line of the block's first word
    uint32_t next_line = 0;                                                    // next line (relative to line0) to fetch
    bool ring_cold = true;
    PT_DECL

    while (sIndex < mflimit) {
        PT_MARK(0)
        if (smc <= 96u && sIndex + 67 <= sEnd && sIndex + 32 <= limit) {
            const int32_t w = sIndex;
            const uint32_t wmis = (uint32_t)((reinterpret_cast<uintptr_t>(base) + (uint32_t)w) & 3u);
            const int32_t wa = w - (int32_t)wmis;                                   // word-aligned window base
            const uintptr_t waddr = gaddr + (intptr_t)wa;
            const uint32_t L = (uint32_t)((waddr >> 7) - line0);                    // line holding wa, relative to line0
            if (ring_cold || next_line < L + 3u) {
                if (ring_cold || next_line < L) next_line = L;                      // first window / jumped past the ring
                ring_cold = false;
                const bool one_ahead = next_line > L + 1u;                          // this refill only fetches line L+2
                do {
                    const int32_t idx = wlo - (int32_t)((gaddr + (uint32_t)wlo) & 127u) + (int32_t)(next_line << 7) + 4 * (int32_t)lane;
                    const bool in = idx >= wlo && idx < whi;
                    cp_async4(ring_s + (next_line % (uint32_t)kRingLines) * 128u + 4u * lane, base + (in ? idx : wlo), in ? 4u : 0u);
                    cp_async_commit();
                    ++next_line;
                } while (next_line < L + 3u);
                if (one_ahead) cp_async_wait<1>(); else cp_async_wait<0>();        // lines L and L+1 have landed
                __syncwarp();
            }
            PT_MARK(1)
            // ---- (A) source bytes, lookup, candidate loads
            const uint32_t wo = (uint32_t)(waddr & 127u) / 4u + lane;             // word offset from the start of line L
            const uint32_t Tw = ring[((L + (wo >> 5)) % (uint32_t)kRingLines) * 32u + (wo & 31u)];   // word (wa/4 + lane)
            const int32_t p = w + (int32_t)lane;
            const uint32_t o = wmis + lane, wi = o >> 2, sh = (o & 3u) * 8u;
            uint32_t tw[9];
#pragma unroll
            for (int k = 0; k < 9; ++k) tw[k] = __shfl_sync(FULL, Tw, wi + k);
            uint32_t Sw[8];                                                         // bytes p .. p+31
#pragma unroll
            for (int k = 0; k < 8; ++k) Sw[k] = __funnelshift_r(tw[k], tw[k + 1], sh);
            const uint32_t h = (Sw[0] * 2654435761u) >> 18;
            PT_USE(h) PT_MARK(12)
            const uint32_t old = tab_raw(T, h);
            const int32_t cand = tab_dec(T, old);
            const bool ok = cand >= 0 && cand != p && (((uint32_t)(p - cand)) >> 16) == 0;
            PT_USE(ok) PT_MARK(13)
            // candidate bytes cand .. cand+35 as three aligned 16-byte loads (3 L1 wavefronts per lane instead of 9)
            uint4 q0 = make_uint4(0, 0, 0, 0), q1 = q0, q2 = q0;
            uint32_t cs = 0;
            // split source: a candidate whose 48-byte read would leave the prefix (or start before it) sends the window to
            // the batch step, which reads byte-exact across the seam
            const bool seam = kSplit && ok && cand < plen && (cand + 48 > plen || cand < 16);
            if (ok && !seam) {              // cand + 35 < p + 35 <= w + 66 < sEnd, and the 16-byte granules holding them
                const uint8_t *cb = (kSplit && cand < plen) ? pre + cand : base + cand;
                cs = (uint32_t)(reinterpret_cast<uintptr_t>(cb) & 15u);
                const uint4 *cq = reinterpret_cast<const uint4 *>(cb - cs);
                q0 = __ldg(cq); q1 = __ldg(cq + 1);
                if (cs + 36u > 32u) q2 = __ldg(cq + 2);
            }
            PT_MARK(2)
            // two lanes of the window in one slot?  Then a later lane's candidate depends on the parse -> batch step.
            // Nothing is inserted yet, so the table is still the exact pre-window state either way.
            const uint32_t mine = tab_enc(T, p);
            const uint32_t conflict = __ballot_sync(FULL, __match_any_sync(FULL, h) != (1u << lane) || seam);
            PT_MARK(3)
            if (conflict) {
                PT_COUNT(10, 1)
            } else {
                bool hit = false;
                int32_t ml = 0;
                if (ok) {
                    // words at byte offset cs of (q0,q1,q2): shift by whole words with two select levels, then by bits
                    uint32_t v[12] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x, q2.y, q2.z, q2.w};
                    if (cs & 8u) {
#pragma unroll
                        for (int k = 0; k < 10; ++k) v[k] = v[k + 2];
                    }
                    if (cs & 4u) {
#pragma unroll
                        for (int k = 0; k < 9; ++k) v[k] = v[k + 1];
                    }
                    const uint32_t csh = (cs & 3u) * 8u;
                    if (__funnelshift_r(v[0], v[1], csh) == Sw[0]) {
                        hit = true;
                        int32_t n = 28;
#pragma unroll
                        for (int k = 7; k >= 1; --k) {
                            const uint32_t x = Sw[k] ^ __funnelshift_r(v[k], v[k + 1], csh);
                            if (x) n = 4 * (k - 1) + ((__ffs(x) - 1) >> 3);
                        }
                        const int32_t lim = matchLimit - p;          // >= 31 here
                        ml = 4 + n;
                        ml = ml < lim ? ml : lim;
                    }
                }
                PT_MARK(4)
                // ---- (B) resolve
                const uint32_t hm = __ballot_sync(FULL, hit);
                const int32_t a_rel0 = anchor - w;               // <= 0: literals pending from earlier windows
                int32_t a_rel = a_rel0;
                uint32_t cur = 0, heads = 0, inside = 0, smc_cur = smc;
                uint32_t myD = 0, myLit = 0, myMl = 0;
                while (cur < 32u) {
                    const uint32_t m = hm & (FULL << cur);
                    if (!m) break;
                    const int hl = __ffs(m) - 1;
                    int32_t mlh = __shfl_sync(FULL, ml, hl);
                    const int32_t s0 = w + hl;
                    if (mlh == 32 && matchLimit - s0 > 32) {
                        // long match: continue cooperatively, 128 bytes per round
                        const int32_t m0 = __shfl_sync(FULL, cand, hl);
                        for (int32_t eb = 32;; eb += 128) {
                            const int32_t q = s0 + eb + 4 * (int32_t)lane;
                            int32_t nv = matchLimit - q;
                            nv = nv > 4 ? 4 : nv;
                            int32_t eq = 0;
                            if (nv > 0) {
                                const uint32_t x = S.ld32(q) ^ S.ld32(m0 + eb + 4 * (int32_t)lane);
                                eq = x ? ((__ffs(x) - 1) >> 3) : 4;
                                eq = eq < nv ? eq : nv;
                            }
                            const uint32_t stop = __ballot_sync(FULL, eq < 4);
                            if (stop) {
                                const int l = __ffs(stop) - 1;
                                mlh = eb + 4 * l + __shfl_sync(FULL, eq, l);
                                break;
                            }
                        }
                    }
                    const uint32_t lit = (uint32_t)(hl - a_rel);
                    const uint32_t code = (uint32_t)(mlh - 4);
                    uint32_t litx = 0, mlx = code >= 15u;            // a match inside the window is <= 32 bytes: one length byte at most
                    if (lit >= 15u) litx = 1u + (lit - 15u) / 255u;  // uniform and rare (3 % of sequences on text)
                    if (code >= 15u + 255u) mlx = 1u + (code - 15u) / 255u;     // long match (continued above)
                    if (lane == (uint32_t)hl) { myD = D; myLit = lit; myMl = (uint32_t)mlh; }
                    D += 3u + litx + lit + mlx;
                    heads |= 1u << hl;
                    a_rel = hl + mlh;
                    cur = (uint32_t)a_rel;
                    inside |= (cur < 32u ? (1u << cur) : 0u) - (2u << hl);      // bits hl+1 .. cur-1 (to the top when the match leaves the window)
                    smc_cur = 67;
                }
                PT_MARK(5)
                // ---- (D) insert exactly the positions the serial loop probed: every lane of the window that is not inside a
                //      match (heads and literals; lanes behind the last match are literals).  One store per probed lane, no
                //      speculative insert to undo.
                if (!((inside >> lane) & 1u)) tab_set_raw(T, h, mine);
                // ---- (C) parallel emission
                if (heads) {
                  if (kEmit) {
                    const int fh = __ffs(heads) - 1, lh = 31 - __clz(heads);
                    const uint32_t lit0 = __shfl_sync(FULL, myLit, fh);
                    if (a_rel0 < 0 && lit0 >= 15u) {
                        // the open run reached 15 literals: its provisional bytes sit one length field too low -> re-copy them
                        const uint32_t D0 = __shfl_sync(FULL, myD, fh);
                        warp_copy(out + D0 + 2u + (lit0 - 15u) / 255u, base + anchor, (uint32_t)(-a_rel0), lane);
                    }
                    const uint32_t above = (heads >> lane) >> 1;
                    const int nh = (int)lane + __ffs(above);                 // next head above this lane (if any)
                    const uint32_t Dn = __shfl_sync(FULL, myD, nh & 31), litn = __shfl_sync(FULL, myLit, nh & 31);
                    const uint32_t is_lit = ~inside & ~heads & ((1u << lh) - 1u);
                    if ((is_lit >> lane) & 1u) {
                        const uint32_t litx = litn >= 15u ? 1u + (litn - 15u) / 255u : 0u;
                        out[Dn + 1u + litx + litn - (uint32_t)(nh - (int)lane)] = (uint8_t)Sw[0];
                    }
                    if ((heads >> lane) & 1u) {
                        uint8_t *q = out + myD;
                        const uint32_t code = myMl - 4u;
                        q[0] = (uint8_t)(((myLit < 15u ? myLit : 15u) << 4) | (code < 15u ? code : 15u));
                        q += 1;
                        if (myLit >= 15u) {
                            uint32_t rest = myLit - 15u;
                            while (rest >= 255u) { *q++ = 255; rest -= 255u; }
                            *q++ = (uint8_t)rest;
                        }
                        q += myLit;
                        const uint32_t offset = (uint32_t)(p - cand);
                        q[0] = (uint8_t)offset;
                        q[1] = (uint8_t)(offset >> 8);
                        if (code >= 15u) {
                            uint32_t rest = code - 15u;
                            q += 2;
                            while (rest >= 255u) { *q++ = 255; rest -= 255u; }
                            *q = (uint8_t)rest;
                        }
                    }
                  }
                    anchor = w + a_rel;
                    pend = 0;
                    smc = 67;
                }
                PT_MARK(6)
                // literal lanes behind the last match: provisional bytes of the still-open sequence
                if (cur < 32u) {
                    if (kEmit && lane >= cur) out[D + 1u + pend + (lane - cur)] = (uint8_t)Sw[0];
                    pend += 32u - cur;
                    smc = smc_cur + (32u - cur);
                    cur = 32;
                }
                __syncwarp();
                sIndex = w + (int32_t)cur;
                PT_MARK(7)
                PT_COUNT(9, 1)
                continue;
            }
        }

        // ---- batch step (identical to compress_block_warp's loop body)
        const uint32_t base_sum = skip_sum(smc);
        const int32_t p = sIndex + (int32_t)(skip_sum(smc + lane) - base_sum);
        const bool valid = p < mflimit;
        uint32_t seq = 0, h = 0x10000u + lane;
        int32_t cand = -1;
        if (valid) {
            seq = S.ld32(p);
            h = (seq * 2654435761u) >> 18;
            cand = T.get(h);
        }
        const uint32_t same = __match_any_sync(FULL, h);
        const uint32_t prev = same & lt;
        const int j = prev ? 31 - __clz(prev) : (int)lane;
        const int32_t pj = __shfl_sync(FULL, p, j);
        const uint32_t sj = __shfl_sync(FULL, seq, j);
        uint32_t cseq = sj;
        if (prev) cand = pj;
        const bool ok = valid && cand >= 0 && cand != p && (((uint32_t)(p - cand)) >> 16) == 0;
        if (ok && !prev) cseq = S.ld32(cand);
        const bool hit = ok && cseq == seq;
        const uint32_t hits = __ballot_sync(FULL, hit);
        const uint32_t vmask = __ballot_sync(FULL, valid);
        const int hl = __ffs(hits) - 1;
        const uint32_t commit = hits ? ((2u << hl) - 1u) : vmask;
        if (((commit >> lane) & 1u) && ((same & commit) >> lane) == 1u) T.put(h, p);
        __syncwarp();
        if (!hits) {
            if (vmask != FULL) break;                            // ran into mflimit: loop ends
            sIndex += (int32_t)(skip_sum(smc + 32u) - base_sum);
            smc += 32u;
            continue;
        }
        const int32_t s0 = __shfl_sync(FULL, p, hl);
        const int32_t m0 = __shfl_sync(FULL, cand, hl);
        smc = 67;
        int32_t ml;
        for (int32_t eb = 4;; eb += 128) {
            const int32_t q = s0 + eb + 4 * (int32_t)lane;
            int32_t nv = matchLimit - q;
            nv = nv > 4 ? 4 : nv;
            int32_t eq = 0;
            if (nv > 0) {
                const uint32_t x = S.ld32(q) ^ S.ld32(m0 + eb + 4 * (int32_t)lane);
                eq = x ? ((__ffs(x) - 1) >> 3) : 4;
                eq = eq < nv ? eq : nv;
            }
            const uint32_t stop = __ballot_sync(FULL, eq < 4);
            if (stop) {
                const int l = __ffs(stop) - 1;
                ml = eb + 4 * l + __shfl_sync(FULL, eq, l);
                break;
            }
        }
        if (kEmit) {
            const uint32_t code = (uint32_t)(ml - 4);
            uint8_t *d = emit_literals(out + D, S, anchor, (uint32_t)(s0 - anchor), code < 15u ? code : 15u, lane);
            const uint32_t offset = (uint32_t)(s0 - m0);
            if (lane == 0) { d[0] = (uint8_t)offset; d[1] = (uint8_t)(offset >> 8); }
            d += 2;
            if (code >= 15u) {
                const uint32_t rest = code - 15u, n255 = rest / 255u;
                for (uint32_t i = lane; i < n255; i += 32) d[i] = 255;
                if (lane == 0) d[n255] = (uint8_t)(rest - n255 * 255u);
                d += n255 + 1;
            }
            D = (uint32_t)(d - out);
        }
        pend = 0;
        sIndex = anchor = s0 + ml;
        PT_MARK(8)
        PT_COUNT(11, 1)
        if (s0 >= limit) {                   // first sequence that starts in the next segment: hand the state over
            st.sIndex = sIndex; st.anchor = anchor; st.smc = smc; st.D = D; st.pend = 0; st.head = s0;
            PT_FLUSH
            return kSpanStopped;
        }
    }
    PT_FLUSH
    if (!kEmit) return 0u;
    uint8_t *d = emit_literals(out + D, S, anchor, (uint32_t)(sEnd - anchor), 0u, lane);
    return (uint32_t)(d - out);
}

// One LZ4 block by one warp, from a fresh parse state (see compress_span_warp).
template <class Tab>
__device__ __forceinline__ uint32_t compress_block_warp_v2(const uint8_t *__restrict__ base, const int32_t start, const int32_t len,
                                                           Tab &T, uint8_t *const out, uint32_t *const ring) {
    SpanState st{start, start, 67u, 0u, 0u, -1};
    return compress_span_warp<Tab, true>(base, start, len, T, out, ring, st, INT_MAX);
}

}  // namespace dlz4
#include "dlz4_wide.cuh"
namespace dlz4 {

// ------------------------------------------------------------------ compress kernels
__device__ __forceinline__ uint32_t next_block(uint32_t *counter, uint32_t lane) {
    uint32_t b = 0;
    if (lane == 0) b = atomicAdd(counter, 1u);
    return __shfl_sync(FULL, b, 0);
}

}  // namespace dlz4
#include "dlz4_parse.cuh"
#include "dlz4_pw.cuh"
namespace dlz4 {

// Round-1 kernel for fresh blocks <= 64 KiB (kept as the A/B baseline, DLZ4_SPLIT=0).  The parse is latency-bound (one dependent chain per block) and
// shared memory holds only 7 tables per SM, so most chains keep their table in L2-resident global scratch instead
// (TabG16): a CTA is 7 warps = 1 chain on a shared-memory table + 6 chains on L2 tables, and 4 such CTAs share an SM
// (28 chains, 64 registers each).  Small CTAs let the chunks of the host pipeline -- launched on different streams --
// co-reside on an SM.  `active_warps` < 7 spreads a small batch over more SMs, shared-memory warp first.
constexpr int kHyWarps = 7;                        // warps per CTA: warp 0 shared-memory table, warps 1..6 L2 tables
constexpr int kHyGlWarps = kHyWarps - 1;
constexpr int kHyCtasPerSm = 4;
constexpr int kHySmemBytes = kHashEntries * 2 + kHyWarps * kRingBytes;
__global__ void __launch_bounds__(kHyWarps * 32, kHyCtasPerSm)
k_compress_fresh16h(const uint8_t *__restrict__ src, const uint64_t *__restrict__ src_off,
                    const uint32_t *__restrict__ src_len, uint32_t nblocks, uint8_t *__restrict__ dst,
                    const uint64_t *__restrict__ dst_off, uint32_t *__restrict__ comp_len, uint32_t *counter,
                    uint16_t *gtabs /* gridDim.x * kHyGlWarps tables */, uint32_t active_warps) {
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    if (warp >= active_warps) return;
    uint32_t *ring = reinterpret_cast<uint32_t *>(smem + kHashEntries * 2 + warp * kRingBytes);
    const bool in_smem = warp == 0;
    uint16_t *tab = in_smem ? reinterpret_cast<uint16_t *>(smem)
                            : gtabs + ((size_t)blockIdx.x * kHyGlWarps + (warp - 1)) * kHashEntries;
    uint32_t epoch = 15;                           // small-block epoch (Tab12e); 15 forces a clear before the first use
    for (;;) {
        const uint32_t b = next_block(counter, lane);
        if (b >= nblocks) break;
        const uint32_t len = src_len[b];
        if (len > 65536u) { if (lane == 0) comp_len[b] = 0xFFFFFFFFu; continue; }
        uint4 *t4 = reinterpret_cast<uint4 *>(tab);
        const bool small = len <= 4096u;
        if (!small || ++epoch > 15u) {
            if (in_smem) { for (uint32_t i = lane; i < kHashEntries * 2 / 16; i += 32) t4[i] = make_uint4(0, 0, 0, 0); }
            else { for (uint32_t i = lane; i < kHashEntries * 2 / 16; i += 32) __stcg(t4 + i, make_uint4(0, 0, 0, 0)); }
            __syncwarp();
            epoch = small ? 1u : 15u;              // a 16-bit-position block leaves arbitrary epochs behind: clear again next time
        }
        uint32_t c;
        if (small) {
            if (in_smem) { Tab12e<false> T{tab, 0, epoch}; c = compress_block_warp_v2(src + src_off[b], 0, (int32_t)len, T, dst + dst_off[b], ring); }
            else { Tab12e<true> T{tab, 0, epoch}; c = compress_block_warp_v2(src + src_off[b], 0, (int32_t)len, T, dst + dst_off[b], ring); }
        } else if (in_smem) {
            Tab16 T{tab, 0};
            c = compress_block_warp_v2(src + src_off[b], 0, (int32_t)len, T, dst + dst_off[b], ring);
        } else {
            TabG16 T{tab, 0};
            c = compress_block_warp_v2(src + src_off[b], 0, (int32_t)len, T, dst + dst_off[b], ring);
        }
        if (lane == 0) comp_len[b] = c;
        __syncwarp();
    }
}

// Blocks of <= 4096 bytes behind a shared prefix, all starting from the same initial table (TabOv).  Same CTA shape as
// k_compress_fresh16h: warp 0 keeps its overlay in shared memory, warps 1..6 in L2-resident global scratch.
__global__ void __launch_bounds__(kHyWarps * 32, kHyCtasPerSm)
k_compress_overlay(const uint8_t *__restrict__ src, const uint64_t *__restrict__ src_off, const uint32_t *__restrict__ src_len,
                   uint32_t nblocks, const uint8_t *__restrict__ prefix, uint32_t prefix_len, const int32_t *__restrict__ init_table,
                   uint8_t *__restrict__ dst, const uint64_t *__restrict__ dst_off, uint32_t *__restrict__ comp_len, uint32_t *counter,
                   uint16_t *gtabs, uint32_t active_warps) {
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    if (warp >= active_warps) return;
    uint32_t *ring = reinterpret_cast<uint32_t *>(smem + kHashEntries * 2 + warp * kRingBytes);
    const bool in_smem = warp == 0;
    uint16_t *tab = in_smem ? reinterpret_cast<uint16_t *>(smem)
                            : gtabs + ((size_t)blockIdx.x * kHyGlWarps + (warp - 1)) * kHashEntries;
    const int32_t plen = (int32_t)prefix_len;
    uint32_t epoch = 15;
    for (;;) {
        const uint32_t b = next_block(counter, lane);
        if (b >= nblocks) break;
        const uint32_t len = src_len[b];
        if (len > 4096u) { if (lane == 0) comp_len[b] = 0xFFFFFFFFu; continue; }
        if (++epoch > 15u) {
            uint4 *t4 = reinterpret_cast<uint4 *>(tab);
            if (in_smem) { for (uint32_t i = lane; i < kHashEntries * 2 / 16; i += 32) t4[i] = make_uint4(0, 0, 0, 0); }
            else { for (uint32_t i = lane; i < kHashEntries * 2 / 16; i += 32) __stcg(t4 + i, make_uint4(0, 0, 0, 0)); }
            __syncwarp();
            epoch = 1;
        }
        const uint8_t *vbase = src + src_off[b] - plen;           // virtual index plen = first byte of the message
        SpanState st{plen, plen, 67u, 0u, 0u, -1};
        uint32_t c;
        if (in_smem) {
            TabOv<false> T{tab, init_table, plen, epoch};
            c = compress_span_warp<TabOv<false>, true, true>(vbase, plen, (int32_t)len, T, dst + dst_off[b], ring, st, INT_MAX, prefix, plen);
        } else {
            TabOv<true> T{tab, init_table, plen, epoch};
            c = compress_span_warp<TabOv<true>, true, true>(vbase, plen, (int32_t)len, T, dst + dst_off[b], ring, st, INT_MAX, prefix, plen);
        }
        if (lane == 0) comp_len[b] = c;
        __syncwarp();
    }
}

// Independent blocks of any size, optional shared prefix and initial table: the reference's Int32 table,
// 64 KiB of shared memory per warp.
template <int WARPS>
__global__ void __launch_bounds__(WARPS * 32, 1)
k_compress_generic32(const uint8_t *__restrict__ src, const uint64_t *__restrict__ src_off,
                     const uint32_t *__restrict__ src_len, uint32_t nblocks, const uint8_t *__restrict__ prefix,
                     uint32_t prefix_len, const int32_t *__restrict__ init_table, uint8_t *__restrict__ dst,
                     const uint64_t *__restrict__ dst_off, uint32_t *__restrict__ comp_len, uint32_t *counter) {
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    int32_t *tab = reinterpret_cast<int32_t *>(smem) + warp * kHashEntries;
    uint32_t *ring = reinterpret_cast<uint32_t *>(smem + WARPS * kHashEntries * 4 + warp * kRingBytes);
    for (;;) {
        const uint32_t b = next_block(counter, lane);
        if (b >= nblocks) break;
        uint4 *t4 = reinterpret_cast<uint4 *>(tab);
        if (init_table) {
            const uint4 *i4 = reinterpret_cast<const uint4 *>(init_table);
            for (uint32_t i = lane; i < kHashEntries * 4 / 16; i += 32) t4[i] = i4[i];
        } else {
            for (uint32_t i = lane; i < kHashEntries * 4 / 16; i += 32) t4[i] = make_uint4(0, 0, 0, 0);
        }
        __syncwarp();
        Tab32 T{tab};
        uint32_t c;
        if (prefix_len) {
            SrcSplit S{prefix, (int32_t)prefix_len, src + src_off[b]};
            c = compress_block_warp(S, (int32_t)prefix_len, (int32_t)src_len[b], T, dst + dst_off[b]);
        } else {
            c = compress_block_warp_v2(src + src_off[b], 0, (int32_t)src_len[b], T, dst + dst_off[b], ring);
        }
        if (lane == 0) comp_len[b] = c;
        __syncwarp();
    }
}

// ------------------------------------------------------------------ segment-parallel compression (large blocks, linked chains)
// The greedy parse forgets its past: a table entry older than 65535 bytes is rejected forever (blockCompress.js:62), and
// slots are overwritten as the parse goes on, so a parse started from an EMPTY table a few hundred KiB early converges to
// exactly the state of the true parse (tools/resync_stats.c: 384 KiB of warm-up suffice in 97 %, 512 KiB in > 99 % of the
// cases on the synthetic corpora).  A chain of blocks that carry the table (linked blocks, bufferCompress.js:182,219,234)
// or one large block is therefore cut into segments; one warp per segment
//   1. warms up: parses [seg_begin - W, seg_begin) from an empty table without output, up to the first sequence that
//      starts at or behind seg_begin, and snapshots that state (next position, head, whole table),
//   2. parses on with output up to the first sequence that starts at or behind seg_end; the state it ends in stays in its
//      table buffer.
// k_seg_verify then compares every segment's snapshot with its predecessor's end state (entries older than 65535 bytes count
// as empty).  Equal states make the speculative segment exact by induction from the chain's first segment, which starts
// from the true initial table; a segment whose snapshot differs is re-run from its predecessor's end state (host loop),
// so the bytes are always those of the serial loop -- speculation only decides how much runs in parallel.
struct SegJob {
    int32_t chain_start, chain_end;      // the chain: consecutive blocks of block_size from chain_start (the last may be short)
    int32_t warm_begin;                  // where the warm-up parse starts (== seg_begin: no warm-up, exact start)
    int32_t seg_begin, seg_end;
    uint32_t first_slot;                 // piece slot of the first block this segment overlaps
    uint32_t first_block;                // global index of that block
    uint32_t flags;                      // kSegFirst | kSegLast | kSegRerun
};
enum : uint32_t { kSegFirst = 1u, kSegLast = 2u, kSegRerun = 4u,
                  kSegCont = 8u,       // first launch: starts from its predecessor's end state (same warp ran it just before)
                  kSegMore = 16u };    // first launch: the warp goes on with the next segment (which has kSegCont)
struct SegState { int32_t s, head; };    // next probe position (== anchor, searchMatchCount == 67 there) and the stopping head
                                         // (-1: fresh start of the block that begins at s)
// offset of the piece that starts at source offset x of its block (pieces of one block never overlap: a run of complete
// sequences over n >= 4 source bytes takes at most n + n/255 bytes)
__device__ __host__ __forceinline__ uint64_t seg_piece_offset(uint64_t x) { return x + (x >> 3); }

template <class Tab, bool kEmit>
__device__ __forceinline__ void seg_run(const uint8_t *__restrict__ base, const SegJob &J, int32_t block_size, Tab &T,
                                        uint32_t *ring, SegState &S, int32_t limit, uint8_t *blockbuf, uint64_t blockbuf_stride,
                                        uint32_t *piece_off, uint32_t *piece_len, int32_t stop_fresh_at) {
    // Runs blocks from state S until a span stops at `limit` (S = hand-over state) or a fresh block start >= stop_fresh_at
    // (or the chain's end) is reached.
    const uint32_t lane = lane_id();
    for (;;) {
        if (S.s >= J.chain_end) break;
        const int32_t bi = (S.s - J.chain_start) / block_size;
        const int32_t bstart = J.chain_start + bi * block_size;
        const int32_t blen = (J.chain_end - bstart) < block_size ? (J.chain_end - bstart) : block_size;
        const bool fresh = S.head < 0;
        if (fresh && bstart >= stop_fresh_at) break;
        if (!fresh && S.head >= limit) break;                    // the hand-over sequence already lies behind this segment
        SpanState st{S.s, S.s, 67u, 0u, 0u, -1};
        uint32_t r;
        if (kEmit) {
            const int32_t bfirst = (J.seg_begin - J.chain_start) / block_size;
            const uint32_t slot = J.first_slot + (uint32_t)(bi - bfirst);
            const uint32_t off = (uint32_t)seg_piece_offset((uint64_t)(S.s - bstart));
            uint8_t *out = blockbuf + (uint64_t)(J.first_block + (uint32_t)(bi - bfirst)) * blockbuf_stride + off;
            r = compress_span_warp<Tab, true>(base, bstart, blen, T, out, ring, st, limit);
            if (lane == 0) { piece_off[slot] = off; piece_len[slot] = r == kSpanStopped ? st.D : r; }
        } else {
            r = compress_span_warp<Tab, false>(base, bstart, blen, T, nullptr, ring, st, limit);
        }
        if (r == kSpanStopped) { S.s = st.sIndex; S.head = st.head; break; }
        S.s = bstart + blen; S.head = -1;                        // block finished: the next one starts fresh (table carried)
    }
}

// One segment by one warp.  kSmem: the live table is in shared memory (twice as fast a chain; 3 per SM) and is written to
// tables[j] at the end, where the verification and a re-run of the successor read it; otherwise tables[j] itself is live.
template <class Tab, bool kSmem>
__device__ __forceinline__ void seg_job(const uint8_t *__restrict__ base, const SegJob &J, uint32_t j, int32_t block_size,
                                        const int32_t *__restrict__ init_table, int32_t *live, int32_t *tables, int32_t *snaps,
                                        SegState *snap_state, SegState *end_state, uint8_t *blockbuf, uint64_t blockbuf_stride,
                                        uint32_t *piece_off, uint32_t *piece_len, uint32_t *ring) {
    const uint32_t lane = lane_id();
    uint4 *l4 = reinterpret_cast<uint4 *>(live);
    auto put = [&](uint32_t i, const uint4 &v) { if (kSmem) l4[i] = v; else __stcg(l4 + i, v); };
    auto get = [&](uint32_t i) -> uint4 { return kSmem ? l4[i] : __ldcg(l4 + i); };
    constexpr uint32_t kVec = kHashEntries * 4 / 16;
    Tab T{live};
    SegState S;
    if (J.flags & (kSegRerun | kSegCont)) {
        // exact start: the predecessor's end state (its table buffer is final, nobody writes it during this launch --
        // a re-run -- or this warp has just written it -- a group of segments run back to back)
        const uint4 *p4 = reinterpret_cast<const uint4 *>(tables + (size_t)(j - 1) * kHashEntries);
        uint4 *s4 = reinterpret_cast<uint4 *>(snaps + (size_t)j * kHashEntries);
        for (uint32_t i = lane; i < kVec; i += 32) { const uint4 v = __ldcg(p4 + i); put(i, v); __stcg(s4 + i, v); }
        S = end_state[j - 1];
        if (lane == 0) snap_state[j] = S;                        // the start is now exact as long as the predecessor's end stands
        __syncwarp();
    } else if (J.flags & kSegFirst) {
        if (init_table && j == 0) {
            const uint4 *i4 = reinterpret_cast<const uint4 *>(init_table);
            for (uint32_t i = lane; i < kVec; i += 32) put(i, i4[i]);
        } else {
            for (uint32_t i = lane; i < kVec; i += 32) put(i, make_uint4(0, 0, 0, 0));
        }
        S.s = J.seg_begin; S.head = -1;
        __syncwarp();
    } else {
        for (uint32_t i = lane; i < kVec; i += 32) put(i, make_uint4(0, 0, 0, 0));
        __syncwarp();
        S.s = J.warm_begin; S.head = -1;
        seg_run<Tab, false>(base, J, block_size, T, ring, S, J.seg_begin, nullptr, 0, nullptr, nullptr, J.seg_begin);
        __syncwarp();
        uint4 *s4 = reinterpret_cast<uint4 *>(snaps + (size_t)j * kHashEntries);
        for (uint32_t i = lane; i < kVec; i += 32) __stcg(s4 + i, get(i));
        if (lane == 0) snap_state[j] = S;
    }
    const bool last = (J.flags & kSegLast) != 0;
    seg_run<Tab, true>(base, J, block_size, T, ring, S, last ? INT_MAX : J.seg_end, blockbuf, blockbuf_stride, piece_off, piece_len,
                       last ? INT_MAX : J.seg_end);
    if (lane == 0) end_state[j] = S;
    __syncwarp();
    if (kSmem) {
        uint4 *t4 = reinterpret_cast<uint4 *>(tables + (size_t)j * kHashEntries);
        for (uint32_t i = lane; i < kVec; i += 32) __stcg(t4 + i, l4[i]);
        __syncwarp();
    }
}

// Does the start state segment j+1 ran from (snapshot) differ from the end state of segment j?  (Same rule as k_seg_verify:
// entries older than 65535 bytes count as empty.)  Whole warp.
__device__ __forceinline__ bool seg_differs(const SegState *snap_next, const SegState *end_prev, const int32_t *tab_snap,
                                            const int32_t *tab_end, uint32_t lane) {
    const int2 a = __ldcg(reinterpret_cast<const int2 *>(snap_next)), b = __ldcg(reinterpret_cast<const int2 *>(end_prev));
    int d = (a.x != b.x) | (a.y != b.y);
    const int32_t horizon = b.x - 65535;
    const int4 *A4 = reinterpret_cast<const int4 *>(tab_snap), *B4 = reinterpret_cast<const int4 *>(tab_end);
    auto norm = [&](int32_t v) { v -= 1; return v < horizon ? -1 : v; };
    for (uint32_t i = lane; i < kHashEntries / 4; i += 32) {
        const int4 x = __ldcg(A4 + i), y = __ldcg(B4 + i);
        d |= (norm(x.x) != norm(y.x)) | (norm(x.y) != norm(y.y)) | (norm(x.z) != norm(y.z)) | (norm(x.w) != norm(y.w));
    }
    return __any_sync(FULL, d) != 0;
}

constexpr int kSegWarps = 7;                       // warp 0: shared-memory table (64 KiB), warps 1..6: tables in L2
constexpr int kSegCtasPerSm = 3;
constexpr int kSegSmemBytes = kHashEntries * 4 + kSegWarps * kRingBytes;
__global__ void __launch_bounds__(kSegWarps * 32, kSegCtasPerSm)
k_compress_segments(const uint8_t *__restrict__ base, const SegJob *__restrict__ jobs, const uint32_t *__restrict__ job_list,
                    uint32_t njobs, int32_t block_size, const int32_t *__restrict__ init_table /* nullable: chain 0 */,
                    int32_t *tables, int32_t *snaps, SegState *snap_state, SegState *end_state,
                    uint8_t *blockbuf, uint64_t blockbuf_stride, uint32_t *piece_off, uint32_t *piece_len, uint32_t *counter,
                    uint32_t active_warps,
                    const uint32_t *landed /* nullable: flag per 2^land_shift input bytes, set once they are in memory */,
                    int32_t land_origin, uint32_t land_shift,
                    uint32_t nbig /* > 0: job_list[0, nbig) are heads of segment groups meant for the shared-memory warps */,
                    uint32_t follow /* first launch: a warp runs on through kSegMore */,
                    const uint8_t *chase_bad /* re-run launch: k_seg_verify's verdicts; a warp runs on while its new end state
                                                differs from the next segment's snapshot (nullable) */,
                    uint32_t total_jobs, uint32_t *chased /* count of segments re-run that way */) {
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    if (warp >= active_warps) return;
    uint32_t *ring = reinterpret_cast<uint32_t *>(smem + kHashEntries * 4 + warp * kRingBytes);
    for (;;) {
        uint32_t q;
        if (nbig) {
            // two queues (counter[0]: groups, counter[1]: single segments); a warp drains its own kind first
            const bool fast = warp == 0;
            const uint32_t n_own = fast ? nbig : njobs - nbig, n_other = njobs - n_own;
            q = next_block(counter + (fast ? 0 : 1), lane);
            if (q < n_own) {
                q += fast ? 0u : nbig;
            } else {
                q = next_block(counter + (fast ? 1 : 0), lane);
                if (q >= n_other) break;
                q += fast ? nbig : 0u;
            }
        } else {
            q = next_block(counter, lane);
            if (q >= njobs) break;
        }
        bool chasing = false;
        for (uint32_t j = job_list ? job_list[q] : q;; ++j) {
            SegJob J = jobs[j];
            if (chasing) J.flags |= kSegRerun;
            if (landed) {
                // the input is still arriving (chunked host-to-device copy on another stream, flags written in copy order):
                // wait for everything this segment can read -- up to the end of the block that holds seg_end, as far as the
                // stopping sequence's match may run
                int32_t need = J.chain_end;
                if (!(J.flags & kSegLast)) {
                    const int32_t be = J.chain_start + (J.seg_end - J.chain_start + block_size - 1) / block_size * block_size;
                    need = be < need ? be : need;
                }
                if (lane == 0) {
                    const volatile uint32_t *f = landed + ((uint32_t)(need - 1 - land_origin) >> land_shift);
                    const long long t0 = clock64();
                    while (*f == 0u) {
                        __nanosleep(500);
                        if (clock64() - t0 > (8ll << 30)) __trap();          // seconds without the copy: fail the call, do not hang
                    }
                    __threadfence_system();
                }
                __syncwarp();
            }
            {   // this run's pieces replace whatever an earlier run of the segment left in its slots
                const int32_t last_pos = (J.seg_end < J.chain_end ? J.seg_end : J.chain_end) - 1;
                const uint32_t nslots = (uint32_t)((last_pos - J.chain_start) / block_size - (J.seg_begin - J.chain_start) / block_size) + 1u;
                for (uint32_t i = lane; i < nslots; i += 32) piece_len[J.first_slot + i] = 0;
            }
            if (warp == 0)
                seg_job<Tab32, true>(base, J, j, block_size, init_table, reinterpret_cast<int32_t *>(smem), tables, snaps, snap_state, end_state,
                                     blockbuf, blockbuf_stride, piece_off, piece_len, ring);
            else
                seg_job<TabG32, false>(base, J, j, block_size, init_table, tables + (size_t)j * kHashEntries, tables, snaps, snap_state,
                                       end_state, blockbuf, blockbuf_stride, piece_off, piece_len, ring);
            __syncwarp();                        // the next segment reads this one's end state and table back
            if (follow) {
                if (!(J.flags & kSegMore)) break;
            } else if (chase_bad) {
                // re-run launch: go on into the successor while it did not start from the state this segment now ends in --
                // unless it heads this launch's list itself (bad, predecessor fine: another warp is on it)
                if (j + 1 >= total_jobs || (jobs[j + 1].flags & kSegFirst)) break;
                if (chase_bad[j + 1] && !chase_bad[j]) break;
                if (!seg_differs(snap_state + j + 1, end_state + j, snaps + (size_t)(j + 1) * kHashEntries,
                                 tables + (size_t)j * kHashEntries, lane)) break;
                chasing = true;
                if (lane == 0) atomicAdd(chased, 1u);
            } else {
                break;
            }
        }
    }
}

// bad[j] = 1 when segment j's warm-up snapshot differs from its predecessor's end state (j not first in its chain).
__global__ void __launch_bounds__(256)
k_seg_verify(const SegJob *__restrict__ jobs, uint32_t njobs, const int32_t *__restrict__ tables, const int32_t *__restrict__ snaps,
             const SegState *__restrict__ snap_state, const SegState *__restrict__ end_state, uint8_t *bad) {
    const uint32_t j = blockIdx.x;
    if (j >= njobs) return;
    __shared__ int diff;
    if (threadIdx.x == 0) diff = 0;
    __syncthreads();
    if (jobs[j].flags & kSegFirst) { if (threadIdx.x == 0) bad[j] = 0; return; }
    const SegState a = snap_state[j], b = end_state[j - 1];
    int d = (a.s != b.s) | (a.head != b.head);
    const int32_t horizon = b.s - 65535;                         // older entries can never pass blockCompress.js:62 again
    const int32_t *ta = snaps + (size_t)j * kHashEntries, *tb = tables + (size_t)(j - 1) * kHashEntries;
    for (uint32_t i = threadIdx.x; i < kHashEntries; i += blockDim.x) {
        int32_t x = ta[i] - 1, y = tb[i] - 1;
        if (x < horizon) x = -1;
        if (y < horizon) y = -1;
        d |= x != y;
    }
    if (d) atomicOr(&diff, 1);
    __syncthreads();
    if (threadIdx.x == 0) bad[j] = (uint8_t)diff;
}

// Concatenates the pieces of every block (slots [slot_first[b], +slot_count[b]), in order) into dst + dst_off[b].
// gridDim.y CTAs share a block: CTA y copies the 4 KiB stripes y, y + gridDim.y, ... of the block's compressed stream.
__global__ void __launch_bounds__(256)
k_seg_assemble(const uint8_t *__restrict__ blockbuf, uint64_t blockbuf_stride, const uint32_t *__restrict__ slot_first,
               const uint32_t *__restrict__ slot_count, const uint32_t *__restrict__ piece_off, const uint32_t *__restrict__ piece_len,
               uint32_t nblocks, uint8_t *__restrict__ dst, const uint64_t *__restrict__ dst_off, uint32_t *__restrict__ comp_len) {
    constexpr uint32_t kStripe = 4096;
    for (uint32_t b = blockIdx.x; b < nblocks; b += gridDim.x) {
        const uint8_t *src = blockbuf + (uint64_t)b * blockbuf_stride;
        uint8_t *d = dst + dst_off[b];
        uint32_t pos = 0;
        for (uint32_t k = 0; k < slot_count[b]; ++k) {
            const uint32_t sl = slot_first[b] + k, n = piece_len[sl];
            const uint8_t *s = src + piece_off[sl];
            // stripes are counted along the assembled stream so that the CTAs of a block stay balanced
            for (uint32_t st0 = ((pos / kStripe + gridDim.y - 1 - blockIdx.y) / gridDim.y * gridDim.y + blockIdx.y) * kStripe; st0 < pos + n;
                 st0 += gridDim.y * kStripe) {
                const uint32_t lo = st0 > pos ? st0 : pos, hi = st0 + kStripe < pos + n ? st0 + kStripe : pos + n;
                for (uint32_t i = lo + threadIdx.x; i < hi; i += blockDim.x) d[i] = s[i - pos];
            }
            pos += n;
        }
        if (threadIdx.x == 0 && blockIdx.y == 0) comp_len[b] = pos;
    }
}

// Serial chain: ONE warp walks consecutive blocks of one contiguous working buffer, carrying the table
// (linked blocks, bufferCompress.js:182,219,234; and the single-block compressRaw entry).  `work` is the
// reference's workingBuffer (dictionary ++ input); block k covers [start + k*block_size, ...).
// With nblocks == 1 it is also block 0 of an independent-mode frame that has a dictionary (the only block that
// sees the warmed table, bufferCompress.js:186-204,234-236).
__global__ void __launch_bounds__(32, 1)
k_compress_chain(const uint8_t *__restrict__ work, int32_t start, int32_t total_len, int32_t block_size, uint32_t nblocks,
                 int32_t *table_io /* global int32[16384], read at entry, written at exit */,
                 uint8_t *__restrict__ dst, uint64_t dst_stride, uint32_t *__restrict__ comp_len) {
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t lane = lane_id();
    int32_t *tab = reinterpret_cast<int32_t *>(smem);
    uint4 *t4 = reinterpret_cast<uint4 *>(tab);
    uint4 *g4 = reinterpret_cast<uint4 *>(table_io);
    for (uint32_t i = lane; i < kHashEntries * 4 / 16; i += 32) t4[i] = g4[i];
    __syncwarp();
    Tab32 T{tab};
    const int32_t end = start + total_len;
    for (uint32_t k = 0; k < nblocks; ++k) {
        const int32_t pos = start + (int32_t)k * block_size;
        const int32_t blen = (end - pos) < block_size ? (end - pos) : block_size;
        const uint32_t c = compress_block_warp_v2(work, pos, blen, T, dst + (uint64_t)k * dst_stride,
                                                  reinterpret_cast<uint32_t *>(smem + kHashEntries * 4));
        if (lane == 0) comp_len[k] = c;
        __syncwarp();
    }
    for (uint32_t i = lane; i < kHashEntries * 4 / 16; i += 32) g4[i] = t4[i];
}

// Jenkins warm-up of the table from the dictionary prefix (bufferCompress.js:186-204): table[slot(seq_i)] = i+1
// for ascending i, i.e. the largest i per slot -> atomicMax on a zeroed table.
__global__ void k_warm_jenkins(const uint8_t *__restrict__ work, int32_t dict_len, int32_t *table) {
    const int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > dict_len - 4) return;
    uint32_t h = ld32u(work + i);
    h = h + 2127912214u + (h << 12);
    h = h ^ 3345072700u ^ (h >> 19);
    h = h + 374761393u + (h << 5);
    h = (h + 3550635116u) ^ (h << 9);
    h = h + 4251993797u + (h << 3);
    h = h ^ 3042594569u ^ (h >> 16);
    atomicMax(&table[(h >> 18) & 16383u], i + 1);
}

// ------------------------------------------------------------------ decompress
// Forward byte-order copy of n bytes from d - offset to d (LZ4 match copy, any overlap).
__device__ __forceinline__ void warp_match_copy(uint8_t *d, uint32_t offset, uint32_t n, uint32_t lane) {
    if (offset >= 32u) {
        const uint8_t *s = d - offset;
        if (offset >= n) { warp_copy(d, s, n, lane); return; }
        for (uint32_t base = 0; base < n; base += 32) {          // each round reads only bytes of earlier rounds
            const uint32_t k = base + lane;
            if (k < n) d[k] = s[k];
            __syncwarp();
        }
    } else {
        // period < 32: every output byte equals one of the `offset` bytes before d.  With a stride that is a
        // multiple of the period each lane keeps writing the same byte.
        const uint32_t step = 32u - (32u % offset);
        if (lane < step) {
            const uint8_t v = d[(int32_t)(lane % offset) - (int32_t)offset];
            for (uint32_t k = lane; k < n; k += step) d[k] = v;
        }
    }
}

// One sequence at in[ip], uniform across the warp (the loop body of blockDecompress.js:55-271).  Returns false when the block
// ends here (last sequence or error, `st` set).
__device__ __forceinline__ bool dec_one_sequence(const uint8_t *__restrict__ in, const uint32_t n, uint8_t *const ob, const uint32_t cap,
                                                 const uint32_t hist, const uint8_t *__restrict__ dict, const uint32_t dict_len,
                                                 uint32_t &ip, uint32_t &op, uint32_t &st, const uint32_t lane) {
    const uint32_t token = in[ip++];                             // :58
    uint32_t lit = token >> 4;                                   // :61
    if (lit == 15u) {                                            // :62-68
        uint32_t b;
        do {
            if (ip >= n) { st = ST_MALFORMED; return false; }
            b = in[ip++]; lit += b;
        } while (b == 255u);
    }
    if ((uint64_t)op + lit > cap) { st = ST_OUTPUT_TOO_SMALL; return false; }      // :74
    if ((uint64_t)ip + lit > n) { st = ST_MALFORMED; return false; }              // :75
    const uint32_t litp = ip;
    ip += lit;
    if (ip >= n) {                                               // :123 last sequence: literals only
        if (lit) warp_copy(ob + op, in + litp, lit, lane);
        op += lit;
        return false;
    }
    if (ip + 2 > n) { if (lit) warp_copy(ob + op, in + litp, lit, lane); st = ST_MALFORMED; return false; }
    const uint32_t offset = (uint32_t)in[ip] | ((uint32_t)in[ip + 1] << 8);   // :126
    ip += 2;
    if (offset == 0) { st = ST_OFFSET_ZERO; return false; }      // :128
    uint32_t ml = token & 15u;                                   // :131
    if (ml == 15u) {                                             // :132-138
        uint32_t b;
        do {
            if (ip >= n) { st = ST_MALFORMED; return false; }
            b = in[ip++]; ml += b;
        } while (b == 255u);
    }
    ml += 4;                                                     // :139
    const int64_t src_rel = (int64_t)op + lit - offset;          // :142, relative to ob
    if (src_rel < -(int64_t)hist) {
        // :145-200 the match starts in the dictionary (ob - hist is output index 0)
        if (lit) warp_copy(ob + op, in + litp, lit, lane);
        op += lit;
        const int64_t cs = src_rel + hist;                       // < 0
        int64_t from_dict = -cs;
        if (from_dict > ml) from_dict = ml;
        const int64_t di = (int64_t)dict_len + cs;
        if (di < 0 || di + from_dict > dict_len) { st = ST_DICT_OOB; return false; }   // :150-152
        if ((uint64_t)op + ml > cap) { st = ST_OUTPUT_TOO_SMALL; return false; }
        warp_copy(ob + op, dict + di, (uint32_t)from_dict, lane);
        op += (uint32_t)from_dict;
        const uint32_t rem = ml - (uint32_t)from_dict;
        __syncwarp();
        if (rem) warp_match_copy(ob + op, offset, rem, lane);
        op += rem;
        __syncwarp();
        return true;
    }
    const uint32_t total = lit + ml;
    if ((uint64_t)op + total > cap) {                            // literals fit (checked above), the match does not
        st = ST_OUTPUT_TOO_SMALL;
        return false;
    }
    if (offset >= (total < 32u ? total : 32u)) {
        // merged pass: every source byte of a round was written before that round
        uint8_t *const d = ob + op;
        const uint8_t *const ls = in + litp;
        const uint8_t *const ms = d - offset;                    // ms[j] is the match source of output byte j (j >= lit)
        for (uint32_t base = 0; base < total; base += 32) {
            const uint32_t j = base + lane;
            if (j < total) d[j] = j < lit ? ls[j] : ms[j];
            __syncwarp();
        }
    } else {
        if (lit) warp_copy(ob + op, in + litp, lit, lane);
        __syncwarp();
        warp_match_copy(ob + op + lit, offset, ml, lane);
        __syncwarp();
    }
    op += total;
    return true;
}

// decompressBlock, the formulation the kernels use: 32-bit indices relative to the block's own output start `ob`, `hist` =
// bytes of earlier output directly before `ob` that may serve as history (frame mode; at most 65536 matter because offsets are
// 16-bit), literals + match of a sequence written in ONE merged pass whenever the match source lies entirely before the bytes
// of that pass (offset >= min(lit + matchLen, 32), the common case on text).
// The token chain is serial (a token's position follows from the previous sequence's lengths): three dependent loads per
// sequence.  So the warp speculates: lane l sizes the sequence that WOULD start at byte ip + l of the window, the warp hops from
// lane 0 along the `next` links (two shuffles per real token) and the visited lanes -- the real tokens -- check themselves in
// the reference's order (:74, :75, :128, ...).  Their copies then run in order, one sequence per step.  Tokens the window
// cannot size (length runs of more than 3 bytes, sources that straddle the dictionary, anything malformed) take dec_one_sequence, also
// what decides every error, so the first error reported is the reference's.
template <bool kDict>                       // kDict: a dictionary exists, matches that lie inside it take the window path too
__device__ uint32_t decompress_block_warp_v2(const uint8_t *__restrict__ in, const uint32_t n, uint8_t *const ob,
                                             const uint32_t cap, const uint32_t hist, const uint8_t *__restrict__ dict,
                                             const uint32_t dict_len, uint32_t *status) {
    const uint32_t lane = lane_id();
    uint32_t ip = 0, op = 0;
    uint32_t st = ST_OK;
    while (ip < n) {
        // ---- every lane sizes "its" sequence
        const uint32_t q = ip + lane;
        uint32_t lit = 0, ml = 0, offset = 1, litp = 0, nxt = 1;
        bool stop = true, last = false;                          // stop: the serial form decides (or the block ends)
        if (q < n) {
            const uint32_t token = in[q];
            uint32_t p = q + 1;
            lit = token >> 4;
            bool ok = true;
            if (lit == 15u) {                                    // at most 3 length bytes speculatively
                uint32_t v = 255u;
                for (int k = 0; k < 3 && v == 255u; ++k) {
                    if (p >= n) { ok = false; v = 0; break; }
                    v = in[p++]; lit += v;
                }
                if (v == 255u) ok = false;
            }
            litp = p;
            const uint64_t endlit = (uint64_t)p + lit;
            if (ok && endlit + 2 <= n) {
                offset = (uint32_t)in[endlit] | ((uint32_t)in[endlit + 1] << 8);
                p = (uint32_t)endlit + 2;
                ml = token & 15u;
                if (offset == 0) ok = false;
                else if (ml == 15u) {
                    uint32_t v = 255u;
                    for (int k = 0; k < 3 && v == 255u; ++k) {
                        if (p >= n) { ok = false; v = 0; break; }
                        v = in[p++]; ml += v;
                    }
                    if (v == 255u) ok = false;
                }
                ml += 4;
                nxt = p - ip;
            } else ok = false;                                   // last sequence, or malformed: serial form
            stop = !ok;
        }
        // ---- hop along the real tokens
        uint32_t cur = 0, real = 0, myop = 0, opw = op;
        const uint32_t adv = lit + ml;
        const uint32_t stopper = __ballot_sync(FULL, stop);
        while (cur < 32u) {
            if ((stopper >> cur) & 1u) break;
            real |= 1u << cur;
            if (lane == cur) myop = opw;
            opw += __shfl_sync(FULL, adv, cur);
            cur = __shfl_sync(FULL, nxt, cur);
        }
        // ---- the visited lanes check capacity and history themselves; the first one that fails goes to the serial form
        bool fine = (real >> lane) & 1u;
        uint32_t dsrc = 0;                                       // 1 + index into `dict` when the whole match lies in the dictionary
        if (fine) {
            const int64_t srel = (int64_t)myop + lit - offset;   // match source relative to ob (:142)
            if ((uint64_t)myop + lit + ml > cap) fine = false;                                 // :74 / match capacity
            else if (srel < -(int64_t)hist) {
                // :145-200 the source starts in the dictionary (ob - hist is output index 0).  Entirely inside it (config 4:
                // every message reads the shared dictionary): a plain copy from `dict`.  Crossing into the output or out of
                // bounds: serial form.
                const int64_t di = (int64_t)dict_len + srel + hist;
                if (kDict && di >= 0 && srel + hist + (int64_t)ml <= 0) dsrc = (uint32_t)di + 1u;
                else fine = false;
            }
#if DLZ4_DEC_PREFETCH
            // the match source is output this warp wrote a while ago: it sits in L2, one round trip per sequence.  Start all
            // round trips of the window now; the copies below then find the lines on their way (or in L1).
            else asm volatile("prefetch.global.L1 [%0];" ::"l"(ob + srel));
#endif
        }
        const uint32_t notfine = real & ~__ballot_sync(FULL, fine);
        const uint32_t good = notfine ? (real & ((notfine & (0u - notfine)) - 1u)) : real;
        // ---- copies, in order
        const uint32_t pack = lit | (ml << 16);                  // both < 1024 here
        const bool anydict = kDict && __ballot_sync(FULL, dsrc != 0) != 0;
        // ---- quick form: every sequence of the window is at most 32 bytes and its match source lies in front of the
        //      window's own output (text: offsets of hundreds of bytes, sequences of ~15).  Then no copy of the window reads what
        //      another one writes: two sequences per step, their loads issued together before the stores (the load-to-store
        //      dependency of one sequence at a time was a third of the kernel's stall samples), two shuffles per sequence.
        const uint32_t rel_o = myop - op;
        const bool quick = adv <= 32u && offset >= rel_o + adv && dsrc == 0u;
        if (good && !(good & ~__ballot_sync(FULL, quick))) {
            const uint32_t pa = adv | (lit << 6) | ((litp - ip) << 12) | (rel_o << 18);      // 6 + 6 + 6 + 10 bits
            uint8_t *const dw = ob + op + lane;
            const uint8_t *const iw = in + ip + lane;
            uint32_t m = good;
            constexpr int kQ = DLZ4_DEC_Q;                                // sequences per step (4: 48 registers, fewer resident warps)
            while (m) {
                const uint8_t *sp[kQ];
                uint8_t *dp[kQ];
                bool pr[kQ];
#pragma unroll
                for (int u = 0; u < kQ; ++u) {
                    const bool valid = m != 0u;
                    const int l = valid ? __ffs(m) - 1 : 0;
                    m &= m - 1u;
                    const uint32_t a = __shfl_sync(FULL, pa, l), of = __shfl_sync(FULL, offset, l);
                    const uint32_t tot = a & 63u, li = (a >> 6) & 63u;
                    pr[u] = valid && lane < tot;
                    dp[u] = dw + (a >> 18);
                    sp[u] = lane < li ? iw + ((a >> 12) & 63u) : dp[u] - of;
                }
                uint8_t v[kQ];
#pragma unroll
                for (int u = 0; u < kQ; ++u) v[u] = pr[u] ? *sp[u] : (uint8_t)0;
#pragma unroll
                for (int u = 0; u < kQ; ++u) if (pr[u]) *dp[u] = v[u];
            }
            __syncwarp();
        } else
        for (uint32_t m = good; m; m &= m - 1u) {
            const int l = __ffs(m) - 1;
            const uint32_t pk = __shfl_sync(FULL, pack, l), off_ = __shfl_sync(FULL, offset, l);
            const uint32_t lp = __shfl_sync(FULL, litp, l), o_ = __shfl_sync(FULL, myop, l);
            const uint32_t lit_ = pk & 0xFFFFu, total = lit_ + (pk >> 16);
            uint8_t *const d = ob + o_;
            if (kDict && anydict) {                              // uniform: some sequence of this window reads the dictionary
                const uint32_t ds = __shfl_sync(FULL, dsrc, l);
                if (ds) {
                    const uint8_t *dsp = dict + (ds - 1u) - lit_;                 // dsp[j] = dictionary byte of output byte j >= lit_
                    for (uint32_t base = 0; base < total; base += 32) {
                        const uint32_t j = base + lane;
                        if (j < total) d[j] = j < lit_ ? in[lp + j] : dsp[j];
                    }
                    __syncwarp();
                    continue;
                }
            }
            if (off_ >= (total < 32u ? total : 32u)) {
                // lane j's source: literal j of the sequence, or the match byte `offset` behind its own output byte
                const uint8_t *sp = lane < lit_ ? in + (lp + lane) : d + ((int32_t)lane - (int32_t)off_);
                uint8_t *dp = d + lane;
                if (total <= 32u) {                              // the common case: one round, no loop
                    if (lane < total) *dp = *sp;
                } else {
#pragma unroll 1
                    for (uint32_t base = 0; base < total; base += 32) {          // uniform trip count: every round ends in a barrier
                        const uint32_t j = base + lane;
                        if (j < total) *dp = *sp;
                        dp += 32;
                        sp = j + 32 < lit_ ? in + (lp + j + 32) : d + ((int32_t)(j + 32) - (int32_t)off_);
                        __syncwarp();
                    }
                }
                __syncwarp();
            } else {
                if (lit_) warp_copy(d, in + lp, lit_, lane);
                __syncwarp();
                warp_match_copy(d + lit_, off_, total - lit_, lane);
                __syncwarp();
            }
        }
        if (good) {
            const int hi = 31 - __clz(good);
            op = __shfl_sync(FULL, myop, hi) + __shfl_sync(FULL, adv, hi);
            ip += __shfl_sync(FULL, nxt, hi);
        }
        if (good != real || cur < 32u) {
            // the next token is one the window could not take (or the walk stopped at one): serial form
            if (ip >= n) break;
            if (!dec_one_sequence(in, n, ob, cap, hist, dict, dict_len, ip, op, st, lane)) break;
        }
    }
    *status = st;
    return op;
}

// Batched decode, one warp per block, blocks handed out by an atomic counter.
// hist_frame != 0: block i's output array starts at dst[0] (history = dict ++ dst[0..dst_off[i]));
// otherwise each block's array starts at its own dst_off[i].
template <int WARPS, bool kDict>
__global__ void __launch_bounds__(WARPS * 32, DLZ4_DEC_MINB)
k_decompress_blocks(const uint8_t *__restrict__ src, const uint64_t *__restrict__ src_off,
                    const uint32_t *__restrict__ src_len, uint32_t nblocks, uint8_t *dst,
                    const uint64_t *__restrict__ dst_off, const uint32_t *__restrict__ dst_cap,
                    const uint8_t *__restrict__ dict, uint32_t dict_len, int hist_frame,
                    const uint8_t *__restrict__ stored /* nullable: 1 = raw copy (frame stored block) */,
                    uint32_t *__restrict__ out_len, uint8_t *__restrict__ status, uint32_t *counter) {
    const uint32_t lane = lane_id();
    // Queue order: a block of text keeps its warp busy for milliseconds -- about as long as the whole kernel runs on a mixed
    // batch -- while runs and incompressible blocks take microseconds, so the queue is walked twice: first the blocks that
    // look like work (compressed size between 1/16 and 15/16 of the room for the decoded bytes), then the rest, which fill the
    // tail.  Only the order changes; with frame history one warp takes the blocks in their own order.
    const bool twice = !hist_frame && nblocks <= 0x7FFFFFFFu;
    const uint32_t qlen = twice ? 2u * nblocks : nblocks;
    for (;;) {
        const uint32_t qi = next_block(counter, lane);
        if (qi >= qlen) break;
        const uint32_t b = qi < nblocks ? qi : qi - nblocks;
        if (twice) {
            const uint32_t cl = src_len[b], room = dst_cap[b];
            const bool work = !(stored && stored[b]) && cl > (room >> 4) && cl + (room >> 4) < room;
            if (work != (qi < nblocks)) continue;
        }
        uint32_t st;
        uint32_t w;
        if (stored && stored[b]) {                               // bufferDecompress.js:147-149
            w = src_len[b];
            st = ST_OK;
            if (w > dst_cap[b]) { st = ST_OUTPUT_TOO_SMALL; w = 0; }
            else warp_copy(dst + dst_off[b], src + src_off[b], w, lane);
        } else {
            const uint64_t o = dst_off[b];
            const uint32_t hist = hist_frame ? (uint32_t)(o < 65536ull ? o : 65536ull) : 0u;
            w = decompress_block_warp_v2<kDict>(src + src_off[b], src_len[b], dst + o, dst_cap[b], hist, dict, dict_len, &st);
        }
        if (lane == 0) { out_len[b] = w; status[b] = (uint8_t)st; }
    }
}

// Serial chain decode: one warp, consecutive blocks of one frame in order (linked blocks read the previous
// blocks' output, bufferDecompress.js:153).  kind[k]: bit31 of the frame's size word (stored block).
__global__ void __launch_bounds__(32)
k_decompress_chain(const uint8_t *__restrict__ src, const uint64_t *__restrict__ src_off,
                   const uint32_t *__restrict__ src_len, const uint8_t *__restrict__ stored, uint32_t nblocks,
                   uint8_t *dst, uint64_t dst_total, uint32_t block_max, const uint8_t *__restrict__ dict, uint32_t dict_len,
                   uint32_t *__restrict__ out_len, uint8_t *__restrict__ status, uint64_t *total_out) {
    const uint32_t lane = lane_id();
    int64_t op = 0;
    uint32_t st = ST_OK;
    for (uint32_t b = 0; b < nblocks; ++b) {
        uint32_t w = 0;
        if (st == ST_OK) {
            // a block never decodes past blockMaxSize, like the jump decoder's (LZ4 frame format; liblz4 enforces it too)
            const uint64_t left = dst_total - (uint64_t)op, room = left < block_max ? left : block_max;
            if (stored[b]) {
                w = src_len[b];
                if (w > room) { st = ST_OUTPUT_TOO_SMALL; w = 0; }
                else warp_copy(dst + op, src + src_off[b], w, lane);
                __syncwarp();
            } else {
                w = decompress_block_warp_v2<true>(src + src_off[b], src_len[b], dst + op, (uint32_t)room,
                                             (uint32_t)(op < 65536 ? op : 65536), dict, dict_len, &st);
            }
        }
        if (lane == 0) { out_len[b] = w; status[b] = (uint8_t)st; }
        op += w;
    }
    if (lane == 0) *total_out = (uint64_t)op;
}

// ------------------------------------------------------------------ jump decoder (linked frames, large blocks)
// A linked-block frame (bufferDecompress.js:153, block k reads the output of block k-1) and a block of several MiB are one
// dependent stream for the warp-per-block decoder above.  Every output byte, though, is either a literal of the compressed
// stream or a copy of an EARLIER output byte, so decoding is pointer chasing and pointer chasing parallelises by doubling:
//   k_jd_scan     one warp per block walks the tokens only (no copies) and writes one record per sequence;
//   k_jd_bases    exclusive scan of the decoded block lengths, history / capacity checks in the reference's error order;
//   per unit of <= 16 MiB of consecutive blocks (its 4-byte-per-byte pointer array stays in L2):
//     k_jd_fill   P[x] = ~literal, or ~out[q] when the source q lies before the unit (already final), or q itself;
//     k_jd_round  P[x] = P[P[P[P[x]]]] for unresolved x, repeated until none is left (chain depth quarters per round);
//     k_jd_emit   out[x] = ~P[x].
// Units run in stream order, so a unit's sources in earlier units are final bytes.  Nothing here depends on how the
// frame was parsed: the result is the byte-exact LZ4 decode whatever the dependency structure.
struct JdSeq { uint32_t op, ip, lit, ml, off, m0, pad1, pad2; };      // block-relative output / input positions; m0 = first
                                                                      // output byte of the WHOLE match (chunked records share it)
constexpr int kJdHopBits = 4;
constexpr int kJdHops = 1 << kJdHopBits;                                // pointer links followed per element per round
constexpr uint32_t kJdChunk = 4096;                                    // long literal runs / matches are recorded in chunks

__device__ __forceinline__ void jd_emit_rec(JdSeq *rec, uint32_t &ns, uint32_t op, uint32_t ip, uint32_t lit, uint32_t ml, uint32_t off,
                                            uint32_t lane) {
    // literals in chunks, then the match in chunks (each record is one warp-pass of work in k_jd_fill)
    while (lit > kJdChunk) {
        if (lane == 0) rec[ns] = JdSeq{op, ip, kJdChunk, 0u, 0u, 0u, 0u, 0u};
        ++ns; op += kJdChunk; ip += kJdChunk; lit -= kJdChunk;
    }
    uint32_t first = ml > kJdChunk ? kJdChunk : ml;
    const uint32_t m0 = op + lit;
    if (lane == 0) rec[ns] = JdSeq{op, ip, lit, first, off, m0, 0u, 0u};
    ++ns; op += lit + first; ml -= first;
    while (ml) {
        first = ml > kJdChunk ? kJdChunk : ml;
        if (lane == 0) rec[ns] = JdSeq{op, 0u, 0u, first, off, m0, 0u, 0u};
        ++ns; op += first; ml -= first;
    }
}

// One token, uniform across the warp (the serial form of blockDecompress.js:55-139 without the copies): used for tokens the
// speculative window below cannot size (long length runs, chunked records).  Returns false when the block ends here.
__device__ __forceinline__ bool jd_scan_one(const uint8_t *__restrict__ in, uint32_t n, uint32_t block_max, JdSeq *rec, uint32_t &ns,
                                            uint32_t &ip, uint64_t &op, uint32_t &rch, uint32_t &st, uint32_t lane) {
    const uint32_t token = in[ip++];                             // :58
    uint32_t lit = token >> 4;                                   // :61
    if (lit == 15u) {                                            // :62-68
        uint32_t v;
        do {
            if (ip >= n) { st = ST_MALFORMED; return false; }
            v = in[ip++]; lit += v;
        } while (v == 255u);
    }
    if (op + lit > block_max) { st = ST_OUTPUT_TOO_SMALL; return false; }              // :74 (a block never decodes past blockMaxSize)
    if ((uint64_t)ip + lit > n) { st = ST_MALFORMED; return false; }                   // :75
    const uint32_t litp = ip;
    ip += lit;
    if (ip >= n) {                                               // :123 last sequence: literals only
        jd_emit_rec(rec, ns, (uint32_t)op, litp, lit, 0u, 0u, lane);
        op += lit;
        return false;
    }
    if (ip + 2 > n) { st = ST_MALFORMED; return false; }
    const uint32_t offset = (uint32_t)in[ip] | ((uint32_t)in[ip + 1] << 8);             // :126
    ip += 2;
    if (offset == 0) { st = ST_OFFSET_ZERO; return false; }                            // :128
    uint32_t ml = token & 15u;                                   // :131
    if (ml == 15u) {                                             // :132-138
        uint32_t v;
        do {
            if (ip >= n) { st = ST_MALFORMED; return false; }
            v = in[ip++]; ml += v;
        } while (v == 255u);
    }
    ml += 4;                                                     // :139
    if (op + lit + ml > block_max) { st = ST_OUTPUT_TOO_SMALL; return false; }
    const int64_t src_rel = (int64_t)op + lit - offset;          // :142
    if (src_rel < 0 && (uint32_t)(-src_rel) > rch) rch = (uint32_t)(-src_rel);
    jd_emit_rec(rec, ns, (uint32_t)op, litp, lit, ml, offset, lane);
    op += lit + ml;
    return true;
}

// Token walk of every block, one warp per block.  The token chain is serial (a token's position follows from the previous
// token's lengths), so the warp speculates: lane l sizes the sequence that WOULD start at byte ip + l; the warp then hops
// from lane 0 along the `next` links (two shuffles per real token instead of three dependent loads) and the lanes it
// visited -- the real tokens -- check themselves in the reference's order and write their records together.
// reach[b] = how far before its own start the block's matches read (checked against the history in k_jd_bases).
__global__ void __launch_bounds__(128)
k_jd_scan(const uint8_t *__restrict__ src, const uint64_t *__restrict__ src_off, const uint32_t *__restrict__ src_len,
          const uint8_t *__restrict__ stored, uint32_t nblocks, uint32_t block_max, JdSeq *seqs, const uint64_t *__restrict__ seq_base,
          uint32_t *nseq, uint32_t *out_len, uint32_t *reach, uint8_t *status, uint32_t *counter,
          const uint8_t *__restrict__ only /* nullable: scan only blocks with only[b] != 0 (fallback of the chunked scan) */) {
    const uint32_t lane = lane_id();
    const uint32_t lt = (1u << lane) - 1u;
    for (;;) {
        const uint32_t b = next_block(counter, lane);
        if (b >= nblocks) break;
        if (only && !only[b]) continue;
        if (only && lane == 0) reach[b] = 0;
        __syncwarp();
        const uint8_t *in = src + src_off[b];
        const uint32_t n = src_len[b];
        JdSeq *rec = seqs + seq_base[b];
        uint32_t ns = 0, ip = 0, rch = 0, st = ST_OK;
        uint64_t op = 0;
        if (stored[b]) {                                         // bufferDecompress.js:147-149: raw bytes
            jd_emit_rec(rec, ns, 0u, 0u, n, 0u, 0u, lane);
            op = n;
            if (n > block_max) st = ST_OUTPUT_TOO_SMALL;
        } else {
            while (ip < n) {
                // ---- every lane sizes "its" sequence
                const uint32_t q = ip + lane;
                uint32_t lit = 0, ml = 0, offset = 1, litp = 0, nxt = 1, err = ST_OK;
                bool slow = false, last = false;
                if (q < n) {
                    const uint32_t token = in[q];
                    uint32_t p = q + 1;
                    lit = token >> 4;
                    if (lit == 15u) {                            // at most 3 length bytes speculatively
                        uint32_t v = 255u;
                        for (int k = 0; k < 3 && v == 255u; ++k) {
                            if (p >= n) { err = ST_MALFORMED; v = 0; break; }
                            v = in[p++]; lit += v;
                        }
                        if (v == 255u) slow = true;
                    }
                    litp = p;
                    const uint64_t endlit = (uint64_t)p + lit;
                    if (!err && !slow) {
                        if (endlit > n) err = ST_MALFORMED | 0x100u;          // :75 -- comes after the :74 capacity check
                        else if (endlit == n) { last = true; nxt = n - ip; }
                        else if (endlit + 2 > n) err = ST_MALFORMED | 0x200u;
                        else {
                            offset = (uint32_t)in[endlit] | ((uint32_t)in[endlit + 1] << 8);
                            p = (uint32_t)endlit + 2;
                            ml = token & 15u;
                            if (offset == 0) err = ST_OFFSET_ZERO | 0x200u;
                            else if (ml == 15u) {
                                uint32_t v = 255u;
                                for (int k = 0; k < 3 && v == 255u; ++k) {
                                    if (p >= n) { err = ST_MALFORMED | 0x200u; v = 0; break; }
                                    v = in[p++]; ml += v;
                                }
                                if (v == 255u) slow = true;
                            }
                            ml += 4;
                            nxt = p - ip;
                        }
                    }
                    if (lit > kJdChunk || ml > kJdChunk) slow = true;         // chunked records: serial form
                }
                // ---- hop along the real tokens
                uint32_t cur = 0, real = 0, myop = 0;
                uint64_t opw = op;
                const uint32_t adv = lit + ml;
                const uint32_t stopper = __ballot_sync(FULL, slow || err != ST_OK || last || q >= n);
                while (cur < 32u) {
                    real |= 1u << cur;
                    if (lane == cur) myop = (uint32_t)opw;
                    if ((stopper >> cur) & 1u) break;
                    opw += __shfl_sync(FULL, adv, cur);
                    cur = __shfl_sync(FULL, nxt, cur);
                }
                // ---- the visited lanes check themselves (reference order: :74 capacity, :75 fit, :128 offset, match capacity)
                const bool mine = (real >> lane) & 1u;
                uint32_t verdict = ST_OK;
                if (mine && !slow && q < n) {
                    if ((err & 0xFFu) && !(err & 0x300u)) verdict = err;                       // length bytes ran out
                    else if ((uint64_t)myop + lit > block_max) verdict = ST_OUTPUT_TOO_SMALL;   // :74
                    else if (err) verdict = err & 0xFFu;
                    else if (!last && (uint64_t)myop + lit + ml > block_max) verdict = ST_OUTPUT_TOO_SMALL;
                }
                const uint32_t bad = __ballot_sync(FULL, verdict != ST_OK);
                const uint32_t slowm = __ballot_sync(FULL, mine && (slow || q >= n));
                // tokens in front of the first bad / slow one are good
                const uint32_t cut = bad | slowm;
                const uint32_t good = cut ? (real & ((cut & (0u - cut)) - 1u)) : real;
                if ((good >> lane) & 1u) {
                    rec[ns + __popc(good & lt)] = JdSeq{myop, litp, lit, last ? 0u : ml, last ? 0u : offset, myop + lit, 0u, 0u};
                    if (!last) {
                        const int64_t src_rel = (int64_t)myop + lit - offset;                 // :142
                        if (src_rel < 0) atomicMax(&reach[b], (uint32_t)(-src_rel));
                    }
                }
                ns += __popc(good);
                bool ended = false;
                if (good) {
                    const int hi = 31 - __clz(good);
                    op = (uint64_t)__shfl_sync(FULL, myop, hi) + __shfl_sync(FULL, adv, hi);
                    ip += __shfl_sync(FULL, nxt, hi);
                    ended = __shfl_sync(FULL, (int)last, hi) != 0;
                }
                if (bad && (!slowm || (bad & (0u - bad)) < (slowm & (0u - slowm)))) {
                    st = __shfl_sync(FULL, verdict, __ffs(bad) - 1);
                    break;
                }
                if (ended) break;
                if (slowm && ip < n) {
                    if (!jd_scan_one(in, n, block_max, rec, ns, ip, op, rch, st, lane)) break;
                }
            }
        }
        __syncwarp();
        if (lane == 0) { nseq[b] = ns; out_len[b] = (uint32_t)op; atomicMax(&reach[b], rch); status[b] = (uint8_t)st; }
    }
}

// ---- chunked token scan (blocks > 64 KiB): the token chain of ONE block in parallel.
//   k_jdp_next   one thread per compressed byte i sizes the sequence that would start there: nx[i] = bytes to the next token
//                (0: not sizeable here -- long length runs, the last sequence, anything malformed), adv[i] = lit + match length;
//   k_jdp_exit   per 2048-byte chunk, pointer doubling in shared memory: from every i, where does the chain leave the chunk
//                (or which unsizeable token stops it), how many tokens and output bytes on the way;
//   k_jdp_hop    one thread per block hops chunk to chunk along the real chain (one 16-byte load per chunk), sizes the
//                unsizeable tokens serially, and lists runs (entry, first record index, output offset) and slow tokens;
//   k_jdp_emit   one warp per run walks its tokens (nx links, two shuffles per token) and writes the records; one warp per
//                slow token writes its chunked records.
// Anything irregular (malformed input, capacity overflow, list overflow) flags the block for the serial scan above, which
// reproduces the reference's error order; the chunked scan only ever handles well-formed blocks.
constexpr uint32_t kJdpChunk = 2048;
constexpr uint32_t kJdpSlowBit = 0x80000000u;
struct JdpExit { uint32_t ex, ca; };      // ex: position where the chain leaves the chunk | kJdpSlowBit; ca = hops:10 | output bytes:22
struct JdpRun { uint32_t pos, ns, op, pad; };
struct JdpSlow { uint32_t op, litp, lit, ml, off, ns, pad0, pad1; };

__device__ __forceinline__ uint32_t jd_rec_count(uint32_t lit, uint32_t ml) {      // records jd_emit_rec writes
    uint32_t c = 1;
    if (lit > kJdChunk) c += (lit - 1) / kJdChunk;
    if (ml > kJdChunk) c += (ml - 1) / kJdChunk;
    return c;
}

__global__ void __launch_bounds__(256)
k_jdp_next(const uint8_t *__restrict__ src, const uint64_t *__restrict__ src_off, const uint32_t *__restrict__ src_len,
           const uint8_t *__restrict__ stored, uint16_t *nx, uint16_t *adv) {
    const uint32_t b = blockIdx.y;
    const uint32_t n = src_len[b];
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || stored[b]) return;
    const uint64_t g = src_off[b];
    const uint8_t *in = src + g;
    const uint32_t token = in[i];
    uint32_t p = i + 1, lit = token >> 4, ml = 0;
    bool ok = true;
    if (lit == 15u) {
        uint32_t v = 255u;
        for (int k = 0; k < 16 && v == 255u; ++k) {
            if (p >= n) { ok = false; v = 0; break; }
            v = in[p++]; lit += v;
        }
        if (v == 255u) ok = false;
    }
    const uint64_t endlit = (uint64_t)p + lit;
    if (ok && endlit + 2 <= n) {                                 // endlit >= n: last sequence or malformed -> serial
        const uint32_t offset = (uint32_t)in[endlit] | ((uint32_t)in[endlit + 1] << 8);
        p = (uint32_t)endlit + 2;
        ml = token & 15u;
        if (offset == 0) ok = false;
        else if (ml == 15u) {
            uint32_t v = 255u;
            for (int k = 0; k < 16 && v == 255u; ++k) {
                if (p >= n) { ok = false; v = 0; break; }
                v = in[p++]; ml += v;
            }
            if (v == 255u) ok = false;
        }
        ml += 4;
    } else ok = false;
    if (lit > kJdChunk || ml > kJdChunk || p - i > 0xFFFFu) ok = false;
    nx[g + i] = ok ? (uint16_t)(p - i) : (uint16_t)0;
    adv[g + i] = ok ? (uint16_t)(lit + ml) : (uint16_t)0;
}

__global__ void __launch_bounds__(256)
k_jdp_exit(const uint64_t *__restrict__ src_off, const uint32_t *__restrict__ src_len, const uint8_t *__restrict__ stored,
           const uint16_t *__restrict__ nx, const uint16_t *__restrict__ adv, JdpExit *exits) {
    // per entry: where its chain stands (tgt: index inside the chunk, 0xFFFF once it has left), hops so far, the exit position
    // and the output bytes so far; (hops << 16 | tgt) share a word so that a doubling step is three loads and three stores
    __shared__ uint32_t ct[kJdpChunk], ex[kJdpChunk], av[kJdpChunk];
    const uint32_t b = blockIdx.y, n = src_len[b];
    const uint32_t c0 = blockIdx.x * kJdpChunk;
    if (c0 >= n || stored[b]) return;
    const uint64_t g = src_off[b];
    const uint32_t cend = c0 + kJdpChunk < n ? c0 + kJdpChunk : n;
    constexpr int PER = kJdpChunk / 256;
    for (int k = 0; k < PER; ++k) {
        const uint32_t i = threadIdx.x + k * 256, a = c0 + i;
        uint32_t t = 0xFFFFu, e = 0, c = 0, v = 0;
        if (a < cend) {
            const uint32_t j = nx[g + a];
            if (j == 0) e = a | kJdpSlowBit;
            else {
                c = 1; v = adv[g + a];
                if (a + j >= cend) e = a + j; else t = i + j;
            }
        }
        ct[i] = (c << 16) | t; ex[i] = e; av[i] = v;
    }
    __syncthreads();
    for (int round = 0; round < 11; ++round) {                   // a hop is >= 3 bytes: <= 683 hops per chunk
        uint32_t ct2[PER], e2[PER], v2[PER];
        for (int k = 0; k < PER; ++k) {
            const uint32_t i = threadIdx.x + k * 256;
            const uint32_t c = ct[i], t = c & 0xFFFFu;
            ct2[k] = c; e2[k] = ex[i]; v2[k] = av[i];
            if (t != 0xFFFFu) { const uint32_t d = ct[t]; ct2[k] = (c & 0xFFFF0000u) + d; e2[k] = ex[t]; v2[k] += av[t]; }
        }
        __syncthreads();
        int open = 0;
        for (int k = 0; k < PER; ++k) {
            const uint32_t i = threadIdx.x + k * 256;
            ct[i] = ct2[k]; ex[i] = e2[k]; av[i] = v2[k];
            open |= (ct2[k] & 0xFFFFu) != 0xFFFFu;
        }
        if (!__syncthreads_or(open)) break;                      // every chain has left the chunk
    }
    for (int k = 0; k < PER; ++k) {
        const uint32_t i = threadIdx.x + k * 256, a = c0 + i;
        if (a < cend) {
            // 8 bytes per compressed byte.  A chain that would overflow the 22 bits (> 4 MiB out of one 2 KiB chunk, i.e.
            // never in a valid 4 MiB block) is handed to the serial form token by token, which is exact for any token
            const bool fits = av[i] < (1u << 22);
            exits[g + a] = fits ? JdpExit{ex[i], ((ct[i] >> 16) << 22) | av[i]} : JdpExit{a | kJdpSlowBit, 0u};
        }
    }
}

// Sum of a length run (bytes of 255 closed by one smaller byte), 32 bytes per step.  Returns false when the input ends first.
__device__ __forceinline__ bool jd_length_run(const uint8_t *__restrict__ in, uint32_t &ip, uint32_t n, uint32_t &acc, uint32_t lane) {
    for (;;) {
        const uint32_t q = ip + lane;
        const uint32_t v = q < n ? (uint32_t)in[q] : 0x100u;
        const uint32_t stop = __ballot_sync(FULL, v != 255u);
        if (!stop) { acc += 255u * 32u; ip += 32u; continue; }
        const int l = __ffs(stop) - 1;
        const uint32_t vv = __shfl_sync(FULL, v, l);
        if (vv == 0x100u) return false;
        acc += 255u * (uint32_t)l + vv;
        ip += (uint32_t)l + 1u;
        return true;
    }
}

// One warp per block (uniform control flow; lane 0 writes).
__global__ void __launch_bounds__(256)
k_jdp_hop(const uint8_t *__restrict__ src, const uint64_t *__restrict__ src_off, const uint32_t *__restrict__ src_len,
          const uint8_t *__restrict__ stored, uint32_t nblocks, uint32_t block_max, const JdpExit *__restrict__ exits,
          JdpRun *runs, JdpSlow *slows, const uint64_t *__restrict__ list_base, uint32_t *nruns, uint32_t *nslow,
          uint32_t *nseq, uint32_t *out_len, uint32_t *reach, uint8_t *status, uint8_t *fallback) {
    const uint32_t lane = lane_id();
    const uint32_t b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (b >= nblocks) return;
    const uint32_t n = src_len[b];
    const uint64_t g = src_off[b];
    const uint8_t *in = src + g;
    JdpRun *R = runs + list_base[b];
    JdpSlow *S = slows + list_base[b];
    const uint32_t cap = (uint32_t)(list_base[b + 1] - list_base[b]);
    uint32_t nr = 0, nsl = 0, ns = 0, pos = 0, rch = 0;
    uint64_t op = 0;
    bool fb = false;
    if (stored[b]) {
        if (lane == 0) S[0] = JdpSlow{0u, 0u, n, 0u, 0u, 0u, 0u, 0u};
        nsl = 1;
        ns = jd_rec_count(n, 0); op = n;
        if (n > block_max) fb = true;
    } else {
        while (pos < n) {
            const uint2 raw = __ldg(reinterpret_cast<const uint2 *>(exits + g + pos));
            const JdpExit E{raw.x, raw.y};
            if (E.ca >> 22) {
                if (nr >= cap) { fb = true; break; }
                if (lane == 0) R[nr] = JdpRun{pos, ns, (uint32_t)op, 0u};
                ++nr;
                ns += E.ca >> 22; op += E.ca & ((1u << 22) - 1u);
                if (op > block_max) { fb = true; break; }
            }
            if (!(E.ex & kJdpSlowBit)) { pos = E.ex; continue; }
            // a token the per-byte pass could not size: serial form (any error -> the serial scan decides the status)
            uint32_t ip = E.ex & ~kJdpSlowBit;
            const uint32_t token = in[ip++];
            uint32_t lit = token >> 4;
            if (lit == 15u && !jd_length_run(in, ip, n, lit, lane)) { fb = true; break; }
            if (op + lit > block_max || (uint64_t)ip + lit > n) { fb = true; break; }
            const uint32_t litp = ip;
            ip += lit;
            uint32_t ml = 0, offset = 0;
            const bool last = ip >= n;
            if (!last) {
                if (ip + 2 > n) { fb = true; break; }
                offset = (uint32_t)in[ip] | ((uint32_t)in[ip + 1] << 8);
                ip += 2;
                if (offset == 0) { fb = true; break; }
                ml = token & 15u;
                if (ml == 15u && !jd_length_run(in, ip, n, ml, lane)) { fb = true; break; }
                ml += 4;
                if (op + lit + ml > block_max) { fb = true; break; }
                const int64_t src_rel = (int64_t)op + lit - offset;
                if (src_rel < 0 && (uint32_t)(-src_rel) > rch) rch = (uint32_t)(-src_rel);
            }
            if (nsl >= cap) { fb = true; break; }
            if (lane == 0) S[nsl] = JdpSlow{(uint32_t)op, litp, lit, ml, offset, ns, 0u, 0u};
            ++nsl;
            ns += jd_rec_count(lit, ml);
            op += lit + ml;
            if (last) break;
            pos = ip;
        }
    }
    if (lane == 0) {
        nruns[b] = fb ? 0u : nr; nslow[b] = fb ? 0u : nsl;
        nseq[b] = ns; out_len[b] = (uint32_t)op; reach[b] = rch; status[b] = ST_OK; fallback[b] = fb ? 1 : 0;
    }
}

__global__ void __launch_bounds__(256)
k_jdp_emit(const uint8_t *__restrict__ src, const uint64_t *__restrict__ src_off, const uint32_t *__restrict__ src_len,
           const uint16_t *__restrict__ nx, const uint16_t *__restrict__ adv, const JdpRun *__restrict__ runs,
           const JdpSlow *__restrict__ slows, const uint64_t *__restrict__ list_base, const uint32_t *__restrict__ nruns,
           const uint32_t *__restrict__ nslow, JdSeq *seqs, const uint64_t *__restrict__ seq_base, uint32_t *reach) {
    const uint32_t lane = lane_id(), b = blockIdx.y;
    const uint32_t lt = (1u << lane) - 1u;
    const uint32_t gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), nw = gridDim.x * (blockDim.x >> 5);
    const uint32_t n = src_len[b];
    const uint64_t g = src_off[b];
    const uint8_t *in = src + g;
    JdSeq *rec = seqs + seq_base[b];
    const uint32_t nr = nruns[b], nsl = nslow[b];
    uint32_t rch = 0;
    for (uint32_t w = gw; w < nr + nsl; w += nw) {
        if (w >= nr) {                                           // slow token: chunked records
            const JdpSlow q = slows[list_base[b] + (w - nr)];
            uint32_t ns = q.ns;
            jd_emit_rec(rec, ns, q.op, q.litp, q.lit, q.ml, q.off, lane);
            continue;
        }
        const JdpRun r = runs[list_base[b] + w];
        const uint32_t cend = ((r.pos / kJdpChunk) + 1) * kJdpChunk < n ? ((r.pos / kJdpChunk) + 1) * kJdpChunk : n;
        uint32_t ip = r.pos, ns = r.ns, op = r.op;
        bool done = false;
        while (!done) {
            const uint32_t q = ip + lane;
            const uint32_t j = q < cend ? (uint32_t)nx[g + q] : 0u;     // 0 also behind the chunk: the run ends there
            const uint32_t a = q < cend ? (uint32_t)adv[g + q] : 0u;
            uint32_t cur = 0, real = 0, myop = 0, opw = op, last_hop = 0;
            while (cur < 32u) {
                const uint32_t jj = __shfl_sync(FULL, j, cur);
                if (jj == 0) { done = true; break; }             // unsizeable token or end of the chunk: k_jdp_hop continues
                real |= 1u << cur;
                if (lane == cur) myop = opw;
                opw += __shfl_sync(FULL, a, cur);
                last_hop = cur + jj;
                cur = last_hop;
            }
            if ((real >> lane) & 1u) {                           // visited lanes = real tokens: parse and write the record
                const uint32_t token = in[q];
                uint32_t p = q + 1, lit = token >> 4;
                if (lit == 15u) { uint32_t v; do { v = in[p++]; lit += v; } while (v == 255u); }
                const uint32_t litp = p;
                p += lit;
                const uint32_t offset = (uint32_t)in[p] | ((uint32_t)in[p + 1] << 8);
                p += 2;
                uint32_t ml = token & 15u;
                if (ml == 15u) { uint32_t v; do { v = in[p++]; ml += v; } while (v == 255u); }
                ml += 4;
                rec[ns + __popc(real & lt)] = JdSeq{myop, litp, lit, ml, offset, myop + lit, 0u, 0u};
                const int64_t src_rel = (int64_t)myop + lit - offset;
                if (src_rel < 0 && (uint32_t)(-src_rel) > rch) rch = (uint32_t)(-src_rel);
            }
            ns += __popc(real);
            op = opw;
            if (!done) {
                ip += last_hop;
                if (ip >= cend) done = true;
            }
        }
    }
    rch = __reduce_max_sync(FULL, rch);
    if (lane == 0 && rch) atomicMax(&reach[b], rch);
}

// base[b] = decoded bytes before block b (base[nblocks] = total); a block that reads further back than its history
// (dictionary, plus the earlier output when linked) gets the reference's "Dictionary Offset Out of Bounds" (:150-152).
__global__ void __launch_bounds__(32)
k_jd_bases(const uint32_t *__restrict__ out_len, const uint32_t *__restrict__ reach, uint32_t nblocks, uint32_t dict_len, int linked,
           uint64_t cap_total, uint64_t *base, uint8_t *status) {
    if (threadIdx.x) return;
    uint64_t acc = 0;
    for (uint32_t b = 0; b < nblocks; ++b) {
        base[b] = acc;
        if (status[b] == ST_OK) {
            const uint64_t hist = (uint64_t)dict_len + (linked ? acc : 0ull);
            if (reach[b] > hist) status[b] = ST_DICT_OOB;
            else if (acc + out_len[b] > cap_total) status[b] = ST_OUTPUT_TOO_SMALL;
        }
        acc += out_len[b];
    }
    base[nblocks] = acc;
}

// Error path of the jump decoder: the first block with any problem (the host finds it in k_jd_bases's statuses) gets the
// status the reference's token loop reaches first -- dec_one_sequence without the copies.  The scans and k_jd_bases test
// capacity, lengths, offsets and history at different times, so they may name a later error of that block (or another
// block's).  A status depends only on lengths, offsets and positions, never on decoded bytes.  hist = how far before the
// block's output its history reaches (dictionary, plus the earlier output when linked); room = the block's capacity.
// Blocks before this one are clean: scan OK, reach within their history, output within the capacity.
__global__ void __launch_bounds__(32)
k_jd_status(const uint8_t *__restrict__ src, const uint64_t *__restrict__ src_off, const uint32_t *__restrict__ src_len,
            const uint8_t *__restrict__ stored, uint64_t hist, uint64_t room, uint8_t *status) {
    if (threadIdx.x) return;
    const uint8_t *in = src + *src_off;
    const uint32_t n = *src_len;
    uint32_t st = ST_OK;
    if (*stored) {
        if (n > room) st = ST_OUTPUT_TOO_SMALL;
    } else {
        uint32_t ip = 0;
        uint64_t op = 0;
        while (ip < n) {
            const uint32_t token = in[ip++];                     // :58
            uint64_t lit = token >> 4;
            if (lit == 15u) {                                    // :62-68
                uint32_t v;
                do {
                    if (ip >= n) { st = ST_MALFORMED; goto done; }
                    v = in[ip++]; lit += v;
                } while (v == 255u);
            }
            if (op + lit > room) { st = ST_OUTPUT_TOO_SMALL; break; }                     // :74
            if ((uint64_t)ip + lit > n) { st = ST_MALFORMED; break; }                    // :75
            ip += (uint32_t)lit;
            op += lit;
            if (ip >= n) break;                                  // :123
            if (ip + 2 > n) { st = ST_MALFORMED; break; }
            const uint32_t offset = (uint32_t)in[ip] | ((uint32_t)in[ip + 1] << 8);      // :126
            ip += 2;
            if (offset == 0) { st = ST_OFFSET_ZERO; break; }    // :128
            uint64_t ml = token & 15u;
            if (ml == 15u) {                                     // :132-138
                uint32_t v;
                do {
                    if (ip >= n) { st = ST_MALFORMED; goto done; }
                    v = in[ip++]; ml += v;
                } while (v == 255u);
            }
            ml += 4;
            if (op + hist < offset) { st = ST_DICT_OOB; break; }                        // :150-152, before the match capacity
            if (op + ml > room) { st = ST_OUTPUT_TOO_SMALL; break; }
            op += ml;
        }
    }
done:
    if (st != ST_OK) *status = (uint8_t)st;                      // (the walk finds an error whenever k_jd_bases did)
}

// One unit = blocks [b0, b1).  P is indexed from the unit's first output byte.
__global__ void __launch_bounds__(256)
k_jd_fill(const uint8_t *__restrict__ src, const uint64_t *__restrict__ src_off, const JdSeq *__restrict__ seqs,
          const uint64_t *__restrict__ seq_base, const uint32_t *__restrict__ nseq, const uint64_t *__restrict__ base, uint32_t b0,
          uint32_t ctas_per_block, const uint8_t *out /* final bytes before the unit */, const uint8_t *__restrict__ dict,
          uint32_t dict_len, int linked, int32_t *P, uint32_t *unresolved) {
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    const uint32_t b = b0 + blockIdx.x / ctas_per_block;
    const uint32_t gw = (blockIdx.x % ctas_per_block) * 8u + warp, nw = ctas_per_block * 8u;
    const uint8_t *in = src + src_off[b];
    const JdSeq *rec = seqs + seq_base[b];
    const uint64_t ustart = base[b0], bstart = base[b];
    const int32_t brel = (int32_t)(bstart - ustart);             // the block's start relative to the unit (units are <= 64 MiB)
    const uint32_t ns = nseq[b];
    uint32_t pending = 0;
    for (uint32_t si = gw; si < ns; si += nw) {
        const JdSeq q = rec[si];
        const uint32_t total = q.lit + q.ml;
        const int32_t xr0 = brel + (int32_t)q.op;                // the sequence's first output byte, relative to the unit
        for (uint32_t j = lane; j < total; j += 32) {
            const int32_t xr = xr0 + (int32_t)j;
            int32_t v;
            if (j < q.lit) {
                v = ~(int32_t)in[q.ip + j];
            } else {
                // a match longer than its offset repeats the `off` bytes in front of it: point every byte straight at them
                // (a zero run of a whole block is then one link deep instead of a chain as long as the run)
                const uint32_t dm = q.op + j - q.m0;             // distance into the whole match
                const int32_t sr = dm < q.off ? xr - (int32_t)q.off
                                              : brel + (int32_t)q.m0 - (int32_t)q.off + (int32_t)(dm % q.off);   // source, relative to the unit
                const int32_t sb = sr - brel;                    // relative to the block's start
                if (sr >= 0 && (linked || sb >= 0)) {
                    v = sr;                                      // inside the unit: resolve by doubling
                    ++pending;
                } else {
                    const int64_t sg = (int64_t)ustart + sr;     // global output position
                    if (linked ? sg >= 0 : sb >= 0) {
                        v = ~(int32_t)out[sg];                   // earlier unit: final already
                    } else {
                        // dictionary: directly before output position 0 (linked) / before every block (independent)
                        v = ~(int32_t)dict[(int64_t)dict_len + (linked ? sg : (int64_t)sb)];
                    }
                }
            }
            P[xr] = v;
        }
    }
    pending = __reduce_add_sync(FULL, pending);
    if (lane == 0 && pending) atomicAdd(unresolved, pending);
}

// Tiles of 4096 elements that had nothing unresolved in the previous round are skipped (tile_todo, reset to 1 per unit).
constexpr uint32_t kJdTile = 4096;
__global__ void __launch_bounds__(256)
k_jd_round(int32_t *P, const uint64_t *__restrict__ base, uint32_t b0, uint32_t b1, const uint32_t *todo, uint32_t *next_todo,
           uint8_t *tile_todo) {
    if (*todo == 0) return;                                      // everything resolved in an earlier round
    const uint64_t len = base[b1] - base[b0];
    const uint32_t ntiles = (uint32_t)((len + kJdTile - 1) / kJdTile);
    uint32_t pending_total = 0;
    for (uint32_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        if (!tile_todo[t]) continue;                             // uniform per CTA
        uint32_t pending = 0;
        const uint64_t t0 = (uint64_t)t * kJdTile;
#pragma unroll 4
        for (uint32_t k = threadIdx.x; k < kJdTile; k += 256) {
            const uint64_t i = t0 + k;
            if (i >= len) break;
            int32_t v = P[i];
            if (v >= 0) {
                // up to kJdHops links per round (v < i: an earlier byte of the unit).  Every link read spans >= kJdHops^round original
                // hops, whether it is this round's value or the last one's, so log4(unit bytes) rounds resolve any chain.
#pragma unroll
                for (int h = 0; h < kJdHops && v >= 0; ++h) v = P[v];
                P[i] = v;
                pending += v >= 0;
            }
        }
        const int any = __syncthreads_or((int)pending);
        if (threadIdx.x == 0) tile_todo[t] = any ? 1 : 0;
        pending_total += pending;
        __syncthreads();
    }
    pending_total = __reduce_add_sync(FULL, pending_total);
    if (lane_id() == 0 && pending_total) atomicAdd(next_todo, pending_total);
}

__global__ void __launch_bounds__(256)
k_jd_emit(const int32_t *__restrict__ P, const uint64_t *__restrict__ base, uint32_t b0, uint32_t b1, uint8_t *out) {
    const uint64_t ustart = base[b0], len = base[b1] - ustart;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (uint64_t)gridDim.x * blockDim.x)
        out[ustart + i] = (uint8_t)~P[i];
}

// ------------------------------------------------------------------ xxHash32 (src/xxhash32/xxhash32.js:21-97)
constexpr uint32_t P32_1 = 2654435761u, P32_2 = 2246822519u, P32_3 = 3266489917u, P32_4 = 668265263u, P32_5 = 374761393u;
__device__ __forceinline__ uint32_t rotl32(uint32_t x, int r) { return __funnelshift_l(x, x, r); }
__device__ __forceinline__ uint32_t xxh_round(uint32_t v, uint32_t w) { return rotl32(v + w * P32_2, 13) * P32_1; }   // :40-42

// tail after the 16-byte stripes (:70-95); executed by one lane
__device__ __forceinline__ uint32_t xxh_finish(uint32_t h, const uint8_t *p, const uint8_t *end, uint32_t len) {
    h += len;
    while (p + 4 <= end) { h = rotl32(h + ld32u(p) * P32_3, 17) * P32_4; p += 4; }
    while (p < end) { h = rotl32(h + (uint32_t)(*p) * P32_5, 11) * P32_1; ++p; }
    h ^= h >> 15; h *= P32_2; h ^= h >> 13; h *= P32_3; h ^= h >> 16;
    return h;
}

// A quad of lanes hashes one item: lane a (0..3) owns accumulator v_{a+1} and reads word a of every stripe.
// The four accumulators are independent serial chains (non-associative), so an item cannot be split further.
__device__ __forceinline__ uint32_t xxh32_quad(const uint8_t *p, uint32_t len, uint32_t seed, uint32_t a, uint32_t quad_mask) {
    const uint8_t *end = p + len;
    uint32_t h;
    uint32_t nstripes = len >> 4;
    if (nstripes) {
        uint32_t v = a == 0 ? seed + P32_1 + P32_2 : a == 1 ? seed + P32_2 : a == 2 ? seed : seed - P32_1;   // :29-32
        const uint8_t *q = p + 4 * a;
        uint32_t s = 0;
        // eight stripes per step, their loads issued together; two dependent operations per stripe (see k_xxh32_stream):
        // a' = (a >> 19)*P1 + (a*(P1 << 13) + x'*P2)
        auto eight = [&](const uint32_t (&x)[8]) {
            constexpr uint32_t K1 = P32_1 << 13;
            uint32_t acc = v + x[0] * P32_2;
#pragma unroll
            for (int u = 1; u < 8; ++u) {
                const uint32_t y = x[u] * P32_2;
                uint32_t c;
                asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(c) : "r"(acc), "r"(K1), "r"(y));
                asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(acc) : "r"(acc >> 19), "r"(P32_1), "r"(c));
            }
            v = rotl32(acc, 13) * P32_1;
        };
        const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(p) & 3u);
        if (mis == 0) {
            const uint32_t *w = reinterpret_cast<const uint32_t *>(q);
            for (; s + 8 <= nstripes; s += 8) {
                uint32_t x[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) x[u] = w[(s + u) * 4];
                eight(x);
            }
            for (; s < nstripes; ++s) v = xxh_round(v, w[s * 4]);
        } else {
            // any alignment (the packed payloads of a frame body): the word from the two aligned words around it; the step that
            // would read behind the last stripe is left to the loop below
            const uint32_t *w = reinterpret_cast<const uint32_t *>(q - mis);
            const uint32_t sh = mis * 8u;
            for (; s + 8 < nstripes; s += 8) {
                uint32_t lo[8], hi[8], x[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) { lo[u] = w[(s + u) * 4]; hi[u] = w[(s + u) * 4 + 1]; }
#pragma unroll
                for (int u = 0; u < 8; ++u) x[u] = __funnelshift_r(lo[u], hi[u], sh);
                eight(x);
            }
            for (; s < nstripes; ++s) v = xxh_round(v, ld32u(q + 16 * s));
        }
        const uint32_t base = lane_id() & ~3u;
        const uint32_t v1 = __shfl_sync(quad_mask, v, base), v2 = __shfl_sync(quad_mask, v, base + 1);
        const uint32_t v3 = __shfl_sync(quad_mask, v, base + 2), v4 = __shfl_sync(quad_mask, v, base + 3);
        h = rotl32(v1, 1) + rotl32(v2, 7) + rotl32(v3, 12) + rotl32(v4, 18);                  // :59-65
    } else {
        h = seed + P32_5;                                                                      // :67
    }
    return xxh_finish(h, p + (size_t)nstripes * 16, end, len);
}

// out[i] = xxh32(base + off[i], len[i]); if append != 0 the hash is also stored little-endian right after the
// item's bytes (LZ4 frame block checksum).
__global__ void __launch_bounds__(256)
k_xxh32_batch(const uint8_t *__restrict__ base, const uint64_t *__restrict__ off, const uint32_t *__restrict__ len,
              uint32_t n, uint32_t seed, uint32_t *__restrict__ out, uint8_t *append_base) {
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t item = tid >> 2, a = tid & 3u;
    const uint32_t quad_mask = 0xFu << (lane_id() & ~3u);
    if (item >= n) return;
    const uint32_t h = xxh32_quad(base + off[item], len[item], seed, a, quad_mask);
    if (a == 0) {
        if (out) out[item] = h;
        if (append_base) {
            uint8_t *q = append_base + off[item] + len[item];
            q[0] = (uint8_t)h; q[1] = (uint8_t)(h >> 8); q[2] = (uint8_t)(h >> 16); q[3] = (uint8_t)(h >> 24);
        }
    }
}

// One hash over one long buffer: a single quad is the whole parallelism the algorithm has.  The other 28
// lanes of the warp stage the stream through shared memory so the four chain lanes never wait on HBM.
// kAhead: chunks of 4 KiB held in registers ahead of the chain -- 1 for device memory, 3 for page-locked HOST memory read
// over PCIe (the content checksum of a frame whose bytes the caller already holds in pinned memory: ~2 us per round trip).
template <int kAhead>
__global__ void __launch_bounds__(32)
k_xxh32_stream(const uint8_t *__restrict__ data, uint64_t len, uint32_t seed, uint32_t *out,
               const uint32_t *__restrict__ acc_in /* nullable: resume from 4 accumulators */,
               uint32_t *acc_out /* nullable: stop after the stripes and store the accumulators (stateful update) */) {
    __shared__ __align__(16) uint32_t buf[2][1024];              // 2 x 4 KiB = 2 x 256 stripes
    const uint32_t lane = lane_id();
    const uint64_t nstripes = len >> 4;
    uint32_t v = lane == 0 ? seed + P32_1 + P32_2 : lane == 1 ? seed + P32_2 : lane == 2 ? seed : seed - P32_1;
    if (acc_in && lane < 4) v = acc_in[lane];
    const bool aligned = (reinterpret_cast<uintptr_t>(data) & 15u) == 0;
    uint64_t s = 0;
    if (aligned) {
        const uint4 *g = reinterpret_cast<const uint4 *>(data);
        const uint64_t nchunks = nstripes >> 8;                  // 256 stripes per chunk
        uint4 r[kAhead][8];
#pragma unroll
        for (int j = 0; j < kAhead; ++j) {
            if ((uint64_t)j < nchunks) {
#pragma unroll
                for (int u = 0; u < 8; ++u) r[j][u] = g[j * 256 + u * 32 + lane];
            }
        }
        for (uint64_t c = 0; c < nchunks; ++c) {
            // staged as x * P2 (:36-39's multiply, done here by all 32 lanes): the four chain lanes are left with a load and
            // the two dependent multiply-adds per stripe
            uint4 *b4 = reinterpret_cast<uint4 *>(buf[c & 1]);
#pragma unroll
            for (int u = 0; u < 8; ++u) b4[u * 32 + lane] = make_uint4(r[0][u].x * P32_2, r[0][u].y * P32_2, r[0][u].z * P32_2, r[0][u].w * P32_2);
#pragma unroll
            for (int j = 0; j + 1 < kAhead; ++j) {
#pragma unroll
                for (int u = 0; u < 8; ++u) r[j][u] = r[j + 1][u];
            }
            if (c + kAhead < nchunks) {
                const uint4 *gn = g + (c + kAhead) * 256;
#pragma unroll
                for (int u = 0; u < 8; ++u) r[kAhead - 1][u] = gn[u * 32 + lane];
            }
            __syncwarp();
            if (lane < 4) {
                // v' = rotl(v + x*P2, 13) * P1 is three dependent operations per stripe.  With a = v + x*P2 and
                // rotl(a,13) = (a << 13) + (a >> 19):  a' = (a >> 19)*P1 + (a*(P1 << 13) + x'*P2) -- the shift and the
                // second multiply-add run side by side, two dependent operations per stripe.
                const uint32_t *w = buf[c & 1] + lane;
                constexpr uint32_t K1 = P32_1 << 13;
                uint32_t a = v + w[0];
#pragma unroll 16
                for (int t = 1; t < 256; ++t) {
                    const uint32_t y = w[t * 4];
                    uint32_t c;                                 // fixed association (nvcc would re-order the sum into three links)
                    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(c) : "r"(a), "r"(K1), "r"(y));
                    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(a) : "r"(a >> 19), "r"(P32_1), "r"(c));
                }
                v = rotl32(a, 13) * P32_1;
            }
            __syncwarp();
        }
        s = nchunks << 8;
    }
    if (lane < 4) {
        const uint8_t *q = data + 4 * lane;
        for (; s < nstripes; ++s) v = xxh_round(v, ld32u(q + 16 * s));
    }
    if (acc_out) {                                               // stateful update: the caller keeps the tail and the total length
        if (lane < 4) acc_out[lane] = v;
        return;
    }
    const uint32_t v1 = __shfl_sync(FULL, v, 0), v2 = __shfl_sync(FULL, v, 1), v3 = __shfl_sync(FULL, v, 2), v4 = __shfl_sync(FULL, v, 3);
    if (lane == 0) {
        uint32_t h = nstripes ? rotl32(v1, 1) + rotl32(v2, 7) + rotl32(v3, 12) + rotl32(v4, 18) : seed + P32_5;
        *out = xxh_finish(h, data + nstripes * 16, data + len, (uint32_t)len);
    }
}

// ------------------------------------------------------------------ frame packing (bufferCompress.js:209-239)
// uniform block table for a contiguous buffer: off[i] = first + i*block, len[i] = min(block, total - i*block)
__global__ void k_uniform_blocks(uint64_t first, uint64_t total, uint32_t block, uint32_t n, uint64_t *off, uint32_t *len,
                                 uint64_t *dst_off, uint64_t dst_stride) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t o = (uint64_t)i * block;
    off[i] = first + o;
    len[i] = (uint32_t)((total - o) < block ? (total - o) : block);
    if (dst_off) dst_off[i] = (uint64_t)i * dst_stride;
}

// Stored-block rule (:221-231): compressed iff 0 < comp < len.  body[i] = 4 + size (+4 with block checksum).
// Single CTA: sizes + exclusive scan into pos[0..n] in one pass (n is at most a few hundred thousand).
// raw != 0: plain concatenation of the compressed blocks (packed batch output): body[i] = comp_len[i], no size word.
__global__ void __launch_bounds__(1024)
k_frame_layout(const uint32_t *__restrict__ src_len, const uint32_t *__restrict__ comp_len, uint32_t n, int block_checksum,
               uint64_t *pos /* n+1 */, uint64_t *data_off /* n: pos+4 */, uint32_t *data_len /* n */, int raw) {
    __shared__ uint64_t warp_tot[32];
    __shared__ uint64_t carry_s;
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    if (tid == 0) carry_s = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n; base += 1024) {
        const uint32_t i = base + tid;
        uint64_t body = 0;
        uint32_t sz = 0;
        if (i < n) {
            const uint32_t c = comp_len[i], L = src_len[i];
            sz = raw ? c : ((c > 0 && c < L) ? c : L);
            body = raw ? (uint64_t)sz : 4ull + sz + (block_checksum ? 4ull : 0ull);
        }
        uint64_t x = body;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint64_t y = __shfl_up_sync(FULL, x, o); if (lane >= (uint32_t)o) x += y; }
        if (lane == 31) warp_tot[warp] = x;
        __syncthreads();
        if (warp == 0) {
            uint64_t t = warp_tot[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const uint64_t y = __shfl_up_sync(FULL, t, o); if (lane >= (uint32_t)o) t += y; }
            warp_tot[lane] = t;                                   // inclusive over warps
        }
        __syncthreads();
        const uint64_t carry = carry_s;
        const uint64_t excl = carry + (warp ? warp_tot[warp - 1] : 0) + x - body;
        if (i < n) { pos[i] = excl; if (data_off) { data_off[i] = excl + 4; data_len[i] = sz; } }
        __syncthreads();
        if (tid == 1023) carry_s = carry + warp_tot[31];
        __syncthreads();
    }
    if (tid == 0) pos[n] = carry_s;
}

// One CTA per block: size word + payload (compressed bytes, or the raw block when stored) into the segment.
__global__ void __launch_bounds__(256)
k_frame_gather(const uint8_t *__restrict__ src, const uint64_t *__restrict__ src_off, const uint32_t *__restrict__ src_len,
               const uint8_t *__restrict__ comp, const uint64_t *__restrict__ comp_off, const uint32_t *__restrict__ comp_len,
               uint32_t n, const uint64_t *__restrict__ pos, uint8_t *__restrict__ seg, int raw) {
    for (uint32_t b = blockIdx.x; b < n; b += gridDim.x) {
        const uint32_t c = comp_len[b], L = src_len[b];
        const bool compressed = raw || (c > 0 && c < L);
        const uint32_t sz = compressed ? c : L;
        const uint8_t *s = compressed ? comp + comp_off[b] : src + src_off[b];
        uint8_t *d = seg + pos[b];
        if (!raw) {
            if (threadIdx.x < 4) {
                const uint32_t word = compressed ? sz : (sz | 0x80000000u);
                d[threadIdx.x] = (uint8_t)(word >> (8 * threadIdx.x));
            }
            d += 4;
        }
        // bytes up to the destination's next 16-byte boundary, then 16-byte stores whose source bytes come from aligned
        // 16-byte loads realigned in registers, then the last bytes (all loads stay inside [s, s + sz))
        const uint32_t head = static_cast<uint32_t>(-reinterpret_cast<intptr_t>(d)) & 15u;
        const uint32_t h = head < sz ? head : sz;
        if (threadIdx.x < h) d[threadIdx.x] = s[threadIdx.x];
        const uint8_t *sb = s + h;
        const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(sb) & 15u);
        uint32_t nv = (sz - h) >> 4;
        if (mis && nv) --nv;                                     // (the realigned form reads the granule behind each vector)
        uint4 *dv = reinterpret_cast<uint4 *>(d + h);
        if (mis == 0u) {
            const uint4 *sv = reinterpret_cast<const uint4 *>(sb);
            for (uint32_t i = threadIdx.x; i < nv; i += blockDim.x) dv[i] = __ldg(sv + i);
        } else {
            const uint4 *sv = reinterpret_cast<const uint4 *>(sb - mis);
            const uint32_t wsel = mis >> 2, sh = (mis & 3u) * 8u;
            for (uint32_t i = threadIdx.x; i < nv; i += blockDim.x) {
                const uint4 a = __ldg(sv + i), c4 = __ldg(sv + i + 1);
                const uint32_t v[8] = {a.x, a.y, a.z, a.w, c4.x, c4.y, c4.z, c4.w};
                uint32_t t[5];
#pragma unroll
                for (int k = 0; k < 5; ++k) t[k] = wsel == 0 ? v[k] : wsel == 1 ? v[k + 1] : wsel == 2 ? v[k + 2] : v[k + 3];
                dv[i] = make_uint4(__funnelshift_r(t[0], t[1], sh), __funnelshift_r(t[1], t[2], sh),
                                   __funnelshift_r(t[2], t[3], sh), __funnelshift_r(t[3], t[4], sh));
            }
        }
        const uint32_t done = h + (nv << 4);                     // at most 31 bytes left
        if (threadIdx.x < sz - done) d[done + threadIdx.x] = s[done + threadIdx.x];
    }
}

}  // namespace dlz4
