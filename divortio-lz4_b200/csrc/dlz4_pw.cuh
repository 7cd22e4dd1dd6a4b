// dlz4_pw.cuh -- the match finder of compressBlock (blockCompress.js:48-71,143-150) as a producer/walker pipeline.
//
// Why: the exact greedy parse is one dependent chain per block, and a chain's table is 32 KiB whatever is done, so an SM holds
// at most six or seven chains with their tables on chip.  One warp per chain (k_parse_fresh16) leaves that warp alone with
// both halves of the work -- the memory round trips (table entry -> candidate bytes -> compare) and the decisions (which
// position is probed next) -- and the chain runs at the SUM of their latencies with the SM's issue slots 30 % used.  Here a
// chain is a team of warps and the two halves overlap:
//
//   producers (kNP warps)   walk a FIXED grid of 32-position windows ahead of the parse, two windows per iteration, two positions
//                           per lane.  For every position p of a window: hash (:53), the table entry as it is at that
//                           moment, the candidate's bytes, verification of the first 32 bytes (:63, :147-150).  Then the
//                           producer RESOLVES THE SERIAL LOOP'S WALK through its window from every entry position at once
//                           (pw_resolve, pointer doubling over next(i) = i + (match ? length : 1)): the set of positions the
//                           loop probes if it arrives at p, and where it leaves the window.  One ring entry per position in
//                           tensor memory: x = {slot, match length}, y = {entry seen, exit}, z = probed set, and one ready
//                           word per ring slot in shared memory (the window number the slot holds).
//                           Nothing a producer does depends on the parse except the table entry it happened to read.
//   walker (1 warp)         the serial loop itself.  Per step it reads the entries of the window it stands in, takes the probed
//                           set and the exit of its own position, and lets the probed lanes validate and insert themselves:
//                           if every probed slot still holds what the producer saw, and no two probed positions share a slot
//                           (tags read back), the producer's walk is the serial loop's -- the hits among the probed positions
//                           are the records, the exit is the next position.  A same-slot pair or a stale entry cuts the step
//                           in front of it; the position behind the cut is probed the slow way, from global memory.  Matches of
//                           32 bytes and more end a walk and are measured by the walker (pw_extend).  Measured on log text:
//                           34 bytes per step, 3 % of the steps cut with producers <= 7 windows ahead.
//
// The walker never waits for global memory on its common path (ring in tensor memory, table in shared memory), the producers
// never wait for the walker except for ring space.  Sparse stretches (searchMatchCount > kPwRingSmc: incompressible data) and
// the last bytes of a block are probed by the walker alone with the batch step of dlz4_parse.cuh while the producers sleep.
//
// CTA shape: the table of a chain is 32 KiB whatever is done, and seven of them fill the shared memory of an SM; the rings
// live in tensor memory (TMEM), which nothing else uses.  A warp's tcgen05.ld/st reaches only the TMEM lanes
// 32 (w % 4) .. +31 of its lane quarter, so the three warps of a team share w % 4: 24 warps, two team slots per quarter,
// warp w is role (w / 4) % 3 of team (w % 4) + 4 (w / 12).  Slot 7 has no table and no work.  A ring entry's lane is
// position & 31, the lane of the 32x32b shape.
//
// Exactness: a producer's entry is used only under `slot value now == slot value seen`; everything else is decided by the
// walker from the table it alone writes, in probe order.  Output: the match records of dlz4_parse.cuh (k_encode_blocks
// turns them into the block's bytes).
#pragma once

namespace dlz4 {

constexpr int kPwChains = 7;                  // chains (teams) per CTA: 7 x (32 KiB table + 64 B control) of 227 KiB
constexpr int kPwProducers = 2;               // producer warps per team
constexpr int kPwThreads = 8 * (1 + kPwProducers) * 32;     // 8 team slots (2 per TMEM lane quarter), the last one idle
constexpr int kPwWin = 14;                    // windows of 32 positions in a chain's ring
constexpr uint32_t kPwTmemCols = 128;         // per CTA: 2 teams per lane quarter x 14 windows x 4 columns (x, y, z, unused) = 112
constexpr int kPwCtl = 64;                    // control bytes per chain (PwCtl)
constexpr int kPwChainBytes = kHashEntries * 2 + kPwCtl;
constexpr int kPwSmemBytes = kPwChains * kPwChainBytes + 16;  // + the TMEM address
constexpr uint32_t kPwRingSmc = 160u;         // the walker uses the ring while searchMatchCount <= this (steps of 1 and 2)
constexpr uint32_t kPwDone = 0x80000000u, kPwSparse = 0x40000000u;
constexpr bool kPwPrefetch = true;            // producers prefetch the second stage's lines and the next window pair's source lines
#ifndef DLZ4_PW_CAP
#define DLZ4_PW_CAP 32
#endif
constexpr uint32_t kPwCap = DLZ4_PW_CAP;              // producers pre-extend a match to this many bytes; the walker continues a longer one

struct PwCtl {                                // one per chain, in shared memory
    uint32_t w_pos;                           // walker's position (block-relative) | kPwSparse | kPwDone
    volatile uint32_t block;                  // block index of the team, 0xFFFFFFFF: no more work
    uint32_t ready[kPwWin];                   // ring slot ws holds the entries of window ready[ws] - 1 (0: none yet)
};
static_assert(sizeof(PwCtl) <= kPwCtl, "PwCtl");

__device__ __forceinline__ void pw_bar(uint32_t id, uint32_t nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
// The control words order the TMEM accesses of the team's warps: a write is released after tcgen05.wait + fence::before_thread_sync,
// and a read is acquired before fence::after_thread_sync + the tcgen05 access that depends on it.
__device__ __forceinline__ uint32_t pw_ld_acquire(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(v) : "r"((uint32_t)__cvta_generic_to_shared(p)) : "memory");
    return v;
}
__device__ __forceinline__ void pw_st_release(uint32_t *p, const uint32_t v) {
    asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(p)), "r"(v) : "memory");
}
__device__ __forceinline__ void pw_st_release2(uint32_t *p, const uint32_t v0, const uint32_t v1) {   // p 8-byte aligned
    asm volatile("st.release.cta.shared.v2.u32 [%0], {%1, %2};" ::"r"((uint32_t)__cvta_generic_to_shared(p)), "r"(v0), "r"(v1) : "memory");
}
__device__ __forceinline__ void pw_prefetch(const void *p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
__device__ __forceinline__ void tm_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tm_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// entries x, y, z of two windows (columns t .. t+7, lane = position & 31): complete when this returns
__device__ __forceinline__ void tm_st8(const uint32_t t, const uint32_t x0, const uint32_t y0, const uint32_t z0, const uint32_t x1,
                                       const uint32_t y1, const uint32_t z1) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %3, %4, %5, %6, %6};\n\t"
                 "tcgen05.wait::st.sync.aligned;" ::"r"(t), "r"(x0), "r"(y0), "r"(z0), "r"(x1), "r"(y1), "r"(z1) : "memory");
}
// loads that complete, and are ordered before what follows, when these return
__device__ __forceinline__ void tm_ld4(const uint32_t t, uint32_t &x, uint32_t &y, uint32_t &z) {
    uint32_t u;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];\n\t"
                 "tcgen05.wait::ld.sync.aligned;\n\t"
                 "tcgen05.fence::before_thread_sync;" : "=r"(x), "=r"(y), "=r"(z), "=r"(u) : "r"(t) : "memory");
}
__device__ __forceinline__ void tm_ld2(const uint32_t t, uint32_t &x, uint32_t &y) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];\n\t"
                 "tcgen05.wait::ld.sync.aligned;\n\t"
                 "tcgen05.fence::before_thread_sync;" : "=r"(x), "=r"(y) : "r"(t) : "memory");
}
// ring slot of window w (< 2048): w mod 14
__device__ __forceinline__ uint32_t pw_ws(const uint32_t w) { return w - (uint32_t)kPwWin * ((w * 74899u) >> 20); }
// Waits (whole warp) until ring slot ws holds window w, then orders the TMEM reads behind.
__device__ __forceinline__ void pw_wait_ready(const PwCtl *ctl, const uint32_t ws, const uint32_t w, const uint32_t ns) {
    while (!__all_sync(FULL, pw_ld_acquire(ctl->ready + ws) == w + 1u)) __nanosleep(ns);
    tm_fence_after();
}
// The walk of the serial loop through one aligned window of 32 positions, from every entry position at once (pointer
// doubling, all lanes): lane i holds the match length ml of position i (0: miss, kPwCap: 64 or more bytes -- the walk ends
// there, the walker measures the match).  Returns the set of positions the walk from position i probes (bit j = position j)
// and, in `exitp`, where it leaves the window: 32..94 window-relative, or 255 for a walk that ended at a capped match.
__device__ __forceinline__ uint32_t pw_resolve(const uint32_t ml, const uint32_t lane, uint32_t &exitp) {
    uint32_t n = ml == kPwCap ? 255u : lane + (ml ? ml : 1u);
    uint32_t m = 1u << lane;
#pragma unroll
    for (int r = 0; r < 5; ++r) {
        const uint32_t mj = __shfl_sync(FULL, m, n), nj = __shfl_sync(FULL, n, n);      // (source lane = n mod 32)
        if (n < 32u) { m |= mj; n = nj; }
    }
    exitp = n;
    return m;
}

// common prefix of base[s0 + eb ..] and base[m0 + eb ..] from byte eb on, bounded by matchLimit (:147-150); all lanes.
// First 128 bytes four at a time per lane (most matches end there); a match that is still running is compared 16 bytes
// per lane from a 16-byte-aligned source address on, 2 KiB per memory round trip (zero runs, periodic data).
__device__ __forceinline__ uint32_t pw_extend(const uint8_t *__restrict__ base, int32_t s0, int32_t m0, int32_t eb,
                                              int32_t matchLimit, uint32_t lane) {
    const int32_t back = s0 - m0;
    auto round4 = [&](int32_t e0, uint32_t &res) -> bool {                     // 128 bytes from e0; true: the match ends in them
        const int32_t q = s0 + e0 + 4 * (int32_t)lane;
        int32_t nv = matchLimit - q;
        nv = nv > 4 ? 4 : nv;
        int32_t eq = 0;
        if (nv > 0) {
            const uint32_t x = ld32u(base + q) ^ ld32u(base + q - back);
            const int32_t e = x ? ((__ffs(x) - 1) >> 3) : 4;
            eq = e < nv ? e : nv;
        }
        const uint32_t stop = __ballot_sync(FULL, eq < 4);
        if (!stop) return false;
        const int l = __ffs(stop) - 1;
        res = (uint32_t)(e0 + 4 * l + __shfl_sync(FULL, eq, l));
        return true;
    };
    uint32_t res = 0;
    if (round4(eb, res)) return res;
    eb += 128;
    // up to the next 16-byte boundary of the source address (at most one more round of 128 covers it)
    const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(base + s0 + eb) & 15u);
    if (mis) {
        if (round4(eb, res)) return res;
        eb += 128 - (int32_t)mis;                                                // bytes [eb, eb + 128) are equal; resume aligned inside them
        eb -= 112;                                                               // (eb + 128 - mis) - 112: first aligned address behind the old eb
    }
    // aligned phase: lane compares bytes [q, q+16), q = s0 + eb + 16 lane (+ 512 u); candidate bytes from two aligned granules
    const uint8_t *cb = base + s0 + eb - back;
    const uint32_t cmis = (uint32_t)(reinterpret_cast<uintptr_t>(cb) & 15u);
    const uint32_t wsel = cmis >> 2, bsh = (cmis & 3u) * 8u;
    for (;; eb += 2048) {
        uint32_t eqb[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int32_t q = s0 + eb + 512 * u + 16 * (int32_t)lane;
            int32_t nv = matchLimit - q;
            nv = nv > 16 ? 16 : nv;
            eqb[u] = 0;
            if (nv > 0) {
                const uint4 a = __ldg(reinterpret_cast<const uint4 *>(base + q));
                const uint4 *cp = reinterpret_cast<const uint4 *>(base + q - back - (int32_t)cmis);
                const uint4 c0 = __ldg(cp), c1 = __ldg(cp + 1);
                uint32_t v[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
                uint32_t t[5];
#pragma unroll
                for (int i = 0; i < 5; ++i) t[i] = wsel == 0 ? v[i] : wsel == 1 ? v[i + 1] : wsel == 2 ? v[i + 2] : v[i + 3];
                const uint32_t x0 = a.x ^ __funnelshift_r(t[0], t[1], bsh), x1 = a.y ^ __funnelshift_r(t[1], t[2], bsh);
                const uint32_t x2 = a.z ^ __funnelshift_r(t[2], t[3], bsh), x3 = a.w ^ __funnelshift_r(t[3], t[4], bsh);
                uint32_t e = x0 ? ((uint32_t)(__ffs(x0) - 1) >> 3) : x1 ? 4u + ((uint32_t)(__ffs(x1) - 1) >> 3)
                           : x2 ? 8u + ((uint32_t)(__ffs(x2) - 1) >> 3) : x3 ? 12u + ((uint32_t)(__ffs(x3) - 1) >> 3) : 16u;
                eqb[u] = e < (uint32_t)nv ? e : (uint32_t)nv;
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const uint32_t stop = __ballot_sync(FULL, eqb[u] < 16u);
            if (stop) { const int l = __ffs(stop) - 1; return (uint32_t)(eb + 512 * u + 16 * l) + __shfl_sync(FULL, eqb[u], l); }
        }
    }
}

// ring entry: x = slot (14 bits) | match length (7) << 14; y = entry seen | exit << 16; z = probed set (pw_resolve)

// candidate bytes (three aligned 16-byte granules, `cs` = byte offset of the first wanted byte inside the first) against
// the 32 bytes Sw[0..7]: number of equal leading bytes, 0..32.  Branch-free like wide_verify.
__device__ __forceinline__ uint32_t pw_count32(const uint4 &q0, const uint4 &q1, const uint4 &q2, const uint32_t cs, const uint32_t *Sw) {
    uint32_t v[12] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x, q2.y, q2.z, q2.w};
    const bool s8 = (cs & 8u) != 0, s4 = (cs & 4u) != 0;
#pragma unroll
    for (int k = 0; k < 10; ++k) v[k] = s8 ? v[k + 2] : v[k];
#pragma unroll
    for (int k = 0; k < 9; ++k) v[k] = s4 ? v[k + 1] : v[k];
    const uint32_t csh = (cs & 3u) * 8u;
    uint32_t x[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) x[k] = Sw[k] ^ __funnelshift_r(v[k], v[k + 1], csh);
    const bool h4 = (x[0] | x[1] | x[2] | x[3]) == 0u;
    const uint32_t y0 = h4 ? x[4] : x[0], y1 = h4 ? x[5] : x[1], y2 = h4 ? x[6] : x[2], y3 = h4 ? x[7] : x[3];
    const bool h2 = (y0 | y1) == 0u;
    const uint32_t z0 = h2 ? y2 : y0, z1 = h2 ? y3 : y1;
    const bool h1 = z0 == 0u;
    const uint32_t zz = h1 ? z1 : z0;
    return (h4 ? 16u : 0u) + (h2 ? 8u : 0u) + (h1 ? 4u : 0u) + (zz ? ((uint32_t)(__ffs(zz) - 1) >> 3) : 4u);
}

// ---- producer: the windows k and k+1 (positions 32k .. 32k+63) of the block at `base`, two positions per lane -- two
//      independent instruction streams, so the memory round trips (source words, table entry, candidate bytes) overlap.
//      two == false: window k only (the last window of a block).
__device__ __forceinline__ void pw_produce2(const uint8_t *__restrict__ base, const uint32_t k, const bool two, const uint16_t *tab,
                                            const uint32_t tcol, PwCtl *ctl, const uint32_t lane) {
    const uint32_t pa = 32u * k + lane, pb = pa + 32u;
    const uintptr_t ba = reinterpret_cast<uintptr_t>(base);
    const uint32_t a = (uint32_t)(ba & 3u) + pa;
    const uint32_t *wp = reinterpret_cast<const uint32_t *>(ba & ~(uintptr_t)3) + (a >> 2);
    const uint32_t sh = (a & 3u) * 8u;
    uint32_t w[17];
#pragma unroll
    for (int i = 0; i < 9; ++i) w[i] = __ldg(wp + i);
#pragma unroll
    for (int i = 9; i < 17; ++i) w[i] = two ? __ldg(wp + i) : 0u;
    uint32_t S[16];                                                             // bytes pa .. pa+63 (pb = pa + 32)
#pragma unroll
    for (int i = 0; i < 16; ++i) S[i] = __funnelshift_r(w[i], w[i + 1], sh);
    const uint32_t ha = (S[0] * 2654435761u) >> 18, hb = (S[8] * 2654435761u) >> 18;   // :53
    const uint32_t seena = *reinterpret_cast<const volatile uint16_t *>(tab + ha);     // the slots as they are right now
    const uint32_t seenb = *reinterpret_cast<const volatile uint16_t *>(tab + hb);
    const bool oka = seena != pa, okb = two && seenb != pb;                      // :62 with the 16-bit table (Tab16: 0 = position 0)
    const uint32_t la = oka ? seena : pa, lb = okb ? seenb : pa;                // no candidate: read at an own address
    const uint32_t csa = ((uint32_t)(ba & 15u) + la) & 15u, csb = ((uint32_t)(ba & 15u) + lb) & 15u;
    const uint4 *cqa = reinterpret_cast<const uint4 *>(base + la - csa), *cqb = reinterpret_cast<const uint4 *>(base + lb - csb);
    const uint4 qa0 = __ldg(cqa), qa1 = __ldg(cqa + 1), qa2 = __ldg(cqa + 2);
    const uint4 qb0 = __ldg(cqb), qb1 = __ldg(cqb + 1), qb2 = __ldg(cqb + 2);
    if (kPwPrefetch) {
        // what the second stage reads if 32 bytes match (granules 3, 4 and the source words behind +64): start the round trip now
        pw_prefetch(cqa + 4);
        if (two) { pw_prefetch(cqb + 4); pw_prefetch(wp + 24); }
    }
    const uint32_t va = wide_verify(qa0, qa1, qa2, csa, S), vb = wide_verify(qb0, qb1, qb2, csb, S + 8);     // 0 or 4..32
    uint32_t mla = oka ? va : 0u, mlb = okb ? vb : 0u;
    if (kPwCap > 32u && __any_sync(FULL, mla == 32u || mlb == 32u)) {
        // second stage for the positions whose 32 bytes all matched: bytes 32..63 (:147-150 continued)
        if (mla == 32u) {
            const uint4 q3 = __ldg(cqa + 3), q4 = __ldg(cqa + 4);
            mla += two ? pw_count32(qa2, q3, q4, csa, S + 8) : 0u;               // (one window only: no bytes behind +32 loaded; stays 32,
        }                                                                        //  fixed below)
        if (mlb == 32u) {
            uint32_t w2[9], S2[8];
#pragma unroll
            for (int i = 0; i < 9; ++i) w2[i] = __ldg(wp + 16 + i);
#pragma unroll
            for (int i = 0; i < 8; ++i) S2[i] = __funnelshift_r(w2[i], w2[i + 1], sh);
            const uint4 q3 = __ldg(cqb + 3), q4 = __ldg(cqb + 4);
            mlb += pw_count32(qb2, q3, q4, csb, S2);
        }
    }
    if (kPwCap > 32u && !two && mla == 32u) {
        // last window of the block, produced alone: its bytes 32..63 come from a direct load
        uint32_t w2[9], S2[8];
#pragma unroll
        for (int i = 0; i < 9; ++i) w2[i] = __ldg(wp + 8 + i);
#pragma unroll
        for (int i = 0; i < 8; ++i) S2[i] = __funnelshift_r(w2[i], w2[i + 1], sh);
        const uint4 q3 = __ldg(cqa + 3), q4 = __ldg(cqa + 4);
        mla += pw_count32(qa2, q3, q4, csa, S2);
    }
    uint32_t exa, exb;
    const uint32_t pma = pw_resolve(mla, lane, exa), pmb = pw_resolve(mlb, lane, exb);
    // k is even, so the pair's ring slots ws, ws + 1 are adjacent (kPwWin is even): one store.  The walker has left the
    // windows these slots held behind (w_pos, read before this call; the fence orders the store after that read).
    const uint32_t ws = pw_ws(k);
    __syncwarp();                                                               // (tcgen05.st is warp-collective)
    tm_fence_after();
    tm_st8(tcol + 4u * ws, ha | (mla << 14), seena | (exa << 16), pma, hb | (mlb << 14), seenb | (exb << 16), pmb);
    tm_fence_before();
    if (two) pw_st_release2(ctl->ready + ws, k + 1u, k + 2u);
    else pw_st_release(ctl->ready + ws, k + 1u);
}

// Producer j of kNP takes the window pairs (2j, 2j+1), (2j + 2 kNP, ...), ... -- skipping those the walker has left behind -- and
// stays at most `lead` windows ahead of the walker's window.
__device__ __forceinline__ void pw_producer(const uint8_t *__restrict__ base, const uint32_t nwin, const uint32_t lead,
                                            const uint32_t j, const uint16_t *tab, const uint32_t tcol, PwCtl *ctl, const uint32_t lane,
                                            const uint32_t full_ns) {
    constexpr int kNP = kPwProducers;
    uint32_t k = 2u * j;
    PT_DECL
    for (;;) {
        const uint32_t wpos = pw_ld_acquire(&ctl->w_pos);
        if (wpos & kPwDone) break;
        if (wpos & kPwSparse) { __nanosleep(1024); PT_MARK(8) continue; }
        const uint32_t wk = wpos >> 5;
        // skip the window pairs the walker has left behind (a long match moves it by hundreds of windows at once)
        if (k + 1u < wk) k += (wk - k - 2u + 2u * (uint32_t)kNP) / (2u * (uint32_t)kNP) * (2u * (uint32_t)kNP);
        if (k >= nwin) { __nanosleep(1024); PT_MARK(8) continue; }
        if (k + 1u >= wk + lead) { __nanosleep(full_ns); PT_MARK(7) continue; }
        if (kPwPrefetch && lane < 2u && k + 2u * (uint32_t)kNP < nwin) pw_prefetch(base + 32u * (k + 2u * (uint32_t)kNP) + 128u * lane);
        pw_produce2(base, k, k + 1u < nwin, tab, tcol, ctl, lane);
        PT_MARK(6) PT_COUNT(13, 1)
        k += 2u * (uint32_t)kNP;
    }
    PT_FLUSH
}

// ---- walker: the serial loop.  Returns the number of records written.
__device__ __forceinline__ uint32_t pw_walker(const uint8_t *__restrict__ base, const int32_t len, const uint32_t nwin, uint16_t *tab,
                                              const uint32_t tcol, PwCtl *ctl, uint64_t *__restrict__ rec, const uint32_t lane) {
    const uint32_t lt = (1u << lane) - 1u;
    const int32_t sEnd = len;
    const int32_t mflimit = sEnd - 12;                                          // blockCompress.js:34
    const int32_t matchLimit = sEnd - 5;                                        // :35
    const int32_t plimit = (int32_t)(32u * nwin);                               // positions below have ring entries
    const int32_t rlimit = plimit < mflimit ? plimit : mflimit;
    int32_t sIndex = 0;
    uint32_t smc = 67;                                                          // :40 searchMatchCount
    uint32_t nrec = 0;
    uint32_t pub = 0;                                                           // what ctl->w_pos holds
    const SrcFlat S{base};
    Tab16 T{tab, 0};
    uint2 *const rec2 = reinterpret_cast<uint2 *>(rec);
    PT_DECL

    while (sIndex < mflimit) {                                                  // :48
        if (smc <= 96u && (sIndex | 31) < rlimit) {
            // ---- path step: while searchMatchCount stays below 128 the schedule steps by 1 (:66-67), so the parse inside an
            //      aligned window of 32 positions is a walk over the producers' match lengths: from a hit to the position
            //      behind its match, from a miss to the next position.  The PRODUCER of the window has already resolved that
            //      walk from every possible entry position (pw_resolve); the walker reads the walk that starts at its own
            //      position -- the set PM of PROBED positions and where the walk leaves the window -- from that position's
            //      ring entry.  The probed lanes validate (slot unchanged since the producer looked, no two of them in one
            //      slot) and insert themselves; the hits among them are the records.
            const uint32_t s = (uint32_t)sIndex, wbase = s & ~31u, sl = s & 31u;
            if (pub != wbase) { pub = wbase; if (lane == 0) pw_st_release(&ctl->w_pos, wbase); }
            const uint32_t p = wbase + lane;
            const uint32_t w = wbase >> 5, ws = pw_ws(w);
            PT_MARK(14)
            while (!__all_sync(FULL, pw_ld_acquire(ctl->ready + ws) == w + 1u)) {
                __nanosleep(32);
                PT_COUNT(15, 1)
            }
            tm_fence_after();
            uint32_t ex, ey, ez;
            tm_ld4(tcol + 4u * ws, ex, ey, ez);
            PT_MARK(1)
            const uint32_t PM = __shfl_sync(FULL, ez, sl), exitp = __shfl_sync(FULL, ey, sl) >> 16;     // entry of position s
            const uint32_t seen = ey & 0xFFFFu;
            const uint32_t h = ex & 0x3FFFu, ml = (ex >> 14) & 127u;
            const uint32_t cur = tab[h];                                       // :54 (state before this step)
            const uint32_t claim = __ballot_sync(FULL, ml != 0u);
            const bool probed = (PM >> lane) & 1u;
            const uint32_t tag = p & 0xFFFFu;
            // two probed positions in one slot (the later one would find the earlier one's insert, not what its producer saw)
            // show up when the tags are read back (match.any instead of the read-back: 920 against 500 cycles for this part)
            __syncwarp();                                                      // every lane holds its `cur` before any slot changes
            if (probed) tab[h] = (uint16_t)tag;                                 // :55
            __syncwarp();
            const uint32_t r = probed ? (uint32_t)tab[h] : tag;
            const uint32_t bad = __ballot_sync(FULL, probed && (r != tag || cur != seen));
            if (!bad) {
                const uint32_t HM = PM & claim;                                // the matches, in order
                const uint32_t nh = (uint32_t)__popc(HM);
                if (((HM >> lane) & 1u) && ml != kPwCap) rec2[nrec + (uint32_t)__popc(HM & lt)] = rec_pack(p, ml, p - cur);
                if (exitp == 255u) {
                    // the walk ended at a match of 32 or more bytes (the last probed position): its real length (:147-150)
                    const uint32_t c = 31u - (uint32_t)__clz(PM);
                    const uint32_t pc = wbase + c, curc = __shfl_sync(FULL, cur, c);
                    const uint32_t mlx = pw_extend(base, (int32_t)pc, (int32_t)curc, (int32_t)kPwCap, matchLimit, lane);
                    if (lane == 0) rec2[nrec + nh - 1u] = rec_pack(pc, mlx, pc - curc);
                    sIndex = (int32_t)(pc + mlx);
                    smc = 67u;
                } else {
                    sIndex = (int32_t)(wbase + exitp);
                    if (HM) smc = 67u + (uint32_t)__popc(PM & ~((2u << (31 - __clz(HM))) - 1u));      // misses behind the last match
                    else smc += (uint32_t)__popc(PM);
                }
                nrec += nh;
                PT_MARK(0) PT_COUNT(9, 1)
                continue;
            }
            // ---- a same-slot pair or a stale entry among the probed positions: the probed positions in front of the first
            //      such position are still the serial loop's (validated one by one, pairwise different slots); keep them, undo
            //      the rest, and probe the first position behind them the slow way
            const uint32_t inv = (probed && r != tag) ? min(tag, r) : 0xFFFFFFFFu;              // lower position of a pair
            const uint32_t cutpos = __reduce_min_sync(FULL, inv);
            const uint32_t stale = __ballot_sync(FULL, probed && cur != seen);
            const uint32_t Bl = min(cutpos == 0xFFFFFFFFu ? 32u : ((cutpos - wbase) & 0xFFFFu) + 1u, stale ? (uint32_t)__ffs(stale) - 1u : 32u);
            const uint32_t below = (1u << Bl) - 1u;                            // Bl <= 31
            if (probed && lane >= Bl) tab[h] = (uint16_t)cur;                   // undo
            __syncwarp();
            if (probed && lane < Bl) tab[h] = (uint16_t)tag;                    // (a kept lane may share its slot with an undone one)
            __syncwarp();
            const uint32_t keep = PM & below, HMk = keep & claim;
            if ((HMk >> lane) & 1u) rec2[nrec + (uint32_t)__popc(HMk & lt)] = rec_pack(p, ml, p - cur);
            nrec += (uint32_t)__popc(HMk);
            if (HMk) smc = 67u + (uint32_t)__popc(keep & ~((2u << (31 - __clz(HMk))) - 1u));
            else smc += (uint32_t)__popc(keep);
            sIndex = (int32_t)(wbase + (uint32_t)__ffs(PM & ~below) - 1u);
            // one position, :50-71
            const uint32_t hx = __shfl_sync(FULL, h, (uint32_t)sIndex - wbase);
            const uint32_t cand = tab[hx];
            __syncwarp();
            if (lane == 0) tab[hx] = (uint16_t)sIndex;
            __syncwarp();
            uint32_t mlx = 0;
            if (cand != (uint32_t)sIndex) mlx = pw_extend(base, sIndex, (int32_t)cand, 0, matchLimit, lane);
            if (mlx >= 4u) {
                if (lane == 0) rec2[nrec] = rec_pack((uint32_t)sIndex, mlx, (uint32_t)sIndex - cand);
                ++nrec;
                sIndex += (int32_t)mlx;
                smc = 67u;
            } else {
                sIndex += (int32_t)(smc >> 6);
                ++smc;
            }
            PT_MARK(4) PT_COUNT(10, 1)
            continue;
        }
        if (smc <= kPwRingSmc && sIndex < rlimit) {
            // ---- ring step: the next 32 probe positions of the skip schedule
            const uint32_t bs = skip_sum(smc);
            const int32_t p = sIndex + (int32_t)(skip_sum(smc + lane) - bs);
            const bool valid = p < rlimit;
            if (pub != (uint32_t)sIndex) { pub = (uint32_t)sIndex; if (lane == 0) pw_st_release(&ctl->w_pos, pub); }
            // the valid probes (steps of 1 and 2) lie in at most three windows: each lane takes its entry from the
            // window's lane p & 31
            const uint32_t w0 = (uint32_t)sIndex >> 5;
            const uint32_t wl = (uint32_t)min(__shfl_sync(FULL, p, 31), rlimit - 1) >> 5;
            uint32_t lo = 0, ye = 0;
            for (uint32_t w = w0; w <= wl; ++w) {
                const uint32_t ws = pw_ws(w);
                pw_wait_ready(ctl, ws, w, 20);
                uint32_t xw, yw;
                tm_ld2(tcol + 4u * ws, xw, yw);
                xw = __shfl_sync(FULL, xw, (uint32_t)p & 31u);
                yw = __shfl_sync(FULL, yw, (uint32_t)p & 31u);
                if (((uint32_t)p >> 5) == w) { lo = xw; ye = yw; }
            }
            const uint32_t seen = ye & 0xFFFFu;
            const uint32_t h = lo & 0x3FFFu, ml = (lo >> 14) & 127u;
            const uint32_t cur = tab[h];                                       // :54 (state before this step)
            const uint32_t claim = __ballot_sync(FULL, valid && ml != 0u);
            const uint32_t f = claim ? (uint32_t)__ffs(claim) - 1u : 32u;
            const bool active = valid && lane <= f;
            const uint32_t tag = (uint32_t)p & 0xFFFFu;
            __syncwarp();                                                      // every lane holds its `cur` before any slot changes
            if (active) tab[h] = (uint16_t)tag;                                 // :55
            __syncwarp();
            const uint32_t r = active ? (uint32_t)tab[h] : tag;
            const uint32_t bad = __ballot_sync(FULL, active && (r != tag || cur != seen));
            if (!bad) {
                if (claim) {
                    // lanes below f: misses; lane f: the match (:71, :143-174)
                    const int32_t pf = sIndex + (int32_t)(skip_sum(smc + f) - bs);
                    const uint32_t curf = __shfl_sync(FULL, cur, f);
                    uint32_t mlf = __shfl_sync(FULL, ml, f);
                    if (mlf == kPwCap) mlf = pw_extend(base, pf, (int32_t)curf, (int32_t)kPwCap, matchLimit, lane);
                    if (lane == 0) rec2[nrec] = rec_pack((uint32_t)pf, mlf, (uint32_t)pf - curf);
                    ++nrec;
                    sIndex = pf + (int32_t)mlf;
                    smc = 67u;
                } else {
                    const uint32_t nv = (uint32_t)__popc(__ballot_sync(FULL, valid));
                    sIndex += (int32_t)(skip_sum(smc + nv) - bs);
                    smc += nv;
                }
                PT_MARK(2) PT_COUNT(11, 1)
                continue;
            }
            // ---- cut: the lanes in front of the first same-slot pair / stale entry are plain misses
            const uint32_t inv = (active && r != tag) ? min((uint32_t)p, r) : 0xFFFFFFFFu;      // lower position of the pair
            const uint32_t cutpos = __reduce_min_sync(FULL, inv);
            const uint32_t grp = __ballot_sync(FULL, active && (uint32_t)p <= cutpos);
            const uint32_t stale = __ballot_sync(FULL, active && cur != seen);
            const uint32_t c = min((uint32_t)__popc(grp), stale ? (uint32_t)__ffs(stale) - 1u : 32u);
            if (active && lane >= c) tab[h] = (uint16_t)cur;                    // undo
            __syncwarp();
            if (active && lane < c) tab[h] = (uint16_t)tag;                     // (a kept lane may share its slot with an undone one)
            __syncwarp();
            if (c != 0u) {
                sIndex += (int32_t)(skip_sum(smc + c) - bs);
                smc += c;
                PT_MARK(2) PT_COUNT(11, 1)
                continue;
            }
            // ---- the position at the head of the step is stale: probe it the slow way (one position, :50-71)
            const uint32_t h0 = __shfl_sync(FULL, h, 0);
            const uint32_t cand = tab[h0];
            __syncwarp();
            if (lane == 0) tab[h0] = (uint16_t)sIndex;
            __syncwarp();
            uint32_t ml0 = 0;
            if (cand != (uint32_t)sIndex) ml0 = pw_extend(base, sIndex, (int32_t)cand, 0, matchLimit, lane);
            if (ml0 >= 4u) {
                if (lane == 0) rec2[nrec] = rec_pack((uint32_t)sIndex, ml0, (uint32_t)sIndex - cand);
                ++nrec;
                sIndex += (int32_t)ml0;
                smc = 67u;
            } else {
                sIndex += (int32_t)(smc >> 6);
                ++smc;
            }
            PT_MARK(2) PT_COUNT(11, 1)
            continue;
        }

        // ---- batch step (sparse schedule, block tail): the walker alone, from global memory; producers sleep
        if (smc > kPwRingSmc && sIndex < rlimit) {
            const uint32_t v = (uint32_t)sIndex | kPwSparse;
            if (pub != v) { pub = v; if (lane == 0) pw_st_release(&ctl->w_pos, pub); }
        }
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
            PT_MARK(3) PT_COUNT(12, 1)
            continue;
        }
        const int32_t s0 = __shfl_sync(FULL, p, hl);
        const int32_t m0 = __shfl_sync(FULL, cand, hl);
        smc = 67;
        const uint32_t ml = pw_extend(base, s0, m0, 4, matchLimit, lane);
        if (lane == 0) rec2[nrec] = rec_pack((uint32_t)s0, ml, (uint32_t)(s0 - m0));
        ++nrec;
        sIndex = s0 + (int32_t)ml;
        PT_MARK(3) PT_COUNT(12, 1)
    }
    PT_MARK(5)
    PT_FLUSH
    return nrec;
}

// Fresh independent blocks <= 64 KiB as producer/walker teams.  CTA = kPwChains teams (warp -> team: header); role 0 of a
// team = walker, 1..kPwProducers = producers.  Output: the match records of every block and their number, for
// k_encode_blocks.  (An encoder warp inside the team was measured: it delays the team's next block; the encoder stays a
// kernel of its own.)
__global__ void __launch_bounds__(kPwThreads, 1)
k_parse_pw(const uint8_t *__restrict__ src, const uint64_t *__restrict__ src_off, const uint32_t *__restrict__ src_len,
           uint32_t nblocks, uint64_t *__restrict__ rec_base, uint64_t rec_stride /* records per block */,
           uint32_t *__restrict__ nrec_out, uint32_t *counter, uint32_t lead,
           uint32_t full_ns /* a producer with a full ring sleeps this long: the ring buffers several windows */) {
    extern __shared__ __align__(16) uint8_t smem[];
    constexpr uint32_t kRoles = 1 + kPwProducers;
    constexpr uint32_t kTeam = kRoles * 32;
    const uint32_t lane = lane_id(), warp = threadIdx.x >> 5;
    const uint32_t quarter = warp & 3u, tslot = (warp >> 2) / kRoles, role = (warp >> 2) % kRoles;
    const uint32_t chain = quarter + 4u * tslot;
    uint32_t *const taddr_smem = reinterpret_cast<uint32_t *>(smem + kPwChains * kPwChainBytes);
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n\t"
                     "tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;"
                     ::"r"((uint32_t)__cvta_generic_to_shared(taddr_smem)), "r"(kPwTmemCols) : "memory");
    }
    tm_fence_before();
    __syncthreads();
    tm_fence_after();
    const uint32_t taddr = *taddr_smem;
    // column 0 of the team's ring in its lane quarter
    const uint32_t tcol = taddr + ((32u * quarter) << 16) + tslot * (uint32_t)(kPwWin * 4);
    if (chain < (uint32_t)kPwChains) {
        const uint32_t tid = role * 32u + lane;                                 // thread index inside the team
        uint8_t *const cb = smem + (size_t)chain * kPwChainBytes;
        uint16_t *const tab = reinterpret_cast<uint16_t *>(cb);
        PwCtl *const ctl = reinterpret_cast<PwCtl *>(cb + kHashEntries * 2);
        const uint32_t bar = 1u + chain;
        // first block of a team: spread over the CTAs first, then over the teams of a CTA; later ones from the queue
        uint32_t first = chain * gridDim.x + blockIdx.x;
        const uint32_t qbase = gridDim.x * (uint32_t)kPwChains;
        bool have_first = true;
        for (;;) {
            pw_bar(bar, kTeam);                                                // everyone is done with the previous block
            if (role == 0 && lane == 0) {
                uint32_t b;
                if (have_first) b = first; else b = qbase + atomicAdd(counter, 1u);
                ctl->block = b < nblocks ? b : 0xFFFFFFFFu;
                ctl->w_pos = 0u;
            }
            have_first = false;
            pw_bar(bar, kTeam);
            const uint32_t b = ctl->block;
            if (b == 0xFFFFFFFFu) break;
            const uint32_t len = src_len[b];
            if (len > 65536u) {
                if (role == 0 && lane == 0) nrec_out[b] = 0xFFFFFFFFu;
                continue;
            }
            {   // empty table (bufferCompress.js:182 / :235), empty ring (the ready words gate every TMEM read)
                uint4 *z = reinterpret_cast<uint4 *>(cb);
                for (uint32_t i = tid; i < kHashEntries * 2 / 16; i += kTeam) z[i] = make_uint4(0, 0, 0, 0);
                if (tid < (uint32_t)kPwWin) ctl->ready[tid] = 0u;
            }
            pw_bar(bar, kTeam);
            const uint8_t *base = src + src_off[b];
            uint64_t *const rec = rec_base + (uint64_t)b * rec_stride;
            // windows whose loads stay inside the block: position 32k+31 reads its own bytes up to +71 and, for a candidate
            // right below it, 16-byte granules up to +79
            const uint32_t nwin = len >= 112u ? (len - 111u) / 32u + 1u : 0u;
            if (role == 0) {
                const uint32_t n = pw_walker(base, (int32_t)len, nwin, tab, tcol, ctl, rec, lane);
                if (lane == 0) {
                    nrec_out[b] = n;
                    pw_st_release(&ctl->w_pos, kPwDone);
                }
            } else {
                pw_producer(base, nwin, lead, role - 1u, tab, tcol, ctl, lane, full_ns);
            }
        }
    }
    // every warp, the idle slot's too: the TMEM is freed when no team uses it any more (a CTA that exits without the
    // dealloc leaves its columns taken for the next kernel on the SM)
    tm_fence_before();
    __syncthreads();
    tm_fence_after();
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(kPwTmemCols) : "memory");
}

}  // namespace dlz4
