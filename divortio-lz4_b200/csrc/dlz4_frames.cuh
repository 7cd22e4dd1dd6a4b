// dlz4_frames.cuh -- sm_100a kernels of the batched frame calls (dlz4_frames_*_batch*): many independent LZ4 frames in one pass.
//
// Frames are independent, so every per-frame step is one thread or one warp per frame; inside a frame the block table stays a
// short serial loop.  The blocks themselves go through the existing compressors (launch_compress, and a chain kernel with one
// CTA per linked frame) and the existing block decoder (decompress_block_warp_v2).
//
//   scan        k_scan_local / k_scan_add      exclusive scan of u64 counts, any length (multi-pass)
//   compress    k_fb_count -> scan -> k_fb_blocks -> scan of the compressed bounds -> k_fb_lists -> compressors ->
//               k_fb_layout -> scan (frame_off) -> k_fb_place -> k_frame_gather [+ k_xxh32_batch] -> k_fb_headers
//   decompress  k_fd_parse -> scan -> k_fd_parse (block table) -> k_fd_decode [+ k_xxh32_batch] -> k_fd_finish
#pragma once
#include "dlz4_kernels.cuh"

namespace dlz4 {

constexpr uint32_t kFbFrameMax = 0x7FFF0000u;           // frames of this size and more: DLZ4_E_TOO_LARGE (bufferCompress.js:127)

// ------------------------------------------------------------------ exclusive scan (u64), in place allowed
// Each CTA scans 1024 items; part[blockIdx.x] receives the CTA's total.
__global__ void __launch_bounds__(1024) k_scan_local(const uint64_t *in, uint64_t *out, uint64_t *part, uint32_t n) {
    __shared__ uint64_t warp_tot[32];
    const uint32_t tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const uint64_t i = (uint64_t)blockIdx.x * 1024u + tid;
    const uint64_t v = i < n ? in[i] : 0;
    uint64_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint64_t y = __shfl_up_sync(FULL, x, o); if (lane >= (uint32_t)o) x += y; }
    if (lane == 31) warp_tot[warp] = x;
    __syncthreads();
    if (warp == 0) {
        uint64_t t = warp_tot[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint64_t y = __shfl_up_sync(FULL, t, o); if (lane >= (uint32_t)o) t += y; }
        warp_tot[lane] = t;
    }
    __syncthreads();
    if (i < n) out[i] = (warp ? warp_tot[warp - 1] : 0) + x - v;
    if (tid == 0) part[blockIdx.x] = warp_tot[31];
}

__global__ void __launch_bounds__(1024) k_scan_add(uint64_t *out, const uint64_t *part, uint32_t n, uint32_t nparts) {
    const uint64_t i = (uint64_t)blockIdx.x * 1024u + threadIdx.x;
    if (i < n) out[i] += part[blockIdx.x];
    if (i == 0) out[n] = part[nparts];
}

// ------------------------------------------------------------------ compress
struct FbStats {
    unsigned long long src_bytes, bound_bytes, chain_blocks;
    uint32_t too_large, chains, first_blocks, pad;
};

// Blocks per frame (an empty frame has none), the linked frames of more than one block (one chain each) and the totals the
// host needs to size its scratch.
__global__ void __launch_bounds__(256) k_fb_count(const uint32_t *__restrict__ src_len, uint32_t nframes, uint32_t B, int linked,
                                                  int dict, uint64_t *nblk, uint32_t *chain_frames, FbStats *stats) {
    const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t lane = lane_id();
    uint64_t len = 0, nb = 0;
    uint32_t chain = 0, big = 0, first = 0;
    if (f < nframes) {
        len = src_len[f];
        nb = (len + B - 1) / B;
        nblk[f] = nb;
        big = len >= kFbFrameMax;
        chain = linked && nb > 1;
        first = dict && nb && !chain;                            // block 0 behind the dictionary, not part of a chain
    }
    const uint32_t cm = __ballot_sync(FULL, chain);
    uint32_t base = 0;
    if (lane == 0 && cm) base = atomicAdd(&stats->chains, (uint32_t)__popc(cm));
    base = __shfl_sync(FULL, base, 0);
    if (chain) chain_frames[base + __popc(cm & ((1u << lane) - 1u))] = f;
    uint64_t a = len, b = f < nframes ? 19 + len + (len / 65536 + 1) * 8 + 8 + 64 : 0, c = chain ? nb : 0;   // dlz4_frame_bound
#pragma unroll
    for (int o = 16; o; o >>= 1) {
        a += __shfl_xor_sync(FULL, a, o); b += __shfl_xor_sync(FULL, b, o); c += __shfl_xor_sync(FULL, c, o);
    }
    const uint32_t bigs = __popc(__ballot_sync(FULL, big)), firsts = __popc(__ballot_sync(FULL, first));
    if (lane == 0) {
        if (a) atomicAdd(&stats->src_bytes, (unsigned long long)a);
        if (b) atomicAdd(&stats->bound_bytes, (unsigned long long)b);
        if (c) atomicAdd(&stats->chain_blocks, (unsigned long long)c);
        if (bigs) atomicAdd(&stats->too_large, bigs);
        if (firsts) atomicAdd(&stats->first_blocks, firsts);
    }
}

// Block table of the batch: one warp per frame.  cls: 0 fresh block, 1 block 0 behind the dictionary, 2 part of a chain.
// Fresh and dictionary blocks are appended to their list (order is irrelevant: every block has its own output slot).
__global__ void __launch_bounds__(256) k_fb_blocks(const uint64_t *__restrict__ src_off, const uint32_t *__restrict__ src_len,
                                                   uint32_t nframes, uint32_t B, int linked, int dict,
                                                   const uint64_t *__restrict__ bfirst, uint64_t *soff, uint32_t *slen,
                                                   uint32_t *bframe, uint64_t *cbound, uint32_t *list, uint32_t list1_base,
                                                   uint32_t *list_count) {
    const uint32_t lane = lane_id();
    const uint32_t f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (f >= nframes) return;
    const uint64_t len = src_len[f], first = bfirst[f], nb = bfirst[f + 1] - first;
    const bool chain = linked && nb > 1;
    for (uint64_t k = lane; k < nb; k += 32) {
        const uint64_t b = first + k, o = k * B;
        const uint32_t l = (uint32_t)(len - o < B ? len - o : B);
        soff[b] = src_off[f] + o;
        slen[b] = l;
        bframe[b] = f;
        cbound[b] = ((uint64_t)l + l / 255 + 16 + 15) & ~15ull;
        if (!chain) {
            const uint32_t cls = (dict && k == 0) ? 1u : 0u;
            list[(cls ? list1_base : 0u) + atomicAdd(&list_count[cls], 1u)] = (uint32_t)b;
        }
    }
}

// Descriptors of one list for launch_compress: block list[j] -> (soff, slen, coff) at j.
__global__ void __launch_bounds__(256) k_fb_lists(const uint32_t *__restrict__ list, uint32_t n, const uint64_t *__restrict__ soff,
                                                  const uint32_t *__restrict__ slen, const uint64_t *__restrict__ coff,
                                                  uint64_t *l_soff, uint32_t *l_slen, uint64_t *l_coff) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const uint32_t b = list[j];
    l_soff[j] = soff[b]; l_slen[j] = slen[b]; l_coff[j] = coff[b];
}

__global__ void __launch_bounds__(256) k_fb_unlist(const uint32_t *__restrict__ list, uint32_t n, const uint32_t *__restrict__ l_clen,
                                                   uint32_t *clen) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) clen[list[j]] = l_clen[j];
}

// Staging of a linked frame for its chain: dictionary window ++ input, the input 16-byte aligned (the single-frame call's
// working buffer, bufferCompress.js:121-124).  One CTA per chain; the region comes from a bump allocator.
__global__ void __launch_bounds__(256) k_fb_stage(const uint8_t *__restrict__ src, const uint64_t *__restrict__ src_off,
                                                  const uint32_t *__restrict__ src_len, const uint32_t *__restrict__ chain_frames,
                                                  uint32_t nchains, const uint8_t *__restrict__ dwin, uint32_t dwin_len,
                                                  uint8_t *stage, unsigned long long *bump, uint64_t *stage_off) {
    __shared__ uint64_t base;
    const uint32_t c = blockIdx.x;
    if (c >= nchains) return;
    const uint32_t f = chain_frames[c];
    const uint64_t len = src_len[f];
    const uint64_t dpad = (dwin_len + 15u) & ~15u;
    if (threadIdx.x == 0) {
        base = atomicAdd(bump, (unsigned long long)(dpad + ((len + 15) & ~15ull) + 16));
        stage_off[c] = base + dpad - dwin_len;                   // where the window starts; the input follows at + dwin_len
    }
    __syncthreads();
    uint8_t *w = stage + base + dpad - dwin_len;
    for (uint32_t i = threadIdx.x; i < dwin_len; i += blockDim.x) w[i] = dwin[i];
    const uint8_t *s = src + src_off[f];
    uint8_t *d = w + dwin_len;
    for (uint64_t i = threadIdx.x; i < len; i += blockDim.x) d[i] = s[i];
}

// Linked frames of more than one block: one warp per chain walks the frame's blocks, table (zero, or the Jenkins-warmed
// dictionary table) and history (dictionary window ++ the frame's own input) carried across blocks -- k_compress_chain with
// per-chain descriptors and per-block output slots.
__global__ void __launch_bounds__(32, 1)
k_fb_chains(const uint8_t *__restrict__ stage, const uint64_t *__restrict__ stage_off, const uint32_t *__restrict__ chain_frames,
            const uint32_t *__restrict__ src_len, const uint64_t *__restrict__ bfirst, uint32_t B, uint32_t dwin_len,
            const int32_t *__restrict__ init_table /* nullable: zero table */, uint8_t *__restrict__ comp,
            const uint64_t *__restrict__ coff, uint32_t *__restrict__ clen) {
    extern __shared__ __align__(16) uint8_t smem[];
    const uint32_t lane = lane_id();
    const uint32_t c = blockIdx.x, f = chain_frames[c];
    int32_t *tab = reinterpret_cast<int32_t *>(smem);
    uint4 *t4 = reinterpret_cast<uint4 *>(tab);
    const uint4 *g4 = reinterpret_cast<const uint4 *>(init_table);
    for (uint32_t i = lane; i < kHashEntries * 4 / 16; i += 32) t4[i] = init_table ? g4[i] : make_uint4(0, 0, 0, 0);
    __syncwarp();
    Tab32 T{tab};
    const uint8_t *work = stage + stage_off[c];
    const int32_t start = (int32_t)dwin_len, end = start + (int32_t)src_len[f];
    const uint64_t first = bfirst[f], nb = bfirst[f + 1] - first;
    for (uint64_t k = 0; k < nb; ++k) {
        const int32_t pos = start + (int32_t)(k * B);
        const int32_t blen = (end - pos) < (int32_t)B ? (end - pos) : (int32_t)B;
        const uint32_t n = compress_block_warp_v2(work, pos, blen, T, comp + coff[first + k],
                                                  reinterpret_cast<uint32_t *>(smem + kHashEntries * 4));
        if (lane == 0) clen[first + k] = n;
        __syncwarp();
    }
}

// Per frame (one warp): position of every block's size word inside the frame and the frame's length
// header + sum(4 + payload [+ 4]) + EndMark [+ content checksum].  Stored-block rule of k_frame_layout: compressed iff 0 < comp < len.
__global__ void __launch_bounds__(256) k_fb_layout(uint32_t nframes, const uint64_t *__restrict__ bfirst, const uint32_t *__restrict__ slen,
                                                   const uint32_t *__restrict__ clen, uint32_t hdr_len, int block_checksum,
                                                   int content_checksum, uint64_t *bpos, uint64_t *frame_len) {
    const uint32_t lane = lane_id();
    const uint32_t f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (f >= nframes) return;
    const uint64_t first = bfirst[f], nb = bfirst[f + 1] - first;
    uint64_t run = hdr_len;
    for (uint64_t k0 = 0; k0 < nb; k0 += 32) {
        const uint64_t k = k0 + lane;
        uint64_t piece = 0;
        if (k < nb) {
            const uint32_t c = clen[first + k], L = slen[first + k];
            piece = 4ull + ((c > 0 && c < L) ? c : L) + (block_checksum ? 4ull : 0ull);
        }
        uint64_t x = piece;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint64_t y = __shfl_up_sync(FULL, x, o); if (lane >= (uint32_t)o) x += y; }
        if (k < nb) bpos[first + k] = run + x - piece;
        run += __shfl_sync(FULL, x, 31);
    }
    if (lane == 0) frame_len[f] = run + 4 + (content_checksum ? 4 : 0);
}

// Absolute block positions in dst, and the payload ranges the block checksums hash.
__global__ void __launch_bounds__(256) k_fb_place(uint64_t nblocks, const uint32_t *__restrict__ bframe, const uint64_t *__restrict__ frame_off,
                                                  const uint32_t *__restrict__ slen, const uint32_t *__restrict__ clen, uint64_t *bpos,
                                                  uint64_t *data_off, uint32_t *data_len) {
    const uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nblocks) return;
    const uint64_t p = frame_off[bframe[b]] + bpos[b];
    bpos[b] = p;
    if (data_off) {
        const uint32_t c = clen[b], L = slen[b];
        data_off[b] = p + 4;
        data_len[b] = (c > 0 && c < L) ? c : L;
    }
}

// xxh32 of the <= 14 header bytes FLG..dictID (bufferCompress.js:177-178): no stripes, seed 0.
__device__ __forceinline__ uint32_t xxh32_small(const uint8_t *p, uint32_t len) { return xxh_finish(P32_5, p, p + len, len); }

// Header (dlz4_frame_header's bytes), EndMark and [content checksum] of every frame: one thread per frame.
__global__ void __launch_bounds__(256) k_fb_headers(uint32_t nframes, const uint32_t *__restrict__ src_len, const uint64_t *__restrict__ frame_off,
                                                    uint8_t flg, uint8_t bd, int add_content_size, int have_dict,
                                                    const uint32_t *__restrict__ dict_id, const uint32_t *__restrict__ content_hash,
                                                    uint8_t *dst) {
    const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= nframes) return;
    uint8_t h[19];
    uint32_t hp = 0;
    auto put32 = [&](uint32_t v) { h[hp] = (uint8_t)v; h[hp + 1] = (uint8_t)(v >> 8); h[hp + 2] = (uint8_t)(v >> 16); h[hp + 3] = (uint8_t)(v >> 24); hp += 4; };
    put32(0x184D2204u);
    h[hp++] = flg;
    h[hp++] = bd;
    if (add_content_size) { put32(src_len[f]); put32(0); }
    if (have_dict) put32(*dict_id);
    h[hp] = (uint8_t)((xxh32_small(h + 4, hp - 4) >> 8) & 0xFF);
    ++hp;
    uint8_t *d = dst + frame_off[f];
    for (uint32_t i = 0; i < hp; ++i) d[i] = h[i];
    uint8_t *e = dst + frame_off[f + 1] - (content_hash ? 8 : 4);
    e[0] = e[1] = e[2] = e[3] = 0;                               // EndMark (:244)
    if (content_hash) {
        const uint32_t v = content_hash[f];
        e[4] = (uint8_t)v; e[5] = (uint8_t)(v >> 8); e[6] = (uint8_t)(v >> 16); e[7] = (uint8_t)(v >> 24);
    }
}

// ------------------------------------------------------------------ decompress
__device__ __forceinline__ uint32_t ld32b(const uint8_t *p) {
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}

struct FdFrame {                                                 // what the decoder needs of a parsed frame
    uint64_t cap;                                                // min(content size or block bound, dst_cap)
    uint64_t end;                                                // frame-relative position behind the EndMark
    uint32_t block_max;
    uint8_t linked, has_bc, has_cc, pad;
};

// One thread per frame: parse_header + walk_blocks of the single-frame call (api_frame_decompress.inc), in its order.
// info_status is dlz4_frame_info's status (adds "frame bytes beyond the input"); dec_status what dlz4_frame_decompress
// returns before decoding (adds the header checksum with flag bit 2).  With `blocks` set (second pass) the block table is
// written at bfirst[f].
__global__ void __launch_bounds__(256) k_fd_parse(const uint8_t *__restrict__ src, const uint64_t *__restrict__ frame_off,
                                                  const uint64_t *__restrict__ frame_len, uint32_t nframes, uint32_t flags,
                                                  const uint64_t *__restrict__ dst_cap, uint64_t *max_decoded, uint8_t *info_status,
                                                  uint8_t *dec_status, uint64_t *nblk, FdFrame *meta, const uint64_t *__restrict__ bfirst,
                                                  uint64_t *b_soff, uint32_t *b_slen, uint8_t *b_stored) {
    const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= nframes) return;
    const uint8_t *p = src + frame_off[f];
    const uint64_t len = frame_len[f];
    uint32_t st = 0;
    uint64_t pos = 4, content = 0, bound = 0, count = 0;
    uint8_t flg = 0;
    uint32_t bmax = 4194304u;
    if (len < 4 || ld32b(p) != 0x184D2204u) st = 5;              // bufferDecompress.js:59-61
    else if (len < 5) st = 6;
    else {
        flg = p[pos++];
        if (((flg & 0xC0) >> 6) != 1) st = 6;                    // :67
        else if (pos >= len) st = 2;
        else {
            const uint32_t bid = (p[pos++] >> 4) & 7;
            bmax = bid >= 4 ? (65536u << (2 * (bid - 4))) : 4194304u;
            if (flg & 0x08) {
                if (pos + 8 > len) st = 2;
                else { content = (uint64_t)ld32b(p + pos) | ((uint64_t)ld32b(p + pos + 4) << 32); pos += 8; }
            }
            if (!st && (flg & 0x01)) { if (pos + 4 > len) st = 2; else pos += 4; }
            if (!st) { pos += 1; if (pos > len) st = 2; }
        }
    }
    uint32_t dst_st = st;
    const bool write = bfirst != nullptr && !st && dec_status[f] == 0;
    if (!st && (flags & 4u) && (uint8_t)((xxh32_small(p + 4, (uint32_t)(pos - 5)) >> 8) & 0xFF) != p[pos - 1]) dst_st = 9;
    if (!st) {
        const bool bc = (flg & 0x10) != 0;
        uint64_t b = write ? bfirst[f] : 0;
        while (pos < len) {                                      // :133
            if (pos + 4 > len) { st = 2; break; }
            const uint32_t bs = ld32b(p + pos);
            pos += 4;
            if (bs == 0) break;                                  // :139 EndMark
            const uint32_t actual = bs & 0x7FFFFFFFu;
            if (pos + actual > len) { st = 2; break; }
            const bool stored = (bs >> 31) != 0;
            if (write) { b_soff[b] = frame_off[f] + pos; b_slen[b] = actual; b_stored[b] = stored; ++b; }
            bound += stored ? actual : ((uint64_t)actual * 255 < bmax ? (uint64_t)actual * 255 : bmax);
            ++count;
            pos += actual;
            if (bc) { if (pos + 4 > len) { st = 2; break; } pos += 4; }
        }
        if (!dst_st) dst_st = st;
    }
    if (bfirst) return;
    const uint64_t md = content ? content : bound;
    uint32_t ist = st;
    if (!ist && pos + ((flg & 0x04) ? 4 : 0) > len) ist = 2;     // dlz4_frame_info: frame_bytes > frame_len
    if (max_decoded) max_decoded[f] = ist ? 0 : md;
    if (info_status) info_status[f] = (uint8_t)ist;
    if (dec_status) dec_status[f] = (uint8_t)dst_st;
    if (nblk) nblk[f] = dst_st ? 0 : count;
    if (meta) {
        FdFrame m;
        const uint64_t cap = dst_cap ? dst_cap[f] : 0;
        m.cap = md < cap ? md : cap;
        m.end = pos;
        m.block_max = bmax;
        m.linked = (flg & 0x20) == 0;
        m.has_bc = (flg & 0x10) != 0;
        m.has_cc = (flg & 0x04) != 0;
        m.pad = 0;
        meta[f] = m;
    }
}

// One warp per frame (atomic queue): its blocks in order at running offsets, the block loop of bufferDecompress.js:133-192.
// A block's room is min(frame room left, blockMaxSize); linked blocks see min(op, 64 KiB) of the frame's own output after the
// dictionary, independent blocks the dictionary only.  The first failing block ends the frame.
template <bool kDict>
__global__ void __launch_bounds__(256)
k_fd_decode(const uint8_t *__restrict__ src, uint32_t nframes, const FdFrame *__restrict__ meta, const uint8_t *__restrict__ dec_status,
            const uint64_t *__restrict__ bfirst, const uint64_t *__restrict__ b_soff, const uint32_t *__restrict__ b_slen,
            const uint8_t *__restrict__ b_stored, uint8_t *dst, const uint64_t *__restrict__ dst_off, const uint8_t *__restrict__ dict,
            uint32_t dict_len, uint64_t *total, uint8_t *status, uint32_t *counter) {
    const uint32_t lane = lane_id();
    for (;;) {
        const uint32_t f = next_block(counter, lane);
        if (f >= nframes) break;
        uint32_t st = dec_status[f];
        uint64_t op = 0;
        if (!st) {
            const FdFrame m = meta[f];
            uint8_t *out = dst + dst_off[f];
            const uint64_t first = bfirst[f], nb = bfirst[f + 1] - first;
            for (uint64_t k = 0; k < nb && st == ST_OK; ++k) {
                const uint64_t b = first + k;
                const uint64_t left = m.cap - op, room = left < m.block_max ? left : m.block_max;
                uint32_t w;
                if (b_stored[b]) {
                    w = b_slen[b];
                    if (w > room) { st = ST_OUTPUT_TOO_SMALL; w = 0; }
                    else warp_copy(out + op, src + b_soff[b], w, lane);
                    __syncwarp();
                } else {
                    const uint32_t hist = m.linked ? (uint32_t)(op < 65536 ? op : 65536) : 0u;
                    w = decompress_block_warp_v2<kDict>(src + b_soff[b], b_slen[b], out + op, (uint32_t)room, hist, dict, dict_len, &st);
                }
                op += w;
            }
        }
        if (lane == 0) { total[f] = op; status[f] = (uint8_t)st; }
    }
}

// Content-checksum lengths: decoded bytes of the frames whose checksum is checked, 0 for the others.
__global__ void __launch_bounds__(256) k_fd_hash_len(uint32_t nframes, const FdFrame *__restrict__ meta, const uint8_t *__restrict__ status,
                                                     const uint64_t *__restrict__ total, uint32_t *hlen) {
    const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= nframes) return;
    hlen[f] = (!status[f] && meta[f].has_cc) ? (uint32_t)total[f] : 0u;
}

// The checks after decoding, in the single-frame order: block status (already there), block checksums (flag bit 1), content
// checksum (flag bit 0), then the caller's capacity.  out_len = 0 on error.
__global__ void __launch_bounds__(256) k_fd_finish(const uint8_t *__restrict__ src, const uint64_t *__restrict__ frame_off,
                                                   const uint64_t *__restrict__ frame_len, uint32_t nframes, uint32_t flags,
                                                   const FdFrame *__restrict__ meta, const uint64_t *__restrict__ bfirst,
                                                   const uint64_t *__restrict__ b_soff, const uint32_t *__restrict__ b_slen,
                                                   const uint32_t *__restrict__ bhash, const uint32_t *__restrict__ chash,
                                                   const uint64_t *__restrict__ dst_cap, const uint64_t *__restrict__ total,
                                                   uint8_t *status, uint64_t *out_len) {
    const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= nframes) return;
    uint32_t st = status[f];
    const FdFrame m = meta[f];
    if (!st && (flags & 2u) && m.has_bc && bhash) {
        for (uint64_t b = bfirst[f]; b < bfirst[f + 1]; ++b)
            if (ld32b(src + b_soff[b] + b_slen[b]) != bhash[b]) { st = 8; break; }
    }
    if (!st && (flags & 1u) && m.has_cc) {                       // :213-217
        if (m.end + 4 > frame_len[f]) st = 7;
        else if (ld32b(src + frame_off[f] + m.end) != chash[f]) st = 7;
    }
    if (!st && total[f] > dst_cap[f]) st = 1;
    status[f] = (uint8_t)st;
    out_len[f] = st ? 0 : total[f];
}

// ------------------------------------------------------------------ frame sequences (dlz4_frames_*_dev, api_frames_dev.inc)
struct FsWalk {                                                  // what k_fs_walk found
    unsigned long long count, max_decoded;                       // LZ4 frames before the first error, sum of their max_decoded
    uint32_t status, pad;                                        // for_each_frame's status
};

// One thread: for_each_frame over data[0, len) (skippable frames skipped) with dlz4_frame_info per LZ4 frame, in the host
// order; stops at the first error.  Frame k (k < cap) gets its offset, frame_bytes and max_decoded; `count` is the true number
// of frames, so a caller whose arrays were too small can grow them and run the walk again.  Reads bytewise: any alignment,
// nothing behind data + len.
__global__ void __launch_bounds__(32) k_fs_walk(const uint8_t *__restrict__ data, uint64_t len, uint32_t cap, uint64_t *frame_off,
                                                uint64_t *frame_len, uint64_t *max_decoded, FsWalk *res) {
    if (threadIdx.x != 0) return;
    uint64_t pos = 0, count = 0, sum = 0;
    uint32_t st = 0;
    while (pos < len) {
        if (pos + 4 > len) { st = 5; break; }
        if ((ld32b(data + pos) & 0xFFFFFFF0u) == 0x184D2A50u) {  // skippable frame: magic, u32 size, payload
            if (pos + 8 > len) { st = 2; break; }
            const uint64_t sz = ld32b(data + pos + 4);
            if (pos + 8 + sz > len) { st = 2; break; }
            pos += 8 + sz;
            continue;
        }
        const uint8_t *p = data + pos;                           // dlz4_frame_info(p, L): parse_header, walk_blocks, frame_bytes
        const uint64_t L = len - pos;
        if (ld32b(p) != 0x184D2204u) { st = 5; break; }
        if (L < 5) { st = 6; break; }
        uint64_t q = 4, content = 0, bound = 0;
        const uint8_t flg = p[q++];
        if (((flg & 0xC0) >> 6) != 1) { st = 6; break; }
        if (q >= L) { st = 2; break; }
        const uint32_t bid = (p[q++] >> 4) & 7;
        const uint32_t bmax = bid >= 4 ? (65536u << (2 * (bid - 4))) : 4194304u;
        if (flg & 0x08) {
            if (q + 8 > L) { st = 2; break; }
            content = (uint64_t)ld32b(p + q) | ((uint64_t)ld32b(p + q + 4) << 32);
            q += 8;
        }
        if (flg & 0x01) { if (q + 4 > L) { st = 2; break; } q += 4; }
        q += 1;
        if (q > L) { st = 2; break; }
        while (q < L) {
            if (q + 4 > L) { st = 2; break; }
            const uint32_t bs = ld32b(p + q);
            q += 4;
            if (bs == 0) break;
            const uint32_t actual = bs & 0x7FFFFFFFu;
            if (q + actual > L) { st = 2; break; }
            bound += (bs >> 31) ? actual : ((uint64_t)actual * 255 < bmax ? (uint64_t)actual * 255 : bmax);
            q += actual;
            if (flg & 0x10) { if (q + 4 > L) { st = 2; break; } q += 4; }
        }
        if (st) break;
        const uint64_t fb = q + ((flg & 0x04) ? 4 : 0);
        if (fb > L) { st = 2; break; }
        const uint64_t md = content ? content : bound;
        if (count < cap) { frame_off[count] = pos; frame_len[count] = fb; max_decoded[count] = md; }
        ++count;
        sum += md;
        pos += fb;
    }
    res->count = count;
    res->max_decoded = sum;
    res->status = st;
    res->pad = 0;
}

// One warp per frame: the out_len[f] bytes decoded into scratch at soff[f] move to dst at doff[f] (a group of small frames
// decoded at a scan of their max_decoded, gathered to their running offsets).
__global__ void __launch_bounds__(256) k_fs_gather(const uint8_t *__restrict__ scratch, const uint64_t *__restrict__ soff,
                                                   const uint64_t *__restrict__ out_len, const uint64_t *__restrict__ doff, uint32_t n,
                                                   uint8_t *dst) {
    const uint32_t lane = lane_id();
    for (uint32_t f = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; f < n; f += (gridDim.x * blockDim.x) >> 5) {
        const uint8_t *s = scratch + soff[f];
        uint8_t *d = dst + doff[f];
        const uint64_t len = out_len[f];
        for (uint64_t o = 0; o < len; o += 1u << 20)
            warp_copy(d + o, s + o, (uint32_t)(len - o < (1u << 20) ? len - o : (1u << 20)), lane);
        __syncwarp();
    }
}

}  // namespace dlz4
