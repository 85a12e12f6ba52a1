// rx_kernels.cuh -- receive chain of wifi_phy_hier as batch kernels over many frames.
// Reference stages (gnu_radio/wifi_phy_hier.grc, SURVEY.md 8a R1-R6):
//   k_detect      R1  autocorrelation front-end (:100-260) + threshold compare of sync_short (:716-734)
//   k_select      R2  sync_short plateau / MIN_GAP / MAX_SAMPLES state machine over the flag bitmap
//   k_sync_long   R2+R3  coarse CFO, derotation, 64-tap LTS matched filter, top-4 peak pairing (:698-715)
//   k_demod       R3 COPY + R4 FFT (:480-500) + R5 frame_equalizer (:550-569), one warp per frame
//   k_signal      R5f SIGNAL deinterleave + Viterbi + parse
//   k_plan        R6 decode_mac tag / symbol collection state machine (:533-549)
//   k_pack        R6 unpack bits, deinterleave, depuncture -> 2-bit symbols, 8 trellis steps per word
//   k_viterbi     R6a-c Viterbi, descramble, CRC-32 -> PSDU bytes
#pragma once
#include <cuda_pipeline.h>
#include "viterbi.cuh"

// ------------------------------------------------------------------ R1 front-end
// sample j of a link; samples before the start of the stream (beyond the stored history) are zeros
__device__ __forceinline__ cf fe_at(const cf *x, int64_t j, int hist) { return j < -(int64_t)hist ? cf{0.f, 0.f} : x[j]; }

__device__ __forceinline__ int find_link(const LinkDesc *links, int n_links, int64_t chunk)
{
    int lo = 0, hi = n_links - 1;
    while (lo < hi) {
        int mid = (lo + hi + 1) >> 1;
        if (links[mid].chunk_base <= chunk) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// DET_SPLIT blocks per tile of DET_TILE samples of one link (DET_BLOCK chunks each), one thread per FE_CHUNK samples.
//
// Data movement: a block's chunks plus two chunks of history (DET_BLOCK + 2 rows of 64 samples) are fetched by 1-D bulk copies
// (cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes, one 512-byte row per copy, issued by one warp, one
// mbarrier per consumer warp: a warp starts as soon as its rows have arrived) -- the copy engine does the work that used
// to cost 15 instructions per sample.  Rows are 66 samples (528 bytes) apart in shared memory: 16-byte aligned, as bulk
// copies require, and 33 16-byte units apart, so the threads' 16-byte loads (two samples each) of a warp are
// bank-conflict free.  A block that touches the start or the end of its stream, or whose samples are not 16-byte
// aligned in global memory, is staged element-wise (zeros outside the stream: that makes every "index < 0" case of
// the oracle an exact no-op, x + 0 == x).
//
// Arithmetic: each thread re-seeds the two running sums exactly as the oracle does at every multiple of FE_CHUNK
// and walks its 64 samples.  The walk is fully unrolled over a register ring of the last 64 samples: sample n is
// loaded once (32 loads of the previous row for the history, 32 of its own row) and the three delayed taps
// x[n-16], x[n-47], x[n-63] are register reads.  Flag n = |a[n]|^2 > thr^2 p[n]^2 (oracle rx_link).
// A block is DET_BLOCK threads -- ONE warp -- and works on a quarter of a tile (its 32 chunks plus two chunks of history,
// 18 KB of shared memory): twelve blocks fit an SM, so twelve loads are in different phases.  Measured per 229.6 Msamples:
// 128 threads per block 0.51 ms, 64: 0.42 ms, 32: 0.36 ms (the history rows are read 1.06 times, mostly from L2).
#ifndef DET_BLOCK
#define DET_BLOCK 32
#endif
#define DET_SPLIT (DET_THREADS / DET_BLOCK)               // blocks per tile
#define DET_ROWS (DET_BLOCK + 2)
#define DET_STRIDE 66                                        // samples between rows in shared memory
#define DET_SMEM_BYTES (DET_ROWS * DET_STRIDE * (int)sizeof(cf) + 32)   // + one mbarrier per warp

__device__ __forceinline__ uint32_t det_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
// bit 0 / bit 1: the first / second sample of the pair at p (shared memory) is not an exact zero (-0 is a zero, NaN is not).
// Volatile loads, here and below: the compiler must not keep the walk's samples alive in registers to reuse them here.
__device__ __forceinline__ uint32_t det_nonzero_pair(const cf *p)
{
    uint32_t a, b, c, d;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(det_smem_u32(p)));
    return (((a | b) << 1) != 0u ? 1u : 0u) | (((c | d) << 1) != 0u ? 2u : 0u);
}
__device__ __forceinline__ bool det_nonzero_one(const cf *p)
{
    uint32_t a, b;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(a), "=r"(b) : "r"(det_smem_u32(p)));
    return ((a | b) << 1) != 0u;
}

__global__ void __launch_bounds__(DET_BLOCK, 384 / DET_BLOCK) k_detect(const cf *__restrict__ iq, const LinkDesc *__restrict__ links, int n_links,
                                                         int64_t tile_base, int64_t total_tiles, float thr_f, uint32_t *__restrict__ flags,
                                                         uint32_t *__restrict__ summary)
{
    extern __shared__ __align__(128) unsigned char det_raw[];
    cf *sx = reinterpret_cast<cf *>(det_raw);                                         // DET_ROWS x DET_STRIDE
    uint64_t *bar = reinterpret_cast<uint64_t *>(det_raw + DET_ROWS * DET_STRIDE * sizeof(cf));
    const int64_t tile = tile_base + blockIdx.x / DET_SPLIT;   // links / n_links: the link group of this launch; tiles are numbered over the whole call
    const int half = blockIdx.x % DET_SPLIT;                   // which DET_BLOCK chunks of the tile
    if (tile >= total_tiles) return;
    const int tid = threadIdx.x;
    int l = find_link(links, n_links, tile * DET_THREADS);
    const LinkDesc L = links[l];
    const cf *x = iq + L.x_off;
    const int64_t T0 = (tile * DET_THREADS - L.chunk_base + half * DET_BLOCK) * FE_CHUNK;   // first sample of this block's chunks in the link
    const int64_t lo = -(int64_t)L.hist, hi = L.len;
    const int64_t g0 = T0 - 2 * FE_CHUNK;                                // first staged sample
    const bool bulk = g0 >= lo && g0 + DET_ROWS * FE_CHUNK <= hi && ((reinterpret_cast<uintptr_t>(x + g0) & 15) == 0);
    if (bulk) {
        // one mbarrier per warp of consumers: rows [0, 34) complete the first, the next 32 rows the second.  Warp w walks
        // the rows 32 w + 1 .. 32 w + 33, i.e. it waits for its own barrier and the one before: the first warp starts
        // its walk when half of the rows have arrived.
        const uint32_t bar_a = det_smem_u32(bar);
        if (tid == 0) {
#pragma unroll
            for (int b = 0; b < DET_BLOCK / 32; ++b) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_a + 8 * b));
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
        if (tid < 32) {
            if (tid < DET_BLOCK / 32)
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a + 8 * tid), "r"((tid == 0 ? 34 : 32) * FE_CHUNK * (int)sizeof(cf)) : "memory");
            __syncwarp();
            for (int r = tid; r < DET_ROWS; r += 32)
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(det_smem_u32(sx + r * DET_STRIDE)),
                             "l"(x + g0 + (int64_t)r * FE_CHUNK), "r"(FE_CHUNK * (int)sizeof(cf)), "r"(bar_a + 8 * (r < 34 ? 0 : (r - 2) >> 5))
                             : "memory");
        }
        const int wq = tid >> 5;
        for (int b = (wq > 0 ? wq - 1 : 0); b <= wq; ++b) {
            uint32_t done = 0;
            while (!done)
                asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(done) : "r"(bar_a + 8 * b) : "memory");
        }
    } else {
        for (int q = tid; q < DET_ROWS * FE_CHUNK; q += DET_BLOCK) {
            const int64_t g = g0 + q;
            sx[(q >> 6) * DET_STRIDE + (q & 63)] = (g >= lo && g < hi) ? x[g] : cf{0.f, 0.f};
        }
        __syncthreads();
    }
    uint32_t w0 = 0u, w1 = 0u;
    if (T0 + (int64_t)tid * FE_CHUNK < hi) {
        // ring[i & 63] = sample i of the chunk for i in [-63, 63]: history sample -k sits in ring[64 - k]
        const float4 *prev = reinterpret_cast<const float4 *>(sx + (tid + 1) * DET_STRIDE);
        const float4 *own = reinterpret_cast<const float4 *>(sx + (tid + 2) * DET_STRIDE);
        cf ring[64];
#pragma unroll
        for (int m = 0; m < 32; ++m) {
            const float4 v = prev[m];
            ring[2 * m] = cf{v.x, v.y};              // ring[0] (sample -64) is not used; overwritten by sample 0
            ring[2 * m + 1] = cf{v.z, v.w};
        }
        cf sa = {0.f, 0.f};
        float sp = 0.f;
#pragma unroll
        for (int j = -47; j <= -1; ++j) sa = wdm_cmacc(sa, ring[64 + j], ring[48 + j]);
#pragma unroll
        for (int j = -63; j <= -1; ++j) sp = wdm_norm_add(sp, ring[64 + j]);
        const float thr2 = thr_f * thr_f;
        cf nxt = {0.f, 0.f};
#pragma unroll
        for (int n = 0; n < 64; ++n) {
            cf xn;
            if ((n & 1) == 0) {
                const float4 v = own[n >> 1];
                xn = cf{v.x, v.y};
                nxt = cf{v.z, v.w};
            } else {
                xn = nxt;
            }
            const cf xd = ring[(n + 48) & 63], xo = ring[(n + 17) & 63], xod = ring[(n + 1) & 63];   // n-16, n-47, n-63
            sa = wdm_cmacc(sa, xn, xd);              // fused multiply-add chains, as the oracle's FrontEnd::step
            const float m2 = wdm_norm(sa);
            sa = wdm_cmsubc(sa, xo, xod);
            sp = wdm_norm_add(sp, xn);
            const float p = sp;
            sp = wdm_norm_sub(sp, xod);
            if (m2 > thr2 * (p * p)) {
                if (n < 32) w0 |= 1u << n; else w1 |= 1u << (n - 32);
            }
            ring[n] = xn;                            // replaces sample n - 64
        }
        // silence is silence (oracle FrontEnd): no flag where the 64-sample window n-63 .. n holds only exact zeros (the
        // running sums may keep a rounding residue there).  If the first flagged sample is nonzero, every flagged window
        // holds it or a later own sample: one load settles the chunk.  Otherwise, bit k of nzh / nzo: sample k - 64 /
        // sample k is nonzero; the window holds one iff n is at or after the first nonzero own sample, or before the last
        // nonzero history sample (k in 1 .. 63, k > n).
        if ((w0 | w1) != 0u && !det_nonzero_one(sx + (tid + 2) * DET_STRIDE + (w0 ? __ffs((int)w0) - 1 : 31 + __ffs((int)w1)))) {
            uint64_t nzh = 0ull, nzo = 0ull;
#pragma unroll 8
            for (int m = 0; m < 32; ++m) {
                nzh |= (uint64_t)det_nonzero_pair(sx + (tid + 1) * DET_STRIDE + 2 * m) << (2 * m);
                nzo |= (uint64_t)det_nonzero_pair(sx + (tid + 2) * DET_STRIDE + 2 * m) << (2 * m);
            }
            nzh &= ~1ull;                            // sample -64 is outside every window of the chunk
            const uint64_t occ = (0ull - (nzo & (0ull - nzo))) | (nzh ? (~0ull >> __clzll((long long)nzh)) >> 1 : 0ull);
            w0 &= (uint32_t)occ;
            w1 &= (uint32_t)(occ >> 32);
        }
    }
    const int64_t chunk = tile * DET_THREADS + half * DET_BLOCK + tid;
    reinterpret_cast<uint2 *>(flags)[chunk] = make_uint2(w0, w1);
    uint32_t any = __ballot_sync(0xffffffffu, (w0 | w1) != 0u);
    if ((tid & 31) == 0) summary[chunk >> 5] = any;
}

// ------------------------------------------------------------------ R2 sync_short selection
// One warp per link.  cand(m) = flag[m] & flag[m-1] & .. & flag[m-min_plateau] (plateau counter
// reached min_plateau before m); triggers are the greedy chain "first candidate more than MIN_GAP
// after the previous trigger" (the COPY-state retrigger and the SEARCH-state trigger coincide, see
// DESIGN.md).  The scan walks the one-bit-per-chunk summary and opens only chunks that hold a flag.
__device__ __forceinline__ int64_t next_candidate(const uint32_t *__restrict__ fw, const uint32_t *__restrict__ sm, int64_t chunk_base,
                                                  int64_t n_chunks, int64_t pos, int lane, int min_plateau)
{
    int64_t c = pos >> 6;
    while (c < n_chunks) {
        // next chunk >= c with any flag: 32 summary words (1024 chunks) per iteration
        int64_t gb = chunk_base + c;                 // global chunk index = summary bit index
        int64_t wbase = gb >> 5;
        int64_t wi = wbase + lane;
        uint32_t sw = (wi * 32 < chunk_base + n_chunks) ? sm[wi] : 0u;
        if (lane == 0) sw &= 0xffffffffu << (gb & 31);
        uint32_t any = __ballot_sync(0xffffffffu, sw != 0u);
        if (!any) { c = (wbase + 32) * 32 - chunk_base; continue; }
        int src = __ffs((int)any) - 1;
        uint32_t hit = __shfl_sync(0xffffffffu, sw, src);
        int64_t ch = (wbase + src) * 32 + (__ffs((int)hit) - 1) - chunk_base;
        if (ch >= n_chunks) return -1;
        // open chunk ch: 64 flags + the last bits of the previous chunk
        uint2 w = reinterpret_cast<const uint2 *>(fw)[ch];
        uint32_t pw = ch > 0 ? fw[2 * ch - 1] : 0u;
        unsigned long long f64 = ((unsigned long long)w.y << 32) | w.x, cand = f64;
        for (int k = 1; k <= min_plateau; ++k) cand &= (f64 << k) | ((unsigned long long)pw >> (32 - k));
        int64_t first = ch * 64;
        if (first < pos) {
            int64_t d = pos - first;
            cand = d >= 64 ? 0ull : (cand & (~0ull << d));
        }
        if (cand) return first + (__ffsll((long long)cand) - 1);
        c = ch + 1;
    }
    return -1;
}

// Speculative pass: one warp per 8192-sample segment (= one detect tile) walks the greedy chain inside
// its segment as if no earlier trigger constrained it.  Chains started at different points merge at
// their first common trigger, so the sequential pass below only has to re-walk a segment whose first
// speculative trigger is closer than MIN_GAP to the true trigger before it.
#define SEG_CHUNKS DET_THREADS          // chunks per segment
#define SEG_CAP 20                      // >= 8192 / 481 + 1 triggers per segment
__global__ void __launch_bounds__(128) k_select_spec(const uint32_t *__restrict__ flags, const uint32_t *__restrict__ summary,
                                                      const LinkDesc *__restrict__ links, int n_links, int64_t seg_base, int64_t total_segs, int min_plateau,
                                                      int *__restrict__ spec_trig, int4 *__restrict__ spec_meta)
{
    int64_t seg = seg_base + (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (seg >= total_segs) return;
    const int l = find_link(links, n_links, seg * SEG_CHUNKS);
    const LinkDesc L = links[l];
    const uint32_t *fw = flags + L.chunk_base * 2;
    const int64_t n_chunks = (L.len + FE_CHUNK - 1) / FE_CHUNK;
    const int64_t c0 = seg * SEG_CHUNKS - L.chunk_base;            // first chunk of the segment in the link
    const int64_t c1 = (c0 + SEG_CHUNKS < n_chunks) ? c0 + SEG_CHUNKS : n_chunks;
    int64_t pos = c0 * FE_CHUNK;
    if (pos < L.min_pos) pos = L.min_pos;
    const int64_t end = (c1 * FE_CHUNK < L.len) ? c1 * FE_CHUNK : L.len;
    int k = 0, first = 0, last = 0;
    while (pos < end) {
        int64_t m = next_candidate(fw, summary, L.chunk_base, c1, pos, lane, min_plateau);
        if (m < 0 || m >= end) break;
        if (lane == 0 && k < SEG_CAP) spec_trig[seg * SEG_CAP + k] = (int)m;
        if (k == 0) first = (int)m;
        last = (int)m;
        ++k;
        pos = m + SS_MIN_GAP + 1;
    }
    // (count, first, last) in one 16-byte record: all the sequential pass needs for a regular segment
    if (lane == 0) spec_meta[seg] = make_int4(k < SEG_CAP ? k : SEG_CAP, first, last, 0);
}

// Second speculative pass, one warp per segment: a segment whose first speculative trigger lies inside the MIN_GAP of the
// LAST speculative trigger of the segment before it (an STS plateau near or across the segment boundary: 7 % of the
// segments of back-to-back traffic) walks its chain again from behind that trigger -- in parallel, into a second trigger
// array.  Unless the segment before changes its own last trigger in this very pass (second order), the sequential pass then
// finds every segment acceptable: without this pass one long stream spent 7 ms per 900 Msamples re-walking there.
// meta2[seg] = (count, first, last, w): w = 0: the unconstrained chain of the first pass (in spec_trig), valid whenever its
// first trigger is more than MIN_GAP behind the true previous trigger; w = p + 1: the chain walked from behind trigger p (in
// spec_trig2), valid exactly when the true previous trigger IS p.
__global__ void __launch_bounds__(128) k_select_fix(const uint32_t *__restrict__ flags, const uint32_t *__restrict__ summary,
                                                     const LinkDesc *__restrict__ links, int n_links, int64_t seg_base, int64_t total_segs, int min_plateau,
                                                     const int *__restrict__ spec_trig, const int4 *__restrict__ spec_meta, int *__restrict__ spec_trig2,
                                                     int4 *__restrict__ meta2)
{
    int64_t seg = seg_base + (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (seg >= total_segs) return;
    const int l = find_link(links, n_links, seg * SEG_CHUNKS);
    const LinkDesc L = links[l];
    const int4 me = spec_meta[seg];
    const int64_t c0 = seg * SEG_CHUNKS - L.chunk_base;            // first chunk of the segment in the link
    bool redo = false;
    int64_t p = 0;
    if (c0 > 0 && me.x > 0) {
        const int4 pv = spec_meta[seg - 1];                        // same link: its segments are consecutive
        if (pv.x > 0) { p = pv.z; redo = !((int64_t)me.y > p + SS_MIN_GAP); }
    }
    if (!redo) {
        if (lane == 0) meta2[seg] = make_int4(me.x, me.y, me.z, 0);
        return;
    }
    const uint32_t *fw = flags + L.chunk_base * 2;
    const int64_t n_chunks = (L.len + FE_CHUNK - 1) / FE_CHUNK;
    const int64_t c1 = (c0 + SEG_CHUNKS < n_chunks) ? c0 + SEG_CHUNKS : n_chunks;
    const int64_t end = (c1 * FE_CHUNK < L.len) ? c1 * FE_CHUNK : L.len;
    int64_t pos = p + SS_MIN_GAP + 1;
    int k = 0, first = 0, last = 0;
    while (pos < end) {
        int64_t m = next_candidate(fw, summary, L.chunk_base, c1, pos, lane, min_plateau);
        if (m < 0 || m >= end) break;
        if (lane == 0 && k < SEG_CAP) spec_trig2[seg * SEG_CAP + k] = (int)m;
        if (k == 0) first = (int)m;
        last = (int)m;
        ++k;
        pos = m + SS_MIN_GAP + 1;
    }
    if (lane == 0) meta2[seg] = make_int4(k < SEG_CAP ? k : SEG_CAP, first, last, (int)p + 1);
}

// Sequential pass, one warp per link: accepts speculative segments 32 at a time while each first
// trigger is more than MIN_GAP after the last trigger before it, re-walks the flags otherwise.
// Leaves the triggers in trig_tmp and their count in links[].frame_count.
__global__ void __launch_bounds__(128) k_select(const uint32_t *__restrict__ flags, const uint32_t *__restrict__ summary, LinkDesc *links,
                                                 int n_links, int min_plateau, int *trig_tmp,
                                                 const int *__restrict__ spec_trig, const int4 *__restrict__ spec_meta, const int *__restrict__ spec_trig2)
{
    // spec_meta here is k_select_fix's output: .w says which of the two trigger arrays holds a segment's chain
    int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= n_links) return;
    LinkDesc L = links[warp];
    const uint32_t *fw = flags + L.chunk_base * 2;
    const int64_t n_chunks = (L.len + FE_CHUNK - 1) / FE_CHUNK;
    const int64_t seg0 = L.chunk_base / SEG_CHUNKS;
    const int64_t n_segs = (n_chunks + SEG_CHUNKS - 1) / SEG_CHUNKS;
    int *tmp = trig_tmp + L.chunk_base / 4;   // triggers are > 480 samples apart: at most one per 7 chunks
    int64_t t_prev = (L.min_pos > 0 ? L.min_pos : 0) - SS_MIN_GAP - 1;   // "last trigger" entering the buffer
    int k = 0;
    int64_t s = 0;
    // prefetch of the next group's records (the common case advances by exactly 128 segments)
    int4 nxt[4];
    int64_t nxt_s = -1;
    auto load_group = [&](int64_t s0, int4 *m) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            int64_t si = s0 + lane * 4 + q;
            m[q] = (si < n_segs) ? spec_meta[seg0 + si] : make_int4(0, 0, 0, 0);
        }
    };
    while (s < n_segs) {
        // look at up to 128 segments at once, four consecutive ones per lane
        int4 meta[4];
        if (nxt_s == s) {
#pragma unroll
            for (int q = 0; q < 4; ++q) meta[q] = nxt[q];
        } else {
            load_group(s, meta);
        }
        nxt_s = s + 128;
        load_group(nxt_s, nxt);
        int cnt[4], first[4], last[4];
        const int *src[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) { cnt[q] = meta[q].x; first[q] = meta[q].y; last[q] = meta[q].z; src[q] = meta[q].w ? spec_trig2 : spec_trig; }
        // last trigger before each segment, assuming every earlier segment of the group is accepted
        const int64_t NONE = -(1ll << 40);
        int64_t lane_last = NONE;
#pragma unroll
        for (int q = 0; q < 4; ++q) if (cnt[q]) lane_last = last[q];      // triggers ascend with the segment index
        int64_t run = lane_last;
        for (int o = 1; o < 32; o <<= 1) {
            int64_t v = __shfl_up_sync(0xffffffffu, run, o);
            if (lane >= o && v > run) run = v;
        }
        int64_t before = __shfl_up_sync(0xffffffffu, run, 1);
        if (lane == 0 || before < t_prev) before = t_prev;
        int my_bad = 4;                                                  // first segment of this lane that is not acceptable
        int64_t b4 = before;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            if (meta[q].w) {                                             // second-pass chain: right iff the trigger before it is the assumed one
                if (my_bad == 4 && b4 != (int64_t)meta[q].w - 1) my_bad = q;
            } else if (cnt[q]) {
                if (my_bad == 4 && !((int64_t)first[q] > b4 + SS_MIN_GAP)) my_bad = q;
            }
            if (cnt[q]) b4 = last[q];
        }
        unsigned badm = __ballot_sync(0xffffffffu, my_bad < 4);
        int n_ok;                                                        // segments s .. s+n_ok-1 are accepted as speculated
        if (badm) {
            int bl = __ffs((int)badm) - 1;
            n_ok = bl * 4 + __shfl_sync(0xffffffffu, my_bad, bl);
        } else {
            n_ok = 128;
        }
        if (s + n_ok > n_segs) n_ok = (int)(n_segs - s);
        const bool bad = badm != 0u;
        // append their triggers
        int mine = 0;
#pragma unroll
        for (int q = 0; q < 4; ++q) if (lane * 4 + q < n_ok) mine += cnt[q];
        int incl = mine;
        for (int o = 1; o < 32; o <<= 1) {
            int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        int wpos = k + incl - mine;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            if (lane * 4 + q < n_ok) {
                int64_t si = s + lane * 4 + q;
                if (cnt[q] > 0) tmp[wpos] = first[q];
                if (cnt[q] > 1) tmp[wpos + cnt[q] - 1] = last[q];
                for (int j = 1; j < cnt[q] - 1; ++j) tmp[wpos + j] = src[q][(seg0 + si) * SEG_CAP + j];
                wpos += cnt[q];
            }
        }
        int total = __shfl_sync(0xffffffffu, incl, 31);
        if (total > 0) {
            // last accepted trigger: the largest `last` among accepted segments
            int64_t acc_last = NONE;
#pragma unroll
            for (int q = 0; q < 4; ++q) if (lane * 4 + q < n_ok && cnt[q]) acc_last = last[q];
            for (int o = 16; o > 0; o >>= 1) {
                int64_t v = __shfl_xor_sync(0xffffffffu, acc_last, o);
                if (v > acc_last) acc_last = v;
            }
            if (acc_last > t_prev) t_prev = acc_last;
        }
        k += total;
        s += n_ok;
        if (bad && s < n_segs) {
            // segment s starts inside the gap of the previous trigger: walk the true chain through it
            const int64_t c1 = ((s + 1) * SEG_CHUNKS < n_chunks) ? (s + 1) * SEG_CHUNKS : n_chunks;
            const int64_t end = (c1 * FE_CHUNK < L.len) ? c1 * FE_CHUNK : L.len;
            const int scnt = spec_meta[seg0 + s].x;
            const int *strig = (spec_meta[seg0 + s].w ? spec_trig2 : spec_trig) + (seg0 + s) * SEG_CAP;
            int64_t pos = t_prev + SS_MIN_GAP + 1;
            while (pos < end) {
                int64_t m = next_candidate(fw, summary, L.chunk_base, c1, pos, lane, min_plateau);
                if (m < 0 || m >= end) break;
                // merged with the speculative chain?  then the rest of it is true as well
                int at = -1;
                for (int j = 0; j < scnt; ++j)
                    if (strig[j] == (int)m) at = j;
                if (at >= 0) {
                    for (int j = at + lane; j < scnt; j += 32) tmp[k + j - at] = strig[j];
                    k += scnt - at;
                    t_prev = strig[scnt - 1];
                    break;
                }
                if (lane == 0) tmp[k] = (int)m;
                ++k;
                t_prev = m;
                pos = m + SS_MIN_GAP + 1;
            }
            ++s;
        }
    }
    __syncwarp();
    if (lane == 0) links[warp].frame_count = k;     // k_reserve turns the counts into ranges
}

// Frame-record and equalizer-row ranges of all links: an exclusive prefix sum over the links in link order, so
// the frame table is ordered by (link, trigger) on every run.  Row offsets inside a link need no scan: bursts
// do not overlap, so frame i may start at row floor(t_i / 80) + i of the link's range (its burst_len/80 + 1
// rows end before the next frame's first row); the range is floor(len / 80) + k + 1 rows.
__global__ void __launch_bounds__(1024) k_reserve(LinkDesc *links, int n_links, int *counters, unsigned long long *row_counter,
                                                   int64_t max_frames, int *err, long long frame_base, long long row_base)
{
    __shared__ long long s_f[1024], s_r[1024];
    const int tid = threadIdx.x;
    const int per = (n_links + 1023) / 1024;
    const int l0 = tid * per < n_links ? tid * per : n_links, l1 = l0 + per < n_links ? l0 + per : n_links;
    long long f = 0, r = 0;
    for (int l = l0; l < l1; ++l) {
        f += links[l].frame_count;
        r += links[l].len / 80 + links[l].frame_count + 1;
    }
    s_f[tid] = f;
    s_r[tid] = r;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
        const long long af = tid >= o ? s_f[tid - o] : 0, ar = tid >= o ? s_r[tid - o] : 0;
        __syncthreads();
        s_f[tid] += af;
        s_r[tid] += ar;
        __syncthreads();
    }
    long long bf = frame_base + s_f[tid] - f, br = row_base + s_r[tid] - r;      // bases: the link groups before this one
    const long long total_f = frame_base + s_f[1023];
    const bool ovf = total_f > max_frames;
    for (int l = l0; l < l1; ++l) {
        const int k = links[l].frame_count;
        links[l].frame_first = (int)bf;
        links[l].row_base = br;
        if (ovf) links[l].frame_count = 0;
        bf += k;
        br += links[l].len / 80 + k + 1;
    }
    if (tid == 0) {
        counters[0] = total_f > 0x7fffffffll ? 0x7fffffff : (int)total_f;
        *row_counter = (unsigned long long)(row_base + s_r[1023]);
        if (ovf) atomicExch(err, WIFI_E_OVERFLOW);

    }
}

// frame records of all links, one thread per frame (grid.y = link)
__global__ void __launch_bounds__(128) k_frames_init(const LinkDesc *__restrict__ links, const int *__restrict__ trig_tmp, wifi_b200_frame *frames,
                                                      int link_base)
{
    const int l = blockIdx.y;
    const LinkDesc L = links[l];
    const int *tmp = trig_tmp + L.chunk_base / 4;
    const int k = L.frame_count;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < k; i += gridDim.x * blockDim.x) {
        const int64_t t = tmp[i];
        const int64_t endp = (i + 1 < k) ? (int64_t)tmp[i + 1] : L.len;
        wifi_b200_frame f;
        f.trigger = t; f.link = link_base + l;
        f.burst_len = (int)((endp - t) < SS_MAX_SAMPLES ? (endp - t) : SS_MAX_SAMPLES);
        // Streaming: the newest burst of a link is complete once MAX_SAMPLES of the stream lie behind its trigger
        // (sync_short's COPY state has ended whatever follows); until then a later trigger may still cut it short,
        // so it is held: no samples (burst_len 0: every later stage skips it) and n_syms = -1 as the marker.
        const bool held = L.hold_last && i == k - 1 && (L.len - t) < SS_MAX_SAMPLES;
        if (held) f.burst_len = 0;
        f.freq_short = 0.f; f.freq_long = 0.f;
        f.found = 0; f.frame_start = SYNC_LENGTH; f.n_syms = held ? -1 : 0; f.sig_ok = 0; f.encoding = 0; f.length = 0;
        f.frame_symbols = 0; f.n_rows = 0; f.accepted = 0; f.decoded = 0; f.crc_ok = 0; f.snr = 0.0;
        f.row_off = L.row_base + t / 80 + i; f.psdu_off = -1;
        frames[L.frame_first + i] = f;
    }
}

// ------------------------------------------------------------------ R2/R3 sync_long search
// One block of SL_THREADS threads per frame.  The 320 x 64 matched filter is register blocked: a thread owns five
// consecutive lags, keeps the five samples under the current tap in registers and loads ONE new sample per tap
// (20 fused multiply-adds per load instead of 4); the taps are compile-time offsets into constant memory, i.e.
// operands of the multiply-adds, not loads.  Each lag still accumulates its 64 taps in ascending order (the contract).
#define SL_THREADS 64
#define SL_LAGS 5                       // SYNC_LENGTH / SL_THREADS
// (f0, n_frames) here and below: the frame range of the link group a launch works on; `links` is the whole call's table
__global__ void __launch_bounds__(SL_THREADS) k_sync_long(const cf *__restrict__ iq, const LinkDesc *__restrict__ links, wifi_b200_frame *frames, int f0, int n_frames)
{
    static_assert(SL_THREADS * SL_LAGS == SYNC_LENGTH, "lags per thread");
    __shared__ cf sb[SYNC_LENGTH + 64];
    __shared__ cf scorr[SYNC_LENGTH];
    __shared__ float smag[SYNC_LENGTH];
    __shared__ float s_freq;
    __shared__ float rmax[SL_THREADS / 32];
    __shared__ int ridx[SL_THREADS / 32];
    __shared__ int top[4];
    int f = f0 + blockIdx.x;
    if (f >= n_frames) return;
    wifi_b200_frame F = frames[f];
    const LinkDesc L = links[F.link];
    const cf *x = iq + L.x_off;
    const int tid = threadIdx.x;
    const int hist = L.hist;
    int64_t t = F.trigger;
    {
        // a[t]: the moving_average_cc value sync_short sees on its port 1 at the trigger, recomputed on
        // the oracle's chunk grid: the samples are staged in parallel, the running sum (a chain of fused
        // multiply-adds whose order is the contract) is walked by one thread from shared memory.
        const int64_t i0 = t & ~(int64_t)(FE_CHUNK - 1);
        cf *sx = sb;         // scratch, reused later: samples i0 - 63 .. t
        const int cnt = (int)(t - i0) + 64;
        for (int q = tid; q < cnt; q += SL_THREADS) sx[q] = fe_at(x, i0 - 63 + q, hist);
        __syncthreads();
        if (tid == 0) {
            cf sa = {0.f, 0.f};
            for (int q = 16; q < 63; ++q) sa = wdm_cmacc(sa, sx[q], sx[q - 16]);                  // seed: lags i0-47 .. i0-1
            for (int q = 63; q < cnt; ++q) {
                sa = wdm_cmacc(sa, sx[q], sx[q - 16]);
                if (q < cnt - 1) sa = wdm_cmsubc(sa, sx[q - 47], sx[q - 63]);
            }
            s_freq = wdm_atan2f(sa.im, sa.re) / 16;
        }
    }
    __syncthreads();
    const float freq = s_freq;
    if (tid == 0) frames[f].freq_short = freq;
    if (F.burst_len < SYNC_LENGTH + 63) return;   // SYNC never completes (end of stream)
    for (int j = tid; j < SYNC_LENGTH + 63; j += SL_THREADS) {
        int64_t src = t + j - 16;
        cf s = src >= -(int64_t)hist ? x[src] : cf{0.f, 0.f};
        sb[j] = cmul(s, crot(-freq * (float)j));
    }
    __syncthreads();
    {
        const int i0 = SL_LAGS * tid;
        cf acc[SL_LAGS], win[SL_LAGS];
#pragma unroll
        for (int q = 0; q < SL_LAGS; ++q) { acc[q] = cf{0.f, 0.f}; win[q] = q < SL_LAGS - 1 ? sb[i0 + q] : cf{0.f, 0.f}; }
#pragma unroll
        for (int m = 0; m < 64; ++m) {
            win[(m + SL_LAGS - 1) % SL_LAGS] = sb[i0 + m + SL_LAGS - 1];      // the window is a ring: sample i0 + m + q sits in win[(m + q) % 5]
            const cf tap = c_tab.long_taps[63 - m];
#pragma unroll
            for (int q = 0; q < SL_LAGS; ++q) acc[q] = wdm_cmac(acc[q], tap, win[(m + q) % SL_LAGS]);
        }
#pragma unroll
        for (int q = 0; q < SL_LAGS; ++q) {
            scorr[i0 + q] = acc[q];
            smag[i0 + q] = wdm_norm(acc[q]);
        }
    }
    __syncthreads();
    // four largest |corr|^2, earlier index first on ties (stable descending sort)
    for (int r = 0; r < 4; ++r) {
        float bm = -1.f;
        int bi = 0x7fffffff;
        for (int i = tid; i < SYNC_LENGTH; i += SL_THREADS) {
            float v = smag[i];
            if (v > bm) { bm = v; bi = i; }   // ascending i per thread: first max kept
        }
        for (int o = 16; o > 0; o >>= 1) {
            float om = __shfl_xor_sync(0xffffffffu, bm, o);
            int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (om > bm || (om == bm && oi < bi)) { bm = om; bi = oi; }
        }
        if ((tid & 31) == 0) { rmax[tid >> 5] = bm; ridx[tid >> 5] = bi; }
        __syncthreads();
        if (tid == 0) {
            for (int w = 1; w < SL_THREADS / 32; ++w)
                if (rmax[w] > bm || (rmax[w] == bm && ridx[w] < bi)) { bm = rmax[w]; bi = ridx[w]; }
            top[r] = bi;
            smag[bi] = -2.f;
        }
        __syncthreads();
    }
    if (tid == 0) {
        int found = 0, fs = SYNC_LENGTH;
        float fo = 0.f;
        for (int i = 0; i < 3 && found != 64; ++i)
            for (int k = i + 1; k < 4; ++k) {
                int lo = min(top[i], top[k]), hi = max(top[i], top[k]);
                int diff = hi - lo;
                if (diff == 63 || diff == 64 || diff == 65) {
                    cf first = scorr[lo], second = scorr[hi];
                    cf pr = wdm_cmulc(first, second);
                    fs = lo;
                    fo = wdm_atan2f(pr.im, pr.re) / (float)diff;
                    found = diff;
                    if (diff == 64) break;
                }
            }
        frames[f].found = found;
        frames[f].frame_start = fs;
        frames[f].freq_long = fo;   // provisional: resolved against the carry in k_demod
    }
}

#ifndef DEMOD_MINB
#define DEMOD_MINB 5
#endif
// ------------------------------------------------------------------ R3 COPY + R4 + R5
struct DemodParams {
    double bw, freq;
    int algo;
    int want_carrier;
    int soft;          // also emit int8 soft values (soft rows + soft trellis words)
};

__device__ __forceinline__ int emitted_symbols(int avail, int fs, bool last)
{
    int R = avail - fs;
    if (R <= 0) return 0;
    int E = R <= 128 ? R : 128 + 64 * ((R - 128) / 80) + max(0, ((R - 128) % 80) - 16);
    return last ? E / 64 : (E + 63) / 64;
}

// phase 0: symbols 0..2 (LTS1, LTS2, SIGNAL) -> EqState ; phase 1: data symbols -> rows
// ALGO: the equalizer (WIFI_EQ_*) as a template parameter: the symbol loop carries only its own update rule
// PHASE: 0 = LTS1, LTS2, SIGNAL -> EqState ; 1 = data symbols -> rows (and trellis words)
template <bool SOFT, int ALGO, int PHASE>
__global__ void __launch_bounds__(128, DEMOD_MINB) k_demod(const cf *__restrict__ iq, const LinkDesc *__restrict__ links, wifi_b200_frame *frames, int f0, int n_frames,
                                                EqState *states, uint8_t *rows, cf *carrier, DemodParams prm,
                                                const uint16_t *__restrict__ depunct_lut, uint32_t *__restrict__ vit_in,
                                                int8_t *__restrict__ soft_rows, uint32_t *__restrict__ vit_soft_in)
{
    __shared__ int8_t s_soft[SOFT ? 4 : 1][SOFT ? 392 : 4];     // soft value of (carrier << 3 | bit); [384] = 0 for erasures
    __shared__ uint16_t s_slut[SOFT ? 4 : 1][SOFT ? 432 : 2];
    __shared__ float s_h2[SOFT ? 4 : 1][SOFT ? 64 : 2];
    __shared__ cf s_hu[4][64];
    __shared__ double s_md[4][64], s_ms[4][64];
    // trellis-word LUT: slots k..k+3 of word w are one uint4 at [k / 4][w], so four offsets come with one load
    __shared__ __align__(16) uint32_t s_lut[4][432];
    // decisions as bit planes: byte (carrier << 3 | bit) = that coded bit (0 / 1), so a LUT entry is the byte
    // offset itself; carrier 48 is a zero slot that the erasure entries point at
    __shared__ __align__(8) uint8_t s_bits[4][49 * 8];
    constexpr int phase = PHASE;
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int f = f0 + blockIdx.x * 4 + wib;
    if (f >= n_frames) return;
    const wifi_b200_frame F = frames[f];
    if (phase == 1 && F.burst_len < SYNC_LENGTH + 63) return;
    const LinkDesc L = links[F.link];
    const cf *x = iq + L.x_off;
    const bool last = L.is_final && (f == L.frame_first + L.frame_count - 1);
    float fo = F.freq_long;
    if (phase == 0) {
        if (!F.found) {   // sync_long keeps d_freq_offset of the last burst that matched
            fo = L.fo_carry;
            for (int g = f - 1; g >= L.frame_first; --g)
                if (frames[g].found) { fo = frames[g].freq_long; break; }
        }
        if (F.burst_len < SYNC_LENGTH + 63) {          // SYNC never completes (end of stream): the record carries the offset in force
            if (lane == 0 && F.n_syms >= 0) frames[f].freq_long = fo;
            return;
        }
    }
    const int avail = F.burst_len - SYNC_LENGTH;
    const int fs = F.frame_start;
    const int n_syms = emitted_symbols(avail, fs, last);
    const float fshort = F.freq_short;
    const float delta = fo - fshort;
    const cf w1 = crot(delta);
    const int64_t t = F.trigger;
    const int hist = L.hist;

    const int iA = lane + 32, iB = lane;      // shifted bin of FFT outputs a (X[lane]) and b (X[lane+32])
    const bool usedA = (iA <= 58), usedB = (iB >= 6);   // iA in 32..63 (32 = DC), iB in 0..31
    const bool dcA = (iA == 32);
    const int carA = c_tab.carrier_of[iA], carB = c_tab.carrier_of[iB];
    const float ltsA = c_tab.lts[iA], ltsB = c_tab.lts[iB];
    const int q0 = warp_fft_in(lane);
    const WarpTw tw = warp_tw(lane, false);

    cf HA = {0.f, 0.f}, HB = {0.f, 0.f};
    cf pp[4] = {{0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}};
    double d_er = 0.0, eps0, snr = 0.0;
    float havg = 1.f, w0A = 1.f, w0B = 1.f;
    int frame_symbols = 0, enc = 0, nb = 1;
    int n_begin, n_end;
    EqState *st = states + f;
    if (phase == 0) {
        eps0 = ((double)fshort - (double)fo) * prm.bw / (2 * M_PI * prm.freq);
        n_begin = 0;
        n_end = n_syms < 3 ? n_syms : 3;
        if (lane == 0) { frames[f].freq_long = fo; frames[f].n_syms = n_syms; }
    } else {
        if (!F.sig_ok) return;
        frame_symbols = F.frame_symbols;
        enc = F.encoding;
        nb = c_tab.mcs[enc].n_bpsc;
        HA = st->H[iA]; HB = st->H[iB];
#pragma unroll
        for (int q = 0; q < 4; ++q) pp[q] = st->prev_pil[q];
        d_er = st->d_er; eps0 = st->eps0;
        if (SOFT) { havg = st->havg; w0A = st->w0[iA]; w0B = st->w0[iB]; }
        n_begin = 3;
        n_end = n_syms < frame_symbols + 3 ? n_syms : frame_symbols + 3;
    }
    // data phase: the warp also depunctures each symbol into the decoder's trellis words (R6
    // unpack + deinterleave + depuncture), 8 steps per 32-bit word, words_per_sym = N_DBPS/8.
    // BPSK 3/4 (N_DBPS 36) does not fill whole words per symbol and goes through k_pack.
    const int ndbps = c_tab.mcs[enc].n_dbps;
    // (frames decode_mac will refuse -- more than 511 symbols / 1528 bytes -- would not fit the per-frame
    // word slot and are never decoded from it, so they are not packed)
    const int wps = (phase == 1 && (ndbps & 7) == 0 && frame_symbols <= WIFI_MAX_SYM && F.length <= WIFI_MAX_PSDU) ? ndbps >> 3 : 0;
    // erasure positions are fixed per (MCS, word): they become a constant OR pattern per lane and their
    // LUT entries point at a zero byte, so the inner loop has no test
    uint32_t era_word = 0;
    if (wps) {
        for (int i = lane; i < 2 * ndbps; i += 32) {
            uint16_t e = depunct_lut[enc * 432 + i];
            s_lut[wib][((i & 15) >> 2) * 108 + (i >> 4) * 4 + (i & 3)] = (e == 0xffffu) ? 48u << 3 : e;   // conflict-free reads
        }
        if (lane < wps)
            for (int k = 0; k < 16; ++k)
                if (depunct_lut[enc * 432 + 16 * lane + k] == 0xffffu) era_word |= 2u << (2 * k);
        if (lane == 0) *reinterpret_cast<uint2 *>(&s_bits[wib][48 * 8]) = make_uint2(0u, 0u);
        __syncwarp();
    }
    uint32_t *vw = vit_in + (int64_t)f * VIT_MAXW;
    // soft mode: N_DBPS/2 words per symbol (2 steps x 2 int8 each); every MCS fills whole words
    const bool soft_on = SOFT && phase == 1;
    const int swps = (soft_on && frame_symbols <= WIFI_MAX_SYM && F.length <= WIFI_MAX_PSDU) ? ndbps >> 1 : 0;
    if (SOFT && soft_on) {
        for (int i = lane; i < 2 * ndbps; i += 32) {
            uint16_t e = depunct_lut[enc * 432 + i];
            s_slut[wib][i] = (e == 0xffffu) ? 384 : e;
        }
        if (lane == 0) s_soft[wib][384] = 0;
        __syncwarp();
    }
    uint32_t *vsw = vit_soft_in ? vit_soft_in + (int64_t)f * SOFT_MAXW : nullptr;
    int n_rows = 0;
    // raw samples of symbol n for this lane (burst positions j0, j0 + 1); the loads of symbol n + 1 are
    // issued before symbol n is processed so that their latency hides behind a whole symbol of arithmetic
    auto sym_j0 = [&](int n) { return fs + ((n < 2) ? 64 * n + q0 : 128 + 80 * (n - 2) + 16 + q0); };
    auto fetch_raw = [&](int n, cf (&raw)[2]) {
        const int j0 = sym_j0(n);
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int j = j0 + u;
            const int64_t src = t + j - 16;
            raw[u] = (j < avail && src >= -(int64_t)hist) ? x[src] : cf{0.f, 0.f};
        }
    };
    cf raw[2] = {{0.f, 0.f}, {0.f, 0.f}};
    if (n_begin < n_end) fetch_raw(n_begin, raw);
    int pidx = n_begin >= 2 ? (n_begin - 2) % 127 : 0;
    for (int n = n_begin; n < n_end; ++n) {
        if (PHASE == 1) __builtin_assume(n >= 3);
        // ---- sync_long COPY: the symbol's samples, both derotations ----
        cf a, b;
        {
            const int j0 = sym_j0(n);
            const cf s0 = raw[0], s1 = raw[1];
            if (n + 1 < n_end) fetch_raw(n + 1, raw);
            // one rotation by delta = freq_long - freq_short: the even sample by exp(j delta j0), the odd one behind
            // it by that times exp(j delta) (oracle: sync_long COPY)
            const cf r0 = crot(delta * (float)j0);
            const cf r1 = cmul(r0, w1);
            a = (j0 < avail) ? cmul(s0, r0) : cf{0.f, 0.f};
            b = (j0 + 1 < avail) ? cmul(s1, r1) : cf{0.f, 0.f};
        }
        warp_fft64(a, b, lane, tw);
        // a = cur[iA], b = cur[iB] (fftshift)
        {
            double k = 2 * M_PI * n * 80 * (eps0 + d_er);
            double phA = k * (iA - 32) / 64, phB = k * (iB - 32) / 64;
            a = cmul(a, crot((float)phA));
            b = cmul(b, crot((float)phB));
        }
        cf c11 = cshfl(b, 11), c25 = cshfl(b, 25), c39 = cshfl(a, 7), c53 = cshfl(a, 21);
        const float p = (n >= 2) ? c_tab.polarity[pidx] : 1.f;        // pidx = (n - 2) mod 127, kept as a counter
        if (n >= 2) pidx = pidx == 126 ? 0 : pidx + 1;
        cf pil[4];
        double beta;
        cf sbeta;
        if (n < 2) {
            sbeta = cadd(cadd(csub(c11, c25), c39), c53);
            pil[0] = c11; pil[1] = cf{-c25.re, -c25.im}; pil[2] = c39; pil[3] = c53;
        } else {
            pil[0] = cscale(c11, p); pil[1] = cscale(c25, p); pil[2] = cscale(c39, p); pil[3] = cscale(c53, -p);
            sbeta = cadd(cadd(cadd(pil[0], pil[2]), pil[1]), pil[3]);
        }
        // the pilot phase (beta) and the pilot-to-pilot rotation (er) are both one atan2 of a warp-uniform
        // argument: lanes 0-15 evaluate the first, lanes 16-31 the second, one shuffle each hands them out
        cf ser = {0.f, 0.f};
        if (n >= 2) {
#pragma unroll
            for (int q = 0; q < 4; ++q) ser = wdm_cmacc(ser, pil[q], pp[q]);
        }
        const bool up = lane >= 16;
        const float at = wdm_atan2f(up ? ser.im : sbeta.im, up ? ser.re : sbeta.re);
        beta = (double)__shfl_sync(0xffffffffu, at, 0);
        double er = 0.0;
        if (n >= 2) {
            er = (double)__shfl_sync(0xffffffffu, at, 16);
            er *= prm.bw / (2 * M_PI * prm.freq * 80);
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) pp[q] = pil[q];
        const cf wb = crot((float)(-beta));
        a = cmul(a, wb);
        b = cmul(b, wb);
        if (n >= 2) d_er = (1 - 0.1) * d_er + 0.1 * er;

        // ---- equalizer::equalize ----
        if (ALGO == WIFI_EQ_COMB) {
            cf r11 = cmul(c11, wb), r25 = cmul(c25, wb), r39 = cmul(c39, wb), r53 = cmul(c53, wb);
            cf cp[4];
            if (n < 2) { cp[0] = r11; cp[1] = cf{-r25.re, -r25.im}; cp[2] = r39; cp[3] = r53; }
            else { cp[0] = cscale(r11, p); cp[1] = cscale(r25, p); cp[2] = cscale(r39, p); cp[3] = cscale(r53, -p); }
            cf avg = cscale(cadd(cadd(cadd(cp[0], cp[1]), cp[2]), cp[3]), 0.25f);
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                int i = u ? iB : iA;
                cf G;
                if (i <= 11) G = cadd(cscale(avg, (float)(11 - i) / 11.0f), cscale(cp[0], (float)i / 11.0f));
                else if (i <= 25) G = cadd(cscale(cp[0], (float)(25 - i) / 14.0f), cscale(cp[1], (float)(i - 11) / 14.0f));
                else if (i <= 39) G = cadd(cscale(cp[1], (float)(39 - i) / 14.0f), cscale(cp[2], (float)(i - 25) / 14.0f));
                else if (i <= 53) G = cadd(cscale(cp[2], (float)(53 - i) / 14.0f), cscale(cp[3], (float)(i - 39) / 14.0f));
                else G = cadd(cscale(cp[3], (float)(64 - i) / 11.0f), cscale(avg, (float)(i - 53) / 11.0f));
                if (u) b = cdiv(b, G); else a = cdiv(a, G);
            }
        }
        // (PHASE == 0 spelt out: on the n >= 3 assumption alone the compiler keeps the LTS blocks in the data loop)
        if (PHASE == 0 && n == 0) {
            HA = a; HB = b;
        } else if (PHASE == 0 && n == 1) {
            {
                cf d = csub(HA, a), s = cadd(HA, a);
                float md = sqrtf(d.re * d.re + d.im * d.im), ms = sqrtf(s.re * s.re + s.im * s.im);
                s_md[wib][iA] = (double)md * (double)md; s_ms[wib][iA] = (double)ms * (double)ms;
                if (usedA && !dcA) HA = cdiv(s, cf{ltsA * 2.0f, 0.f});
                d = csub(HB, b); s = cadd(HB, b);
                md = sqrtf(d.re * d.re + d.im * d.im); ms = sqrtf(s.re * s.re + s.im * s.im);
                s_md[wib][iB] = (double)md * (double)md; s_ms[wib][iB] = (double)ms * (double)ms;
                if (usedB) HB = cdiv(s, cf{ltsB * 2.0f, 0.f});
            }
            if (SOFT) {
                s_h2[wib][iA] = HA.re * HA.re + HA.im * HA.im;
                s_h2[wib][iB] = HB.re * HB.re + HB.im * HB.im;
            }
            __syncwarp();
            if (lane == 0) {
                double signal = 0, noise = 0;
                float acc = 0.f;
                for (int i = 6; i <= 58; ++i) {
                    if (i == 32) continue;
                    noise += s_md[wib][i];
                    signal += s_ms[wib][i];
                    if (SOFT) acc += s_h2[wib][i];
                }
                snr = 10 * log10(signal / noise / 2);
                havg = acc / 52.0f;
            }
            if (SOFT) {
                havg = __shfl_sync(0xffffffffu, havg, 0);
                w0A = s_h2[wib][iA] / havg;
                w0B = s_h2[wib][iB] / havg;
            }
            __syncwarp();
        } else {
            // Straight-line carrier path: every lane equalizes and decides both of its bins, and the results of a
            // bin that is no data carrier (pilot, DC, guard) are never stored or selected into H.  Branching per
            // carrier instead made the warp run both sides of every test.
            cf ptA, ptB;
            int bitsA, bitsB;
            const cf symA = cdiv(a, HA), symB = cdiv(b, HB);
            dev_decide_point(nb, symA, bitsA, ptA);
            dev_decide_point(nb, symB, bitsB, ptB);
            SoftQ sqA = {}, sqB = {};
            if (SOFT && soft_on) { sqA = dev_soft_demap(nb, symA, w0A); sqB = dev_soft_demap(nb, symB, w0B); }
            if (ALGO == WIFI_EQ_LMS) {
                const cf qA = cdiv(a, ptA), qB = cdiv(b, ptB);
                const cf nA = cadd(cscale(HA, 0.5f), cscale(qA, 0.5f)), nB = cadd(cscale(HB, 0.5f), cscale(qB, 0.5f));
                HA = carA >= 0 ? nA : HA;
                HB = carB >= 0 ? nB : HB;
            }
            cf huA = {0.f, 0.f}, huB = {0.f, 0.f};
            if (ALGO == WIFI_EQ_STA) {
                const cf dA = cdiv(a, ptA), dB = cdiv(b, ptB);
                const cf pA = cscale(a, iA == 53 ? -p : p), pB = cscale(b, p);
                huA = carA >= 0 ? dA : (iA == 39 || iA == 53) ? pA : huA;
                huB = carB >= 0 ? dB : (iB == 11 || iB == 25) ? pB : huB;
            }
            if (ALGO == WIFI_EQ_STA) {
                s_hu[wib][iA] = huA; s_hu[wib][iB] = huB;
                __syncwarp();
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    int i = u ? iB : iA;
                    if (i < 6 || i > 58 || i == 32) continue;
                    cf sum = {0.f, 0.f};
                    int cnt = 0;
                    for (int k = i - 2; k <= i + 2; ++k) {
                        if (k == 32 || k < 6 || k > 58) continue;
                        sum = cadd(sum, s_hu[wib][k]);
                        ++cnt;
                    }
                    cf avg = {sum.re / (float)cnt, sum.im / (float)cnt};
                    if (u) HB = cadd(cscale(HB, 0.5f), cscale(avg, 0.5f));
                    else HA = cadd(cscale(HA, 0.5f), cscale(avg, 0.5f));
                }
                __syncwarp();
            }
            if (PHASE == 0) {   // n == 2: SIGNAL
                if (carA >= 0) st->sig_bits[carA] = (uint8_t)bitsA;
                if (carB >= 0) st->sig_bits[carB] = (uint8_t)bitsB;
            } else {
                int64_t row = F.row_off + (n - 3);
                if (carA >= 0) rows[row * 48 + carA] = (uint8_t)bitsA;
                if (carB >= 0) rows[row * 48 + carB] = (uint8_t)bitsB;
                if (prm.want_carrier) {
                    if (carA >= 0) carrier[row * 48 + carA] = symA;
                    if (carB >= 0) carrier[row * 48 + carB] = symB;
                }
                if (wps) {
                    // spread the six decision bits over six bytes: (x & 15) * (1 + 2^7 + 2^14 + 2^21) puts bit j at bit 8 j
                    if (carA >= 0)
                        *reinterpret_cast<uint2 *>(&s_bits[wib][carA * 8]) =
                            make_uint2((((uint32_t)bitsA & 15u) * 0x00204081u) & 0x01010101u, (((uint32_t)bitsA >> 4) * 0x81u) & 0x0101u);
                    if (carB >= 0)
                        *reinterpret_cast<uint2 *>(&s_bits[wib][carB * 8]) =
                            make_uint2((((uint32_t)bitsB & 15u) * 0x00204081u) & 0x01010101u, (((uint32_t)bitsB >> 4) * 0x81u) & 0x0101u);
                    __syncwarp();
                    if (lane < wps) {
                        uint32_t word = era_word;
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const uint4 e = reinterpret_cast<const uint4 *>(s_lut[wib])[j * 27 + lane];
                            // disjoint bit positions: + is |
                            word += ((uint32_t)s_bits[wib][e.x] << (8 * j)) + ((uint32_t)s_bits[wib][e.y] << (8 * j + 2)) +
                                    ((uint32_t)s_bits[wib][e.z] << (8 * j + 4)) + ((uint32_t)s_bits[wib][e.w] << (8 * j + 6));
                        }
                        vw[(n - 3) * wps + lane] = word;
                    }
                    __syncwarp();
                }
                if (SOFT && soft_on) {
                    const int hb = nb > 1 ? nb >> 1 : 1;
#pragma unroll
                    for (int u = 0; u < 2; ++u)
#pragma unroll
                        for (int t = 0; t < 3; ++t) {
                            if (t < hb && (u == 0 || nb > 1)) {
                                const int k = u * hb + t;
                                if (carA >= 0) { s_soft[wib][(carA << 3) | k] = (int8_t)sqA.q[u][t]; soft_rows[row * SOFT_ROW + carA * nb + k] = (int8_t)sqA.q[u][t]; }
                                if (carB >= 0) { s_soft[wib][(carB << 3) | k] = (int8_t)sqB.q[u][t]; soft_rows[row * SOFT_ROW + carB * nb + k] = (int8_t)sqB.q[u][t]; }
                            }
                        }
                    __syncwarp();
                    for (int w = lane; w < swps; w += 32) {
                        uint32_t word = 0;
#pragma unroll
                        for (int k = 0; k < 4; ++k) word |= (uint32_t)(uint8_t)s_soft[wib][s_slut[wib][4 * w + k]] << (8 * k);
                        vsw[(n - 3) * swps + w] = word;
                    }
                    __syncwarp();
                }
                ++n_rows;
            }
        }
    }
    if (phase == 0) {
        st->H[iA] = HA; st->H[iB] = HB;
        if (SOFT) { st->w0[iA] = w0A; st->w0[iB] = w0B; }
        if (lane == 0) {
#pragma unroll
            for (int q = 0; q < 4; ++q) st->prev_pil[q] = pp[q];
            st->d_er = d_er; st->eps0 = eps0; st->snr = snr; st->havg = havg;
        }
    } else if (lane == 0) {
        frames[f].n_rows = n_rows;
    }
}

// ------------------------------------------------------------------ R5f SIGNAL field
// One thread per frame: deinterleave 48 hard bits, 62-step Viterbi (ntb 5) on VitCoreH, parse_signal.
__global__ void __launch_bounds__(VIT_BLOCK) k_signal(wifi_b200_frame *frames, int f0, int n_frames, const EqState *states)
{
    __shared__ uint32_t ring[5 * 16 * VIT_BLOCK];
    __shared__ uint4 s_bm[8 * 4 * 16];
    __shared__ uint32_t s_hop[VIT_HOP_ENTRIES];
    const int tid = threadIdx.x;
    for (int i = tid; i < 512; i += VIT_BLOCK) s_bm[i] = VitCoreH::table_entry(i >> 6, (i >> 4) & 3, (uint32_t)(i & 15));
    for (int i = tid; i < VIT_HOP_ENTRIES; i += VIT_BLOCK) s_hop[i] = vit_h_hop_entry(i);
    __syncthreads();
    int f = f0 + blockIdx.x * VIT_BLOCK + tid;
    if (f >= n_frames) return;
    if (frames[f].n_syms < 3) return;
    const EqState *st = states + f;
    // 48 deinterleaved bits as 24 nibbles: step t uses deint[2t], deint[2t+1]; deint[i] = bits[(i%16)*3 + i/16]
    uint64_t lo = 0, hi = 0;   // nibble t at bits 4t (t < 16 in lo, else hi)
    for (int tstep = 0; tstep < 24; ++tstep) {
        int i0 = 2 * tstep, i1 = i0 + 1;
        uint32_t s0 = st->sig_bits[(i0 % 16) * 3 + i0 / 16] & 1u, s1 = st->sig_bits[(i1 % 16) * 3 + i1 / 16] & 1u;
        uint64_t nib = s0 | (s1 << 2);
        if (tstep < 16) lo |= nib << (4 * tstep); else hi |= nib << (4 * (tstep - 16));
    }
    // k_viterbi's decoder, chunk for chunk; (lo, hi) is a 128-bit shift register of nibbles, zeros after step 24.
    // Chunk 0 has 6 steps: two erased steps in front of them leave the all-zero metrics as they are and set bits 0, 1
    // of every path byte, which trace_begin masks off (keep = 0xfc)
    VitCoreH v;
    v.init();
    const uint32_t first = (uint32_t)lo;
    v.step4<0>(s_bm, 0xau, 0xau, first & 0xfu, (first >> 4) & 0xfu);
    v.step4<4>(s_bm, (first >> 8) & 0xfu, (first >> 12) & 0xfu, (first >> 16) & 0xfu, (first >> 20) & 0xfu);
    uint8_t *rbt = reinterpret_cast<uint8_t *>(ring) + 4 * tid;   // the thread's column of slot 0
    const uint32_t rbt_sh = (uint32_t)__cvta_generic_to_shared(rbt), hop_sh = (uint32_t)__cvta_generic_to_shared(s_hop);
    v.trace_begin(rbt + VIT_SLOT_BYTES, rbt_sh + VIT_SLOT_BYTES, s_hop, true, 0xfcu);
    uint32_t dec = 0;   // decoded bit i at bit i
#pragma unroll 1
    for (int chunk = 1; chunk < 8; ++chunk) {
        const uint32_t bits = (uint32_t)(lo >> 24);   // steps 8 * chunk - 2 .. 8 * chunk + 5
        lo = (lo >> 32) | (hi << 32);
        hi >>= 32;
        v.step4<0>(s_bm, bits & 0xfu, (bits >> 4) & 0xfu, (bits >> 8) & 0xfu, (bits >> 12) & 0xfu);
        v.step4<4>(s_bm, (bits >> 16) & 0xfu, (bits >> 20) & 0xfu, (bits >> 24) & 0xfu, bits >> 28);
        int sl = (chunk + 1) % 5;
        uint32_t c = v.trace_begin(rbt + sl * VIT_SLOT_BYTES, rbt_sh + sl * VIT_SLOT_BYTES, s_hop, (chunk & 3) == 0);
        if (chunk >= 5) {
            // four hops back through slots sl - 1 .. sl - 4 (mod 5); the ring byte holds the decisions in ascending
            // bit order, as dec does.  The first hop reads the snapshot just stored: keep the stores ahead of it.
            asm volatile("" ::: "memory");
            for (int i = 0; i < 4; ++i) {
                sl = sl == 0 ? 4 : sl - 1;
                c = VitCoreH::hop(c, hop_sh, rbt_sh + sl * VIT_SLOT_BYTES);
            }
            dec |= VitCoreH::ring_byte(c) << (8 * (chunk - 5));
        }
    }
    int r = 0, len = 0;
    bool parity = false;
    for (int i = 0; i < 17; ++i) {
        bool bit = (dec >> i) & 1u;
        parity ^= bit;
        if (i < 4 && bit) r |= 1 << i;
        if (bit && i > 4) len |= 1 << (i - 5);
    }
    if (parity != (bool)((dec >> 17) & 1u)) return;
    int enc;
    switch (r) {
    case 11: enc = 0; break;
    case 15: enc = 1; break;
    case 10: enc = 2; break;
    case 14: enc = 3; break;
    case 9: enc = 4; break;
    case 13: enc = 5; break;
    case 8: enc = 6; break;
    case 12: enc = 7; break;
    default: return;
    }
    int ndbps = c_tab.mcs[enc].n_dbps;
    frames[f].sig_ok = 1;
    frames[f].encoding = enc;
    frames[f].length = len;
    frames[f].frame_symbols = (16 + 8 * len + 6 + ndbps - 1) / ndbps;
    frames[f].snr = st->snr;
}

// ------------------------------------------------------------------ R6 decode_mac planning
// decode_mac's tag / symbol-collection state machine (see oracle rx_link).  One warp per link.
// A frame is "regular" when its SIGNAL decoded, it passes the size check and it delivered all of
// its symbols: then it resets the collection state whatever came before (unless an older tag is
// still pending) and forms a job on its own.  Groups of 32 frames that are all regular or
// SIGNAL-less are planned in parallel; any other group falls back to the sequential machine.
struct PlanState { int cur, copied, need, pending; JobDesc J; };

__device__ void plan_sequential(PlanState &S, int f0, int f1, wifi_b200_frame *frames, JobDesc *jobs, int *pack_list, int *n_pack, int *err, int soft)
{
    for (int fi = f0; fi < f1; ++fi) {
        wifi_b200_frame F = frames[fi];
        if (!F.sig_ok) continue;
        if (F.n_rows == 0) {
            if (S.pending < 0) S.pending = fi;
            continue;
        }
        int tagf = S.pending >= 0 ? S.pending : fi;
        S.pending = -1;
        int t_sym = frames[tagf].frame_symbols, t_len = frames[tagf].length;
        if (t_sym <= WIFI_MAX_SYM && t_len <= WIFI_MAX_PSDU) {
            frames[tagf].accepted = 1;
            S.cur = tagf;
            S.copied = 0;
            S.need = t_sym;
            S.J.frame = tagf; S.J.enc = frames[tagf].encoding; S.J.len = t_len; S.J.n_sym = t_sym; S.J.n_seg = 0; S.J.need_pack = 0;
        }
        if (S.cur < 0 || S.copied >= S.need) continue;
        int take = F.n_rows < S.need - S.copied ? F.n_rows : S.need - S.copied;
        if (S.J.n_seg < 4) {
            S.J.seg_row[S.J.n_seg] = (int32_t)F.row_off;
            S.J.seg_cnt[S.J.n_seg] = take;
        }
        S.J.n_seg++;              // beyond four the packer walks the frame records (job_row)
        S.copied += take;
        if (S.copied == S.need) {
            S.J.last_frame = fi;
            S.J.pad0 = 0;
            for (int s = S.J.n_seg; s < 4; ++s) { S.J.seg_row[s] = 0; S.J.seg_cnt[s] = 0; }
            bool own = (S.J.n_seg == 1 && fi == S.cur);
            S.J.need_pack = (!own || (!soft && (c_tab.mcs[S.J.enc].n_dbps & 7) != 0)) ? 1 : 0;
            jobs[S.cur] = S.J;
            if (S.J.need_pack) pack_list[atomicAdd(n_pack, 1)] = S.cur;
            frames[S.cur].decoded = 1;
            frames[S.cur].psdu_off = (int64_t)S.cur * PSDU_STRIDE;
        }
    }
}

// Fast path: one thread per frame.  A "regular" frame forms its own job and a SIGNAL-less frame forms
// none, whatever surrounds them -- unless some frame of the link is irregular (SIGNAL ok but no rows,
// too few rows, or an oversize tag), in which case the link is flagged and k_plan replays the exact
// sequential state machine over it, from its first irregular frame on (everything in front of that frame is regular or
// SIGNAL-less, which leaves decode_mac's state closed: the fast path's answer stands there).
__global__ void __launch_bounds__(128) k_plan_fast(wifi_b200_frame *frames, int f0, int n_frames, JobDesc *jobs, int *pack_list, int *n_pack,
                                                    int *link_dirty, int soft)
{
    int fi = f0 + blockIdx.x * blockDim.x + threadIdx.x;
    if (fi >= n_frames) return;
    const wifi_b200_frame *F = frames + fi;
    const int sig = F->sig_ok, nrows = F->n_rows, fsym = F->frame_symbols, len = F->length, enc = F->encoding;
    jobs[fi].n_sym = 0;
    if (!sig) return;
    const bool regular = nrows > 0 && fsym <= WIFI_MAX_SYM && len <= WIFI_MAX_PSDU && nrows >= fsym;
    if (!regular) { atomicMax(&link_dirty[F->link], 0x7fffffff - fi); return; }   // records the link's FIRST irregular frame
    JobDesc J;
    J.frame = fi; J.enc = enc; J.len = len; J.n_sym = fsym; J.n_seg = 1;
    J.seg_row[0] = (int32_t)F->row_off; J.seg_cnt[0] = fsym;
    for (int s = 1; s < 4; ++s) { J.seg_row[s] = 0; J.seg_cnt[s] = 0; }
    J.need_pack = (!soft && (c_tab.mcs[enc].n_dbps & 7) != 0) ? 1 : 0;
    J.last_frame = fi; J.pad0 = 0;
    jobs[fi] = J;
    if (J.need_pack) pack_list[atomicAdd(n_pack, 1)] = fi;
    frames[fi].accepted = 1;
    frames[fi].decoded = 1;
    frames[fi].psdu_off = (int64_t)fi * PSDU_STRIDE;
}

// link_open[l]: frame at which the link's decode_mac state was left open at the end of the buffer (a tag waiting for
// rows, or a collection short of symbols), -1 if closed.  Streaming uses it to defer those frames while the next burst
// is still held back.
__global__ void __launch_bounds__(128) k_plan(const LinkDesc *__restrict__ links, int n_links, wifi_b200_frame *frames, JobDesc *jobs,
                                               int *pack_list, int *n_pack, int *err, int soft, const int *__restrict__ link_dirty,
                                               int *__restrict__ link_open)
{
    int l = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (l >= n_links) return;
    const int dirty = link_dirty[l];
    if (!dirty) return;                  // every frame of the link was regular or SIGNAL-less: k_plan_fast is exact
    const LinkDesc L = links[l];
    PlanState S;
    S.cur = -1; S.copied = 0; S.need = 0; S.pending = -1; S.J.n_seg = 0;
    const int fend = L.frame_first + L.frame_count;
    // start at the group of 32 that holds the first irregular frame: no tag is pending and no collection open in front of
    // it, which is the state above (a long stream cut at an arbitrary sample has ONE irregular frame, its last)
    const int fstart = L.frame_first + (((0x7fffffff - dirty) - L.frame_first) & ~31);
    for (int f0 = fstart; f0 < fend; f0 += 32) {
        int fi = f0 + lane;
        bool valid = fi < fend;
        int sig = 0, nrows = 0, fsym = 0, len = 0, enc = 0;
        long long row_off = 0;
        if (valid) {
            const wifi_b200_frame *F = frames + fi;
            sig = F->sig_ok; nrows = F->n_rows; fsym = F->frame_symbols; len = F->length; enc = F->encoding; row_off = F->row_off;
            jobs[fi].n_sym = 0;          // undo what the fast path wrote for this frame
            frames[fi].accepted = 0; frames[fi].decoded = 0; frames[fi].psdu_off = -1;
        }
        bool regular = valid && sig && nrows > 0 && fsym <= WIFI_MAX_SYM && len <= WIFI_MAX_PSDU && nrows >= fsym;
        bool quiet = !valid || !sig;
        bool all_simple = __all_sync(0xffffffffu, regular || quiet);
        if (all_simple && S.pending < 0) {
            if (regular) {
                JobDesc J;
                J.frame = fi; J.enc = enc; J.len = len; J.n_sym = fsym; J.n_seg = 1;
                J.seg_row[0] = (int32_t)row_off; J.seg_cnt[0] = fsym;
                for (int s = 1; s < 4; ++s) { J.seg_row[s] = 0; J.seg_cnt[s] = 0; }
                J.need_pack = (!soft && (c_tab.mcs[enc].n_dbps & 7) != 0) ? 1 : 0;
                J.last_frame = fi; J.pad0 = 0;
                jobs[fi] = J;
                if (J.need_pack) pack_list[atomicAdd(n_pack, 1)] = fi;
                frames[fi].accepted = 1;
                frames[fi].decoded = 1;
                frames[fi].psdu_off = (int64_t)fi * PSDU_STRIDE;
            }
            unsigned reg = __ballot_sync(0xffffffffu, regular);
            if (reg) {   // state after the last regular frame: its collection is complete
                int lastl = 31 - __clz((int)reg);
                S.cur = f0 + lastl;
                S.need = __shfl_sync(0xffffffffu, fsym, lastl);
                S.copied = S.need;
                S.J.n_seg = 0;
            }
        } else {
            __syncwarp();   // the jobs[].n_sym = 0 defaults above must land before the sequential writes
            if (lane == 0) plan_sequential(S, f0, f0 + 32 < fend ? f0 + 32 : fend, frames, jobs, pack_list, n_pack, err, soft);
            S.cur = __shfl_sync(0xffffffffu, S.cur, 0);
            S.copied = __shfl_sync(0xffffffffu, S.copied, 0);
            S.need = __shfl_sync(0xffffffffu, S.need, 0);
            S.pending = __shfl_sync(0xffffffffu, S.pending, 0);
            // S.J of an open collection lives in lane 0 only; lane 0 is the one that continues it
        }
    }
    if (lane == 0) link_open[l] = S.pending >= 0 ? S.pending : ((S.cur >= 0 && S.copied < S.need) ? S.cur : -1);
}

// ------------------------------------------------------------------ R6 unpack/deinterleave/depuncture
// Only for the jobs k_demod could not pack itself (pack_list): gathered rows, BPSK 3/4.
// depunct_lut[enc][q] for q in [0, 2*n_dbps): 0xffff = erasure, else (carrier << 3) | bit
__global__ void __launch_bounds__(256) k_pack(const JobDesc *__restrict__ jobs, const int *__restrict__ pack_list, const int *__restrict__ n_pack,
                                               const uint8_t *__restrict__ rows, const uint16_t *__restrict__ depunct_lut, uint32_t *__restrict__ vit_in,
                                               const wifi_b200_frame *__restrict__ frames)
{
    const int np = *n_pack;
    for (int e = blockIdx.y; e < np; e += gridDim.y) {
        const JobDesc J = jobs[pack_list[e]];
        if (J.n_sym == 0 || !J.need_pack) continue;     // stale entry of a link that was re-planned
        const int ndbps = c_tab.mcs[J.enc].n_dbps;
        const int per = 2 * ndbps;
        const int n_data = J.n_sym * ndbps;
        const int n_words = (n_data + 7) >> 3;
        const uint16_t *lut = depunct_lut + J.enc * 432;
        uint32_t *vw = vit_in + (int64_t)J.frame * VIT_MAXW;
        for (int w = blockIdx.x * blockDim.x + threadIdx.x; w < n_words; w += gridDim.x * blockDim.x) {
            int tstep = 8 * w;
            int q = 2 * tstep;
            int s = q / per, qi = q - s * per;
            const uint8_t *rp = rows + job_row(J, frames, s) * 48;
            uint32_t word = 0;
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                uint32_t sym = 0;
                if (tstep + (k >> 1) < n_data) {
                    uint16_t en = lut[qi];
                    sym = (en == 0xffffu) ? 2u : ((rp[en >> 3] >> (en & 7)) & 1u);
                }
                word |= sym << (2 * k);
                if (++qi == per) {
                    qi = 0;
                    ++s;
                    if (s < J.n_sym) rp = rows + job_row(J, frames, s) * 48;
                }
            }
            vw[w] = word;
        }
    }
}

// ------------------------------------------------------------------ R6a-c Viterbi + descramble + CRC
// One thread per frame slot; jobs[frame].n_sym == 0 means nothing to decode.  Trellis words of the
// frame are contiguous (in[frame][w]); words past the coded data read as 0 (oracle note 2).
// viterbi_body is the kernel of both one-trellis-per-thread decoders: k_viterbi (hard decisions, VitCoreH) and
// k_viterbi_soft (soft decisions, VitCoreS).  A reader, VitHardIn or VitSoftIn, names the core and feeds it its
// input: chunk 0 (6 steps, run as two erased steps + 6) in first(), then the eight steps of each further chunk as
// fetch() and two four-step halves; prefetch() runs once between them.

// hard decisions (k_pack, k_demod): one word of eight steps x two 2-bit symbols (2 = erased) per word; chunk j >= 1 is
// the last two steps of word j - 1 and the first six of word j.  VitCoreH reads its branch words from the table.
struct VitHardIn {
    using Core = VitCoreH;
    static constexpr int MAXW = VIT_MAXW, BM = 512;   // words per job; entries of the branch-word table
    static __device__ __forceinline__ uint4 table_entry(int i) { return VitCoreH::table_entry(i >> 6, (i >> 4) & 3, (uint32_t)(i & 15)); }
    static __device__ __forceinline__ int words(const JobDesc &J) { return (J.n_sym * c_tab.mcs[J.enc].n_dbps + 7) >> 3; }
    const uint32_t *in;
    int nw;
    const uint4 *bm;
    uint32_t prev, next, bits;
    __device__ __forceinline__ void first(VitCoreH &v)
    {
        prev = in[0];
        v.step4<0>(bm, 0xau, 0xau, prev & 0xfu, (prev >> 4) & 0xfu);
        v.step4<4>(bm, (prev >> 8) & 0xfu, (prev >> 12) & 0xfu, (prev >> 16) & 0xfu, (prev >> 20) & 0xfu);
    }
    // word 1, read ahead for chunk 1.  Loaded here, after chunk 0's snapshot, rather than in first(): the earlier load
    // changes ptxas's register allocation of the whole kernel
    __device__ __forceinline__ void prefetch() { next = 1 < nw ? in[1] : 0u; }
    __device__ __forceinline__ void fetch(int chunk)
    {
        bits = __funnelshift_r(prev, next, 24);
        prev = next;
        next = (chunk + 1 < nw) ? in[chunk + 1] : 0u;
    }
    template <int H>
    __device__ __forceinline__ void half(VitCoreH &v)
    {
        const uint32_t b = bits >> (16 * H);
        v.step4<4 * H>(bm, b & 0xfu, (b >> 4) & 0xfu, (b >> 8) & 0xfu, (b >> 12) & 0xfu);
    }
};

// soft decisions (k_pack_soft, k_demod): one word of two steps x two int8 soft values (0 = erased); chunk j >= 1 is
// words 4j - 1 .. 4j + 2.  No branch-word table.
struct VitSoftIn {
    using Core = VitCoreS;
    static constexpr int MAXW = SOFT_MAXW, BM = 0;
    static __device__ __forceinline__ int words(const JobDesc &J) { return J.n_sym * (c_tab.mcs[J.enc].n_dbps >> 1); }
    const uint32_t *in;
    int nw;
    const uint4 *bm;                      // unused: no branch-word table
    uint32_t w[4];
    __device__ __forceinline__ uint32_t at(int i) const { return i < nw ? in[i] : 0u; }
    __device__ __forceinline__ void first(VitCoreS &v)
    {
        v.step4<0>(0u, at(0));            // soft value 0: every branch value is 254, every candidate ties
        v.step4<4>(at(1), at(2));
    }
    __device__ __forceinline__ void prefetch() {}   // fetch() reads a chunk's words itself
    __device__ __forceinline__ void fetch(int chunk)
    {
#pragma unroll
        for (int k = 0; k < 4; ++k) w[k] = at(4 * chunk - 1 + k);
    }
    template <int H>
    __device__ __forceinline__ void half(VitCoreS &v) { v.step4<4 * H>(w[2 * H], w[2 * H + 1]); }
};

// dynamic shared memory of viterbi_body: ring, CRC table, descrambler table, the reader's branch-word table (16 bytes an
// entry), traceback rows (24 x 48 bytes), hop table (320 words): 52864 bytes for k_viterbi (4 blocks per SM), 44672
// for k_viterbi_soft
template <class In>
constexpr int vit_smem_bytes() { return (VIT_NTB_MAX * 16 * VIT_BLOCK + 256) * 4 + 256 + In::BM * 16 + VIT_ROWS * 48 + VIT_HOP_ENTRIES * 4; }

// tid: threadIdx.x as the kernel reads it, where __launch_bounds__ tells the compiler that it is below VIT_BLOCK
template <class In>
__device__ __forceinline__ void viterbi_body(int tid, const JobDesc *__restrict__ jobs, int f0, int n_frames, const uint32_t *__restrict__ vin,
                                             uint32_t *__restrict__ psdu, wifi_b200_frame *frames)
{
    extern __shared__ uint32_t vsm[];
    uint32_t *ring = vsm;                                   // VIT_NTB_MAX*16*VIT_BLOCK words
    uint32_t *s_crc = vsm + VIT_NTB_MAX * 16 * VIT_BLOCK;   // 256
    uint16_t *s_scr = (uint16_t *)(s_crc + 256);            // 128
    uint4 *s_bm = (uint4 *)(s_crc + 256 + 64);              // branch-word table, In::BM entries (VitCoreH::table_entry)
    uint4 *s_rows = s_bm + In::BM;                          // traceback rows [VIT_ROWS][3] (vit_h_row_entry)
    uint32_t *s_hop = (uint32_t *)(s_rows + 3 * VIT_ROWS);  // hop table (vit_h_hop_entry)
    for (int i = tid; i < 256; i += VIT_BLOCK) s_crc[i] = c_tab.crc_tab[i];
    for (int i = tid; i < 128; i += VIT_BLOCK) s_scr[i] = c_tab.scr_tab[i];
    if constexpr (In::BM > 0)
        for (int i = tid; i < In::BM; i += VIT_BLOCK) s_bm[i] = In::table_entry(i);
    for (int i = tid; i < 12 * VIT_ROWS; i += VIT_BLOCK) ((uint32_t *)s_rows)[i] = vit_h_row_entry(i / 12, i % 12);
    for (int i = tid; i < VIT_HOP_ENTRIES; i += VIT_BLOCK) s_hop[i] = vit_h_hop_entry(i);
    // the identity slot, in every thread's column (a frame with ntb = 10 overwrites it with snapshots and never reads it
    // as such)
    for (int w = 0; w < 16; ++w) ring[(VIT_ID_SLOT * 16 + w) * VIT_BLOCK + tid] = vit_h_identity_word(w);
    __syncthreads();
    const int job = f0 + blockIdx.x * VIT_BLOCK + tid;
    if (job >= n_frames) return;
    const JobDesc J = jobs[job];
    if (J.n_sym == 0) return;
    const int punct = c_tab.mcs[J.enc].punct;
    const int ntb = punct == 0 ? 5 : (punct == 1 ? 9 : 10);   // the three depths the traceback rows know (vit_h_row_entry)
    In f{vin + (int64_t)job * In::MAXW, In::words(J), s_bm};
    uint32_t *out = psdu + (int64_t)job * (PSDU_STRIDE / 4);
    const int L = J.len;
    const int last_chunk = L + 1 + ntb;   // chunk whose traceback yields PSDU byte L-1
    typename In::Core v;
    v.init();
    // chunk 0 has 6 steps: two erased steps in front of them leave all metrics equal and set bits 0, 1 of every path
    // byte, which trace_begin masks off (keep = 0xfc)
    f.first(v);
    // the traceback of chunk j - 1 (snapshot slot s = j mod ntb, row `row`) runs interleaved with the trellis steps of
    // chunk j, three hops before each half and three before the output byte; the cursor `c` is a ring byte offset
    // (VitCoreH), the hops' slots come from the row
    uint8_t *rbt = reinterpret_cast<uint8_t *>(ring) + 4 * tid;   // the thread's column of slot 0
    const uint32_t rbt_sh = (uint32_t)__cvta_generic_to_shared(rbt), hop_sh = (uint32_t)__cvta_generic_to_shared(s_hop);
    int row = 3 * (vit_h_row0(ntb) + 1);
    uint4 r0 = s_rows[row];
    uint32_t c = v.trace_begin(rbt + r0.x, rbt_sh + r0.y, s_hop, true, 0xfcu);
    PsduSink sink;
    sink.init(out, L, s_crc, s_scr);
    f.prefetch();
#pragma unroll 1
    for (int chunk = 1; chunk <= last_chunk; ++chunk) {
        f.fetch(chunk);
        const uint4 r1 = s_rows[row + 1], r2 = s_rows[row + 2];
        c = VitCoreH::hop(c, hop_sh, rbt_sh + r0.z);
        c = VitCoreH::hop(c, hop_sh, rbt_sh + r0.w);
        c = VitCoreH::hop(c, hop_sh, rbt_sh + r1.x);
        f.template half<0>(v);
        c = VitCoreH::hop(c, hop_sh, rbt_sh + r1.y);
        c = VitCoreH::hop(c, hop_sh, rbt_sh + r1.z);
        c = VitCoreH::hop(c, hop_sh, rbt_sh + r1.w);
        f.template half<1>(v);
        c = VitCoreH::hop(c, hop_sh, rbt_sh + r2.x);
        c = VitCoreH::hop(c, hop_sh, rbt_sh + r2.y);
        c = VitCoreH::hop(c, hop_sh, rbt_sh + r2.z);
        if (chunk - 1 >= ntb) sink.push(VitCoreH::trace_finish(c), chunk - 1 - ntb);
        row = (int)r2.w;
        r0 = s_rows[row];
        c = v.trace_begin(rbt + r0.x, rbt_sh + r0.y, s_hop, (chunk & 3) == 0);
    }
    if (last_chunk >= ntb) {
        const uint4 r1 = s_rows[row + 1], r2 = s_rows[row + 2];
        const uint32_t base[9] = {r0.z, r0.w, r1.x, r1.y, r1.z, r1.w, r2.x, r2.y, r2.z};
#pragma unroll
        for (int i = 0; i < 9; ++i) c = VitCoreH::hop(c, hop_sh, rbt_sh + base[i]);
        sink.push(VitCoreH::trace_finish(c), last_chunk - ntb);
    }
    frames[J.frame].crc_ok = sink.crc_ok();
}

__global__ void __launch_bounds__(VIT_BLOCK) k_viterbi(const JobDesc *__restrict__ jobs, int f0, int n_frames, const uint32_t *__restrict__ vit_in,
                                                        uint32_t *__restrict__ psdu, wifi_b200_frame *frames)
{
    viterbi_body<VitHardIn>(threadIdx.x, jobs, f0, n_frames, vit_in, psdu, frames);
}

// soft-decision mode (DESIGN.md 9)
__global__ void __launch_bounds__(VIT_BLOCK) k_viterbi_soft(const JobDesc *__restrict__ jobs, int f0, int n_frames, const uint32_t *__restrict__ vit_soft_in,
                                                             uint32_t *__restrict__ psdu, wifi_b200_frame *frames)
{
    viterbi_body<VitSoftIn>(threadIdx.x, jobs, f0, n_frames, vit_soft_in, psdu, frames);
}

// ------------------------------------------------------------------ R6a-c, four lanes per trellis (middle-sized calls)
// VitQuad (viterbi.cuh): a quarter of the butterflies per lane and two quad exchanges per four steps.  A call with a few
// thousand frames (a streaming run of a hundred links, a link group of a host batch) has one warp per scheduler or
// less in the one-trellis-per-thread kernel and pays that kernel's full ~1.7 ms latency; here the same frames make four
// times the warps, each with a quarter of the dependent work.  Chunk 0 (6 steps) runs as two erased steps + 6: from
// all-zero metrics an erased step leaves the metrics zero and every path's decision bit set, so masking bits 7, 6 of
// the path bytes afterwards gives exactly the 6-step bytes.
__global__ void __launch_bounds__(VQ_BLOCK) k_viterbi_quad(const JobDesc *__restrict__ jobs, int f0, int n_frames, const uint32_t *__restrict__ vit_in,
                                                          uint32_t *__restrict__ psdu, wifi_b200_frame *frames)
{
    __shared__ uint32_t s_ring[VQ_FRAMES * VQ_RSTRIDE];
    __shared__ uint32_t s_crc[256];
    __shared__ uint16_t s_scr[128];
    __shared__ uint2 s_bm[16];
    const int tid = threadIdx.x;
    for (int i = tid; i < 256; i += VQ_BLOCK) s_crc[i] = c_tab.crc_tab[i];
    for (int i = tid; i < 128; i += VQ_BLOCK) s_scr[i] = c_tab.scr_tab[i];
    if (tid < 16) { uint32_t T, E; VitQuad::branch((uint32_t)tid, T, E); s_bm[tid] = make_uint2(T, E); }
    __syncthreads();
    const int job = f0 + blockIdx.x * VQ_FRAMES + (tid >> 2);
    // the quads of a warp stay together (full-mask shuffles): a quad without a frame, or with a shorter one, runs along
    // on zeros and keeps its results to itself
    JobDesc J;
    J.n_sym = 0;
    if (job < n_frames) J = jobs[job];
    const bool active = job < n_frames && J.n_sym != 0;
    if (!__any_sync(0xffffffffu, active)) return;
    const int enc = active ? J.enc : 0;
    const int punct = c_tab.mcs[enc].punct;
    const int ntb = punct == 0 ? 5 : (punct == 1 ? 9 : 10);
    const int nw = active ? (J.n_sym * c_tab.mcs[enc].n_dbps + 7) >> 3 : 0;
    const uint32_t *in = vit_in + (int64_t)(active ? job : f0) * VIT_MAXW;
    const int L = active ? J.len : 0;
    const int last_chunk = active ? L + 1 + ntb : 0;
    const int trips = __reduce_max_sync(0xffffffffu, last_chunk);
    uint32_t *ring = s_ring + (tid >> 2) * VQ_RSTRIDE;
    VitQuad v;
    v.init(tid & 31);
    uint32_t prev = 0 < nw ? in[0] : 0u;
    v.step4<0>(s_bm, 0xau, 0xau, prev & 0xfu, (prev >> 4) & 0xfu);
    v.step4<4>(s_bm, (prev >> 8) & 0xfu, (prev >> 12) & 0xfu, (prev >> 16) & 0xfu, (prev >> 20) & 0xfu);
#pragma unroll
    for (int i = 0; i < 4; ++i) v.p[i] &= 0x3f3f3f3fu;
    int slot = 1 % ntb;
    v.trace_begin(ring, slot, ntb, true);
    PsduSink sink;
    sink.init(psdu + (int64_t)(active ? job : f0) * (PSDU_STRIDE / 4), L, s_crc, s_scr);
    sink.writer = active && (tid & 3) == 0;
    uint32_t next = 1 < nw ? in[1] : 0u;
    VitQuad::Trace tr;
    tr.bs = 0; tr.sl = slot; tr.left = 0;
#pragma unroll 1
    for (int chunk = 1; chunk <= trips; ++chunk) {
        const uint32_t bits = __funnelshift_r(prev, next, 24);
        prev = next;
        next = (chunk + 1 < nw) ? in[chunk + 1] : 0u;
        VitQuad::trace_hops<3>(tr, ring, ntb);
        v.step4<0>(s_bm, bits & 0xfu, (bits >> 4) & 0xfu, (bits >> 8) & 0xfu, (bits >> 12) & 0xfu);
        VitQuad::trace_hops<3>(tr, ring, ntb);
        v.step4<4>(s_bm, (bits >> 16) & 0xfu, (bits >> 20) & 0xfu, (bits >> 24) & 0xfu, bits >> 28);
        VitQuad::trace_hops<3>(tr, ring, ntb);
        // the traceback of chunk - 1 is complete (ntb - 1 <= 9 hops): its byte, if that chunk has one and is this frame's
        if (chunk - 1 >= ntb && chunk - 1 <= last_chunk) sink.push(VitQuad::ring_byte(ring, tr.sl, tr.bs), chunk - 1 - ntb);
        slot = (slot + 1 == ntb) ? 0 : slot + 1;
        tr = v.trace_begin(ring, slot, ntb, (chunk & 3) == 0);
    }
    VitQuad::trace_hops<9>(tr, ring, ntb);
    if (trips == last_chunk && last_chunk >= ntb) sink.push(VitQuad::ring_byte(ring, tr.sl, tr.bs), last_chunk - ntb);
    if (sink.writer) frames[J.frame].crc_ok = sink.crc_ok();
}

// ------------------------------------------------------------------ R6a-c, low-latency form for small batches
// One trellis per WARP: lane l owns states l and l + 32 -- exactly the two inputs of butterfly l -- and the survivors
// 2l, 2l + 1 travel to their new owners by shuffle (state n lives in lane n % 32).  Per-frame latency is a fraction of
// the one-trellis-per-thread kernel's (whose decode of a 1528-byte frame takes ~1.4 ms however idle the GPU is), at
// several times the instructions per decoded bit: it serves the streaming path, where a run holds a handful of frames.
// Same decoder: agreement metrics (kept as plain ints: only differences matter, so no renormalisation), tie -> the
// predecessor k + 32, one path byte per state and chunk, traceback over ntb snapshots from the first best state.
// The tracebacks are DEFERRED and run 32 at a time, one chunk per lane: a traceback is a chain of ntb dependent
// shared-memory reads, a warp issues in order, so doing it after every chunk costs more than the eight trellis steps;
// with the last 32 + ntb snapshots and the per-lane best-state keys parked in shared memory, 32 chains run in lock step.
#define VW_WARPS 4
#define VW_RING 48            // snapshots kept per frame: >= 32 + VIT_NTB_MAX - 1
__global__ void __launch_bounds__(32 * VW_WARPS) k_viterbi_warp(const JobDesc *__restrict__ jobs, int f0, int n_frames, const uint32_t *__restrict__ vit_in,
                                                               uint32_t *__restrict__ psdu, wifi_b200_frame *frames)
{
    __shared__ uint8_t s_ring[VW_WARPS][VW_RING][64];
    __shared__ uint32_t s_keys[VW_WARPS][32 * 33];      // [lane][chunk % 32], rows padded: conflict-free both ways
    __shared__ uint32_t s_crc[256];
    __shared__ uint16_t s_scr[128];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_crc[i] = c_tab.crc_tab[i];
    for (int i = threadIdx.x; i < 128; i += blockDim.x) s_scr[i] = c_tab.scr_tab[i];
    __syncthreads();
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int job = f0 + blockIdx.x * VW_WARPS + wib;
    if (job >= n_frames) return;
    const JobDesc J = jobs[job];
    if (J.n_sym == 0) return;
    const int punct = c_tab.mcs[J.enc].punct;
    const int ntb = punct == 0 ? 5 : (punct == 1 ? 9 : 10);
    const int nw = (J.n_sym * c_tab.mcs[J.enc].n_dbps + 7) >> 3;
    const uint32_t *in = vit_in + (int64_t)job * VIT_MAXW;
    const int L = J.len;
    const int last_chunk = L + 1 + ntb;
    uint8_t (*ring)[64] = s_ring[wib];
    uint32_t *keys = s_keys[wib];
    // this lane's butterfly: expected symbols on the branch from state `lane` to state 2 * lane
    const uint32_t A = vit_par((2u * lane) & 0x6du), B = vit_par((2u * lane) & 0x4fu);
    const int src_lo = lane >> 1, src_hi = 16 + (lane >> 1);
    const bool odd = lane & 1;
    // A survivor is one word: (metric << 9) | path byte, bit 8 free.  The candidate that comes from state k + 32
    // carries bit 8 (and the step's decision bit in its path byte), so ONE unsigned maximum performs compare, tie rule
    // (equal metrics: the k + 32 candidate is larger) and the selection of metric and path together.
    uint32_t wlo = 0, whi = 0;
    auto step = [&](uint32_t nib, uint32_t bit) {
        const uint32_t s0 = nib & 3u, s1 = (nib >> 2) & 3u;
        const uint32_t e0 = s0 != 2u, e1 = s1 != 2u;
        const uint32_t svm = (e0 & (s0 ^ A)) + (e1 & (s1 ^ B));      // disagreements with (A, B); erasures count for nothing
        const uint32_t sv = e0 + e1 - svm;                            // agreements
        const uint32_t hb = 0x100u | bit;
        const uint32_t v0 = max(wlo + (sv << 9), whi + (svm << 9) + hb);     // new state 2 * lane
        const uint32_t v1 = max(wlo + (svm << 9), whi + (sv << 9) + hb);     // new state 2 * lane + 1
        const uint32_t a0 = __shfl_sync(0xffffffffu, v0, src_lo), a1 = __shfl_sync(0xffffffffu, v1, src_lo);
        const uint32_t b0 = __shfl_sync(0xffffffffu, v0, src_hi), b1 = __shfl_sync(0xffffffffu, v1, src_hi);
        wlo = (odd ? a1 : a0) & ~0x100u;
        whi = (odd ? b1 : b0) & ~0x100u;
    };
    // end of chunk c: park the path bytes (slot c % VW_RING) and this lane's best-state key (largest metric, smallest
    // state of its two), clear the path bytes
    auto park = [&](int c) {
        ring[c % VW_RING][lane] = (uint8_t)wlo;
        ring[c % VW_RING][lane + 32] = (uint8_t)whi;
        keys[lane * 33 + (c & 31)] = max(((wlo >> 9) << 6) | (uint32_t)(63 - lane), ((whi >> 9) << 6) | (uint32_t)(31 - lane));
        wlo &= ~0xffu;
        whi &= ~0xffu;
    };
    PsduSink sink;
    sink.init(psdu + (int64_t)job * (PSDU_STRIDE / 4), L, s_crc, s_scr);
    sink.writer = lane == 0;                          // every lane runs the sink (no divergent region), lane 0 stores
    // tracebacks of chunks base .. base + 31 (those in [1, last_chunk]), lane g takes chunk base + g
    auto trace32 = [&](int base) {
        __syncwarp();
        const int k = base + lane;
        uint32_t key = 0;
#pragma unroll 8
        for (int j = 0; j < 32; ++j) key = max(key, keys[j * 33 + (k & 31)]);
        int bs = 63 - (int)(key & 63u), sl = k % VW_RING;
        for (int i = 0; i < ntb - 1; ++i) { bs = ring[sl][bs] >> 2; sl = (sl == 0 ? VW_RING : sl) - 1; }
        const uint32_t byte = ring[sl][bs];
        for (int g = 0; g < 32; ++g) {
            const uint32_t bg = __shfl_sync(0xffffffffu, byte, g);
            const int kg = base + g;
            if (kg >= ntb && kg <= last_chunk) sink.push(bg, kg - ntb);
        }
        __syncwarp();
    };
    uint32_t w = in[0];
#pragma unroll 1
    for (int k = 0; k < 6; ++k) step((w >> (4 * k)) & 0xfu, 1u << (5 - k));
    park(0);                                          // chunk 0 is never traced back (upstream discards its output)
    uint32_t next = 1 < nw ? in[1] : 0u;
#pragma unroll 1
    for (int chunk = 1; chunk <= last_chunk; ++chunk) {
        const uint32_t bits = __funnelshift_r(w, next, 24);
        w = next;
        next = (chunk + 1 < nw) ? in[chunk + 1] : 0u;
#pragma unroll
        for (int s = 0; s < 8; ++s) step((bits >> (4 * s)) & 0xfu, 0x80u >> s);
        park(chunk);
        if ((chunk & 31) == 31) trace32(chunk - 31);
    }
    if ((last_chunk & 31) != 31) trace32(last_chunk & ~31);
    if (lane == 0) frames[J.frame].crc_ok = sink.crc_ok();
}

// ------------------------------------------------------------------ soft-decision variants (DESIGN.md 9)
// trellis words for gathered jobs in soft mode: word = 2 steps x 2 int8 soft symbols, erasure = 0
__global__ void __launch_bounds__(256) k_pack_soft(const JobDesc *__restrict__ jobs, const int *__restrict__ pack_list, const int *__restrict__ n_pack,
                                                    const int8_t *__restrict__ soft_rows, const uint16_t *__restrict__ depunct_lut,
                                                    uint32_t *__restrict__ vit_soft_in, const wifi_b200_frame *__restrict__ frames)
{
    const int np = *n_pack;
    for (int e = blockIdx.y; e < np; e += gridDim.y) {
        const JobDesc J = jobs[pack_list[e]];
        if (J.n_sym == 0 || !J.need_pack) continue;
        const McsDesc m = c_tab.mcs[J.enc];
        const int per = 2 * m.n_dbps;
        const int n_words = J.n_sym * (m.n_dbps >> 1);
        const uint16_t *lut = depunct_lut + J.enc * 432;
        uint32_t *vw = vit_soft_in + (int64_t)J.frame * SOFT_MAXW;
        for (int w = blockIdx.x * blockDim.x + threadIdx.x; w < n_words; w += gridDim.x * blockDim.x) {
            int q = 4 * w;
            int s = q / per, qi = q - s * per;   // 4 positions never straddle a symbol (per % 4 == 0)
            const int8_t *rp = soft_rows + job_row(J, frames, s) * SOFT_ROW;
            uint32_t word = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                uint16_t en = lut[qi + k];
                uint32_t b = (en == 0xffffu) ? 0u : (uint32_t)(uint8_t)rp[(en >> 3) * m.n_bpsc + (en & 7)];
                word |= b << (8 * k);
            }
            vw[w] = word;
        }
    }
}
