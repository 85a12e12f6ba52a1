// viterbi.cuh -- K=7 (133,171) Viterbi decoders, hard and soft decision.
//
// Restates [UPSTREAM] gr-ieee802-11 lib/viterbi_decoder/{base,viterbi_decoder_generic}.cc
// (instance wifi_phy_hier.grc:533-549 decode_mac, and :550-569 frame_equalizer for SIGNAL):
// 8-bit agreement metrics, tie -> predecessor k+32, per-state 8-bit path registers, a
// traceback over `ntb` stored path snapshots every 8 trellis steps (first after 6).
//
// Three forms of the hard-decision decoder, chosen by the number of frames in a call (wifi_b200.cu):
//   VitCoreH  one trellis per THREAD (k_viterbi, and k_signal for the SIGNAL field), metric and path byte of a state in
//             one halfword, two states per register: the add-compare-select of four new states is two VIADDMNMX.U16x2
//             + two adds;
//   VitQuad   one trellis per FOUR lanes (k_viterbi_quad), byte-packed metrics and path bytes (4 states per register),
//             two quad exchanges per 4 steps;
//   (k_viterbi_warp, rx_kernels.cuh: one trellis per warp.)
// VitCoreSoft is the soft-decision decoder (k_viterbi_soft): 16-bit metrics and path halfwords, two states per register.
//
// VitCoreH, VitQuad and VitCoreSoft run the trellis four steps at a time (step4) with one re-layout instead of four.
// A butterfly leaves its survivors split into "new even states" and "new odd states" words; instead of interleaving
// them back to natural order after every step, the next steps pair the split words directly -- the state stride inside
// a word doubles each step: 1 (natural) -> 2 -> 4 -> 8 -> 16 -- and one transpose restores natural order after the
// fourth step.  Chunks are 8 steps, so the best-state search always sees the natural layout, and so do the snapshots
// of VitQuad and VitCoreSoft (VitCoreH snapshots the split layout in front of the transpose).  The path
// bytes are never shifted: step s of a chunk sets its own decision bit.  Chunk 0 has 6 steps; it runs as two erased
// steps + 6, whose two extra decision bits are masked off before the snapshot (see the kernels).
// Path snapshots of the per-thread forms go to shared memory, word-interleaved across the block's threads (bank =
// thread id, conflict free).
#pragma once
#include "wifi_common.cuh"

#define VIT_BLOCK 64
#define VIT_NTB_MAX 10

__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel)
{
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}

// parity of a 7-bit word; butterfly k's expected code bits are A = par(2k & 0x6d), B = par(2k & 0x4f)
__host__ __device__ constexpr uint32_t vit_par(uint32_t v) { return (v ^ (v >> 1) ^ (v >> 2) ^ (v >> 3) ^ (v >> 4) ^ (v >> 5) ^ (v >> 6)) & 1u; }
// selector picking, for two butterflies k0 (low halfword) and k1 (high), halfword (2A+B) of a (Tlo, Thi) register pair
__host__ __device__ constexpr uint32_t vit_sel2(int k0, int k1)
{
    const int k[2] = {k0, k1};
    uint32_t s = 0;
    for (int b = 0; b < 2; ++b) {
        uint32_t idx = 2 * vit_par((2 * k[b]) & 0x6d) + vit_par((2 * k[b]) & 0x4f);
        s |= ((2 * idx) | ((2 * idx + 1) << 4)) << (8 * b);
    }
    return s;
}

// The traceback of one chunk is a chain of dependent shared-memory reads.  trace_begin() stores the snapshot and finds
// the first best state; the hops follow (branch-free, so the scheduler can interleave the chain with the next chunk's
// add-compare-select work); then the output byte is read.  That read must come before the next snapshot is stored:
// the byte lives in the slot it overwrites.  VitQuad and VitCoreSoft keep the cursor as VitTrace (state, ring slot,
// hops left) and step it with trace_hops(); VitCoreH's cursor is a byte address (see there).
struct VitTrace { int bs, sl, left; };
// byte (slot, state) of this thread's ring: the ring is word-interleaved across the block's threads,
// word (slot * 16 + state / 4) * VIT_BLOCK + tid, so the path byte is a single byte load
__device__ __forceinline__ uint32_t vit_ring_byte(const uint32_t *ring, int sl, int bs, int tid)
{
    const uint8_t *rb = reinterpret_cast<const uint8_t *>(ring) + tid * 4;
    return rb[sl * (16 * VIT_BLOCK * 4) + (bs >> 2) * (VIT_BLOCK * 4) + (bs & 3)];
}

// ---------------------------------------------------------------------------------------------------------------
// VitCoreH: the per-thread decoder with metric and path byte of a state in ONE halfword, two states per register:
//     halfword = metric << 8 | path byte,   the decision of step s of a chunk at bit s of the path byte (ascending).
// The candidate that comes from state k + 32 carries the step's decision bit, and every later bit of both candidates'
// path bytes is still zero, so among equal metrics it is the larger halfword: ONE packed 16-bit maximum performs the
// compare, upstream's tie rule (-> k + 32) and the selection of metric and path together -- VIADDMNMX.U16x2 even adds
// one candidate's branch metric on the way.  An add-compare-select of two butterflies (four new states) is two
// alu-pipe instructions + two adds (which ptxas places on the fma pipe), against 8.5 + 5 for four butterflies in the
// byte-packed form of VitQuad::bfly (compare word, sign-replicating permute, two selects per output word), for the
// same 32 registers of state a whole trellis takes in bytes (16 metric words + 16 path words).
// Path bytes are therefore bit-reversed with respect to upstream's shift register (decision of step s at bit 7 - s):
// the traceback follows them through a table (vit_h_hop_entry), and the output byte is reversed once.
// Metrics stay below 12 + 4 * 16 = 76 between renormalisations (every fourth chunk), so 8 bits hold them; their bytes
// never have bit 7 set, which the chunk-final transpose uses to clear the path bytes (trace_begin).
//
// Ring layout and traceback cursor.  The snapshot is taken from the split layout the chunk's last step leaves (Q), so
// a slot's byte order is a fixed permutation of the states: word w = 8j + i (i < 8, m = 2i) holds states 32j + m,
// 32j + 16 + m, 32j + m + 1, 32j + m + 17 in bytes 0..3 (vit_h_off).  The traceback cursor points at the byte; a hop is
//     cursor = hop_base + table[*cursor]
// where table[b] is the in-slot offset of the predecessor state that path byte b names, and hop_base is the thread's
// column of the slot the hop lands in: one byte load, one table load and one add, where following the state and slot
// took ten alu instructions.  Which slot that is does not depend on the data, so the kernels take the bases
// from per-slot rows (k_viterbi) or count them (k_signal).  A hop that must not move (the traceback is shorter than
// the hop slots the schedule has) runs through the identity slot: its byte for state x names x, so a hop whose base
// is the identity slot's lands on the same state there.
__host__ __device__ constexpr uint32_t vit_h_off(uint32_t x)   // in-slot byte offset of state x (thread column 0)
{
    return (8 * (x >> 5) + ((x & 15) >> 1)) * (VIT_BLOCK * 4) + ((x >> 4) & 1) + 2 * (x & 1);
}
#define VIT_SLOT_BYTES (16 * VIT_BLOCK * 4)
#define VIT_HOP_ENTRIES (256 + 64)
// the hop table: entries 0..255 map a path byte to the offset of the state its decisions of steps 0..5 name (the state
// eight steps back: the six bits, reversed); entries 256 + l map a best-state label l = 63 - state to its offset
__device__ __forceinline__ uint32_t vit_h_hop_entry(int i)
{
    return vit_h_off(i < 256 ? __brev((uint32_t)i) >> 26 : 63u - (uint32_t)(i - 256));
}
// word w of the identity slot: byte k holds the path byte whose predecessor is the state stored there
__device__ __forceinline__ uint32_t vit_h_identity_word(int w)
{
    const uint32_t j = (uint32_t)w >> 3, m = 2u * ((uint32_t)w & 7u);
    const uint32_t x[4] = {32 * j + m, 32 * j + 16 + m, 32 * j + m + 1, 32 * j + m + 17};
    uint32_t v = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) v |= (__brev(x[k]) >> 26) << (8 * k);
    return v;
}

// k_viterbi's traceback rows: one per (traceback depth ntb, snapshot slot s), 24 in all (ntb 5: rows 0..4, ntb 9:
// 5..13, ntb 10: 14..23), 12 words each, no thread column:
//   0     the snapshot's slot s
//   1     where the cursor starts: slot s, or the identity slot (9, unused at ntb 5 and 9) for the hops that stand still
//   2..10 the slot each of the chunk's nine hops lands in.  At ntb < 10 the first 10 - ntb hops stand still: they land
//         in the identity slot, the last of them in slot s.  The others land in s - 1, s - 2, ... (mod ntb), the last
//         in slot s - (ntb - 1) = s + 1, the next snapshot's
//   11    the next row (slot s + 1 mod ntb), as its uint4 index
#define VIT_ROWS 24
#define VIT_ID_SLOT 9
// the rows know exactly the traceback depths of the 802.11a/g code rates (1/2: 5, 2/3: 9, 3/4: 10, k_viterbi) and a
// ring of ten slots, the last of which only ntb = 10 writes; another depth or ring size needs new rows
static_assert(VIT_NTB_MAX == 10 && VIT_ID_SLOT == VIT_NTB_MAX - 1, "traceback rows assume ntb in {5, 9, 10}, ten ring slots");
__host__ __device__ constexpr int vit_h_row0(int ntb) { return ntb == 5 ? 0 : (ntb == 9 ? 5 : 14); }
__device__ __forceinline__ uint32_t vit_h_row_entry(int r, int e)
{
    const int ntb = r < 5 ? 5 : (r < 14 ? 9 : 10);
    const int s = r - vit_h_row0(ntb);
    int slot;
    if (e == 0) slot = s;
    else if (e == 1) slot = ntb == 10 ? s : VIT_ID_SLOT;
    else if (e <= 10) {
        const int still = 10 - ntb, i = e - 2;    // hop i; the first `still` hops leave the cursor where it is
        slot = i < still - 1 ? VIT_ID_SLOT : (s - (i - still + 1) + ntb) % ntb;
    } else return (uint32_t)(3 * (vit_h_row0(ntb) + (s + 1) % ntb));
    return (uint32_t)(slot * VIT_SLOT_BYTES);
}

struct VitCoreH {
    uint32_t X[32];                      // natural order: word j = states 2j (low halfword), 2j + 1 (high)
    uint32_t Q[32];                      // after step4<4>: the split layout, Q[16j + m] = states 32j + m (low), 32j + 16 + m

    __device__ __forceinline__ void init()
    {
#pragma unroll
        for (int i = 0; i < 32; ++i) X[i] = 0;
    }
    // per-step branch words: halfword p = 2A + B of (Tlo | Thi) = disagreements with the expected pair (A, B), << 8;
    // Ew = symbols present (not erased) << 8 in both halfwords
    static __device__ __forceinline__ uint4 branch(uint32_t nib)
    {
        const uint32_t s0 = nib & 3u, s1 = (nib >> 2) & 3u;
        const uint32_t e0 = s0 != 2u, e1 = s1 != 2u;
        uint32_t t[4];
#pragma unroll
        for (uint32_t p = 0; p < 4; ++p) t[p] = ((e0 & (s0 ^ (p >> 1))) + (e1 & (s1 ^ (p & 1u)))) << 8;
        return make_uint4(t[0] | (t[1] << 16), t[2] | (t[3] << 16), ((e0 + e1) << 8) * 0x00010001u, 0u);
    }
    // a + b as a multiply-add by one: ptxas then keeps register-register adds as IMAD.IADD (fma pipe) where it would
    // place part of the plain adds on the alu pipe (VIADD) -- the pipe this kernel is bound by
    static __device__ __forceinline__ uint32_t fadd(uint32_t a, uint32_t b)
    {
        uint32_t d;
        asm("mad.lo.u32 %0, %1, 1, %2;" : "=r"(d) : "r"(a), "r"(b));
        return d;
    }
    // ---- branch words from a table ----
    // Every stage of the four-step schedule (the one of VitCoreSoft::step4: stride inside a word 1 -> 2 -> 4 -> 8 -> 16,
    // then a halfword transpose per word pair) uses exactly four selectors (two complementary pairs), distinguished by the
    // expected pair of their low-halfword butterfly (c = 2A + B of k0); the high halfword's is c ^ 1 in stage A, 3 - c in
    // stages B and C, c in stage D.  table[s][c][nibble] = (svm, sv, svm + BIT_s, sv + BIT_s) for step s of a chunk:
    // one LDS.128 replaces the permute and the three adds per selector and step (the lsu pipe is idle, the alu pipe is
    // not): 2.33 -> 2.14 ms per 37888 frames.  Measured alternatives of the add-compare-select itself (tools/ab.sh):
    // separate add + VIMNMX instead of the fused VIADDMNMX 3.08 ms (the adds load the fma pipe, whose IMADs issue at
    // half rate too); plain `+` instead of fadd() 2.55 ms (ptxas places a third of the adds on the alu pipe).
    // two packed butterflies k0 (low halfword), k1 (high): lo = old states k, hi = old states k + 32; v0 = survivors of
    // the new states 2k, v1 of 2k + 1; e = the table entry of their selector.
    static __device__ __forceinline__ uint4 table_entry(int s, int c, uint32_t nib)
    {
        const int st = s & 3;
        const int c1 = st == 0 ? (c ^ 1) : (st == 3 ? c : 3 - c);
        const uint32_t sel = (uint32_t)((2 * c) | ((2 * c + 1) << 4)) | ((uint32_t)((2 * c1) | ((2 * c1 + 1) << 4)) << 8);
        const uint4 b = branch(nib);
        const uint32_t svm = prmt(b.x, b.y, sel), sv = b.z - svm, bit = 0x00010001u << s;
        return make_uint4(svm, sv, svm + bit, sv + bit);
    }
    static __device__ __forceinline__ void bflyt(const uint4 e, uint32_t lo, uint32_t hi, uint32_t &v0, uint32_t &v1)
    {
        v0 = __viaddmax_u16x2(lo, e.y, fadd(hi, e.z));
        v1 = __viaddmax_u16x2(lo, e.x, fadd(hi, e.w));
    }
    static __host__ __device__ constexpr int selc(uint32_t sel) { return (int)((sel & 0xfu) >> 1); }
    // bt: the table, uint4 [8][4][16].  step4<0> ends in natural order (X); step4<4>, the chunk's last four steps,
    // leaves the split layout Q for trace_begin, which snapshots it and transposes it.
    template <int S0>
    __device__ __forceinline__ void step4(const uint4 *bt, uint32_t n0, uint32_t n1, uint32_t n2, uint32_t n3)
    {
        uint32_t S[32];
        uint4 e[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) e[c] = bt[((S0 + 0) * 4 + c) * 16 + n0];
#pragma unroll
        for (int j = 0; j < 16; ++j) bflyt(e[selc(vit_sel2(2 * j, 2 * j + 1))], X[j], X[j + 16], S[j], S[16 + j]);
#pragma unroll
        for (int c = 0; c < 4; ++c) e[c] = bt[((S0 + 1) * 4 + c) * 16 + n1];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            bflyt(e[selc(vit_sel2(4 * j, 4 * j + 2))], S[j], S[j + 8], Q[4 * j], Q[4 * j + 1]);
            bflyt(e[selc(vit_sel2(4 * j + 1, 4 * j + 3))], S[16 + j], S[24 + j], Q[4 * j + 2], Q[4 * j + 3]);
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) e[c] = bt[((S0 + 2) * 4 + c) * 16 + n2];
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int o = 0; o < 4; ++o)
                bflyt(e[selc(vit_sel2(8 * j + o, 8 * j + 4 + o))], Q[4 * j + o], Q[4 * (j + 4) + o], S[8 * j + 2 * o], S[8 * j + 2 * o + 1]);
#pragma unroll
        for (int c = 0; c < 4; ++c) e[c] = bt[((S0 + 3) * 4 + c) * 16 + n3];
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int o = 0; o < 8; ++o)
                bflyt(e[selc(vit_sel2(16 * j + o, 16 * j + 8 + o))], S[8 * j + o], S[8 * (j + 2) + o], Q[16 * j + 2 * o], Q[16 * j + 2 * o + 1]);
        if (S0 == 0) {
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int e2 = 0; e2 < 16; e2 += 2) {
                    X[(32 * j + e2) >> 1] = prmt(Q[16 * j + e2], Q[16 * j + e2 + 1], 0x5410u);
                    X[(32 * j + 16 + e2) >> 1] = prmt(Q[16 * j + e2], Q[16 * j + e2 + 1], 0x7632u);
                }
        }
    }
    // end of a chunk, after step4<4>: snapshot the path bytes (at byte offset `snap` of the ring, the thread's column of
    // the slot; layout see vit_h_off), transpose to natural order with the path bytes cleared, first best state,
    // optional renormalisation.  Returns the traceback cursor: the best state's byte in the slot whose thread column
    // starts at c0_base (the snapshot's, or the identity slot's).  keep: mask applied to the path bytes first (0xff;
    // 0xfc after the 6-step first chunk, which runs as two erased steps + 6).
    __device__ __forceinline__ uint32_t trace_begin(uint8_t *snap, uint32_t c0_base, const uint32_t *hop_tab, bool renorm,
                                                    uint32_t keep = 0xffu)
    {
        const uint32_t keepw = 0xff00ff00u | keep | (keep << 16);
#pragma unroll
        for (int w = 0; w < 16; ++w)
            *reinterpret_cast<uint32_t *>(snap + w * (VIT_BLOCK * 4)) = prmt(Q[2 * w] & keepw, Q[2 * w + 1] & keepw, 0x6420u);
        // the transpose of step4<0>, with selector nibbles 8 | i (replicate the sign bit of byte i) for the path bytes:
        // byte i is the state's metric byte, below 0x80, so the path bytes come out cleared
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int e2 = 0; e2 < 16; e2 += 2) {
                X[(32 * j + e2) >> 1] = prmt(Q[16 * j + e2], Q[16 * j + e2 + 1], 0x5d19u);
                X[(32 * j + 16 + e2) >> 1] = prmt(Q[16 * j + e2], Q[16 * j + e2 + 1], 0x7f3bu);
            }
        // keys (metric << 8) | (63 - state) -- the largest key is the largest metric at the smallest state -- are the
        // cleared words plus the state labels (an add: fma pipe, where a permute would be alu)
        uint32_t key[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) key[j] = fadd(X[j], (uint32_t)(63 - 2 * j) | ((uint32_t)(62 - 2 * j) << 16));
#pragma unroll
        for (int n = 16; n >= 1; n >>= 1)
#pragma unroll
            for (int i = 0; i < n; ++i) key[i] = __vmaxu2(key[i], key[i + n]);
        const uint32_t kbest = max(key[0] & 0xffffu, key[0] >> 16);
        const uint32_t c = c0_base + hop_tab[256 + (kbest & 0xffu)];
        if (renorm) {
            // Only metric differences matter (upstream subtracts the minimum after every chunk).  Any state is reached
            // from any other in K - 1 = 6 steps of at most 2 agreements each, so min >= max - 12: subtracting max - 12
            // keeps every metric non-negative without a search for the minimum.
            const uint32_t mx = kbest >> 8;
            const uint32_t nminw = 0u - (mx > 12u ? ((mx - 12u) << 8) * 0x00010001u : 0u);
#pragma unroll
            for (int i = 0; i < 32; ++i) X[i] = fadd(X[i], nminw);
        }
        return c;
    }
    // Cursors and bases are shared-window addresses, read with explicit ld.shared: as C++ pointers, the compiler
    // re-associates base + table entry into ring + (thread column + slot + entry) and spends a second add per hop.
    // One traceback hop (see the top of VitCoreH): to the byte of the predecessor state in the slot column at `base`.
    // hop_tab: the shared-window address of the hop table.  The first hop after trace_begin reads a byte of the
    // snapshot trace_begin has just stored with plain C++ stores; a caller that does so in straight-line code (k_signal)
    // puts a compiler memory barrier between them.  (In k_viterbi the snapshot is stored at the end of one loop trip and
    // read in the next.)
    static __device__ __forceinline__ uint32_t hop(uint32_t c, uint32_t hop_tab, uint32_t base)
    {
        uint32_t b, t;
        asm volatile("ld.shared.u8 %0, [%1];" : "=r"(b) : "r"(c));
        asm("ld.shared.u32 %0, [%1];" : "=r"(t) : "r"(hop_tab + 4u * b));
        return base + t;
    }
    // the byte at the cursor; the "memory" clobber keeps it ahead of the snapshot that overwrites its slot
    static __device__ __forceinline__ uint32_t ring_byte(uint32_t c)
    {
        uint32_t b;
        asm volatile("ld.shared.u8 %0, [%1];" : "=r"(b) : "r"(c) : "memory");
        return b;
    }
    // the chunk's output byte in upstream's bit order (MSB = earliest decision)
    static __device__ __forceinline__ uint32_t trace_finish(uint32_t c) { return __brev(ring_byte(c)) >> 24; }
};

// ---------------------------------------------------------------------------------------------------------------
// The same decoder with one trellis spread over FOUR lanes (a "quad"), for calls that hold too few frames to fill the
// machine with one thread per trellis (a 1528-byte frame is 12312 dependent trellis steps; one warp per scheduler runs
// them in ~1.7 ms however idle the GPU is).
// Metrics and path bytes are byte-packed: natural word w holds states 4w .. 4w + 3, 16 metric and 16 path words per
// trellis.  Metrics never exceed 12 + 4 * 16 (spread bound of the code + growth between renormalisations, every fourth
// chunk), so bytes cannot carry into each other.  The four-step schedule of the 16 words (b = byte lane, k = butterfly,
// which pairs old states k and k + 32; S and Q are the split layouts between steps):
//   step A  natural: words j, j + 8, k = 4j + b                  -> S[j] = states 8j + 2b, S[8 + j] = states 8j + 2b + 1
//   step B  stride 2: S[j], S[j + 4], k = 8j + 2b (o = 0, 1); S[8 + j], S[12 + j], k = 8j + 2b + 1 (o = 2, 3)
//                                                                -> Q[4j + o] = states 16j + 4b + o
//   step C  stride 4: Q[4j + o], Q[4(j + 2) + o], k = 16j + 4b + o -> S[8j + o'] = states 32j + 8b + o', o' = 2o, 2o + 1
//   step D  stride 8: S[o], S[8 + o], k = 8b + o                  -> Q[o'] = states 16b + o', o' = 2o, 2o + 1
//   stride 16 -> natural: a 4x4 byte transpose per four words, natural word w byte i = Q[4 (w % 4) + i] byte (w / 4)
// Lane g of a quad owns the natural metric words {g, g+4, g+8, g+12} (and the path words), i.e. local word i <-> natural
// word g + 4i.  That ownership makes
//   step A           local: j = g and j = g + 4
//   step B           local
//   step C           one exchange with lane g ^ 2 (two metric + two path words each way)
//   step D           one exchange with lane g ^ 1
//   the transpose    local, and lands on the ownership step A needs
// so four trellis steps cost a quarter of the butterflies plus 8 shuffles per lane.  Which butterflies a lane computes
// depends on g, so the branch selectors are per-lane registers (set up once) instead of immediates.  The eight quads of
// a warp run in lock step (full-mask shuffles): the kernel gives them one trip count.
// Decoded bytes are those of VitCoreH bit for bit: same metrics, same tie rule, same first-best-state search.  The path
// bytes are in upstream's bit order (earliest decision = MSB), VitCoreH's reversed.
#define VQ_BLOCK 64                      // threads per block: 16 quads
#define VQ_FRAMES (VQ_BLOCK / 4)
#define VQ_RSTRIDE (VIT_NTB_MAX * 16 + 4) // ring words per frame; 164 = 4 (mod 32): the 8 quads x 4 lanes of a warp hit 32 banks

struct VitQuad {
    uint32_t m[4], p[4];
    uint32_t selA0, selA1, selB0, selB1, selC0, selC1, selD0, selD1;
    uint32_t keyc[4];                    // state labels (63 - state) of local word i, for the best-state keys
    int g;
    bool hiC, hiD;

    // per-step branch words: T = disagreements per (A,B) pattern, E = symbols present (not erased)
    static __device__ __forceinline__ void branch(uint32_t nib, uint32_t &T, uint32_t &E)
    {
        const uint32_t s0 = nib & 3u, s1 = (nib >> 2) & 3u;
        const uint32_t t0 = (s0 == 2u) ? 0u : (s0 ? 0x00000101u : 0x01010000u);
        const uint32_t t1 = (s1 == 2u) ? 0u : (s1 ? 0x00010001u : 0x01000100u);
        T = t0 + t1;
        E = ((s0 != 2u) ? 0x01010101u : 0u) + ((s1 != 2u) ? 0x01010101u : 0u);
    }
    static __device__ __forceinline__ uint32_t sel4(int k0, int k1, int k2, int k3)
    {
        const int k[4] = {k0, k1, k2, k3};
        uint32_t s = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const uint32_t A = __popc((2u * k[b]) & 0x6du) & 1u, B = __popc((2u * k[b]) & 0x4fu) & 1u;
            s |= (2 * A + B) << (4 * b);
        }
        return s;
    }

    __device__ __forceinline__ void init(int lane_in_warp)
    {
        g = lane_in_warp & 3;
#pragma unroll
        for (int i = 0; i < 4; ++i) { m[i] = 0; p[i] = 0; keyc[i] = 0x3c3d3e3fu - 0x04040404u * (uint32_t)(g + 4 * i); }
        selA0 = sel4(4 * g, 4 * g + 1, 4 * g + 2, 4 * g + 3);
        selA1 = sel4(4 * (g + 4), 4 * (g + 4) + 1, 4 * (g + 4) + 2, 4 * (g + 4) + 3);
        selB0 = sel4(8 * g, 8 * g + 2, 8 * g + 4, 8 * g + 6);
        selB1 = sel4(8 * g + 1, 8 * g + 3, 8 * g + 5, 8 * g + 7);
        hiC = (g >> 1) != 0;
        { const int j = g & 1, o = hiC ? 2 : 0;
          selC0 = sel4(16 * j + o, 16 * j + 4 + o, 16 * j + 8 + o, 16 * j + 12 + o);
          selC1 = sel4(16 * j + o + 1, 16 * j + 5 + o, 16 * j + 9 + o, 16 * j + 13 + o); }
        hiD = (g & 1) != 0;
        { const int o = (g >> 1) * 4 + (g & 1) * 2;
          selD0 = sel4(o, 8 + o, 16 + o, 24 + o);
          selD1 = sel4(o + 1, 9 + o, 17 + o, 25 + o); }
    }

    // four packed butterflies: lo = old states k_b, hi = old states k_b + 32 (same byte lanes);
    // v0/q0 = survivors of new states 2k_b, v1/q1 of 2k_b + 1
    // BIT: the decision bit of this step inside the path byte.  The bytes are never shifted: step s of a
    // chunk ORs its decision in at bit 7 - s (earliest decision = MSB, as upstream's shift register leaves it).
    template <uint32_t BIT>
    static __device__ __forceinline__ void bfly(uint32_t T, uint32_t E, uint32_t sel, uint32_t lo, uint32_t hi, uint32_t plo, uint32_t phi,
                                                uint32_t &v0, uint32_t &v1, uint32_t &q0, uint32_t &q1)
    {
        const uint32_t svm = prmt(T, 0u, sel), sv = E - svm;   // agreements = available symbols - disagreements
        const uint32_t m0 = lo + sv, m1 = hi + svm, m2 = lo + svm, m3 = hi + sv;
        const uint32_t k0 = prmt(m0 + 0x7f7f7f7fu - m1, 0u, 0xba98u);
        const uint32_t k1 = prmt(m2 + 0x7f7f7f7fu - m3, 0u, 0xba98u);
        v0 = (m0 & k0) | (m1 & ~k0);
        v1 = (m2 & k1) | (m3 & ~k1);
        const uint32_t pb = phi + BIT;
        q0 = (plo & k0) | (pb & ~k0);
        q1 = (plo & k1) | (pb & ~k1);
    }

    // the lane that computes the "upper" two pairs keeps x[2], x[3] as the hi inputs and receives its partner's as lo;
    // the other keeps x[0], x[1] as lo and receives hi
    __device__ __forceinline__ void exchange(const uint32_t (&x)[4], bool high, int lane_xor, uint32_t &lo_a, uint32_t &hi_a, uint32_t &lo_b, uint32_t &hi_b) const
    {
        const uint32_t ra = __shfl_xor_sync(0xffffffffu, high ? x[0] : x[2], lane_xor);
        const uint32_t rb = __shfl_xor_sync(0xffffffffu, high ? x[1] : x[3], lane_xor);
        lo_a = high ? ra : x[0]; hi_a = high ? x[2] : ra;
        lo_b = high ? rb : x[1]; hi_b = high ? x[3] : rb;
    }

    template <int S0>
    __device__ __forceinline__ void step4(const uint2 *bm, uint32_t n0, uint32_t n1, uint32_t n2, uint32_t n3)
    {
        constexpr uint32_t B0 = 0x01010101u << (7 - S0), B1 = B0 >> 1, B2 = B0 >> 2, B3 = B0 >> 3;
        uint32_t T, E;
        uint32_t s[4], sp[4], q[4], qp[4];
        // A: pairs j = g -> S[g], S[8+g]; j = g + 4 -> S[g+4], S[12+g]      (s[i] <-> S[g + 4i])
        { const uint2 te = bm[n0]; T = te.x; E = te.y; }
        bfly<B0>(T, E, selA0, m[0], m[2], p[0], p[2], s[0], s[2], sp[0], sp[2]);
        bfly<B0>(T, E, selA1, m[1], m[3], p[1], p[3], s[1], s[3], sp[1], sp[3]);
        // B: even pair j = g: (S[g], S[g+4]) -> Q[4g], Q[4g+1]; odd pair: (S[8+g], S[12+g]) -> Q[4g+2], Q[4g+3]
        { const uint2 te = bm[n1]; T = te.x; E = te.y; }
        bfly<B1>(T, E, selB0, s[0], s[1], sp[0], sp[1], q[0], q[1], qp[0], qp[1]);
        bfly<B1>(T, E, selB1, s[2], s[3], sp[2], sp[3], q[2], q[3], qp[2], qp[3]);
        // C: lanes j and j + 2 share pairs (j, o): the lower lane takes o = 0, 1, the upper one o = 2, 3
        { const uint2 te = bm[n2]; T = te.x; E = te.y; }
        {
            uint32_t la, ha, lb, hb, pla, pha, plb, phb;
            exchange(q, hiC, 2, la, ha, lb, hb);
            exchange(qp, hiC, 2, pla, pha, plb, phb);
            bfly<B2>(T, E, selC0, la, ha, pla, pha, s[0], s[1], sp[0], sp[1]);
            bfly<B2>(T, E, selC1, lb, hb, plb, phb, s[2], s[3], sp[2], sp[3]);
        }
        // now lane 0: S[0..3], lane 2: S[4..7], lane 1: S[8..11], lane 3: S[12..15].  D: pairs (S[o], S[8+o]): lanes g, g ^ 1
        { const uint2 te = bm[n3]; T = te.x; E = te.y; }
        {
            uint32_t la, ha, lb, hb, pla, pha, plb, phb;
            exchange(s, hiD, 1, la, ha, lb, hb);
            exchange(sp, hiD, 1, pla, pha, plb, phb);
            bfly<B3>(T, E, selD0, la, ha, pla, pha, q[0], q[1], qp[0], qp[1]);
            bfly<B3>(T, E, selD1, lb, hb, plb, phb, q[2], q[3], qp[2], qp[3]);
        }
        // lane g holds Q[4g .. 4g+3]: the byte transpose of group g -> natural words g, g+4, g+8, g+12
        uint32_t t0 = prmt(q[0], q[1], 0x5140u), t1 = prmt(q[0], q[1], 0x7362u);
        uint32_t t2 = prmt(q[2], q[3], 0x5140u), t3 = prmt(q[2], q[3], 0x7362u);
        m[0] = prmt(t0, t2, 0x5410u); m[1] = prmt(t0, t2, 0x7632u); m[2] = prmt(t1, t3, 0x5410u); m[3] = prmt(t1, t3, 0x7632u);
        t0 = prmt(qp[0], qp[1], 0x5140u); t1 = prmt(qp[0], qp[1], 0x7362u);
        t2 = prmt(qp[2], qp[3], 0x5140u); t3 = prmt(qp[2], qp[3], 0x7362u);
        p[0] = prmt(t0, t2, 0x5410u); p[1] = prmt(t0, t2, 0x7632u); p[2] = prmt(t1, t3, 0x5410u); p[3] = prmt(t1, t3, 0x7632u);
    }

    // ring: this frame's VIT_NTB_MAX x 16 words (natural order).  All four lanes follow the traceback (same addresses:
    // broadcast reads), so no lane waits for another's result.
    __device__ __forceinline__ VitTrace trace_begin(uint32_t *ring, int slot, int ntb, bool renorm)
    {
        __syncwarp();                                        // the quad is done reading the slot this snapshot replaces
#pragma unroll
        for (int i = 0; i < 4; ++i) ring[slot * 16 + g + 4 * i] = p[i];
        uint32_t key[8];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            key[2 * i] = prmt(m[i], keyc[i], 0x1504u);
            key[2 * i + 1] = prmt(m[i], keyc[i], 0x3726u);
        }
#pragma unroll
        for (int n = 4; n >= 1; n >>= 1)
#pragma unroll
            for (int i = 0; i < n; ++i) key[i] = __vmaxu2(key[i], key[i + n]);
        uint32_t kbest = max(key[0] & 0xffffu, key[0] >> 16);
        kbest = max(kbest, __shfl_xor_sync(0xffffffffu, kbest, 1));
        kbest = max(kbest, __shfl_xor_sync(0xffffffffu, kbest, 2));  // (also orders the snapshot stores before the quad's reads)
        __syncwarp();
        VitTrace t;
        t.bs = 63 - (int)(kbest & 0xffu);
        t.sl = slot;
        t.left = ntb - 1;
        if (renorm) {                                        // by max - 12, as VitCoreH::trace_begin
            const uint32_t mx = kbest >> 8;
            const uint32_t minw = (mx > 12u ? mx - 12u : 0u) * 0x01010101u;
#pragma unroll
            for (int i = 0; i < 4; ++i) m[i] -= minw;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) p[i] = 0;
        return t;
    }
    static __device__ __forceinline__ uint32_t ring_byte(const uint32_t *ring, int sl, int bs)
    {
        return reinterpret_cast<const uint8_t *>(ring)[sl * 64 + bs];
    }
    template <int N>
    static __device__ __forceinline__ void trace_hops(VitTrace &t, const uint32_t *ring, int ntb)
    {
#pragma unroll
        for (int i = 0; i < N; ++i) {
            const bool go = t.left > 0;
            const int nb = (int)(ring_byte(ring, t.sl, t.bs) >> 2);
            const int ns = (t.sl == 0) ? ntb - 1 : t.sl - 1;
            t.bs = go ? nb : t.bs;
            t.sl = go ? ns : t.sl;
            t.left -= go ? 1 : 0;
        }
    }
};

// descramble + CRC-32 + PSDU word assembly shared by the hard and soft decoders
// ([UPSTREAM] decode_mac.cc descramble(), boost::crc_32_type).  push() takes the traceback byte c
// (MSB = earliest bit) of decoded byte index m.
struct PsduSink {
    uint32_t state, crc, accw;
    bool writer = true;            // warp-per-frame decoder: every lane runs the sink, one stores
    uint32_t *out;
    int L;
    const uint32_t *s_crc;
    const uint16_t *s_scr;
    __device__ __forceinline__ void init(uint32_t *o, int len, const uint32_t *crc_tab, const uint16_t *scr_tab)
    {
        state = 0; crc = 0xffffffffu; accw = 0; out = o; L = len; s_crc = crc_tab; s_scr = scr_tab;
    }
    __device__ __forceinline__ void push(uint32_t c, int m)
    {
        if (m == 0) {
            // state from the first 7 decoded bits, bit 7 is the first descrambled bit (SERVICE)
            state = c >> 1;
            uint32_t fb = ((state >> 6) ^ (state >> 3)) & 1u;
            state = ((state << 1) & 0x7eu) | fb;
            return;
        }
        uint32_t tabv = s_scr[state];
        uint32_t byte = (__brev(c) >> 24) ^ (tabv & 0xffu);
        state = tabv >> 8;
        int pidx = m - 2;
        if (pidx >= 0) {
            crc = s_crc[(crc ^ byte) & 0xffu] ^ (crc >> 8);
            accw |= byte << (8 * (pidx & 3));
            if ((pidx & 3) == 3 || pidx == L - 1) { if (writer) out[pidx >> 2] = accw; accw = 0; }
        }
    }
    __device__ __forceinline__ int crc_ok() const { return ((crc ^ 0xffffffffu) == 558161692u) ? 1 : 0; }
};

// Soft-decision variant (oracle viterbi_soft): 16-bit path metrics, two states per register, branch
// metric = correlation of the expected output bits with int8 soft inputs, offset +254 per step.
struct VitCoreSoft {
    uint32_t M[32], P[32];

    __device__ __forceinline__ void init()
    {
#pragma unroll
        for (int i = 0; i < 32; ++i) { M[i] = 0; P[i] = 0; }
    }
    // BIT: position of this step's decision in the path halfword (never shifted, see VitQuad::bfly)
    template <uint32_t BIT>
    static __device__ __forceinline__ void bfly(uint32_t Tlo, uint32_t Thi, uint32_t sel, uint32_t lo, uint32_t hi, uint32_t plo, uint32_t phi,
                                                uint32_t &v0, uint32_t &v1, uint32_t &p0, uint32_t &p1)
    {
        const uint32_t x = prmt(Tlo, Thi, sel), y = 0x01fc01fcu - x;
        const uint32_t m0 = lo + x, m1 = hi + y, m2 = lo + y, m3 = hi + x;
        const uint32_t k0 = prmt(m0 + 0x7fff7fffu - m1, 0u, 0xbb99u);
        const uint32_t k1 = prmt(m2 + 0x7fff7fffu - m3, 0u, 0xbb99u);
        v0 = (m0 & k0) | (m1 & ~k0);
        v1 = (m2 & k1) | (m3 & ~k1);
        const uint32_t pb = phi + BIT;
        p0 = (plo & k0) | (pb & ~k0);
        p1 = (plo & k1) | (pb & ~k1);
    }
    static __device__ __forceinline__ void branch(int q0, int q1, uint32_t &Tlo, uint32_t &Thi)
    {
        const uint32_t t11 = (uint32_t)(q0 + q1 + 254), t00 = 508u - t11;
        const uint32_t t10 = (uint32_t)(q0 - q1 + 254), t01 = 508u - t10;
        Tlo = t00 | (t01 << 16);
        Thi = t10 | (t11 << 16);
    }
    // Four steps with one re-layout (see the top of this file): with two states per word the stride inside a
    // word goes 1 -> 2 -> 4 -> 8 -> 16 and one halfword transpose per word pair restores natural order.
    // w0 / w1: the two input words (2 steps x 2 int8 each).
    template <int S0>
    __device__ __forceinline__ void step4(uint32_t w0, uint32_t w1)
    {
        constexpr uint32_t B0 = 0x00010001u << (7 - S0), B1 = B0 >> 1, B2 = B0 >> 2, B3 = B0 >> 3;
        uint32_t Tlo, Thi;
        uint32_t S[32], SP[32], Q[32], QP[32];
        // A: natural, pair j: k = 2j + b -> S[j] = {4j, 4j+2}, S[16+j] = {4j+1, 4j+3}
        branch((int)(int8_t)(w0 & 0xffu), (int)(int8_t)((w0 >> 8) & 0xffu), Tlo, Thi);
#pragma unroll
        for (int j = 0; j < 16; ++j) bfly<B0>(Tlo, Thi, vit_sel2(2 * j, 2 * j + 1), M[j], M[j + 16], P[j], P[j + 16], S[j], S[16 + j], SP[j], SP[16 + j]);
        // B: stride 2.  even pair j: k = 4j + 2b ; odd pair j: k = 4j + 2b + 1 -> Q[4j + o] = {8j + o, 8j + 4 + o}
        branch((int)(int8_t)((w0 >> 16) & 0xffu), (int)(int8_t)(w0 >> 24), Tlo, Thi);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            bfly<B1>(Tlo, Thi, vit_sel2(4 * j, 4 * j + 2), S[j], S[j + 8], SP[j], SP[j + 8], Q[4 * j], Q[4 * j + 1], QP[4 * j], QP[4 * j + 1]);
            bfly<B1>(Tlo, Thi, vit_sel2(4 * j + 1, 4 * j + 3), S[16 + j], S[24 + j], SP[16 + j], SP[24 + j], Q[4 * j + 2], Q[4 * j + 3], QP[4 * j + 2], QP[4 * j + 3]);
        }
        // C: stride 4.  pair (j, o): k = 8j + 4b + o -> S[8j + o'] = {16j + o', 16j + 8 + o'}, o' = 2o, 2o+1
        branch((int)(int8_t)(w1 & 0xffu), (int)(int8_t)((w1 >> 8) & 0xffu), Tlo, Thi);
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int o = 0; o < 4; ++o)
                bfly<B2>(Tlo, Thi, vit_sel2(8 * j + o, 8 * j + 4 + o), Q[4 * j + o], Q[4 * (j + 4) + o], QP[4 * j + o], QP[4 * (j + 4) + o],
                     S[8 * j + 2 * o], S[8 * j + 2 * o + 1], SP[8 * j + 2 * o], SP[8 * j + 2 * o + 1]);
        // D: stride 8.  pair (j, o'): k = 16j + 8b + o' -> Q[16j + o''] = {32j + o'', 32j + 16 + o''}, o'' = 2o', 2o'+1
        branch((int)(int8_t)((w1 >> 16) & 0xffu), (int)(int8_t)(w1 >> 24), Tlo, Thi);
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int o = 0; o < 8; ++o)
                bfly<B3>(Tlo, Thi, vit_sel2(16 * j + o, 16 * j + 8 + o), S[8 * j + o], S[8 * (j + 2) + o], SP[8 * j + o], SP[8 * (j + 2) + o],
                     Q[16 * j + 2 * o], Q[16 * j + 2 * o + 1], QP[16 * j + 2 * o], QP[16 * j + 2 * o + 1]);
        // stride 16 -> natural: natural word w = {2w, 2w+1}; Q[16j + e], Q[16j + e + 1] (e even) hold them in the same lane
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int e = 0; e < 16; e += 2) {
                M[(32 * j + e) >> 1] = prmt(Q[16 * j + e], Q[16 * j + e + 1], 0x5410u);
                M[(32 * j + 16 + e) >> 1] = prmt(Q[16 * j + e], Q[16 * j + e + 1], 0x7632u);
                P[(32 * j + e) >> 1] = prmt(QP[16 * j + e], QP[16 * j + e + 1], 0x5410u);
                P[(32 * j + 16 + e) >> 1] = prmt(QP[16 * j + e], QP[16 * j + e + 1], 0x7632u);
            }
    }
    // snapshot + first best state (index-carrying tournament over adjacent words) + optional renormalisation
    __device__ __forceinline__ VitTrace trace_begin(uint32_t *ring, int slot, int ntb, int tid, bool renorm)
    {
#pragma unroll
        for (int w = 0; w < 16; ++w) ring[(slot * 16 + w) * VIT_BLOCK + tid] = prmt(P[2 * w], P[2 * w + 1], 0x6420u);
        uint32_t tv[16], ti[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const uint32_t a = M[2 * i], b = M[2 * i + 1];
            const uint32_t k = prmt((a | 0x80008000u) - b, 0u, 0xbb99u);          // 0xffff where a >= b
            tv[i] = (a & k) | (b & ~k);
            ti[i] = ((uint32_t)(2 * i) * 0x00010001u & k) | ((uint32_t)(2 * i + 1) * 0x00010001u & ~k);
        }
#pragma unroll
        for (int n = 8; n >= 1; n >>= 1)
#pragma unroll
            for (int i = 0; i < n; ++i) {
                const uint32_t a = tv[2 * i], b = tv[2 * i + 1];
                const uint32_t k = prmt((a | 0x80008000u) - b, 0u, 0xbb99u);
                tv[i] = (a & k) | (b & ~k);
                ti[i] = (ti[2 * i] & k) | (ti[2 * i + 1] & ~k);
            }
        const int v0 = (int)(tv[0] & 0xffffu), s0 = (int)(ti[0] & 0xffffu) * 2;
        const int v1 = (int)(tv[0] >> 16), s1 = (int)(ti[0] >> 16) * 2 + 1;
        VitTrace t;
        t.bs = (v1 > v0 || (v1 == v0 && s1 < s0)) ? s1 : s0;
        t.sl = slot;
        t.left = ntb - 1;
        if (renorm) {
            uint32_t mn = M[0];
#pragma unroll
            for (int i = 1; i < 32; ++i) mn = vmin2(mn, M[i]);
            mn = vmin2(mn, mn >> 16);
            const uint32_t minw = (mn & 0xffffu) * 0x00010001u;
#pragma unroll
            for (int i = 0; i < 32; ++i) M[i] -= minw;
        }
#pragma unroll
        for (int i = 0; i < 32; ++i) P[i] = 0;
        return t;
    }
    static __device__ __forceinline__ uint32_t vmin2(uint32_t a, uint32_t b)
    {
        uint32_t k = prmt((a | 0x80008000u) - b, 0u, 0xbb99u);
        return (b & k) | (a & ~k);
    }
    // ring bytes hold the decisions MSB first (upstream's order): the state eight steps back is the byte >> 2
    template <int N>
    static __device__ __forceinline__ void trace_hops(VitTrace &t, const uint32_t *ring, int ntb, int tid)
    {
#pragma unroll
        for (int i = 0; i < N; ++i) {
            const bool go = t.left > 0;
            const int nb = (int)(vit_ring_byte(ring, t.sl, t.bs, tid) >> 2);
            const int ns = (t.sl == 0) ? ntb - 1 : t.sl - 1;
            t.bs = go ? nb : t.bs;
            t.sl = go ? ns : t.sl;
            t.left -= go ? 1 : 0;
        }
    }
};
