// wifi_b200.cu -- host side of libwifi_b200.so: handle, workspace, C ABI (include/wifi_b200.h).
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false -lineinfo -O3 -shared -Xcompiler -fPIC
// No CPU fallback anywhere in this file: every entry point that computes launches CUDA kernels.
#include <sched.h>

#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <deque>
#include <vector>

#include "rx_kernels.cuh"
#include "tx_kernels.cuh"


namespace {

const McsDesc H_MCS[8] = {
    {1, 48, 24, 0x0D, 0}, {1, 48, 36, 0x0F, 2}, {2, 96, 48, 0x05, 0}, {2, 96, 72, 0x07, 2},
    {4, 192, 96, 0x09, 0}, {4, 192, 144, 0x0B, 2}, {6, 288, 192, 0x01, 1}, {6, 288, 216, 0x03, 2},
};
const int H_LTS53[53] = {1, 1, -1, -1, 1, 1, -1, 1, -1, 1, 1, 1, 1, 1, 1, -1, -1, 1, 1, -1, 1, -1, 1, 1, 1, 1, 0,
                         1, -1, -1, 1, 1, -1, 1, -1, 1, -1, -1, -1, -1, -1, 1, 1, -1, -1, 1, -1, 1, -1, 1, 1, 1, 1};

inline int h_n_sym(int enc, int len) { return (16 + 8 * len + 6 + H_MCS[enc].n_dbps - 1) / H_MCS[enc].n_dbps; }

uint32_t h_crc_tab[256];
void h_crc_init()
{
    for (uint32_t i = 0; i < 256; ++i) {
        uint32_t c = i;
        for (int k = 0; k < 8; ++k) c = (c & 1) ? (0xEDB88320u ^ (c >> 1)) : (c >> 1);
        h_crc_tab[i] = c;
    }
}
uint32_t h_crc32(const uint8_t *p, int n)
{
    if (!h_crc_tab[1]) h_crc_init();
    uint32_t c = 0xffffffffu;
    for (int i = 0; i < n; ++i) c = h_crc_tab[(c ^ p[i]) & 0xff] ^ (c >> 8);
    return c ^ 0xffffffffu;
}

// Tables are generated from the formulas of the standard / upstream sources, never copied:
// see the matching generator in oracle/wifi_oracle.cpp; tests/test_oracle_kat.py checks both against the standard's
// Annex G/L tables and against the constants written in the reference's wifi_phy_hier.grc.
void build_tables(DevTables &t, std::vector<uint16_t> &depunct)
{
    memset(&t, 0, sizeof t);
    for (int k = -26; k <= 26; ++k) t.lts[k + 32] = (float)H_LTS53[k + 26];
    int state = 0x7f;
    for (int i = 0; i < 127; ++i) {
        int fb = ((state >> 6) & 1) ^ ((state >> 3) & 1);
        t.polarity[i] = fb ? -1.f : 1.f;
        state = ((state << 1) & 0x7e) | fb;
    }
    for (int n = 0; n < 64; ++n) {
        double re = 0, im = 0;
        for (int k = -26; k <= 26; ++k) {
            double ph = 2.0 * M_PI * k * n / 64.0;
            re += H_LTS53[k + 26] * std::cos(ph);
            im += H_LTS53[k + 26] * std::sin(ph);
        }
        re /= std::sqrt(52.0);
        im /= std::sqrt(52.0);
        t.long_taps[63 - n].re = (float)(std::round(re * 1e4) / 1e4);
        t.long_taps[63 - n].im = (float)(std::round(-im * 1e4) / 1e4);
    }
    for (int k = 0; k < 32; ++k) {
        t.tw[k].re = (float)std::cos(2.0 * M_PI * k / 64.0);
        t.tw[k].im = (float)(-std::sin(2.0 * M_PI * k / 64.0));
    }
    t.tw[0] = {1.f, 0.f};
    t.tw[16] = {0.f, -1.f};
    t.win = (float)(1.0 / std::sqrt(52.0));
    const float sv = (float)std::sqrt(13.0 / 6.0);
    const int sts_k[12] = {-24, -20, -16, -12, -8, -4, 4, 8, 12, 16, 20, 24};
    const int sts_s[12] = {1, -1, 1, -1, -1, 1, -1, -1, 1, 1, 1, 1};
    for (int i = 0; i < 12; ++i) t.sts[sts_k[i] + 32] = {sts_s[i] * sv, sts_s[i] * sv};
    for (int i = 0; i < 64; ++i) {
        int k = i - 32, m = ((k % 4) + 4) % 4;
        float v = t.lts[i];
        t.lts_rot[i] = (m == 0) ? cf{v, 0.f} : (m == 1) ? cf{0.f, -v} : (m == 2) ? cf{-v, 0.f} : cf{0.f, v};
    }
    for (int e = 0; e < 8; ++e) {
        t.mcs[e] = H_MCS[e];
        int n_cbps = H_MCS[e].n_cbps, s = std::max(H_MCS[e].n_bpsc / 2, 1);
        int first[288], second[288];
        for (int j = 0; j < n_cbps; ++j) first[j] = s * (j / s) + ((j + (int)std::floor(16.0 * j / n_cbps)) % s);
        for (int i = 0; i < n_cbps; ++i) second[i] = 16 * i - (n_cbps - 1) * (int)std::floor(16.0 * i / n_cbps);
        for (int k = 0; k < n_cbps; ++k) {
            t.P[e][k] = (uint16_t)second[first[k]];
            t.Pinv[e][second[first[k]]] = (uint16_t)k;
        }
        int nb = H_MCS[e].n_bpsc;
        for (int v = 0; v < (1 << nb); ++v) {
            if (nb == 1) { t.cons[e][v] = {v ? 1.f : -1.f, 0.f}; continue; }
            int h = nb / 2;
            float level = (h == 1) ? sqrtf(0.5f) : (h == 2) ? sqrtf(0.1f) : sqrtf(1.0f / 42.0f);
            auto axis = [&](int bits) -> float {
                int b0 = bits & 1, b1 = (bits >> 1) & 1, b2 = (bits >> 2) & 1, mag;
                if (h == 1) mag = 1;
                else if (h == 2) mag = b1 ? 1 : 3;
                else mag = b1 ? (b2 ? 3 : 1) : (b2 ? 5 : 7);
                return (float)(b0 ? mag : -mag) * level;
            };
            t.cons[e][v] = {axis(v & ((1 << h) - 1)), axis(v >> h)};
        }
    }
    h_crc_init();
    memcpy(t.crc_tab, h_crc_tab, sizeof h_crc_tab);
    for (int s0 = 0; s0 < 128; ++s0) {
        int st = s0, fbits = 0;
        for (int i = 0; i < 8; ++i) {
            int fb = ((st >> 6) & 1) ^ ((st >> 3) & 1);
            fbits |= fb << i;
            st = ((st << 1) & 0x7e) | fb;
        }
        t.scr_tab[s0] = (uint16_t)(fbits | (st << 8));
    }
    int c = 0;
    for (int i = 0; i < 64; ++i) {
        if (i < 6 || i > 58 || i == 32 || i == 11 || i == 25 || i == 39 || i == 53) t.carrier_of[i] = -1;
        else t.carrier_of[i] = (int8_t)c++;
    }
    // depuncture + deinterleave + bit-unpack lookup, per symbol: position q of the rate-1/2
    // stream -> (carrier << 3 | bit) of the equalizer's 48-byte row, or 0xffff for an erasure
    depunct.assign(8 * 432, 0xffff);
    for (int e = 0; e < 8; ++e) {
        const McsDesc &m = H_MCS[e];
        int per = 2 * m.n_dbps, cb = 0;
        for (int q = 0; q < per; ++q) {
            bool keep = true;
            if (m.punct == 1) keep = (q % 4) != 3;
            else if (m.punct == 2) keep = !((q % 6) == 3 || (q % 6) == 4);
            if (!keep) continue;
            int k = t.Pinv[e][cb];    // deint[d] = bits[Pinv[d]]
            depunct[e * 432 + q] = (uint16_t)(((k / m.n_bpsc) << 3) | (k % m.n_bpsc));
            ++cb;
        }
    }
}

enum { ST_H2D = 0, ST_DETECT, ST_SELECT, ST_SYNC_LONG, ST_DEMOD_HEAD, ST_SIGNAL, ST_DEMOD_DATA, ST_PLAN, ST_PACK, ST_VITERBI, ST_D2H, ST_COUNT };
const char *STAGE_NAMES[ST_COUNT] = {"h2d", "detect", "select", "sync_long", "demod_head", "signal", "demod_data", "plan", "pack", "viterbi", "d2h"};

#define MAX_LINKS 16384
// Which Viterbi kernel decodes a call's (or a link group's) frames, by their number -- measured on 1528-byte 64-QAM 3/4
// frames (tools/exp_viterbi_forms.sh, profiles/r02_viterbi_forms_sweep.txt, DESIGN.md 4): one trellis per warp 0.68 ms up
// to 592 frames, 0.87 at 1184, 1.45 at 2368; per four lanes 0.93 ms flat up to 4736, 1.38 at 9472, 2.54 at 18944; per
// thread 1.43-1.50 ms up to 18944, 2.34 at 37888 (measured before that kernel's branch-word table: 2.14 at 37888 now).
#ifndef VW_SWITCH
#define VW_SWITCH 1280          // up to here one trellis per warp
#endif
#ifndef VQ_SWITCH
#define VQ_SWITCH 10240         // up to here one trellis per four lanes; above, one per thread
#endif
#define VQ_SPLIT_MAX 4736        // frames beyond a step of the per-thread kernel's staircase that get their own launch (run_rx)
#define DET_SMEM DET_SMEM_BYTES
// k_viterbi: ring, CRC table, descrambler table, branch-word table (8 x 4 x 16 entries of 16 bytes): 50432 bytes, 4 blocks per SM
#define VIT_SMEM_BYTES ((VIT_NTB_MAX * 16 * VIT_BLOCK + 256) * 4 + 256 + 8192)

} // namespace


#define A_SLOTS 3                // asynchronous pushes that may be pending at once (device staging buffers)
struct wifi_b200 {
    wifi_b200_cfg cfg;
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr, d2h_stream = nullptr;   // host input / results of one link group while another is decoded
    cudaStream_t aux_stream = nullptr;     // the Viterbi launch of the frames beyond whole waves, beside the main one
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    int sm_count = 148;
    std::vector<cudaEvent_t> ev_h2d, ev_done;
    std::mutex mu;
    std::string err;
    // device workspace
    cf *d_iq = nullptr;            // staging for host input (max_samples + history)
    int16_t *d_sc16 = nullptr;     // staging for wire-format (int16 I/Q) host input
    uint32_t *d_flags = nullptr;      // 1 bit per sample: c[n] > threshold
    uint32_t *d_summary = nullptr;    // 1 bit per FE_CHUNK chunk: any flag set
    int *d_trig_tmp = nullptr;        // k_select scratch: trigger list per link
    int *d_spec_trig = nullptr;       // speculative triggers per 8192-sample segment
    int4 *d_spec_cnt = nullptr;       // per segment (count, first, last, -)
    int *d_spec_trig2 = nullptr;      // second speculative pass (k_select_fix): chains walked again behind the previous segment's last trigger
    int4 *d_spec_cnt2 = nullptr;      // per segment (count, first, last, which trigger array)
    int *d_pack_list = nullptr;       // frames whose trellis words k_pack must build
    int *d_link_dirty = nullptr;      // links that need the sequential decode_mac replay
    int64_t tile_cap = 0;
    LinkDesc *d_links = nullptr;
    wifi_b200_frame *d_frames = nullptr;
    EqState *d_states = nullptr;
    uint8_t *d_rows = nullptr;
    cf *d_carrier = nullptr;
    JobDesc *d_jobs = nullptr;
    uint32_t *d_vit_in = nullptr;
    int8_t *d_soft = nullptr;          // soft mode: int8 per coded bit, SOFT_ROW per row
    uint32_t *d_vit_soft_in = nullptr; // soft mode trellis words
    uint32_t *d_psdu = nullptr;
    uint16_t *d_depunct = nullptr;
    int *d_counters = nullptr;     // [0] frames [1] pack-list length [2] err ; ints 8..9: row counter (u64)
    int *h_counters = nullptr;     // pinned mirror
    int64_t row_cap = 0;
    // tx workspace
    uint8_t *d_txblob = nullptr;
    TxFrameDesc *d_txdesc = nullptr;
    uint8_t *d_txsym = nullptr;
    cf *d_txiq = nullptr;
    size_t txblob_cap = 0, txiq_cap = 0, txsym_cap = 0;   // bytes, as every capacity grow() keeps
    int64_t tx_sym_bytes = 0;
    int tx_seed = 1;               // [UPSTREAM] mapper.cc d_scrambler: 1, ++ per frame, wraps after 127
    wifi_b200_chan_seg *d_segs = nullptr;
    wifi_b200_fading *d_fades = nullptr;
    size_t segs_cap = 0, fades_cap = 0;
    // last rx call
    const cf *cur_iq = nullptr;
    std::vector<LinkDesc> h_links;
    int64_t n_frames = 0, n_jobs = 0, n_rows = 0, n_samples = 0, n_triggers = 0;
    bool host_mirror = false;      // frame table already copied to host
    bool psdu_mirror = false;      // PSDU store already copied to host
    wifi_b200_frame *h_frames = nullptr;   // pinned
    uint8_t *h_psdu = nullptr;             // pinned
    float *h_iq = nullptr;                 // pinned staging for host input
    cudaEvent_t ev[ST_COUNT + 1];
    bool ev_used[ST_COUNT + 1];
    float stage_ms[ST_COUNT];
    wifi_b200_stats stats;
    // streaming: one state per link (wifi_b200_rx_push = one link, wifi_b200_rx_push_links = many)
    struct StreamLink {
        int64_t fill = 0;          // samples in the link's region of the device arena: history + pending
        int64_t abs0 = 0;          // absolute index of the first non-history sample of the region
        int hist = 0;
        int64_t prev_trigger = -1; // absolute
        float fo_carry = 0.f;
    };
    std::vector<StreamLink> s_links;
    cf *d_stream = nullptr;        // streaming arena: one region of s_cap samples per link; samples go from the caller's buffer
    int64_t s_cap = 0;             //   straight to the device and stay there until their burst is decoded
    struct MoveSeg { int64_t src, dst, n; };
    MoveSeg *d_moves = nullptr;    // tail compaction descriptors
    int64_t group_samples = 0;     // WIFI_P_HOST_GROUP_SAMPLES: samples per link group of the host-input batch calls (0: 128 MB of host bytes)
    int64_t s_batch = 0;           // WIFI_P_STREAM_BATCH: a push only buffers until this many new samples per link wait (0: every push)
    int64_t s_unprocessed = 0;     // samples appended to the fullest link since the last pipeline run
    // results waiting for wifi_b200_rx_pop: the frames of the newest runs stay in the page-locked PSDU mirror they arrived
    // in (one block per run, two mirrors used in turn); a block whose mirror the next run needs is spilled into the
    // packed queue (s_meta / s_bytes), which is always older than every block
    struct StreamBlock { uint8_t *buf = nullptr; std::vector<wifi_b200_frame> meta; size_t next = 0; };
    std::vector<wifi_b200_frame> s_meta;
    std::vector<uint8_t> s_bytes;
    std::deque<StreamBlock> s_blocks;
    uint8_t *h_psdu_alt = nullptr;         // pinned, allocated by the first streaming run
    int view_kind = 0;                     // wifi_b200_rx_pop_view handed out: 1 = the packed queue, 2 = the front block
    size_t view_n = 0, view_bytes = 0;
    // asynchronous pushes (wifi_b200_rx_push_links_async): up to A_SLOTS in flight, each with its device staging buffer
    struct AsyncPush { int slot = 0; int flush = 0; float sc16_scale = 0.f; std::vector<uint64_t> off; };   // sc16_scale != 0: the slot holds int16 I/Q
    std::vector<AsyncPush> a_pending;
    cf *d_stage[A_SLOTS] = {};
    size_t a_cap[A_SLOTS] = {};
    cudaEvent_t a_ev[A_SLOTS] = {};
    int a_next = 0;
    int viterbi_form = 0;          // WIFI_P_VITERBI_FORM
};

namespace {

#define CK(call)                                                                                        \
    do {                                                                                                \
        cudaError_t e_ = (call);                                                                        \
        if (e_ != cudaSuccess) {                                                                        \
            h->err = std::string(#call) + ": " + cudaGetErrorString(e_);                                \
            return WIFI_E_CUDA;                                                                         \
        }                                                                                               \
    } while (0)

std::mutex g_tab_mu;
bool g_tab_done[64];

int upload_tables(wifi_b200 *h)
{
    std::lock_guard<std::mutex> g(g_tab_mu);
    static DevTables t;
    static std::vector<uint16_t> dep;
    if (dep.empty()) build_tables(t, dep);
    if (!g_tab_done[h->device & 63]) {
        CK(cudaMemcpyToSymbol(c_tab, &t, sizeof t));
        g_tab_done[h->device & 63] = true;
    }
    CK(cudaMalloc(&h->d_depunct, dep.size() * sizeof(uint16_t)));
    CK(cudaMemcpy(h->d_depunct, dep.data(), dep.size() * sizeof(uint16_t), cudaMemcpyHostToDevice));
    return WIFI_OK;
}

void free_all(wifi_b200 *h)
{
    cudaSetDevice(h->device);
    // nothing of this handle may still be reading a caller's buffer or writing a pinned mirror when the memory goes away
    if (h->copy_stream) cudaStreamSynchronize(h->copy_stream);
    if (h->d2h_stream) cudaStreamSynchronize(h->d2h_stream);
    if (h->aux_stream) cudaStreamSynchronize(h->aux_stream);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    for (int k = 0; k < A_SLOTS; ++k) if (h->a_ev[k]) cudaEventDestroy(h->a_ev[k]);
    void *ptrs[] = {h->d_stage[0], h->d_stage[1], h->d_stage[2], h->d_stream, h->d_moves, h->d_sc16, h->d_iq, h->d_flags, h->d_links, h->d_frames, h->d_states, h->d_rows, h->d_carrier, h->d_jobs, h->d_vit_in,
                    h->d_psdu, h->d_depunct, h->d_counters, h->d_summary, h->d_trig_tmp, h->d_pack_list, h->d_link_dirty, h->d_spec_trig, h->d_spec_cnt, h->d_spec_trig2, h->d_spec_cnt2, h->d_soft, h->d_vit_soft_in, h->d_txblob, h->d_txdesc, h->d_txsym, h->d_txiq, h->d_segs, h->d_fades};
    for (void *p : ptrs) if (p) cudaFree(p);
    if (h->h_counters) cudaFreeHost(h->h_counters);
    if (h->h_frames) cudaFreeHost(h->h_frames);
    if (h->h_psdu) cudaFreeHost(h->h_psdu);
    if (h->h_psdu_alt) cudaFreeHost(h->h_psdu_alt);
    if (h->h_iq) cudaFreeHost(h->h_iq);
    for (int i = 0; i <= ST_COUNT; ++i) if (h->ev[i]) cudaEventDestroy(h->ev[i]);
    for (cudaEvent_t e : h->ev_h2d) cudaEventDestroy(e);
    for (cudaEvent_t e : h->ev_done) cudaEventDestroy(e);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->d2h_stream) cudaStreamDestroy(h->d2h_stream);
    if (h->aux_stream) cudaStreamDestroy(h->aux_stream);
    if (h->stream) cudaStreamDestroy(h->stream);
}

// Grows the handle buffer *p to hold need bytes, with slack bytes to spare; what it held is not kept.  A failed
// allocation leaves *p null and *cap 0, so the next call allocates again.
int grow(wifi_b200 *h, void **p, size_t *cap, size_t need, size_t slack)
{
    if (need <= *cap) return WIFI_OK;
    if (*p) cudaFree(*p);
    *p = nullptr;
    *cap = 0;
    CK(cudaMalloc(p, need + slack));
    *cap = need + slack;
    return WIFI_OK;
}

int ensure_soft(wifi_b200 *h)
{
    if (!h->d_soft) CK(cudaMalloc(&h->d_soft, (size_t)h->row_cap * SOFT_ROW));
    if (!h->d_vit_soft_in) CK(cudaMalloc(&h->d_vit_soft_in, (size_t)h->cfg.max_frames * SOFT_MAXW * 4));
    return WIFI_OK;
}

int ensure_iq_staging(wifi_b200 *h)
{
    if (!h->d_iq) CK(cudaMalloc(&h->d_iq, (size_t)(h->cfg.max_samples + 512) * sizeof(cf)));
    return WIFI_OK;
}

int ensure_sc16_staging(wifi_b200 *h)
{
    if (!h->d_sc16) CK(cudaMalloc(&h->d_sc16, (size_t)(h->cfg.max_samples + 512) * 2 * sizeof(int16_t)));
    return WIFI_OK;
}

// wire-format ingest: 4 complex samples per thread (16 B in, 32 B out), x = (float)i16 * scale
__global__ void __launch_bounds__(256) k_sc16_to_fc32(const int16_t *__restrict__ in, cf *__restrict__ out, int64_t n, float scale)
{
    const int64_t stride = (int64_t)gridDim.x * blockDim.x * 4;
    for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < n; i += stride) {
        if (i + 4 <= n && (((uintptr_t)(in + 2 * i)) & 15) == 0 && (((uintptr_t)(out + i)) & 15) == 0) {
            const int4 v = *reinterpret_cast<const int4 *>(in + 2 * i);
            const int w[4] = {v.x, v.y, v.z, v.w};
            float4 o[2];
            float *of = reinterpret_cast<float *>(o);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                of[2 * k] = (float)(int16_t)(w[k] & 0xffff) * scale;
                of[2 * k + 1] = (float)(int16_t)(w[k] >> 16) * scale;
            }
            reinterpret_cast<float4 *>(out + i)[0] = o[0];
            reinterpret_cast<float4 *>(out + i)[1] = o[1];
        } else {
            for (int64_t j = i; j < n && j < i + 4; ++j) out[j] = cf{(float)in[2 * j] * scale, (float)in[2 * j + 1] * scale};
        }
    }
}

// streaming: dst[m.dst + i] = src[m.src + i] for segment m = blockIdx.y; run twice (arena -> scratch -> arena) to slide
// every link's retained tail to the front of its region (source and destination ranges of one link may overlap)
__global__ void __launch_bounds__(256) k_move_segments(const cf *__restrict__ src, cf *__restrict__ dst, const wifi_b200::MoveSeg *__restrict__ segs)
{
    const wifi_b200::MoveSeg m = segs[blockIdx.y];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m.n; i += (int64_t)gridDim.x * blockDim.x) dst[m.dst + i] = src[m.src + i];
}

// the same append for a staging buffer in the wire format: x = (float)i16 * scale as k_sc16_to_fc32, converted on the way
// into the arena (one 4-byte load and one 8-byte store per sample, no intermediate fc32 copy)
__global__ void __launch_bounds__(256) k_append_sc16(const int16_t *__restrict__ src, cf *__restrict__ dst, const wifi_b200::MoveSeg *__restrict__ segs, float scale)
{
    const wifi_b200::MoveSeg m = segs[blockIdx.y];
    const int *in = reinterpret_cast<const int *>(src) + m.src;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < m.n; i += (int64_t)gridDim.x * blockDim.x) {
        const int w = in[i];
        dst[m.dst + i] = cf{(float)(int16_t)(w & 0xffff) * scale, (float)(int16_t)(w >> 16) * scale};
    }
}

// element-wise evaluation of the numerical contract on the device (tests/test_detmath.py)
__global__ void __launch_bounds__(256) k_detmath(int fn, const float *__restrict__ a, const float *__restrict__ b, const float *__restrict__ c,
                                                  const float *__restrict__ d, float *o0, float *o1, int64_t n)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float r0 = o0[i], r1 = o1[i];
        wdm_selftest(fn, a[i], b[i], c[i], d[i], &r0, &r1);
        o0[i] = r0;
        o1[i] = r1;
    }
}

// Issue-rate probe of the integer ALU pipe (the pipe k_viterbi is bound by): every thread runs eight independent
// chains of LOP3 (64 alu-pipe instructions per loop iteration, pinned with asm volatile), enough warps per
// scheduler to hide the pipe latency.  warp-instructions / time = the ceiling bench.py's Viterbi roofline is quoted against.
#define ALU_PROBE_OPS 64
__global__ void __launch_bounds__(256) k_alu_peak(int iters, uint32_t seed, uint32_t *sink)
{
    uint32_t r[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) r[k] = seed * (threadIdx.x + 1u) + (uint32_t)k;
    const uint32_t m = seed | 1u;
#pragma unroll 1
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int u = 0; u < ALU_PROBE_OPS / 16; ++u) {
            // (ptxas turns plain integer adds into IMAD.IADD on the fma pipe when the alu pipe is the busier one, so the
            // probe sticks to three-input logic ops, which only the alu pipe executes)
#pragma unroll
            for (int k = 0; k < 8; ++k) asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(r[k]) : "r"(r[(k + 3) & 7]), "r"(m));
#pragma unroll
            for (int k = 0; k < 8; ++k) asm volatile("lop3.b32 %0, %0, %1, %2, 0xe8;" : "+r"(r[k]) : "r"(r[(k + 5) & 7]), "r"(m));
        }
    }
    uint32_t x = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) x ^= r[k];
    if (x == 0x12345u) sink[0] = x;      // keeps the chains alive; practically never taken
}

void mark(wifi_b200 *h, int i)
{
    cudaEventRecord(h->ev[i], h->stream);
    h->ev_used[i] = true;
}

// One host -> device copy of a link group, queued on the copy stream before run_rx is called
struct H2dPlan {
    const void *src = nullptr;     // host buffer (fc32 or sc16) of the first sample of link 0 of the call
    size_t bytes_per_sample = 0;   // 8 (fc32) or 4 (sc16)
    float sc16_scale = 0.f;        // != 0: the group is converted from d_sc16 to d_iq on the compute stream once it has arrived
};

// The receive pipeline over the links in h->h_links.  `iq` is device memory.  The links are processed in GROUPS of
// whole links (one group for device-resident input): with host input (`plan`) the copy of group g + 1 runs on the copy
// stream while group g is decoded, and the results of group g travel back on a third stream while group g + 1 is
// decoded -- one cudaMemcpyAsync per group and direction.  Frame records, rows and PSDU slots of the groups follow each
// other in link order, so the result is the same table as from one pass over all links.
// ---- queued streaming results (see wifi_b200::StreamBlock) ----
void release_view(wifi_b200 *h)
{
    if (h->view_kind == 1) {
        h->s_meta.erase(h->s_meta.begin(), h->s_meta.begin() + h->view_n);
        h->s_bytes.erase(h->s_bytes.begin(), h->s_bytes.begin() + h->view_bytes);
    } else if (h->view_kind == 2 && !h->s_blocks.empty()) {
        h->s_blocks.pop_front();
    }
    h->view_kind = 0;
}

void spill_front_block(wifi_b200 *h)
{
    wifi_b200::StreamBlock &b = h->s_blocks.front();
    for (size_t i = b.next; i < b.meta.size(); ++i) {
        const wifi_b200_frame &f = b.meta[i];
        const uint8_t *p = b.buf + f.psdu_off;
        h->s_bytes.insert(h->s_bytes.end(), p, p + (f.length - 4));
        h->s_meta.push_back(f);
    }
    h->s_blocks.pop_front();
}

// `buf` is about to be overwritten: the blocks that live in it, and the older ones in front of them, move to the packed queue
void spill_blocks_on(wifi_b200 *h, const uint8_t *buf)
{
    release_view(h);
    size_t last = 0;
    for (size_t i = 0; i < h->s_blocks.size(); ++i)
        if (h->s_blocks[i].buf == buf) last = i + 1;
    for (size_t i = 0; i < last; ++i) spill_front_block(h);
}

int run_rx(wifi_b200 *h, const cf *iq, bool mirror, const H2dPlan *plan = nullptr)
{
    spill_blocks_on(h, h->h_psdu);
    const int n_links = (int)h->h_links.size();
    int64_t total_tiles = 0, total = 0;
    for (auto &L : h->h_links) {
        L.chunk_base = total_tiles * DET_THREADS;
        total_tiles += (L.len + DET_TILE - 1) / DET_TILE;
        total += L.len;
    }
    if (total_tiles > h->tile_cap) { h->err = "tile capacity exceeded (too many short links)"; return WIFI_E_OVERFLOW; }
    h->cur_iq = iq;
    h->n_frames = h->n_jobs = h->n_rows = 0;
    h->n_samples = total;
    h->host_mirror = h->psdu_mirror = false;
    for (int i = 0; i <= ST_COUNT; ++i) h->ev_used[i] = false;
    memset(h->stage_ms, 0, sizeof h->stage_ms);
    const double thr = h->cfg.sensitivity;
    float thr_f = (float)thr;   // (double)c > thr  <=>  c > largest float <= thr
    if ((double)thr_f > thr) thr_f = nextafterf(thr_f, -INFINITY);
    cudaStream_t s = h->stream;
    // link groups when the input comes from the host (copy / decode overlap), else one
    std::vector<int> gstart{0};
    if (plan && n_links > 1) {
        // about 128 MB of host bytes per group: its copy then takes longer than its decode (a group costs 1.5 - 3 ms of
        // kernels whatever its size: the Viterbi launch is latency bound), so the decode hides behind the next copy
        const int64_t target = h->group_samples > 0 ? h->group_samples : std::max<int64_t>(((int64_t)128 << 20) / (int64_t)plan->bytes_per_sample, (int64_t)1 << 22);
        int64_t acc = 0;
        for (int l = 0; l < n_links; ++l) {
            acc += h->h_links[l].len;
            if (acc >= target && l + 1 < n_links) { gstart.push_back(l + 1); acc = 0; }
        }
    }
    gstart.push_back(n_links);
    const int n_groups = (int)gstart.size() - 1;
    while ((int)h->ev_h2d.size() < n_groups) {
        cudaEvent_t a = nullptr, b = nullptr;
        CK(cudaEventCreateWithFlags(&a, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&b, cudaEventDisableTiming));
        h->ev_h2d.push_back(a);
        h->ev_done.push_back(b);
    }
    if (plan) {
        mark(h, ST_H2D);
        for (int g = 0; g < n_groups; ++g) {
            const int64_t o0 = h->h_links[gstart[g]].x_off, o1 = h->h_links[gstart[g + 1] - 1].x_off + h->h_links[gstart[g + 1] - 1].len;
            void *dst = plan->bytes_per_sample == 8 ? (void *)(h->d_iq + o0) : (void *)(h->d_sc16 + 2 * o0);
            CK(cudaMemcpyAsync(dst, (const char *)plan->src + (size_t)o0 * plan->bytes_per_sample, (size_t)(o1 - o0) * plan->bytes_per_sample,
                               cudaMemcpyHostToDevice, h->copy_stream));
            CK(cudaEventRecord(h->ev_h2d[g], h->copy_stream));
        }
    }
    CK(cudaMemcpyAsync(h->d_links, h->h_links.data(), n_links * sizeof(LinkDesc), cudaMemcpyHostToDevice, s));
    CK(cudaMemsetAsync(h->d_counters, 0, 64, s));
    const int soft = h->cfg.soft_decision ? 1 : 0;
    if (soft) { int rc_ = ensure_soft(h); if (rc_) return rc_; }
    const DemodParams prm{h->cfg.bandwidth, h->cfg.frequency, h->cfg.chan_est, h->cfg.want_carrier, soft};
    typedef void (*demod_fn)(const cf *, const LinkDesc *, wifi_b200_frame *, int, int, EqState *, uint8_t *, cf *, DemodParams,
                             const uint16_t *, uint32_t *, int8_t *, uint32_t *);
#define DEMOD_ROW(S, P) {k_demod<S, WIFI_EQ_LS, P>, k_demod<S, WIFI_EQ_LMS, P>, k_demod<S, WIFI_EQ_COMB, P>, k_demod<S, WIFI_EQ_STA, P>}
    static const demod_fn demod_tab[2][2][4] = {{DEMOD_ROW(false, 0), DEMOD_ROW(false, 1)}, {DEMOD_ROW(true, 0), DEMOD_ROW(true, 1)}};
#undef DEMOD_ROW
    const demod_fn demod_head = demod_tab[soft][0][prm.algo & 3], demod_data = demod_tab[soft][1][prm.algo & 3];
    const size_t vit_smem_soft = (size_t)(VIT_NTB_MAX * 16 * VIT_BLOCK + 256) * 4 + 256 + 256;   // ring, CRC table, descrambler table, branch words
    const size_t vit_smem = (size_t)VIT_SMEM_BYTES;
    const bool timed = n_groups == 1;              // per-stage events only make sense for a single pass
    int64_t frame_base = 0, row_base = 0, tile_base = 0;
    for (int g = 0; g < n_groups; ++g) {
        const int lb = gstart[g], ng = gstart[g + 1] - gstart[g];
        int64_t tiles_g = 0, samples_g = 0;
        for (int l = lb; l < lb + ng; ++l) { tiles_g += (h->h_links[l].len + DET_TILE - 1) / DET_TILE; samples_g += h->h_links[l].len; }
        LinkDesc *gl = h->d_links + lb;
        if (plan) {
            CK(cudaStreamWaitEvent(s, h->ev_h2d[g], 0));
            if (plan->sc16_scale != 0.f && samples_g > 0) {
                const int64_t o0 = h->h_links[lb].x_off;
                int64_t blocks = std::min<int64_t>((samples_g / 4 + 255) / 256 + 1, 148 * 16);
                k_sc16_to_fc32<<<(unsigned)blocks, 256, 0, s>>>(h->d_sc16 + 2 * o0, h->d_iq + o0, samples_g, plan->sc16_scale);
            }
        }
        if (timed) mark(h, ST_DETECT);
        if (tiles_g > 0)
            k_detect<<<(unsigned)(DET_SPLIT * tiles_g), DET_BLOCK, DET_SMEM, s>>>(iq, gl, ng, tile_base, tile_base + tiles_g, thr_f, h->d_flags, h->d_summary);
        if (timed) mark(h, ST_SELECT);
        if (tiles_g > 0)
            k_select_spec<<<(unsigned)((tiles_g * 32 + 127) / 128), 128, 0, s>>>(h->d_flags, h->d_summary, gl, ng, tile_base, tile_base + tiles_g,
                                                                                h->cfg.min_plateau, h->d_spec_trig, h->d_spec_cnt);
        if (tiles_g > 0)
            k_select_fix<<<(unsigned)((tiles_g * 32 + 127) / 128), 128, 0, s>>>(h->d_flags, h->d_summary, gl, ng, tile_base, tile_base + tiles_g,
                                                                               h->cfg.min_plateau, h->d_spec_trig, h->d_spec_cnt, h->d_spec_trig2, h->d_spec_cnt2);
        k_select<<<(ng * 32 + 127) / 128, 128, 0, s>>>(h->d_flags, h->d_summary, gl, ng, h->cfg.min_plateau, h->d_trig_tmp, h->d_spec_trig, h->d_spec_cnt2,
                                                       h->d_spec_trig2);
        k_reserve<<<1, 1024, 0, s>>>(gl, ng, h->d_counters, (unsigned long long *)(h->d_counters + 8), h->cfg.max_frames, h->d_counters + 2,
                                     (long long)frame_base, (long long)row_base);
        k_frames_init<<<dim3(8, ng), 128, 0, s>>>(gl, h->d_trig_tmp, h->d_frames, lb);
        if (timed) mark(h, ST_SYNC_LONG);
        CK(cudaMemcpyAsync(h->h_counters, h->d_counters, 64, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        if (h->h_counters[2] != 0 || h->h_counters[0] > h->cfg.max_frames) {
            h->err = "more sync_short triggers than max_frames";
            return WIFI_E_OVERFLOW;
        }
        const int64_t f_end = h->h_counters[0], nf = f_end - frame_base;
        const int64_t rows_needed = *(int64_t *)(h->h_counters + 8);
        if (rows_needed > h->row_cap) {
            h->err = "row capacity exceeded";
            return WIFI_E_OVERFLOW;
        }
        const int f0 = (int)frame_base, fe = (int)f_end;
        if (nf > 0) {
            k_sync_long<<<(unsigned)nf, SL_THREADS, 0, s>>>(iq, h->d_links, h->d_frames, f0, fe);
            if (timed) mark(h, ST_DEMOD_HEAD);
            demod_head<<<(unsigned)((nf + 3) / 4), 128, 0, s>>>(iq, h->d_links, h->d_frames, f0, fe, h->d_states, h->d_rows, h->d_carrier, prm,
                                                            h->d_depunct, h->d_vit_in, h->d_soft, h->d_vit_soft_in);
            if (timed) mark(h, ST_SIGNAL);
            k_signal<<<(unsigned)((nf + VIT_BLOCK - 1) / VIT_BLOCK), VIT_BLOCK, 0, s>>>(h->d_frames, f0, fe, h->d_states);
            if (timed) mark(h, ST_DEMOD_DATA);
            demod_data<<<(unsigned)((nf + 3) / 4), 128, 0, s>>>(iq, h->d_links, h->d_frames, f0, fe, h->d_states, h->d_rows, h->d_carrier, prm,
                                                            h->d_depunct, h->d_vit_in, h->d_soft, h->d_vit_soft_in);
            if (timed) mark(h, ST_PLAN);
            CK(cudaMemsetAsync(h->d_link_dirty + lb, 0, (size_t)ng * sizeof(int), s));
            CK(cudaMemsetAsync(h->d_link_dirty + MAX_LINKS + lb, 0xff, (size_t)ng * sizeof(int), s));
            CK(cudaMemsetAsync(h->d_counters + 1, 0, sizeof(int), s));          // the pack list starts over with every group
            k_plan_fast<<<(unsigned)((nf + 127) / 128), 128, 0, s>>>(h->d_frames, f0, fe, h->d_jobs, h->d_pack_list, h->d_counters + 1, h->d_link_dirty, soft);
            k_plan<<<(ng * 32 + 127) / 128, 128, 0, s>>>(gl, ng, h->d_frames, h->d_jobs, h->d_pack_list, h->d_counters + 1,
                                                         h->d_counters + 2, soft, h->d_link_dirty + lb, h->d_link_dirty + MAX_LINKS + lb);
            if (timed) mark(h, ST_PACK);
            if (!soft) {
                k_pack<<<dim3(7, 148), 256, 0, s>>>(h->d_jobs, h->d_pack_list, h->d_counters + 1, h->d_rows, h->d_depunct, h->d_vit_in, h->d_frames);
                if (timed) mark(h, ST_VITERBI);
                // by frame count: one trellis per warp, per four lanes, per thread (WIFI_P_VITERBI_FORM pins one form: the
                // three are the same decoder, bit for bit)
                auto launch_viterbi = [&](cudaStream_t st, int a, int b) {
                    const int64_t n = b - a;
                    const int form = h->viterbi_form ? h->viterbi_form : (n <= VW_SWITCH ? 1 : (n <= VQ_SWITCH ? 2 : 3));
                    if (form == 1) k_viterbi_warp<<<(unsigned)((n + VW_WARPS - 1) / VW_WARPS), 32 * VW_WARPS, 0, st>>>(h->d_jobs, a, b, h->d_vit_in, h->d_psdu, h->d_frames);
                    else if (form == 2) k_viterbi_quad<<<(unsigned)((n + VQ_FRAMES - 1) / VQ_FRAMES), VQ_BLOCK, 0, st>>>(h->d_jobs, a, b, h->d_vit_in, h->d_psdu, h->d_frames);
                    else k_viterbi<<<(unsigned)((n + VIT_BLOCK - 1) / VIT_BLOCK), VIT_BLOCK, vit_smem, st>>>(h->d_jobs, a, b, h->d_vit_in, h->d_psdu, h->d_frames);
                };
                // The per-thread kernel's time is a staircase: 1.5 ms while every scheduler holds at most one of its warps
                // (sm_count x 2 blocks x 64 = 18944 frames), 2.3 ms up to two (37888), and so on -- 18951 frames cost what
                // 37888 do.  A few frames beyond a step (a long stream cut into step-sized segments with an overlap) therefore
                // go to their own launch on a second stream, in the form their number calls for, beside the main grid.
                const int64_t wave = (int64_t)h->sm_count * 2 * VIT_BLOCK;
                int64_t rem = nf % wave;
                if (rem > VQ_SPLIT_MAX) rem = 0;           // a large remainder competes for the same pipes: no gain
                if (h->viterbi_form || nf < wave || rem == 0) {
                    launch_viterbi(s, f0, fe);
                } else {
                    CK(cudaEventRecord(h->ev_fork, s));
                    CK(cudaStreamWaitEvent(h->aux_stream, h->ev_fork, 0));
                    launch_viterbi(h->aux_stream, fe - (int)rem, fe);
                    launch_viterbi(s, f0, fe - (int)rem);
                    CK(cudaEventRecord(h->ev_join, h->aux_stream));
                    CK(cudaStreamWaitEvent(s, h->ev_join, 0));
                }
            } else {
                k_pack_soft<<<dim3(25, 148), 256, 0, s>>>(h->d_jobs, h->d_pack_list, h->d_counters + 1, h->d_soft, h->d_depunct, h->d_vit_soft_in, h->d_frames);
                if (timed) mark(h, ST_VITERBI);
                k_viterbi_soft<<<(unsigned)((nf + VIT_BLOCK - 1) / VIT_BLOCK), VIT_BLOCK, vit_smem_soft, s>>>(h->d_jobs, f0, fe, h->d_vit_soft_in, h->d_psdu, h->d_frames);
            }
            if (mirror) {
                // results of this group go home on their own stream while the next group is decoded
                CK(cudaEventRecord(h->ev_done[g], s));
                CK(cudaStreamWaitEvent(h->d2h_stream, h->ev_done[g], 0));
                CK(cudaMemcpyAsync(h->h_frames + f0, h->d_frames + f0, (size_t)nf * sizeof(wifi_b200_frame), cudaMemcpyDeviceToHost, h->d2h_stream));
                CK(cudaMemcpyAsync(h->h_psdu + (size_t)f0 * PSDU_STRIDE, (const uint8_t *)h->d_psdu + (size_t)f0 * PSDU_STRIDE, (size_t)nf * PSDU_STRIDE,
                                   cudaMemcpyDeviceToHost, h->d2h_stream));
            }
        }
        frame_base = f_end;
        row_base = rows_needed;
        tile_base += tiles_g;
    }
    h->n_triggers = h->n_frames = h->n_jobs = frame_base;       // decode jobs live at the index of their owner frame
    h->n_rows = row_base;
    if (timed) mark(h, ST_D2H);
    mark(h, ST_COUNT);
    CK(cudaMemcpyAsync(h->h_counters, h->d_counters, 64, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (mirror) CK(cudaStreamSynchronize(h->d2h_stream));
    CK(cudaGetLastError());
    if (h->h_counters[2] != 0) {
        h->err = "receive pipeline reported an internal overflow";
        return WIFI_E_OVERFLOW;
    }
    h->host_mirror = h->psdu_mirror = mirror;
    // stage times: difference between consecutive recorded events
    int prev = -1;
    for (int i = 0; i <= ST_COUNT; ++i) {
        if (!h->ev_used[i]) continue;
        if (prev >= 0) cudaEventElapsedTime(&h->stage_ms[prev], h->ev[prev], h->ev[i]);
        prev = i;
    }
    return WIFI_OK;
}

// run_rx with host input: whatever happens, the caller's buffer is no longer being read when the call returns
int run_rx_host(wifi_b200 *h, const H2dPlan &plan)
{
    int rc = run_rx(h, h->d_iq, true, &plan);
    if (rc != WIFI_OK) {
        cudaStreamSynchronize(h->copy_stream);
        cudaStreamSynchronize(h->d2h_stream);
        cudaStreamSynchronize(h->aux_stream);
        cudaStreamSynchronize(h->stream);
    }
    return rc;
}

int fetch_frames(wifi_b200 *h)
{
    if (h->host_mirror || h->n_frames == 0) return WIFI_OK;
    CK(cudaMemcpyAsync(h->h_frames, h->d_frames, h->n_frames * sizeof(wifi_b200_frame), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->host_mirror = true;
    return WIFI_OK;
}

int fetch_psdus(wifi_b200 *h)
{
    if (h->psdu_mirror || h->n_jobs == 0) return WIFI_OK;
    spill_blocks_on(h, h->h_psdu);
    CK(cudaMemcpyAsync(h->h_psdu, h->d_psdu, (size_t)h->n_jobs * PSDU_STRIDE, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->psdu_mirror = true;
    return WIFI_OK;
}

void count_frame(wifi_b200_stats &st, const wifi_b200_frame &f)
{
    st.frames_detected++;
    st.signal_ok += f.sig_ok;
    st.decoded += f.decoded;
    if (f.crc_ok) {
        st.crc_ok++;
        st.pdu_bytes += f.length - 4;
        st.per_mcs_crc_ok[f.encoding & 7]++;
    }
}

void update_stats(wifi_b200 *h)
{
    h->stats.samples += h->n_samples;
    for (int64_t i = 0; i < h->n_frames; ++i) count_frame(h->stats, h->h_frames[i]);
}

int set_links(wifi_b200 *h, const uint64_t *link_off, int n_links, int final)
{
    if (!link_off || n_links <= 0 || n_links > MAX_LINKS) { h->err = "bad link table"; return WIFI_E_ARG; }
    int64_t total = (int64_t)(link_off[n_links] - link_off[0]);
    if (total > h->cfg.max_samples) { h->err = "more samples than max_samples"; return WIFI_E_OVERFLOW; }
    h->h_links.resize(n_links);
    for (int l = 0; l < n_links; ++l) {
        LinkDesc &L = h->h_links[l];
        memset(&L, 0, sizeof L);
        if (link_off[l + 1] < link_off[l]) { h->err = "link offsets not ascending"; return WIFI_E_ARG; }
        L.x_off = (int64_t)link_off[l];
        L.len = (int64_t)(link_off[l + 1] - link_off[l]);
        if (L.len >= (1ll << 31)) { h->err = "a link is limited to 2^31-1 samples (trigger positions are 32-bit inside the library)"; return WIFI_E_TOO_LARGE; }
        L.is_final = final ? 1 : 0;
    }
    return WIFI_OK;
}

} // namespace

extern "C" {

int wifi_b200_abi_version(void) { return WIFI_B200_ABI_VERSION; }

int wifi_b200_device_count(void)
{
    int n = 0, ok = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    for (int i = 0; i < n; ++i) {
        cudaDeviceProp p;
        if (cudaGetDeviceProperties(&p, i) == cudaSuccess && p.major == 10) ++ok;
    }
    return ok;
}

const char *wifi_b200_strerror(int code)
{
    switch (code) {
    case WIFI_OK: return "ok";
    case WIFI_E_ARG: return "bad argument";
    case WIFI_E_TOO_LARGE: return "PSDU too large (max 1528 bytes / 511 symbols)";
    case WIFI_E_CUDA: return "CUDA error";
    case WIFI_E_NOMEM: return "out of memory";
    case WIFI_E_OVERFLOW: return "capacity exceeded";
    case WIFI_E_NODEVICE: return "no sm_100 device";
    default: return "unknown";
    }
}

int wifi_b200_create(const wifi_b200_cfg *cfg_in, wifi_b200_t **out)
{
    if (!cfg_in || !out) return WIFI_E_ARG;
    *out = nullptr;
    wifi_b200_cfg cfg = *cfg_in;
    if (cfg.bandwidth <= 0) cfg.bandwidth = 10e6;
    if (cfg.frequency <= 0) cfg.frequency = 5.89e9;
    if (cfg.sensitivity <= 0) cfg.sensitivity = 0.56;
    if (cfg.min_plateau <= 0) cfg.min_plateau = 2;
    if (cfg.max_samples <= 0) cfg.max_samples = 1 << 22;
    if (cfg.max_frames <= 0) cfg.max_frames = cfg.max_samples / 1000 + 64;
    if (cfg.chan_est < 0 || cfg.chan_est > 3 || cfg.encoding < 0 || cfg.encoding > 7 || cfg.min_plateau > 16) return WIFI_E_ARG;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0 || cfg.device < 0 || cfg.device >= ndev) return WIFI_E_NODEVICE;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, cfg.device) != cudaSuccess || prop.major != 10) return WIFI_E_NODEVICE;
    wifi_b200 *h = new wifi_b200;
    h->cfg = cfg;
    h->device = cfg.device;
    memset(h->ev, 0, sizeof h->ev);
    memset(&h->stats, 0, sizeof h->stats);
    memset(h->stage_ms, 0, sizeof h->stage_ms);
    auto fail = [&](int code) { free_all(h); delete h; return code; };
    if (cudaSetDevice(h->device) != cudaSuccess) return fail(WIFI_E_CUDA);
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) return fail(WIFI_E_CUDA);
    if (cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking) != cudaSuccess) return fail(WIFI_E_CUDA);
    if (cudaStreamCreateWithFlags(&h->d2h_stream, cudaStreamNonBlocking) != cudaSuccess) return fail(WIFI_E_CUDA);
    if (cudaStreamCreateWithFlags(&h->aux_stream, cudaStreamNonBlocking) != cudaSuccess) return fail(WIFI_E_CUDA);
    if (cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming) != cudaSuccess) return fail(WIFI_E_CUDA);
    if (cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming) != cudaSuccess) return fail(WIFI_E_CUDA);
    if (cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, h->device) != cudaSuccess || h->sm_count <= 0) h->sm_count = 148;
    for (int i = 0; i <= ST_COUNT; ++i) if (cudaEventCreate(&h->ev[i]) != cudaSuccess) return fail(WIFI_E_CUDA);
    if (upload_tables(h) != WIFI_OK) return fail(WIFI_E_CUDA);
    if (cudaFuncSetAttribute(k_detect, cudaFuncAttributeMaxDynamicSharedMemorySize, DET_SMEM) != cudaSuccess) return fail(WIFI_E_CUDA);
    if (VIT_SMEM_BYTES > 48 * 1024 && cudaFuncSetAttribute(k_viterbi, cudaFuncAttributeMaxDynamicSharedMemorySize, VIT_SMEM_BYTES) != cudaSuccess) return fail(WIFI_E_CUDA);
    {
        // CUDA loads a kernel on its first launch (milliseconds): do it here, not inside the first live run
        const void *kernels[] = {(const void *)k_detect, (const void *)k_select_spec, (const void *)k_select_fix, (const void *)k_select, (const void *)k_reserve,
                                 (const void *)k_frames_init, (const void *)k_sync_long, (const void *)k_signal, (const void *)k_plan_fast,
                                 (const void *)k_plan, (const void *)k_pack, (const void *)k_viterbi, (const void *)k_viterbi_warp,
                                 (const void *)k_move_segments, (const void *)k_viterbi_quad, (const void *)k_append_sc16, (const void *)k_sc16_to_fc32, (const void *)k_tx, (const void *)k_channel, (const void *)k_channel_fading,
                                 (const void *)k_demod<false, WIFI_EQ_LS, 0>, (const void *)k_demod<false, WIFI_EQ_LS, 1>,
                                 (const void *)k_demod<false, WIFI_EQ_LMS, 0>, (const void *)k_demod<false, WIFI_EQ_LMS, 1>,
                                 (const void *)k_demod<false, WIFI_EQ_COMB, 0>, (const void *)k_demod<false, WIFI_EQ_COMB, 1>,
                                 (const void *)k_demod<false, WIFI_EQ_STA, 0>, (const void *)k_demod<false, WIFI_EQ_STA, 1>};
        cudaFuncAttributes fa;
        for (const void *k : kernels)
            if (cudaFuncGetAttributes(&fa, k) != cudaSuccess) return fail(WIFI_E_CUDA);
    }
    const int64_t S = cfg.max_samples, Fm = cfg.max_frames;
    h->row_cap = S / 80 + Fm + MAX_LINKS + 64;
    bool ok = true;
    auto A = [&](void **p, size_t bytes) { if (ok && cudaMalloc(p, bytes ? bytes : 16) != cudaSuccess) ok = false; };
    h->tile_cap = S / DET_TILE + MAX_LINKS + 1;
    A((void **)&h->d_flags, (size_t)h->tile_cap * DET_THREADS * 8);
    A((void **)&h->d_summary, (size_t)h->tile_cap * (DET_THREADS / 32) * 4 + 256);
    A((void **)&h->d_trig_tmp, (size_t)h->tile_cap * (DET_THREADS / 4) * sizeof(int));
    A((void **)&h->d_spec_trig, (size_t)h->tile_cap * SEG_CAP * sizeof(int));
    A((void **)&h->d_spec_cnt, (size_t)h->tile_cap * sizeof(int4));
    A((void **)&h->d_spec_trig2, (size_t)h->tile_cap * SEG_CAP * sizeof(int));
    A((void **)&h->d_spec_cnt2, (size_t)h->tile_cap * sizeof(int4));
    A((void **)&h->d_pack_list, (size_t)2 * Fm * sizeof(int));
    A((void **)&h->d_link_dirty, (size_t)2 * MAX_LINKS * sizeof(int));   // [0, MAX_LINKS): dirty flags, [MAX_LINKS, 2 MAX_LINKS): open decode_mac state
    A((void **)&h->d_links, (size_t)MAX_LINKS * sizeof(LinkDesc));
    A((void **)&h->d_frames, (size_t)Fm * sizeof(wifi_b200_frame));
    A((void **)&h->d_states, (size_t)Fm * sizeof(EqState));
    A((void **)&h->d_rows, (size_t)h->row_cap * 48);
    if (cfg.want_carrier) A((void **)&h->d_carrier, (size_t)h->row_cap * 48 * sizeof(cf));
    A((void **)&h->d_jobs, (size_t)Fm * sizeof(JobDesc));
    A((void **)&h->d_vit_in, (size_t)Fm * VIT_MAXW * 4);
    A((void **)&h->d_psdu, (size_t)Fm * PSDU_STRIDE);
    A((void **)&h->d_counters, 64);
    if (!ok) return fail(WIFI_E_NOMEM);
    if (cudaMallocHost(&h->h_counters, 64) != cudaSuccess) return fail(WIFI_E_NOMEM);
    if (cudaMallocHost(&h->h_frames, (size_t)Fm * sizeof(wifi_b200_frame)) != cudaSuccess) return fail(WIFI_E_NOMEM);
    if (cudaMallocHost(&h->h_psdu, (size_t)Fm * PSDU_STRIDE) != cudaSuccess) return fail(WIFI_E_NOMEM);
    *out = h;
    return WIFI_OK;
}

void wifi_b200_destroy(wifi_b200_t *h)
{
    if (!h) return;
    free_all(h);
    delete h;
}

int wifi_b200_set_param(wifi_b200_t *h, int id, double v)
{
    if (!h) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    switch (id) {
    case WIFI_P_BANDWIDTH: if (v <= 0) return WIFI_E_ARG; h->cfg.bandwidth = v; break;
    case WIFI_P_FREQUENCY: if (v <= 0) return WIFI_E_ARG; h->cfg.frequency = v; break;
    case WIFI_P_SENSITIVITY: h->cfg.sensitivity = v; break;
    case WIFI_P_CHAN_EST: if (v < 0 || v > 3) return WIFI_E_ARG; h->cfg.chan_est = (int)v; break;
    case WIFI_P_ENCODING: if (v < 0 || v > 7) return WIFI_E_ARG; h->cfg.encoding = (int)v; break;
    case WIFI_P_MIN_PLATEAU: if (v < 1 || v > 16) return WIFI_E_ARG; h->cfg.min_plateau = (int)v; break;
    case WIFI_P_SOFT_DECISION: h->cfg.soft_decision = v != 0; break;
    case WIFI_P_STREAM_BATCH: if (v < 0 || v > (double)h->cfg.max_samples / 2) return WIFI_E_ARG; h->s_batch = (int64_t)v; break;
    case WIFI_P_HOST_GROUP_SAMPLES: if (v < 0) return WIFI_E_ARG; h->group_samples = (int64_t)v; break;
    case WIFI_P_VITERBI_FORM: if (v != 0 && v != 1 && v != 2 && v != 3) return WIFI_E_ARG; h->viterbi_form = (int)v; break;
    case WIFI_P_WANT_CARRIER:
        if (v != 0 && !h->d_carrier) {
            cudaSetDevice(h->device);
            if (cudaMalloc(&h->d_carrier, (size_t)h->row_cap * 48 * sizeof(cf)) != cudaSuccess) return WIFI_E_NOMEM;
        }
        h->cfg.want_carrier = v != 0;
        break;
    default: return WIFI_E_ARG;
    }
    return WIFI_OK;
}

double wifi_b200_get_param(wifi_b200_t *h, int id)
{
    if (!h) return NAN;
    std::lock_guard<std::mutex> g(h->mu);
    switch (id) {
    case WIFI_P_BANDWIDTH: return h->cfg.bandwidth;
    case WIFI_P_FREQUENCY: return h->cfg.frequency;
    case WIFI_P_SENSITIVITY: return h->cfg.sensitivity;
    case WIFI_P_CHAN_EST: return h->cfg.chan_est;
    case WIFI_P_ENCODING: return h->cfg.encoding;
    case WIFI_P_MIN_PLATEAU: return h->cfg.min_plateau;
    case WIFI_P_WANT_CARRIER: return h->cfg.want_carrier;
    case WIFI_P_SOFT_DECISION: return h->cfg.soft_decision;
    case WIFI_P_STREAM_BATCH: return (double)h->s_batch;
    case WIFI_P_HOST_GROUP_SAMPLES: return (double)h->group_samples;
    case WIFI_P_VITERBI_FORM: return h->viterbi_form;
    default: return NAN;
    }
}

const char *wifi_b200_last_error(wifi_b200_t *h) { return h ? h->err.c_str() : "null handle"; }
void *wifi_b200_stream(wifi_b200_t *h) { return h ? (void *)h->stream : nullptr; }
int wifi_b200_sync(wifi_b200_t *h)
{
    if (!h) return WIFI_E_ARG;
    cudaSetDevice(h->device);
    CK(cudaStreamSynchronize(h->stream));
    return WIFI_OK;
}

int wifi_b200_mac_frame(const uint8_t *payload, int n, int seq, const uint8_t src[6], const uint8_t dst[6], const uint8_t bss[6], uint8_t *o)
{
    // [UPSTREAM] mac.cc: fc 0x0008, duration 0, addr1 = dst, addr2 = src, addr3 = bss, seq_ctl = (seq & 0xfff) << 4, FCS
    if (!payload && n > 0) return WIFI_E_ARG;
    if (n < 0 || !o || !src || !dst || !bss) return WIFI_E_ARG;
    if (n > 1500) return WIFI_E_TOO_LARGE;
    o[0] = 0x08; o[1] = 0x00; o[2] = 0x00; o[3] = 0x00;
    memcpy(o + 4, dst, 6);
    memcpy(o + 10, src, 6);
    memcpy(o + 16, bss, 6);
    uint16_t sc = (uint16_t)((seq & 0xfff) << 4);
    o[22] = sc & 0xff; o[23] = sc >> 8;
    if (n) memcpy(o + 24, payload, n);
    uint32_t c = h_crc32(o, 24 + n);
    o[24 + n] = c & 0xff; o[25 + n] = (c >> 8) & 0xff; o[26 + n] = (c >> 16) & 0xff; o[27 + n] = (c >> 24) & 0xff;
    return 28 + n;
}

int wifi_b200_n_sym(int enc, int len) { return (enc < 0 || enc > 7 || len < 0) ? WIFI_E_ARG : h_n_sym(enc, len); }
int wifi_b200_frame_samples(int enc, int len) { return (enc < 0 || enc > 7 || len < 0) ? WIFI_E_ARG : 80 * (5 + h_n_sym(enc, len)) + 1; }

static int64_t tx_common(wifi_b200_t *h, const uint8_t *blob, const uint32_t *off, const uint32_t *len, const uint8_t *enc,
                         const uint8_t *seed, int n, float *iq_out, size_t cap, uint64_t *burst_off, bool out_is_dev)
{
    if (!h || !blob || !off || !len || n <= 0 || !iq_out) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    cudaSetDevice(h->device);
    if (n > h->cfg.max_frames) { h->err = "more PSDUs than max_frames"; return WIFI_E_OVERFLOW; }
    std::vector<TxFrameDesc> descs(n);
    uint64_t pos = 0, spos = 0;
    size_t blob_bytes = 0;
    int seedc = h->tx_seed;
    for (int i = 0; i < n; ++i) {
        int e = enc ? enc[i] : h->cfg.encoding;
        if (e < 0 || e > 7) { h->err = "bad encoding"; return WIFI_E_ARG; }
        int ns = h_n_sym(e, (int)len[i]);
        if (len[i] > WIFI_MAX_PSDU || ns > WIFI_MAX_SYM) { h->err = "PSDU too large"; return WIFI_E_TOO_LARGE; }
        int sd;
        if (seed) { sd = seed[i] & 0x7f; if (sd == 0) { h->err = "scrambler seed 0"; return WIFI_E_ARG; } }
        else { sd = seedc; seedc = seedc >= 127 ? 1 : seedc + 1; }
        descs[i] = {off[i], len[i], (uint32_t)e, (uint32_t)sd, pos, spos};
        if (burst_off) burst_off[i] = pos;
        pos += (uint64_t)(80 * (5 + ns) + 1);
        spos += (uint64_t)ns * 48;
        blob_bytes = std::max(blob_bytes, (size_t)off[i] + len[i]);
    }
    if (burst_off) burst_off[n] = pos;
    if (pos > cap) { h->err = "iq_out too small"; return WIFI_E_OVERFLOW; }
    if (!seed) h->tx_seed = seedc;
    int rc = grow(h, (void **)&h->d_txblob, &h->txblob_cap, blob_bytes, 1024);
    if (rc == WIFI_OK) rc = grow(h, (void **)&h->d_txsym, &h->txsym_cap, spos, 1024);
    if (rc == WIFI_OK && !out_is_dev) rc = grow(h, (void **)&h->d_txiq, &h->txiq_cap, pos * sizeof(cf), 1024 * sizeof(cf));
    if (rc != WIFI_OK) return rc;
    if (!h->d_txdesc) CK(cudaMalloc(&h->d_txdesc, (size_t)h->cfg.max_frames * sizeof(TxFrameDesc)));
    cf *dst = out_is_dev ? (cf *)iq_out : h->d_txiq;
    cudaStream_t s = h->stream;
    CK(cudaMemcpyAsync(h->d_txblob, blob, blob_bytes, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(h->d_txdesc, descs.data(), n * sizeof(TxFrameDesc), cudaMemcpyHostToDevice, s));
    k_tx<<<n, 128, 0, s>>>(h->d_txblob, h->d_txdesc, n, dst, h->d_txsym);
    CK(cudaGetLastError());
    if (!out_is_dev) CK(cudaMemcpyAsync(iq_out, dst, pos * sizeof(cf), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    h->tx_sym_bytes = (int64_t)spos;
    return (int64_t)pos;
}

int64_t wifi_b200_tx(wifi_b200_t *h, const uint8_t *blob, const uint32_t *off, const uint32_t *len, const uint8_t *enc,
                     const uint8_t *seed, int n, float *iq_out, size_t cap, uint64_t *burst_off)
{
    return tx_common(h, blob, off, len, enc, seed, n, iq_out, cap, burst_off, false);
}
int64_t wifi_b200_tx_dev(wifi_b200_t *h, const uint8_t *blob, const uint32_t *off, const uint32_t *len, const uint8_t *enc,
                         const uint8_t *seed, int n, float *iq_out_dev, size_t cap, uint64_t *burst_off)
{
    return tx_common(h, blob, off, len, enc, seed, n, iq_out_dev, cap, burst_off, true);
}
int64_t wifi_b200_tx_symbols(wifi_b200_t *h, uint8_t *out, size_t cap)
{
    if (!h || !out) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    cudaSetDevice(h->device);
    if ((size_t)h->tx_sym_bytes > cap) return WIFI_E_OVERFLOW;
    if (h->tx_sym_bytes) CK(cudaMemcpy(out, h->d_txsym, h->tx_sym_bytes, cudaMemcpyDeviceToHost));
    return h->tx_sym_bytes;
}

static bool fading_ok(const wifi_b200_chan_seg &s, const wifi_b200_fading &f)
{
    if (s.n_taps != 0 || f.n_taps < 1 || f.n_taps > 8 || f.n_sin < 1 || f.n_sin > 16) return false;
    if (!(f.k_factor >= 0.f && f.k_factor <= FLT_MAX) || !(f.doppler >= 0.f && f.doppler <= 0.25f) || !(fabsf(f.los_doppler) <= 0.25f)) return false;
    for (int t = 0; t < f.n_taps; ++t)
        if (f.delay[t] < 0 || !(f.power[t] >= 0.f && f.power[t] <= FLT_MAX)) return false;
    return true;
}

// The argument check of the four channel entry points, made before anything is allocated or written.  fades == nullptr
// selects the fixed taps.  in_len / out_len are the lengths of host buffers, which every segment must lie inside; device
// buffers (in_len == 0) are the caller's to size.
static int check_channel(wifi_b200 *h, const wifi_b200_chan_seg *segs, const wifi_b200_fading *fades, int n_segs, int64_t in_len, int64_t out_len)
{
    if (!segs || n_segs <= 0) { h->err = "no channel segments"; return WIFI_E_ARG; }
    for (int i = 0; i < n_segs; ++i) {
        const wifi_b200_chan_seg &s = segs[i];
        if (s.n < 0 || s.in_len < 0 || (fades ? !fading_ok(s, fades[i]) : (s.n_taps < 0 || s.n_taps > 8))) {
            h->err = fades ? "bad fading channel segment" : "bad channel segment";
            return WIFI_E_ARG;
        }
        if (in_len && (s.in_off < 0 || s.in_off + s.in_len > in_len || s.out_off < 0 || s.out_off + s.n > out_len)) {
            h->err = "channel segment outside the buffers";
            return WIFI_E_ARG;
        }
    }
    return WIFI_OK;
}

// Runs checked segments through k_channel, or k_channel_fading when fades is given, in launches of at most 65535 grid
// rows (one segment per row).  The caller holds h->mu and has made h->device current.
static int run_channel(wifi_b200 *h, const cf *in_dev, cf *out_dev, const wifi_b200_chan_seg *segs, const wifi_b200_fading *fades, int n_segs)
{
    int64_t maxn = 0;
    for (int i = 0; i < n_segs; ++i) maxn = std::max(maxn, segs[i].n);
    int rc = grow(h, (void **)&h->d_segs, &h->segs_cap, (size_t)n_segs * sizeof(wifi_b200_chan_seg), 64 * sizeof(wifi_b200_chan_seg));
    if (rc == WIFI_OK && fades) rc = grow(h, (void **)&h->d_fades, &h->fades_cap, (size_t)n_segs * sizeof(wifi_b200_fading), 64 * sizeof(wifi_b200_fading));
    if (rc != WIFI_OK) return rc;
    CK(cudaMemcpyAsync(h->d_segs, segs, (size_t)n_segs * sizeof(wifi_b200_chan_seg), cudaMemcpyHostToDevice, h->stream));
    if (fades) CK(cudaMemcpyAsync(h->d_fades, fades, (size_t)n_segs * sizeof(wifi_b200_fading), cudaMemcpyHostToDevice, h->stream));
    for (int base = 0; base < n_segs; base += 65535) {
        int cnt = std::min(65535, n_segs - base);
        dim3 grid((unsigned)std::min<int64_t>((maxn + 255) / 256, 4096), cnt);
        if (grid.x == 0) grid.x = 1;
        if (fades) k_channel_fading<<<grid, 256, 0, h->stream>>>(in_dev, out_dev, h->d_segs + base, h->d_fades + base, cnt);
        else k_channel<<<grid, 256, 0, h->stream>>>(in_dev, out_dev, h->d_segs + base, cnt);
    }
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(h->stream));
    return WIFI_OK;
}

static int channel_dev(wifi_b200_t *h, const float *in_dev, float *out_dev, const wifi_b200_chan_seg *segs, const wifi_b200_fading *fades, int n_segs)
{
    if (!h || !in_dev || !out_dev) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    int rc = check_channel(h, segs, fades, n_segs, 0, 0);
    if (rc != WIFI_OK) return rc;
    cudaSetDevice(h->device);
    return run_channel(h, (const cf *)in_dev, (cf *)out_dev, segs, fades, n_segs);
}

// host-buffer forms: stage in/out through temporary device buffers; out is zero where no segment writes
static int channel_host(wifi_b200_t *h, const float *in_host, int64_t in_len, float *out_host, int64_t out_len,
                        const wifi_b200_chan_seg *segs, const wifi_b200_fading *fades, int n_segs)
{
    if (!h || !in_host || !out_host || in_len <= 0 || out_len <= 0) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    int rc = check_channel(h, segs, fades, n_segs, in_len, out_len);
    if (rc != WIFI_OK) return rc;
    cudaSetDevice(h->device);
    cf *d_in = nullptr, *d_out = nullptr;
    CK(cudaMalloc(&d_in, (size_t)in_len * sizeof(cf)));
    if (cudaMalloc(&d_out, (size_t)out_len * sizeof(cf)) != cudaSuccess) { cudaFree(d_in); h->err = "cudaMalloc"; return WIFI_E_NOMEM; }
    if (cudaMemcpy(d_in, in_host, (size_t)in_len * sizeof(cf), cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemset(d_out, 0, (size_t)out_len * sizeof(cf)) != cudaSuccess) {
        h->err = "channel staging copy";
        rc = WIFI_E_CUDA;
    } else if ((rc = run_channel(h, d_in, d_out, segs, fades, n_segs)) == WIFI_OK &&
               cudaMemcpy(out_host, d_out, (size_t)out_len * sizeof(cf), cudaMemcpyDeviceToHost) != cudaSuccess) {
        h->err = "channel staging copy";
        rc = WIFI_E_CUDA;
    }
    cudaFree(d_in);
    cudaFree(d_out);
    return rc;
}

int wifi_b200_channel_dev(wifi_b200_t *h, const float *in_dev, float *out_dev, const wifi_b200_chan_seg *segs, int n_segs)
{
    return channel_dev(h, in_dev, out_dev, segs, nullptr, n_segs);
}

int wifi_b200_channel(wifi_b200_t *h, const float *in_host, int64_t in_len, float *out_host, int64_t out_len,
                      const wifi_b200_chan_seg *segs, int n_segs)
{
    return channel_host(h, in_host, in_len, out_host, out_len, segs, nullptr, n_segs);
}

int wifi_b200_channel_fading_dev(wifi_b200_t *h, const float *in_dev, float *out_dev, const wifi_b200_chan_seg *segs,
                                 const wifi_b200_fading *fades, int n_segs)
{
    return fades ? channel_dev(h, in_dev, out_dev, segs, fades, n_segs) : WIFI_E_ARG;
}

int wifi_b200_channel_fading(wifi_b200_t *h, const float *in_host, int64_t in_len, float *out_host, int64_t out_len,
                             const wifi_b200_chan_seg *segs, const wifi_b200_fading *fades, int n_segs)
{
    return fades ? channel_host(h, in_host, in_len, out_host, out_len, segs, fades, n_segs) : WIFI_E_ARG;
}

int wifi_b200_rx_batch_dev(wifi_b200_t *h, const float *iq_dev, const uint64_t *link_off, int n_links, int final)
{
    if (!h || !iq_dev) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    cudaSetDevice(h->device);
    int rc = set_links(h, link_off, n_links, final);
    if (rc) return rc;
    for (int i = 0; i <= ST_COUNT; ++i) h->ev_used[i] = false;
    rc = run_rx(h, (const cf *)iq_dev, false);
    return rc;
}

int wifi_b200_rx_batch_dev_state(wifi_b200_t *h, const float *iq_dev, const uint64_t *link_off, int n_links, int final,
                                 const wifi_b200_link_state *state)
{
    if (!h || !iq_dev || !state) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    cudaSetDevice(h->device);
    int rc = set_links(h, link_off, n_links, final);
    if (rc) return rc;
    for (int l = 0; l < n_links; ++l) {
        if (state[l].hist < 0 || state[l].hist > 256 || (uint64_t)state[l].hist > link_off[l] || state[l].min_pos < 0) {
            h->err = "bad link state (hist must be 0..256 samples that exist in front of the link)";
            return WIFI_E_ARG;
        }
        LinkDesc &L = h->h_links[l];
        L.hist = state[l].hist;
        L.min_pos = state[l].min_pos;
        L.fo_carry = state[l].fo_carry;
    }
    for (int i = 0; i <= ST_COUNT; ++i) h->ev_used[i] = false;
    return run_rx(h, (const cf *)iq_dev, false);
}

int wifi_b200_rx_batch(wifi_b200_t *h, const float *iq_host, const uint64_t *link_off, int n_links, int final)
{
    if (!h || !iq_host) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    cudaSetDevice(h->device);
    int rc = set_links(h, link_off, n_links, final);
    if (rc) return rc;
    rc = ensure_iq_staging(h);
    if (rc) return rc;
    // rebase the links onto the staging buffer
    uint64_t base = link_off[0];
    for (auto &L : h->h_links) L.x_off -= (int64_t)base;
    H2dPlan plan;
    plan.src = iq_host + 2 * base;
    plan.bytes_per_sample = sizeof(cf);
    rc = run_rx_host(h, plan);
    if (rc) return rc;
    update_stats(h);
    return WIFI_OK;
}

int wifi_b200_rx_batch_sc16(wifi_b200_t *h, const int16_t *iq_host, float scale, const uint64_t *link_off, int n_links, int final)
{
    if (!h || !iq_host) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    cudaSetDevice(h->device);
    int rc = set_links(h, link_off, n_links, final);
    if (rc) return rc;
    rc = ensure_iq_staging(h);
    if (rc) return rc;
    rc = ensure_sc16_staging(h);
    if (rc) return rc;
    uint64_t base = link_off[0];
    for (auto &L : h->h_links) L.x_off -= (int64_t)base;
    H2dPlan plan;
    plan.src = iq_host + 2 * base;
    plan.bytes_per_sample = 2 * sizeof(int16_t);
    if (scale == 0.f) { h->err = "sc16 scale must not be 0"; return WIFI_E_ARG; }
    plan.sc16_scale = scale;
    rc = run_rx_host(h, plan);
    if (rc) return rc;
    update_stats(h);
    return WIFI_OK;
}

int wifi_b200_rx_counts(wifi_b200_t *h, int64_t *n_frames, int64_t *n_rows, int64_t *n_pdus, int64_t *psdu_store_bytes)
{
    if (!h) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    cudaSetDevice(h->device);
    int rc = fetch_frames(h);
    if (rc) return rc;
    int64_t np = 0;
    for (int64_t i = 0; i < h->n_frames; ++i) np += h->h_frames[i].crc_ok;
    if (n_frames) *n_frames = h->n_frames;
    if (n_rows) *n_rows = h->n_rows;
    if (n_pdus) *n_pdus = np;
    if (psdu_store_bytes) *psdu_store_bytes = h->n_jobs * PSDU_STRIDE;
    return WIFI_OK;
}

int wifi_b200_rx_frames(wifi_b200_t *h, wifi_b200_frame *out, int64_t cap)
{
    if (!h || !out) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    cudaSetDevice(h->device);
    if (cap < h->n_frames) return WIFI_E_OVERFLOW;
    int rc = fetch_frames(h);
    if (rc) return rc;
    memcpy(out, h->h_frames, h->n_frames * sizeof(wifi_b200_frame));
    return (int)h->n_frames;
}

int wifi_b200_rx_rows(wifi_b200_t *h, uint8_t *rows, float *carrier, int64_t cap_rows)
{
    if (!h) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    cudaSetDevice(h->device);
    if (cap_rows < h->n_rows) return WIFI_E_OVERFLOW;
    if (rows && h->n_rows) CK(cudaMemcpy(rows, h->d_rows, (size_t)h->n_rows * 48, cudaMemcpyDeviceToHost));
    if (carrier) {
        if (!h->d_carrier || !h->cfg.want_carrier) { h->err = "carrier output not enabled"; return WIFI_E_ARG; }
        if (h->n_rows) CK(cudaMemcpy(carrier, h->d_carrier, (size_t)h->n_rows * 48 * sizeof(cf), cudaMemcpyDeviceToHost));
    }
    return WIFI_OK;
}

int wifi_b200_rx_soft(wifi_b200_t *h, int8_t *soft, int64_t cap_rows)
{
    if (!h || !soft) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    cudaSetDevice(h->device);
    if (!h->cfg.soft_decision || !h->d_soft) { h->err = "soft decisions not enabled"; return WIFI_E_ARG; }
    if (cap_rows < h->n_rows) return WIFI_E_OVERFLOW;
    if (h->n_rows) CK(cudaMemcpy(soft, h->d_soft, (size_t)h->n_rows * SOFT_ROW, cudaMemcpyDeviceToHost));
    return WIFI_OK;
}

int wifi_b200_rx_psdus(wifi_b200_t *h, uint8_t *store, size_t cap)
{
    if (!h || !store) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    cudaSetDevice(h->device);
    if (cap < (size_t)h->n_jobs * PSDU_STRIDE) return WIFI_E_OVERFLOW;
    int rc = fetch_psdus(h);
    if (rc) return rc;
    memcpy(store, h->h_psdu, (size_t)h->n_jobs * PSDU_STRIDE);
    return WIFI_OK;
}

int wifi_b200_rx_flags(wifi_b200_t *h, int link, uint32_t *flags, int64_t cap_words)
{
    if (!h || !flags || link < 0 || link >= (int)h->h_links.size()) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    cudaSetDevice(h->device);
    const LinkDesc &L = h->h_links[link];
    int64_t words = (L.len + 31) / 32;
    if (cap_words < words) return WIFI_E_OVERFLOW;
    CK(cudaMemcpy(flags, h->d_flags + L.chunk_base * (FE_CHUNK / 32), words * 4, cudaMemcpyDeviceToHost));
    return (int)words;
}

// ---- streaming: one continuous stream, arbitrary chunking (samp_in) ----
int wifi_b200_rx_reset(wifi_b200_t *h)
{
    if (!h) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->copy_stream);
    h->a_pending.clear();
    h->s_links.clear();
    h->s_cap = 0;
    h->s_unprocessed = 0;
    h->s_meta.clear(); h->s_bytes.clear();
    h->s_blocks.clear();
    h->view_kind = 0;
    return WIFI_OK;
}

// Streaming over n_links continuous streams: link l receives iq[link_off[l] .. link_off[l+1]) new samples.
// Samples are copied once, from the caller's buffer into the link's region of a device arena (pinned caller memory
// makes that a plain DMA), and stay on the device: a run decodes the regions in place, then every link's retained
// tail (history + held / deferred bursts) slides to the front of its region.
// dev_src != nullptr: the new samples already sit in device memory (the staging buffer of an asynchronous push, link l at
// dev_src[link_off[l]]; as int16 I/Q pairs when sc16_scale != 0) and are appended by a copy kernel; else they are copied
// from the host buffer `iq`.
static int stream_push(wifi_b200 *h, const float *iq, const uint64_t *link_off, int n_links, int flush, const cf *dev_src = nullptr, float sc16_scale = 0.f)
{
    if (n_links <= 0 || n_links > MAX_LINKS) return WIFI_E_ARG;
    cudaSetDevice(h->device);
    if (h->s_links.empty()) {
        h->s_links.resize(n_links);
        h->s_cap = h->cfg.max_samples / n_links;
        if (!h->d_stream) CK(cudaMalloc(&h->d_stream, (size_t)(h->cfg.max_samples + 512) * sizeof(cf)));
        if (!h->d_moves) CK(cudaMalloc(&h->d_moves, (size_t)2 * MAX_LINKS * sizeof(wifi_b200::MoveSeg)));
    }
    if ((int)h->s_links.size() != n_links) { h->err = "the number of streams is fixed until wifi_b200_rx_reset"; return WIFI_E_ARG; }
    int64_t newest = 0, pushed = 0;
    for (int l = 0; l < n_links; ++l) {
        const int64_t n = (int64_t)(link_off[l + 1] - link_off[l]);
        if (h->s_links[l].fill + n > h->s_cap) { h->err = "stream backlog exceeds max_samples / n_links"; return WIFI_E_OVERFLOW; }
        if (n > newest) newest = n;
        pushed += n;
    }
    int64_t have_all = 0, fullest = 0;
    std::vector<wifi_b200::MoveSeg> app;
    for (int l = 0; l < n_links; ++l) {
        auto &S = h->s_links[l];
        const int64_t n = (int64_t)(link_off[l + 1] - link_off[l]);
        if (n && !dev_src) CK(cudaMemcpyAsync(h->d_stream + (int64_t)l * h->s_cap + S.fill, iq + 2 * link_off[l], (size_t)n * sizeof(cf), cudaMemcpyHostToDevice, h->stream));
        if (n && dev_src) app.push_back({(int64_t)link_off[l], (int64_t)l * h->s_cap + S.fill, n});
        S.fill += n;
        have_all += S.fill - S.hist;
        if (S.fill > fullest) fullest = S.fill;
    }
    if (!app.empty()) {
        CK(cudaMemcpyAsync(h->d_moves, app.data(), app.size() * sizeof(wifi_b200::MoveSeg), cudaMemcpyHostToDevice, h->stream));
        unsigned bx = (unsigned)std::min<int64_t>((newest + 2047) / 2048, 64);
        if (sc16_scale != 0.f)
            k_append_sc16<<<dim3(bx ? bx : 1, (unsigned)app.size()), 256, 0, h->stream>>>(reinterpret_cast<const int16_t *>(dev_src), h->d_stream, h->d_moves, sc16_scale);
        else
            k_move_segments<<<dim3(bx ? bx : 1, (unsigned)app.size()), 256, 0, h->stream>>>(dev_src, h->d_stream, h->d_moves);
    }
    h->s_unprocessed += newest;
    // small pushes only buffer: a pipeline run has a fixed cost of about a millisecond (the decoder's latency for the
    // longest frame), so it runs when enough new samples wait, when a region is half full, on an empty push, or on flush
    if (have_all <= 0 || (!flush && pushed != 0 && h->s_unprocessed < h->s_batch && 2 * fullest < h->s_cap)) {
        if (pushed && !dev_src) {
            // The caller's buffer must be free again when the call returns.  A copy from pageable memory has left the
            // source when cudaMemcpyAsync returns (it is staged); only page-locked sources are read asynchronously.
            cudaPointerAttributes at;
            const bool pinned = cudaPointerGetAttributes(&at, iq) == cudaSuccess && at.type != cudaMemoryTypeUnregistered;
            cudaGetLastError();
            if (pinned) CK(cudaStreamSynchronize(h->stream));
        }
        return WIFI_OK;
    }
    h->s_unprocessed = 0;
    h->h_links.resize(n_links);
    for (int l = 0; l < n_links; ++l) {
        auto &S = h->s_links[l];
        LinkDesc &L = h->h_links[l];
        memset(&L, 0, sizeof L);
        L.x_off = (int64_t)l * h->s_cap + S.hist;
        L.len = S.fill - S.hist;
        L.is_final = flush ? 1 : 0;
        L.hold_last = flush ? 0 : 1;     // the newest burst is held back unless flushing (k_frames_init)
        L.hist = S.hist;
        L.fo_carry = S.fo_carry;
        L.min_pos = S.prev_trigger >= 0 ? S.prev_trigger + SS_MIN_GAP + 1 - S.abs0 : 0;
    }
    for (int i = 0; i <= ST_COUNT; ++i) h->ev_used[i] = false;
    int rc = run_rx(h, h->d_stream, true);
    if (rc) {
        // The run failed (more triggers than max_frames, a CUDA error ...).  Keeping the samples would make every later
        // push re-run them and fail again until the backlog overflows, so the buffered region is dropped: the streams
        // continue behind it as after a flush and the caller sees the error code once.
        for (auto &S : h->s_links) {
            const int64_t end_abs = S.abs0 + (S.fill - S.hist);
            S.fill = 0;
            S.abs0 = (end_abs + FE_CHUNK - 1) / FE_CHUNK * FE_CHUNK;
            S.hist = 0; S.prev_trigger = -1; S.fo_carry = 0.f;
        }
        h->err += " (streaming: the buffered samples were discarded)";
        return rc;
    }
    // Frames are ordered by (link, trigger): publish the CRC-ok ones and note from where each link must be kept:
    // its held burst, or -- when decode_mac's state was left open in front of a held burst (a frame cut short by a
    // re-trigger whose symbol collection, or pending tag, continues into that burst) -- the frame that opened it.
    std::vector<int> open_at(n_links, -1);
    if (!flush && h->n_frames > 0)
        CK(cudaMemcpy(open_at.data(), h->d_link_dirty + MAX_LINKS, (size_t)n_links * sizeof(int), cudaMemcpyDeviceToHost));
    std::vector<char> has_held(n_links, 0);
    for (int64_t i = 0; i < h->n_frames; ++i)
        if (h->h_frames[i].n_syms < 0) has_held[h->h_frames[i].link] = 1;
    std::vector<int64_t> keep(n_links, -1);
    wifi_b200::StreamBlock blk;
    h->stats.samples += h->n_samples;             // samples this run looked at (a held burst is looked at again)
    for (int64_t i = 0; i < h->n_frames; ++i) {
        wifi_b200_frame f = h->h_frames[i];
        auto &S = h->s_links[f.link];
        if (keep[f.link] >= 0) continue;          // deferred together with the frame that opened the state
        if (f.n_syms < 0 || (has_held[f.link] && open_at[f.link] >= 0 && i >= open_at[f.link])) {
            keep[f.link] = f.trigger + S.abs0;    // held or deferred: re-detected and decoded by a later run
            continue;
        }
        count_frame(h->stats, f);
        S.prev_trigger = f.trigger + S.abs0;
        S.fo_carry = f.freq_long;
        if (!f.crc_ok) continue;
        f.trigger += S.abs0;
        blk.meta.push_back(f);                    // psdu_off: offset of the PSDU in this run's mirror
    }
    if (!blk.meta.empty()) {
        // the PSDUs stay where the copy engine put them; the next run writes into the other mirror
        if (!h->h_psdu_alt && cudaMallocHost(&h->h_psdu_alt, (size_t)h->cfg.max_frames * PSDU_STRIDE) != cudaSuccess) {
            cudaGetLastError();
            h->h_psdu_alt = nullptr;
        }
        blk.buf = h->h_psdu;
        h->s_blocks.push_back(std::move(blk));
        if (h->h_psdu_alt) {
            std::swap(h->h_psdu, h->h_psdu_alt);
            h->psdu_mirror = false;               // h_psdu no longer holds the last run's PSDUs
        } else {
            spill_blocks_on(h, h->h_psdu);        // no second mirror: packed copy, as a pageable queue
        }
    }
    std::vector<wifi_b200::MoveSeg> moves;         // [0, nm): arena -> scratch, [nm, 2 nm): scratch -> front of the region
    std::vector<wifi_b200::MoveSeg> back;
    int64_t scratch = 0, longest = 0;
    for (int l = 0; l < n_links; ++l) {
        auto &S = h->s_links[l];
        const int64_t have = S.fill - S.hist;
        const int64_t buf_abs = S.abs0 - S.hist;   // absolute index of the region's first sample
        const int64_t end_abs = S.abs0 + have;
        if (flush) {                               // stream ended: nothing is kept
            S.fill = 0;
            S.abs0 = (end_abs + FE_CHUNK - 1) / FE_CHUNK * FE_CHUNK;
            S.hist = 0; S.prev_trigger = -1; S.fo_carry = 0.f;
            continue;
        }
        const int64_t k = keep[l] >= 0 ? keep[l] : end_abs;
        int64_t new_abs0 = (k - FE_CHUNK) / FE_CHUNK * FE_CHUNK;
        if (new_abs0 < S.abs0) new_abs0 = S.abs0;
        int64_t new_hist = new_abs0 - buf_abs;
        if (new_hist > 256) new_hist = 256;
        const int64_t drop = (new_abs0 - new_hist) - buf_abs;   // samples to discard from the front of the region
        if (drop > 0) {
            const int64_t tail = S.fill - drop;
            if (tail > 0) {
                moves.push_back({(int64_t)l * h->s_cap + drop, scratch, tail});
                back.push_back({scratch, (int64_t)l * h->s_cap, tail});
                scratch += tail;
                if (tail > longest) longest = tail;
            }
            S.fill = tail;
        }
        S.abs0 = new_abs0;
        S.hist = (int)new_hist;
    }
    if (!moves.empty()) {
        rc = ensure_iq_staging(h);                 // the batch staging buffer is the scratch space
        if (rc) return rc;
        const int nm = (int)moves.size();
        moves.insert(moves.end(), back.begin(), back.end());
        unsigned bx = (unsigned)((longest + 2047) / 2048);
        if (bx > 64) bx = 64;
        if (bx < 1) bx = 1;
        CK(cudaMemcpyAsync(h->d_moves, moves.data(), moves.size() * sizeof(wifi_b200::MoveSeg), cudaMemcpyHostToDevice, h->stream));
        k_move_segments<<<dim3(bx, nm), 256, 0, h->stream>>>(h->d_stream, h->d_iq, h->d_moves);
        k_move_segments<<<dim3(bx, nm), 256, 0, h->stream>>>(h->d_iq, h->d_stream, h->d_moves + nm);
        CK(cudaStreamSynchronize(h->stream));
        CK(cudaGetLastError());
    }
    return WIFI_OK;
}

int wifi_b200_rx_push(wifi_b200_t *h, const float *iq, size_t n, int flush)
{
    if (!h || (!iq && n)) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    if (h->s_links.size() > 1) { h->err = "this handle streams several links: use wifi_b200_rx_push_links"; return WIFI_E_ARG; }
    const uint64_t off[2] = {0, (uint64_t)n};
    return stream_push(h, iq, off, 1, flush);
}

int wifi_b200_rx_push_links(wifi_b200_t *h, const float *iq, const uint64_t *link_off, int n_links, int flush)
{
    if (!h || !link_off || n_links <= 0) return WIFI_E_ARG;
    for (int l = 0; l < n_links; ++l)
        if (link_off[l + 1] < link_off[l]) return WIFI_E_ARG;
    if (!iq && link_off[n_links] != link_off[0]) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    return stream_push(h, iq, link_off, n_links, flush);
}

static int push_async(wifi_b200 *h, const void *iq, size_t bytes_per_sample, float sc16_scale, const uint64_t *link_off, int n_links, int flush)
{
    if (!h || !link_off || n_links <= 0 || n_links > MAX_LINKS) return WIFI_E_ARG;
    for (int l = 0; l < n_links; ++l)
        if (link_off[l + 1] < link_off[l]) return WIFI_E_ARG;
    const int64_t total = (int64_t)(link_off[n_links] - link_off[0]);
    if (!iq && total) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    cudaSetDevice(h->device);
    if (h->a_pending.size() >= A_SLOTS) { h->err = "three asynchronous pushes are already pending: call wifi_b200_rx_push_wait first"; return WIFI_E_OVERFLOW; }
    if (total > h->cfg.max_samples) { h->err = "push larger than max_samples"; return WIFI_E_OVERFLOW; }
    const int slot = h->a_next % A_SLOTS;
    // slots are sized in fc32 samples: either format fits
    int rc = grow(h, (void **)&h->d_stage[slot], &h->a_cap[slot], (size_t)total * sizeof(cf), 64 * sizeof(cf));
    if (rc != WIFI_OK) return rc;
    if (!h->a_ev[slot]) CK(cudaEventCreateWithFlags(&h->a_ev[slot], cudaEventDisableTiming));
    wifi_b200::AsyncPush job;
    job.slot = slot;
    job.flush = flush;
    job.sc16_scale = sc16_scale;
    job.off.resize(n_links + 1);
    for (int l = 0; l <= n_links; ++l) job.off[l] = link_off[l] - link_off[0];
    // one copy for the whole push (the links lie back to back in the caller's buffer), on the copy stream: it runs while
    // the pipeline of the push before it is still decoding
    if (total) CK(cudaMemcpyAsync(h->d_stage[slot], (const char *)iq + bytes_per_sample * link_off[0], (size_t)total * bytes_per_sample, cudaMemcpyHostToDevice, h->copy_stream));
    CK(cudaEventRecord(h->a_ev[slot], h->copy_stream));
    h->a_pending.push_back(std::move(job));
    h->a_next++;
    return WIFI_OK;
}

int wifi_b200_rx_push_links_async(wifi_b200_t *h, const float *iq, const uint64_t *link_off, int n_links, int flush)
{
    return push_async(h, iq, sizeof(cf), 0.f, link_off, n_links, flush);
}

int wifi_b200_rx_push_links_sc16_async(wifi_b200_t *h, const int16_t *iq, float scale, const uint64_t *link_off, int n_links, int flush)
{
    if (h && scale == 0.f) {
        std::lock_guard<std::mutex> g(h->mu);
        h->err = "sc16 scale must not be 0";
        return WIFI_E_ARG;
    }
    return push_async(h, iq, 2 * sizeof(int16_t), scale, link_off, n_links, flush);
}

int wifi_b200_rx_push_wait(wifi_b200_t *h)
{
    if (!h) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    cudaSetDevice(h->device);
    if (h->a_pending.empty()) return 0;
    wifi_b200::AsyncPush job = std::move(h->a_pending.front());
    h->a_pending.erase(h->a_pending.begin());
    CK(cudaStreamWaitEvent(h->stream, h->a_ev[job.slot], 0));
    int rc = stream_push(h, nullptr, job.off.data(), (int)job.off.size() - 1, job.flush, h->d_stage[job.slot], job.sc16_scale);
    // the staging buffer may be written by the next asynchronous push only after the append kernel has read it
    cudaStreamSynchronize(h->stream);
    return rc < 0 ? rc : 1;
}

int wifi_b200_rx_pop(wifi_b200_t *h, wifi_b200_frame *meta, int cap, uint8_t *psdu_buf, size_t psdu_cap, int *n_out)
{
    if (!h || !n_out) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    release_view(h);
    int k = 0;
    size_t used = 0, consumed_bytes = 0;
    while (k < (int)h->s_meta.size() && k < cap) {
        wifi_b200_frame f = h->s_meta[k];
        size_t nb = (size_t)(f.length - 4);
        if (used + nb > psdu_cap) break;
        if (psdu_buf) memcpy(psdu_buf + used, h->s_bytes.data() + consumed_bytes, nb);
        f.psdu_off = (int64_t)used;
        if (meta) meta[k] = f;
        used += nb;
        consumed_bytes += nb;
        ++k;
    }
    const bool queue_empty = k == (int)h->s_meta.size();
    h->s_meta.erase(h->s_meta.begin(), h->s_meta.begin() + k);
    h->s_bytes.erase(h->s_bytes.begin(), h->s_bytes.begin() + consumed_bytes);
    bool full = !queue_empty;
    while (!full && !h->s_blocks.empty()) {        // then the runs whose PSDUs still sit in their mirror, oldest first
        wifi_b200::StreamBlock &b = h->s_blocks.front();
        while (b.next < b.meta.size()) {
            wifi_b200_frame f = b.meta[b.next];
            size_t nb = (size_t)(f.length - 4);
            if (k >= cap || used + nb > psdu_cap) { full = true; break; }
            if (psdu_buf) memcpy(psdu_buf + used, b.buf + f.psdu_off, nb);
            f.psdu_off = (int64_t)used;
            if (meta) meta[k] = f;
            used += nb;
            ++k;
            ++b.next;
        }
        if (!full) h->s_blocks.pop_front();
    }
    *n_out = k;
    return WIFI_OK;
}

int wifi_b200_rx_pop_view(wifi_b200_t *h, const wifi_b200_frame **meta, const uint8_t **psdu_bytes, size_t *n_bytes, int *n_out)
{
    if (!h || !meta || !psdu_bytes || !n_bytes || !n_out) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    release_view(h);
    *meta = nullptr; *psdu_bytes = nullptr; *n_bytes = 0; *n_out = 0;
    if (!h->s_meta.empty()) {
        size_t used = 0;
        for (auto &f : h->s_meta) { f.psdu_off = (int64_t)used; used += (size_t)(f.length - 4); }
        *meta = h->s_meta.data();
        *psdu_bytes = h->s_bytes.data();
        *n_bytes = used;
        *n_out = (int)h->s_meta.size();
        h->view_kind = 1;
        h->view_n = h->s_meta.size();
        h->view_bytes = used;
    } else if (!h->s_blocks.empty()) {
        wifi_b200::StreamBlock &b = h->s_blocks.front();
        *meta = b.meta.data() + b.next;
        *psdu_bytes = b.buf;
        *n_bytes = (size_t)h->cfg.max_frames * PSDU_STRIDE;
        *n_out = (int)(b.meta.size() - b.next);
        h->view_kind = 2;
    }
    return WIFI_OK;
}

int wifi_b200_selftest_detmath(wifi_b200_t *h, int fn, const float *a, const float *b, const float *c, const float *d, float *o0, float *o1, int64_t n)
{
    if (!h || !a || !b || !c || !d || !o0 || !o1 || n < 0 || fn < 0 || fn >= WDM_T_COUNT) return WIFI_E_ARG;
    if (n == 0) return WIFI_OK;
    std::lock_guard<std::mutex> g(h->mu);
    cudaSetDevice(h->device);
    float *dv = nullptr;
    const size_t bytes = (size_t)n * sizeof(float);
    CK(cudaMalloc(&dv, 6 * bytes));
    const float *src[6] = {a, b, c, d, o0, o1};
    int rc = WIFI_OK;
    for (int k = 0; k < 6 && rc == WIFI_OK; ++k)
        if (cudaMemcpyAsync(dv + (size_t)k * n, src[k], bytes, cudaMemcpyHostToDevice, h->stream) != cudaSuccess) rc = WIFI_E_CUDA;
    if (rc == WIFI_OK) {
        k_detmath<<<(unsigned)std::min<int64_t>((n + 255) / 256, 148 * 8), 256, 0, h->stream>>>(fn, dv, dv + n, dv + 2 * n, dv + 3 * n, dv + 4 * n, dv + 5 * n, n);
        if (cudaMemcpyAsync(o0, dv + 4 * n, bytes, cudaMemcpyDeviceToHost, h->stream) != cudaSuccess ||
            cudaMemcpyAsync(o1, dv + 5 * n, bytes, cudaMemcpyDeviceToHost, h->stream) != cudaSuccess ||
            cudaStreamSynchronize(h->stream) != cudaSuccess || cudaGetLastError() != cudaSuccess) rc = WIFI_E_CUDA;
    }
    cudaFree(dv);
    if (rc) h->err = "selftest_detmath: CUDA error";
    return rc;
}

int wifi_b200_alu_peak(wifi_b200_t *h, int iters, double *warp_inst_per_s, double *ms_out)
{
    if (!h || iters <= 0 || !warp_inst_per_s) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    cudaSetDevice(h->device);
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, h->device));
    const int blocks = prop.multiProcessorCount * 8, threads = 256;      // 64 warps per SM, 16 per scheduler
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    k_alu_peak<<<blocks, threads, 0, h->stream>>>(iters / 8 + 1, 12345u, (uint32_t *)h->d_counters + 12);   // warm-up
    cudaEventRecord(e0, h->stream);
    k_alu_peak<<<blocks, threads, 0, h->stream>>>(iters, 12345u, (uint32_t *)h->d_counters + 12);
    cudaEventRecord(e1, h->stream);
    int rc = WIFI_OK;
    float ms = 0.f;
    if (cudaStreamSynchronize(h->stream) != cudaSuccess || cudaGetLastError() != cudaSuccess || cudaEventElapsedTime(&ms, e0, e1) != cudaSuccess) rc = WIFI_E_CUDA;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (rc) { h->err = "alu_peak: CUDA error"; return rc; }
    *warp_inst_per_s = (double)blocks * (threads / 32) * (double)iters * ALU_PROBE_OPS / (ms * 1e-3);
    if (ms_out) *ms_out = ms;
    return WIFI_OK;
}

// ---- page-locked host memory near the handle's GPU ----
// Reads /sys/bus/pci/devices/<gpu>/local_cpulist: the host cores on the GPU's side of the machine.  The buffer is allocated
// and first touched from those cores, so on a multi-socket box its pages land on the NUMA node whose PCIe root the GPU hangs
// off (Linux places pages on the node of the core that first writes them); the caller's affinity is restored afterwards.
static bool gpu_local_cpus(int device, cpu_set_t *set)
{
    char bdf[32] = {0};
    if (cudaDeviceGetPCIBusId(bdf, sizeof bdf, device) != cudaSuccess) return false;
    for (char *c = bdf; *c; ++c) *c = (char)tolower(*c);
    std::string path = std::string("/sys/bus/pci/devices/") + bdf + "/local_cpulist";
    FILE *f = fopen(path.c_str(), "r");
    if (!f) return false;
    char buf[4096] = {0};
    const bool ok = fgets(buf, sizeof buf, f) != nullptr;
    fclose(f);
    if (!ok) return false;
    CPU_ZERO(set);
    int n = 0;
    for (char *p = buf; *p && *p != '\n';) {                        // "0-15,32-47"
        char *e;
        long a = strtol(p, &e, 10), b = a;
        if (e == p) break;
        if (*e == '-') { p = e + 1; b = strtol(p, &e, 10); }
        for (long c = a; c <= b && c < CPU_SETSIZE; ++c) { CPU_SET((int)c, set); ++n; }
        p = (*e == ',') ? e + 1 : e;
    }
    return n > 0;
}

int wifi_b200_host_alloc(wifi_b200_t *h, size_t bytes, void **out)
{
    if (!h || !out || bytes == 0) return WIFI_E_ARG;
    *out = nullptr;
    std::lock_guard<std::mutex> g(h->mu);
    cudaSetDevice(h->device);
    cpu_set_t old_set, local;
    const bool have_old = sched_getaffinity(0, sizeof old_set, &old_set) == 0;
    bool moved = false;
    if (have_old && gpu_local_cpus(h->device, &local)) {
        cpu_set_t both;
        CPU_AND(&both, &local, &old_set);                             // never leave the cores the caller is allowed on
        if (CPU_COUNT(&both) > 0) moved = sched_setaffinity(0, sizeof both, &both) == 0;
    }
    void *p = nullptr;
    const cudaError_t e = cudaHostAlloc(&p, bytes, cudaHostAllocPortable);
    // first touch from the GPU's side of the machine; the whole buffer, because the driver may hand back pinned pages a
    // previous allocation of this process left data in
    if (e == cudaSuccess) memset(p, 0, bytes);
    if (moved) sched_setaffinity(0, sizeof old_set, &old_set);
    if (e != cudaSuccess) { cudaGetLastError(); h->err = "cudaHostAlloc failed"; return WIFI_E_NOMEM; }
    *out = p;
    return WIFI_OK;
}

int wifi_b200_host_free(wifi_b200_t *h, void *p)
{
    if (!h) return WIFI_E_ARG;
    if (!p) return WIFI_OK;
    std::lock_guard<std::mutex> g(h->mu);
    cudaSetDevice(h->device);
    CK(cudaFreeHost(p));
    return WIFI_OK;
}

int wifi_b200_get_stats(wifi_b200_t *h, wifi_b200_stats *out)
{
    if (!h || !out) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    *out = h->stats;
    return WIFI_OK;
}

int wifi_b200_stage_times(wifi_b200_t *h, float *ms, int cap)
{
    if (!h || !ms) return WIFI_E_ARG;
    std::lock_guard<std::mutex> g(h->mu);
    int n = cap < ST_COUNT ? cap : ST_COUNT;
    for (int i = 0; i < n; ++i) ms[i] = h->stage_ms[i];
    return n;
}
const char *wifi_b200_stage_name(int i) { return (i >= 0 && i < ST_COUNT) ? STAGE_NAMES[i] : ""; }

} // extern "C"
