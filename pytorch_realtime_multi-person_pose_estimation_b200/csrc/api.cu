// C-ABI of libb200pose.so (include/b200pose.h): network object, post-processing object, fused inference and the
// legacy pafprocess surface.  Host-side runtime only; the kernels live in conv_tc.cu, conv_misc.cu, postprocess.cu.
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <set>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/b200pose.h"
#include "conv_misc.cuh"
#include "conv_tc.cuh"
#include "postprocess.cuh"
#include "resize.cuh"
#include "tta.cuh"

using namespace b2p;

namespace {

thread_local std::string g_err;
std::atomic<long> g_launches{0};

int fail(const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return 1;
}
#define CU(x)                                                                                       \
    do {                                                                                            \
        cudaError_t e_ = (x);                                                                       \
        if (e_ != cudaSuccess) return fail("%s failed: %s (%s:%d)", #x, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// ---------------------------------------------------------------- layer table (rtpose_vgg.py:69-127)
struct ConvSpec { int cin, cout, ks; };
const ConvSpec kTrunk[12] = {{3, 64, 3},    {64, 64, 3},   {64, 128, 3},  {128, 128, 3}, {128, 256, 3}, {256, 256, 3},
                             {256, 256, 3}, {256, 256, 3}, {256, 512, 3}, {512, 512, 3}, {512, 256, 3}, {256, 128, 3}};
const bool kPoolAfter[12] = {false, true, false, true, false, false, false, true, false, false, false, false};
constexpr int kPaf = 38, kHeat = 19, kFeat = 128, kCat = kPaf + kHeat + kFeat;
constexpr int kRaggedCap = 4096;       // images per ragged call (size of the net's fixed extent array)

int stage_num_layers(int stage) { return stage == 1 ? 5 : 7; }
ConvSpec stage_layer(int stage, int branch, int li) {
    const int outc = branch == 0 ? kPaf : kHeat;
    if (stage == 1) {
        if (li < 3) return {128, 128, 3};
        if (li == 3) return {128, 512, 1};
        return {512, outc, 1};
    }
    if (li == 0) return {kCat, 128, 7};
    if (li < 5) return {128, 128, 7};
    if (li == 5) return {128, 128, 1};
    return {128, outc, 1};
}
// conv index in state_dict order: trunk 0..11, then branch 0 stages 1..6, then branch 1 stages 1..6
int conv_index(int stage, int branch, int li) {
    int idx = 12;
    for (int b = 0; b < 2; ++b)
        for (int s = 1; s <= 6; ++s) {
            if (b == branch && s == stage) return idx + li;
            idx += stage_num_layers(s);
        }
    return -1;
}
constexpr int kNumConvs = 12 + 2 * (5 + 5 * 7);   // 92
ConvSpec conv_spec(int ci) {
    if (ci < 12) return kTrunk[ci];
    int idx = 12;
    for (int b = 0; b < 2; ++b)
        for (int s = 1; s <= 6; ++s) {
            const int nl = stage_num_layers(s);
            if (ci < idx + nl) return stage_layer(s, b, ci - idx);
            idx += nl;
        }
    return {0, 0, 0};
}
// physical channel of the bf16 concat buffer [paf 0..37, pad, heat 40..58, pad, feat 64..191] for reference
// concat channel c of torch.cat([paf, heat, feat], 1) (rtpose_vgg.py:165)
int cat_phys(int c) { return c < kPaf ? c : (c < kPaf + kHeat ? c + 2 : c + 7); }

uint16_t f2bf(float f) {
    uint32_t u;
    memcpy(&u, &f, 4);
    if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);
    u += 0x7fffu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
}

float bf2f(uint16_t b) {
    uint32_t u = (uint32_t)b << 16;
    float f;
    memcpy(&f, &u, 4);
    return f;
}

template <class T> struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    cudaError_t ensure(size_t count) {
        if (count <= n) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        n = 0;
        cudaError_t e = cudaMalloc(&p, count * sizeof(T));
        if (e == cudaSuccess) n = count;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
};

struct TcLayer {            // one grouped tensor-core launch
    int ks, cin_blocks, groups, n_tile, n_tiles, relu, pool;
    double macs_per_pixel = 0;    // algorithmic (unpadded) MACs per output pixel, all groups
    __nv_bfloat16* w = nullptr;   // [taps][groups*n_tiles*n_tile][cin_blocks*64]
    float* bias = nullptr;        // [groups*n_tiles*n_tile]
};

}  // namespace

struct b200pose_net {
    int device = 0, num_sms = 148;
    bool finalized = false;
    std::vector<std::vector<float>> host_w, host_b;   // per conv
    std::vector<bool> have;                            // per tensor
    float* d_w[kNumConvs] = {};                        // fp32 OIHW (parity mode, conv1_1)
    float* d_b[kNumConvs] = {};
    // tensor-core layers: trunk 1..11 -> tc[0..10]; stage 1: tc[11..15]; stage t>=2: tc[16 + (t-2)*7 + li]
    std::vector<TcLayer> tc;
    // ---- plan (depends on n, H, W)
    int pn = 0, pH = 0, pW = 0, pmode = -1;
    std::vector<ConvTcArgs> plan;
    std::vector<double> plan_flops;   // algorithmic FLOPs per launch of `plan`
    bool plan_split = false;          // the plan was built for the split-precision (bf16x3) mode
    // Plans of other (n, H, W, mode) keys are kept, so that alternating shapes (multi-scale, mixed frame sizes) do not
    // re-encode 51 tensor maps and synchronise the stream.  An entry is valid while the activation buffers it points
    // into have not been reallocated.  B200POSE_PLAN_CACHE=0 (read when the net is created) turns it off.
    struct PlanEntry {
        int n, H, W, mode;
        bool ragged;
        bool split;
        std::vector<ConvTcArgs> plan;
        std::vector<double> flops;
        std::vector<const void*> buffers;
    };
    bool plan_cache_on = true;
    bool conv_pdl = true;             // programmatic dependent launch between the layers of small-batch plans (B200POSE_CONV_PDL=0: never)
    bool conv_narrow = true;          // 8 x 16 pixel tiles for layers that fill less than half of the SMs (B200POSE_CONV_NARROW=0: never)
    bool conv_pair = true;            // tcgen05 cta_group::2 CTA pairs for the N >= 64 layers (B200POSE_CONV_PAIR=0: single CTAs)
    // The 52 launches of a forward pass are captured at the second use of a (shape, mode, input pointer) into a CUDA graph and replayed
    // (B200POSE_GRAPH=0: plain launches).  Graphs embed the tensor maps, i.e. buffer addresses: every plan build drops them.
    // Capture needs a real stream: calls on the legacy default stream (0) launch directly.
    struct GraphKey {
        int n, H, W, mode, in_u8;
        const void* in;
        bool operator<(const GraphKey& o) const {
            if (n != o.n) return n < o.n;
            if (H != o.H) return H < o.H;
            if (W != o.W) return W < o.W;
            if (mode != o.mode) return mode < o.mode;
            if (in_u8 != o.in_u8) return in_u8 < o.in_u8;
            return in < o.in;
        }
    };
    bool use_graph = true;
    std::map<GraphKey, cudaGraphExec_t> graphs;
    std::set<GraphKey> graph_seen;    // a key is captured at its SECOND use: callers that pass a fresh pointer every time never pay a capture
    int kn = 0, kH = 0, kW = 0, kmode = -1;      // key of the plan currently held in `plan`
    bool kragged = false, pragged = false;       // ... and whether it (resp. the last bf16 forward's plan) is a ragged plan
    std::vector<PlanEntry> plan_cache;
    DevBuf<__nv_bfloat16> t1, t2, t3, t4, t5a, t5b, t6, t7, t8, t9, cat, bra, brb, br512;
    // residual ("lo") planes of the same buffers, split-precision mode only
    DevBuf<__nv_bfloat16> l1, l2, l3, l4, l5a, l5b, l6, l7, l8, l9, lcat, lbra, lbrb, lbr512;
    std::map<const void*, __nv_bfloat16*> lo_of;
    DevBuf<float> in_stage, out_f32[12];
    // fp32 parity buffers
    DevBuf<float> f_a, f_b, f_cat, f_x, f_y, f_in, f_u8;
    cudaStream_t own_stream = nullptr;
    const void* last_in = nullptr;    // device pointer of the last forward's input (profiling hook)
    int last_in_u8 = 0;
    DevBuf<unsigned char> in_stage_u8;
    int preprocess = 1;                // normalisation fused into the uint8 entry points (preprocess_core.h; 1 = rtpose)
    DevBuf<unsigned char> raw_stage;   // raw (un-resized) frames of b200pose_*crop* / b200pose_infer_raw_u8
    // Ragged batches: full-resolution (h, w) of every image of the call, uploaded on the caller's stream before its first
    // launch.  Allocated once at kRaggedCap entries: the ragged plans (their ConvTcArgs::ext) point into it.
    DevBuf<int2> ext;
    DevBuf<RaggedCrop> rcrop;          // per-frame crop geometry of b200pose_infer_raw_u8_ragged
};

struct b200pose_post {
    int device = 0;
    PostBuffers pb{};
    DevBuf<float> d_heat, d_paf;
    DevBuf<float> tta_in, tta_out;   // b200pose_flip_merge staging for host pointers
    // Results are copied to pinned host memory by the run itself (second stream, right after the assembly) into one
    // of two slots selected by the run's parity, so the host can fetch run i while run i+1 is in flight.
    cudaStream_t s2 = nullptr;
    cudaEvent_t ev_limbs = nullptr, ev_asm = nullptr, ev_fetch[2] = {nullptr, nullptr};
    long runs = 0;                  // runs submitted so far; ticket of the latest = runs - 1
    int slot_n[2] = {0, 0};
    int* hp_nh[2] = {nullptr, nullptr};
    int* hp_status[2] = {nullptr, nullptr};
    int* hp_counts[2] = {nullptr, nullptr};
    float* hp_humans[2] = {nullptr, nullptr};
    int cur = 0;                    // slot the getters read
    long cur_ticket = -1;
    std::vector<float> h_px_s;
    std::vector<int> h_px, h_py;
    int hw_h = 0, hw_w = 0;
    // Peaks / limbs / assembly of run i all run on the second stream from a private copy of the maps (15 MB at batch 32),
    // so that the caller's stream is free for the convolutions of run i+1: the small kernels (peaks, assembly) co-reside
    // with the conv CTAs and the limbs blocks fill the SMs the conv launches leave idle in their last wave
    // (measured on B200, batch 32: 14.23 -> 13.52 ms per step device-resident, 14.26 -> 13.15 end to end;
    // profiles/r02_variants.txt).  B200POSE_POST_OVERLAP=0 keeps everything on the caller's stream.
    bool overlap = true;
    DevBuf<float> ov_maps[2];                       // [heat | paf] copies, slot = run parity
    DevBuf<int2> dims[2];                           // ragged runs: low-res (h, w) per image, slot = run parity
    cudaEvent_t ev_maps = nullptr, ev_ld[2] = {nullptr, nullptr};   // maps copied (st) / limbs done with a slot (s2)
    bool have_ld[2] = {false, false};
};

namespace {

int pack_tc_layer(b200pose_net* net, TcLayer& L, const std::vector<int>& conv_ids /*per group*/, int n_tile,
                  bool cat_input, int ks, int relu, int pool) {
    const int groups = (int)conv_ids.size();
    const ConvSpec sp = conv_spec(conv_ids[0]);
    const int cin_pad = cat_input ? 192 : sp.cin;
    const int cout_pad = ((sp.cout + n_tile - 1) / n_tile) * n_tile;
    L.ks = ks; L.cin_blocks = cin_pad / 64; L.groups = groups; L.n_tile = n_tile; L.n_tiles = cout_pad / n_tile;
    L.relu = relu; L.pool = pool;
    const int taps = ks * ks, rows = groups * cout_pad;
    L.macs_per_pixel = 0;
    for (int g = 0; g < groups; ++g) L.macs_per_pixel += (double)conv_spec(conv_ids[g]).cin * conv_spec(conv_ids[g]).cout * taps;
    // [hi taps | lo taps]: bf16(w) and the residual bf16(w - hi) (used by the split-precision mode only)
    std::vector<uint16_t> w((size_t)2 * taps * rows * cin_pad, 0);
    std::vector<float> b((size_t)rows, 0.f);
    for (int g = 0; g < groups; ++g) {
        const ConvSpec s = conv_spec(conv_ids[g]);
        const std::vector<float>& hw = net->host_w[conv_ids[g]];
        const std::vector<float>& hb = net->host_b[conv_ids[g]];
        for (int o = 0; o < s.cout; ++o) {
            b[g * cout_pad + o] = hb[o];
            for (int c = 0; c < s.cin; ++c) {
                const int pc = cat_input ? cat_phys(c) : c;
                for (int t = 0; t < taps; ++t) {
                    const float wf = hw[((size_t)o * s.cin + c) * taps + t];
                    const uint16_t hi = f2bf(wf);
                    w[((size_t)t * rows + g * cout_pad + o) * cin_pad + pc] = hi;
                    w[((size_t)(taps + t) * rows + g * cout_pad + o) * cin_pad + pc] = f2bf(wf - bf2f(hi));
                }
            }
        }
    }
    CU(cudaMalloc(&L.w, w.size() * 2));
    CU(cudaMalloc(&L.bias, b.size() * 4));
    CU(cudaMemcpy(L.w, w.data(), w.size() * 2, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(L.bias, b.data(), b.size() * 4, cudaMemcpyHostToDevice));
    return 0;
}

// Small-batch plans: the 46 x 46 stage layers would fill less than half of the SMs with 16 x 16 tiles.  Their launches are the
// launch-bound part of the product: they are chained by PDL and replayed as a CUDA graph; the large plans are GPU-bound and
// get neither (PDL measured -2 % there; a capture only adds a CPU hiccup).
bool small_plan(const b200pose_net* net, int n, int H, int W) {
    return 2 * n * ((H / 8 + kTileH - 1) / kTileH) * ((W / 8 + kTileW - 1) / kTileW) * 2 <= net->num_sms;
}

int add_plan(b200pose_net* net, const TcLayer& L, int n, int H, int W, const __nv_bfloat16* in, int in_cstride,
             int in_ch_base, int in_group_stride, __nv_bfloat16* out, int out_cstride, int off0, int off1, int store0,
             int store1, float* f32_0, float* f32_1, int f32c0, int f32c1) {
    ConvTcArgs a;
    memset(&a, 0, sizeof(a));
    a.n_img = n; a.H = H; a.W = W; a.ksize = L.ks; a.cin_blocks = L.cin_blocks;
    a.in_ch_base = in_ch_base; a.in_ch_group_stride = in_group_stride; a.groups = L.groups;
    a.n_tile = L.n_tile; a.n_tiles = L.n_tiles; a.bias = L.bias; a.relu = L.relu; a.pool = L.pool;
    {   // small batches: while the layer's CTAs fill less than half of the SMs, halve the work per CTA - 128-wide n-tiles
        // become 64-wide, then the 16 x 16 pixel tile becomes 8 x 16 (one UMMA sub-tile), then 64-wide n-tiles become
        // 32-wide (the weight layout does not depend on the n-tile).  B200POSE_CONV_NARROW=0 keeps the 16 x 16 tiles.
        auto ctas = [&](int narrow, int n_tiles) {
            const int pix = n * ((H + kTileH - 1) / kTileH) * ((W + (narrow ? 8 : kTileW) - 1) / (narrow ? 8 : kTileW));
            return (net->conv_pair ? (pix + 1) / 2 * 2 : pix) * L.groups * n_tiles;
        };
        if (L.n_tile == 128 && 2 * ctas(0, a.n_tiles) <= net->num_sms) { a.n_tile = 64; a.n_tiles = L.n_tiles * 2; }
        if (net->conv_narrow && 2 * ctas(0, a.n_tiles) <= net->num_sms) {
            a.narrow = 1;
            if (a.n_tile == 64 && net->conv_pair && 2 * ctas(1, a.n_tiles) <= net->num_sms) { a.n_tile = 32; a.n_tiles *= 2; }
        }
    }
    if (net->plan_split) {     // bf16x3: K-chunked accumulation, one 32-column chunk per epilogue warp, so N <= 64
        a.chunk = 1;
        if (a.n_tile > 64) { a.n_tile = 64; a.n_tiles = L.n_tiles * (L.n_tile / 64); }
    }
    a.out = out; a.out_cstride = out_cstride;
    a.out_ch_off[0] = off0; a.out_ch_off[1] = off1;
    a.store_ch[0] = store0; a.store_ch[1] = store1;
    a.out_f32[0] = f32_0; a.out_f32[1] = f32_1;
    a.f32_ch[0] = f32c0; a.f32_ch[1] = f32c1;
    a.use_base_offset = 0;
    a.pair = (net->conv_pair && a.n_tile % 32 == 0) ? 1 : 0;    // heads (N = 48) stay single-CTA
    // small batches (the 46 x 46 layers fill less than half of the SMs with 16 x 16 tiles): chain the layers with programmatic
    // dependent launches; the first tensor-core layer follows conv1_1, which does not signal
    a.pdl = (net->conv_pdl && !net->plan.empty() && small_plan(net, n, H, W)) ? 1 : 0;
    const __nv_bfloat16* in_lo = nullptr;
    if (net->plan_split) {
        a.split = 1;
        in_lo = net->lo_of.at(in);
        a.out_lo = net->lo_of.at(out);
    }
    cudaError_t e = conv_tc_make_maps(a, in, in_cstride, L.w, in_lo);
    if (e != cudaSuccess) return fail("conv_tc_make_maps failed: %s", cudaGetErrorString(e));
    net->plan.push_back(a);
    net->plan_flops.push_back(2.0 * n * H * W * L.macs_per_pixel);
    return 0;
}

int build_plan_bf16(b200pose_net* net, int n, int H, int W, bool split, bool ragged, cudaStream_t st) {
    const size_t px1 = (size_t)n * H * W, px2 = px1 / 4, px4 = px1 / 16, px8 = px1 / 64;
    const int h = H / 8, w = W / 8;
    CU(net->t1.ensure(px1 * 64)); CU(net->t2.ensure(px2 * 64)); CU(net->t3.ensure(px2 * 128));
    CU(net->t4.ensure(px4 * 128)); CU(net->t5a.ensure(px4 * 256)); CU(net->t5b.ensure(px4 * 256));
    CU(net->t6.ensure(px8 * 256)); CU(net->t7.ensure(px8 * 512)); CU(net->t8.ensure(px8 * 512));
    CU(net->t9.ensure(px8 * 256)); CU(net->cat.ensure(px8 * 192)); CU(net->bra.ensure(px8 * 256));
    CU(net->brb.ensure(px8 * 256)); CU(net->br512.ensure(px8 * 1024));
    // pad lanes of the concat buffer must read as zero; on the caller's stream (a non-blocking stream is not ordered
    // against the legacy default stream a plain cudaMemset would use)
    CU(cudaMemsetAsync(net->cat.p, 0, px8 * 192 * 2, st));
    net->plan_split = split;
    net->lo_of.clear();
    if (split) {
        CU(net->l1.ensure(px1 * 64)); CU(net->l2.ensure(px2 * 64)); CU(net->l3.ensure(px2 * 128));
        CU(net->l4.ensure(px4 * 128)); CU(net->l5a.ensure(px4 * 256)); CU(net->l5b.ensure(px4 * 256));
        CU(net->l6.ensure(px8 * 256)); CU(net->l7.ensure(px8 * 512)); CU(net->l8.ensure(px8 * 512));
        CU(net->l9.ensure(px8 * 256)); CU(net->lcat.ensure(px8 * 192)); CU(net->lbra.ensure(px8 * 256));
        CU(net->lbrb.ensure(px8 * 256)); CU(net->lbr512.ensure(px8 * 1024));
        CU(cudaMemsetAsync(net->lcat.p, 0, px8 * 192 * 2, st));
        DevBuf<__nv_bfloat16>* hi[] = {&net->t1, &net->t2, &net->t3, &net->t4, &net->t5a, &net->t5b, &net->t6, &net->t7,
                                       &net->t8, &net->t9, &net->cat, &net->bra, &net->brb, &net->br512};
        DevBuf<__nv_bfloat16>* lo[] = {&net->l1, &net->l2, &net->l3, &net->l4, &net->l5a, &net->l5b, &net->l6, &net->l7,
                                       &net->l8, &net->l9, &net->lcat, &net->lbra, &net->lbrb, &net->lbr512};
        for (int i = 0; i < 14; ++i) net->lo_of[hi[i]->p] = lo[i]->p;
    }
    for (int i = 0; i < 12; ++i) CU(net->out_f32[i].ensure(px8 * (i % 2 == 0 ? kPaf : kHeat)));
    net->plan.clear();
    net->plan_flops.clear();
    const std::vector<TcLayer>& T = net->tc;
#define PLAN(...) do { if (add_plan(net, __VA_ARGS__)) return 1; } while (0)
    // trunk (conv1_1 runs on CUDA cores before the plan)
    PLAN(T[0], n, H, W, net->t1.p, 64, 0, 0, net->t2.p, 64, 0, 0, 64, 0, nullptr, nullptr, 0, 0);              // conv1_2+pool
    PLAN(T[1], n, H / 2, W / 2, net->t2.p, 64, 0, 0, net->t3.p, 128, 0, 0, 128, 0, nullptr, nullptr, 0, 0);    // conv2_1
    PLAN(T[2], n, H / 2, W / 2, net->t3.p, 128, 0, 0, net->t4.p, 128, 0, 0, 128, 0, nullptr, nullptr, 0, 0);   // conv2_2+pool
    PLAN(T[3], n, H / 4, W / 4, net->t4.p, 128, 0, 0, net->t5a.p, 256, 0, 0, 128, 0, nullptr, nullptr, 0, 0);  // conv3_1
    PLAN(T[4], n, H / 4, W / 4, net->t5a.p, 256, 0, 0, net->t5b.p, 256, 0, 0, 128, 0, nullptr, nullptr, 0, 0); // conv3_2
    PLAN(T[5], n, H / 4, W / 4, net->t5b.p, 256, 0, 0, net->t5a.p, 256, 0, 0, 128, 0, nullptr, nullptr, 0, 0); // conv3_3
    PLAN(T[6], n, H / 4, W / 4, net->t5a.p, 256, 0, 0, net->t6.p, 256, 0, 0, 128, 0, nullptr, nullptr, 0, 0);  // conv3_4+pool
    PLAN(T[7], n, h, w, net->t6.p, 256, 0, 0, net->t7.p, 512, 0, 0, 128, 0, nullptr, nullptr, 0, 0);            // conv4_1
    PLAN(T[8], n, h, w, net->t7.p, 512, 0, 0, net->t8.p, 512, 0, 0, 128, 0, nullptr, nullptr, 0, 0);            // conv4_2
    PLAN(T[9], n, h, w, net->t8.p, 512, 0, 0, net->t9.p, 256, 0, 0, 128, 0, nullptr, nullptr, 0, 0);            // conv4_3_CPM
    PLAN(T[10], n, h, w, net->t9.p, 256, 0, 0, net->cat.p, 192, 64, 0, 128, 0, nullptr, nullptr, 0, 0);         // conv4_4_CPM -> feat slice
    // stage 1 (both branches grouped)
    PLAN(T[11], n, h, w, net->cat.p, 192, 64, 0, net->bra.p, 256, 0, 128, 128, 128, nullptr, nullptr, 0, 0);
    PLAN(T[12], n, h, w, net->bra.p, 256, 0, 128, net->brb.p, 256, 0, 128, 128, 128, nullptr, nullptr, 0, 0);
    PLAN(T[13], n, h, w, net->brb.p, 256, 0, 128, net->bra.p, 256, 0, 128, 128, 128, nullptr, nullptr, 0, 0);
    PLAN(T[14], n, h, w, net->bra.p, 256, 0, 128, net->br512.p, 1024, 0, 512, 128, 128, nullptr, nullptr, 0, 0);
    PLAN(T[15], n, h, w, net->br512.p, 1024, 0, 512, net->cat.p, 192, 0, 40, 40, 24, net->out_f32[0].p,
         net->out_f32[1].p, kPaf, kHeat);
    for (int s = 2; s <= 6; ++s) {
        const int b0 = 16 + (s - 2) * 7;
        PLAN(T[b0 + 0], n, h, w, net->cat.p, 192, 0, 0, net->bra.p, 256, 0, 128, 128, 128, nullptr, nullptr, 0, 0);
        PLAN(T[b0 + 1], n, h, w, net->bra.p, 256, 0, 128, net->brb.p, 256, 0, 128, 128, 128, nullptr, nullptr, 0, 0);
        PLAN(T[b0 + 2], n, h, w, net->brb.p, 256, 0, 128, net->bra.p, 256, 0, 128, 128, 128, nullptr, nullptr, 0, 0);
        PLAN(T[b0 + 3], n, h, w, net->bra.p, 256, 0, 128, net->brb.p, 256, 0, 128, 128, 128, nullptr, nullptr, 0, 0);
        PLAN(T[b0 + 4], n, h, w, net->brb.p, 256, 0, 128, net->bra.p, 256, 0, 128, 128, 128, nullptr, nullptr, 0, 0);
        PLAN(T[b0 + 5], n, h, w, net->bra.p, 256, 0, 128, net->brb.p, 256, 0, 128, 128, 128, nullptr, nullptr, 0, 0);
        PLAN(T[b0 + 6], n, h, w, net->brb.p, 256, 0, 128, net->cat.p, 192, 0, 40, 40, 24,
             net->out_f32[2 * (s - 1)].p, net->out_f32[2 * (s - 1) + 1].p, kPaf, kHeat);
    }
#undef PLAN
    if (ragged)      // every layer masks by the images' extents at its input resolution H >> ext_shift
        for (ConvTcArgs& a : net->plan) {
            a.ext = net->ext.p;
            a.ext_shift = 0;
            while ((H >> a.ext_shift) > a.H) ++a.ext_shift;
        }
    return 0;
}

std::vector<const void*> plan_buffers(const b200pose_net* net) {
    std::vector<const void*> v = {net->t1.p, net->t2.p, net->t3.p, net->t4.p, net->t5a.p, net->t5b.p, net->t6.p, net->t7.p,
                                  net->t8.p, net->t9.p, net->cat.p, net->bra.p, net->brb.p, net->br512.p,
                                  net->l1.p, net->l2.p, net->l3.p, net->l4.p, net->l5a.p, net->l5b.p, net->l6.p, net->l7.p,
                                  net->l8.p, net->l9.p, net->lcat.p, net->lbra.p, net->lbrb.p, net->lbr512.p};
    for (const auto& b : net->out_f32) v.push_back(b.p);
    return v;
}

// plan cache (experiment): returns true when a valid plan for the key was swapped into net->plan
bool plan_cache_swap(b200pose_net* net, int n, int H, int W, int want, bool ragged) {
    if (net->kmode >= 0 && !net->plan.empty()) {      // stash the plan we hold
        b200pose_net::PlanEntry* slot = nullptr;
        for (auto& e : net->plan_cache)
            if (e.n == net->kn && e.H == net->kH && e.W == net->kW && e.mode == net->kmode && e.ragged == net->kragged) slot = &e;
        if (!slot) {
            if (net->plan_cache.size() >= 32) net->plan_cache.erase(net->plan_cache.begin());
            net->plan_cache.emplace_back();
            slot = &net->plan_cache.back();
        }
        slot->n = net->kn; slot->H = net->kH; slot->W = net->kW; slot->mode = net->kmode; slot->ragged = net->kragged;
        slot->split = net->plan_split;
        slot->plan.swap(net->plan);
        slot->flops.swap(net->plan_flops);
        slot->buffers = plan_buffers(net);
        net->plan.clear(); net->plan_flops.clear();
        net->kmode = -1;
    }
    for (auto& e : net->plan_cache)
        if (e.n == n && e.H == H && e.W == W && e.mode == want && e.ragged == ragged && !e.plan.empty() &&
            e.buffers == plan_buffers(net)) {
            net->plan.swap(e.plan);
            net->plan_flops.swap(e.flops);
            net->plan_split = e.split;
            net->kn = n; net->kH = H; net->kW = W; net->kmode = want; net->kragged = ragged;
            return true;
        }
    return false;
}

void drop_graphs(b200pose_net* net) {
    for (auto& kv : net->graphs) cudaGraphExecDestroy(kv.second);
    net->graphs.clear();
    net->graph_seen.clear();
}

int launch_forward_bf16(b200pose_net* net, const void* d_in, int in_u8, int n, int H, int W, cudaStream_t st, bool split,
                        const int2* ext = nullptr) {
    CU(conv_first_launch(d_in, in_u8, net->d_w[0], net->d_b[0], net->t1.p, split ? net->l1.p : nullptr, n, H, W, st, ext));
    for (const ConvTcArgs& a : net->plan) CU(conv_tc_launch(a, net->num_sms, st));
    return 0;
}

// ragged: the images' extents are in net->ext (the plan masks by them); such calls always launch directly, never as a graph
int forward_bf16(b200pose_net* net, const void* d_in, int in_u8, int n, int H, int W, cudaStream_t st, bool split,
                 bool ragged = false) {
    const int want = split ? B200POSE_MODE_BF16X3 : B200POSE_MODE_BF16;
    if (net->pn != n || net->pH != H || net->pW != W || net->pmode != want || net->pragged != ragged) {
        if (!(net->plan_cache_on && plan_cache_swap(net, n, H, W, want, ragged))) {
            CU(cudaStreamSynchronize(st));
            drop_graphs(net);                   // the buffers the captured tensor maps point into may move
            if (build_plan_bf16(net, n, H, W, split, ragged, st)) return 1;
            net->kn = n; net->kH = H; net->kW = W; net->kmode = want; net->kragged = ragged;
        }
        net->pn = n; net->pH = H; net->pW = W; net->pmode = want; net->pragged = ragged;
    }
    const long launches = 1 + (long)net->plan.size();
    if (ragged) {
        if (launch_forward_bf16(net, d_in, in_u8, n, H, W, st, split, net->ext.p)) return 1;
        g_launches += launches;
        return 0;
    }
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (net->use_graph && small_plan(net, n, H, W) && st != nullptr && cudaStreamIsCapturing(st, &cap) == cudaSuccess &&
        cap == cudaStreamCaptureStatusNone) {
        const b200pose_net::GraphKey key{n, H, W, want, in_u8, d_in};
        auto it = net->graphs.find(key);
        if (it == net->graphs.end() && net->graph_seen.insert(key).second) {      // first sight: plain launches
            if (net->graph_seen.size() > 4096) net->graph_seen.clear();
            if (launch_forward_bf16(net, d_in, in_u8, n, H, W, st, split)) return 1;
            g_launches += launches;
            return 0;
        }
        if (it == net->graphs.end()) {
            if (net->graphs.size() >= 64) drop_graphs(net);
            cudaGraph_t graph = nullptr;
            cudaGraphExec_t exec = nullptr;
            CU(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
            const int rc = launch_forward_bf16(net, d_in, in_u8, n, H, W, st, split);
            cudaError_t e = cudaStreamEndCapture(st, &graph);
            if (rc == 0 && e == cudaSuccess) e = cudaGraphInstantiate(&exec, graph, 0);
            if (graph) cudaGraphDestroy(graph);
            if (rc != 0 || e != cudaSuccess) {      // no graph (e.g. a launch attribute the capture refuses): plain launches from now on
                cudaGetLastError();
                fprintf(stderr, "[b200pose] CUDA graph capture of the forward pass failed (%s): launching directly\n",
                        rc ? b200pose_last_error() : cudaGetErrorString(e));
                net->use_graph = false;
                if (launch_forward_bf16(net, d_in, in_u8, n, H, W, st, split)) return 1;
                g_launches += launches;
                return 0;
            }
            it = net->graphs.emplace(key, exec).first;
        }
        CU(cudaGraphLaunch(it->second, st));
        g_launches += launches;
        return 0;
    }
    if (launch_forward_bf16(net, d_in, in_u8, n, H, W, st, split)) return 1;
    g_launches += launches;
    return 0;
}

int forward_fp32(b200pose_net* net, const float* d_in, int n, int H, int W, cudaStream_t st, const int2* ext = nullptr) {
    const size_t px1 = (size_t)n * H * W;
    const int h = H / 8, w = W / 8;
    const size_t px8 = (size_t)n * h * w;
    CU(net->f_in.ensure(px1 * 3));
    CU(net->f_a.ensure(px1 * 64)); CU(net->f_b.ensure(px1 * 64));
    CU(net->f_cat.ensure(px8 * kCat)); CU(net->f_x.ensure(px8 * 512)); CU(net->f_y.ensure(px8 * 512));
    for (int i = 0; i < 12; ++i) CU(net->out_f32[i].ensure(px8 * (i % 2 == 0 ? kPaf : kHeat)));
    net->pmode = B200POSE_MODE_FP32;   // invalidates the bf16 plan's claim on out_f32 (same buffers, same sizes)
    CU(nchw_to_nhwc_f32_launch(d_in, net->f_in.p, n, 3, H, W, 3, 0, st));
    ++g_launches;
    const float* cur = net->f_in.p;
    int cur_c = 3, ch = H, cw = W;
    float* ping = net->f_a.p;
    float* pong = net->f_b.p;
    auto conv = [&](int ci, const float* in, int in_cs, int in_off, float* out, int out_cs, int out_off, int hh, int ww,
                    int relu, float* nchw) -> int {
        const ConvSpec s = conv_spec(ci);
        ConvF32Args a;
        a.in = in; a.in_cstride = in_cs; a.in_ch_off = in_off; a.w = net->d_w[ci]; a.bias = net->d_b[ci];
        a.out = out; a.out_cstride = out_cs; a.out_ch_off = out_off; a.out_nchw = nchw;
        a.n_img = n; a.H = hh; a.W = ww; a.cin = s.cin; a.cout = s.cout; a.ks = s.ks; a.relu = relu;
        a.ext = ext; a.ext_shift = 0;
        while ((H >> a.ext_shift) > hh) ++a.ext_shift;
        CU(conv_f32_launch(a, st));
        ++g_launches;
        return 0;
    };
    for (int i = 0; i < 12; ++i) {
        const ConvSpec s = kTrunk[i];
        const bool last = (i == 11);
        float* dst = last ? net->f_cat.p : ping;
        if (conv(i, cur, cur_c, 0, dst, last ? kCat : s.cout, last ? kPaf + kHeat : 0, ch, cw, 1, nullptr)) return 1;
        cur = dst; cur_c = s.cout;
        std::swap(ping, pong);
        if (kPoolAfter[i]) {
            CU(maxpool_f32_launch(cur, ping, n, ch, cw, cur_c, st));
            ++g_launches;
            cur = ping; ch /= 2; cw /= 2;
            std::swap(ping, pong);
        }
    }
    for (int s = 1; s <= 6; ++s)
        for (int b = 0; b < 2; ++b) {
            const int nl = stage_num_layers(s);
            const float* in = net->f_cat.p;
            int in_cs = kCat, in_off = (s == 1) ? kPaf + kHeat : 0;
            float* bufs[2] = {net->f_x.p, net->f_y.p};
            for (int li = 0; li < nl; ++li) {
                const ConvSpec sp = stage_layer(s, b, li);
                const bool lastl = (li == nl - 1);
                float* nchw = lastl ? net->out_f32[2 * (s - 1) + b].p : nullptr;
                // last layer output goes to a scratch slice; the concat for the next stage is written after both
                // branches are done (the other branch still reads f_cat)
                float* dst = bufs[li & 1];
                if (conv(conv_index(s, b, li), in, in_cs, in_off, dst, sp.cout, 0, h, w, lastl ? 0 : 1, nchw)) return 1;
                in = dst; in_cs = sp.cout; in_off = 0;
            }
            if (b == 1 && s < 6) {
                CU(nchw_to_nhwc_f32_launch(net->out_f32[2 * (s - 1)].p, net->f_cat.p, n, kPaf, h, w, kCat, 0, st));
                CU(nchw_to_nhwc_f32_launch(net->out_f32[2 * (s - 1) + 1].p, net->f_cat.p, n, kHeat, h, w, kCat, kPaf, st));
                g_launches += 2;
            }
        }
    return 0;
}

}  // namespace

extern "C" {

const char* b200pose_last_error(void) { return g_err.c_str(); }
int b200pose_version(void) { return 100; }
long b200pose_launch_count(void) { return g_launches.load(); }

int b200pose_net_tensor_shape(int index, long dims[4]) {
    if (index < 0 || index >= B200POSE_NUM_TENSORS) return -1;
    const ConvSpec s = conv_spec(index / 2);
    if (index % 2 == 0) { dims[0] = s.cout; dims[1] = s.cin; dims[2] = s.ks; dims[3] = s.ks; return 4; }
    dims[0] = s.cout;
    return 1;
}

int b200pose_net_create(b200pose_net** out, int cuda_device) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail("b200pose: no CUDA device available (this library has no CPU fallback)");
    CU(cudaSetDevice(cuda_device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, cuda_device));
    if (prop.major != 10) return fail("b200pose: built for sm_100a (B200); device is sm_%d%d", prop.major, prop.minor);
    b200pose_net* net = new b200pose_net();
    net->device = cuda_device;
    net->num_sms = prop.multiProcessorCount;
    net->host_w.resize(kNumConvs);
    net->host_b.resize(kNumConvs);
    net->have.assign(B200POSE_NUM_TENSORS, false);
    const char* pc = getenv("B200POSE_PLAN_CACHE");
    net->plan_cache_on = !(pc && pc[0] == '0');
    const char* cp = getenv("B200POSE_CONV_PAIR");
    net->conv_pair = !(cp && cp[0] == '0');
    const char* nw = getenv("B200POSE_CONV_NARROW");
    net->conv_narrow = !(nw && nw[0] == '0');
    const char* pd = getenv("B200POSE_CONV_PDL");
    net->conv_pdl = !(pd && pd[0] == '0');
    const char* gr = getenv("B200POSE_GRAPH");
    net->use_graph = !(gr && gr[0] == '0');
    *out = net;
    return 0;
}

void b200pose_net_destroy(b200pose_net* net) {
    if (!net) return;
    cudaSetDevice(net->device);
    drop_graphs(net);
    for (int i = 0; i < kNumConvs; ++i) { if (net->d_w[i]) cudaFree(net->d_w[i]); if (net->d_b[i]) cudaFree(net->d_b[i]); }
    for (TcLayer& L : net->tc) { if (L.w) cudaFree(L.w); if (L.bias) cudaFree(L.bias); }
    DevBuf<__nv_bfloat16>* bb[] = {&net->t1, &net->t2, &net->t3, &net->t4, &net->t5a, &net->t5b, &net->t6,
                                   &net->t7, &net->t8, &net->t9, &net->cat, &net->bra, &net->brb, &net->br512};
    for (auto* b : bb) b->release();
    DevBuf<__nv_bfloat16>* lb[] = {&net->l1, &net->l2, &net->l3, &net->l4, &net->l5a, &net->l5b, &net->l6,
                                   &net->l7, &net->l8, &net->l9, &net->lcat, &net->lbra, &net->lbrb, &net->lbr512};
    for (auto* b : lb) b->release();
    DevBuf<float>* fb[] = {&net->in_stage, &net->f_a, &net->f_b, &net->f_cat, &net->f_x, &net->f_y, &net->f_in, &net->f_u8};
    net->in_stage_u8.release();
    net->raw_stage.release();
    net->ext.release();
    net->rcrop.release();
    for (auto* b : fb) b->release();
    for (auto& b : net->out_f32) b.release();
    delete net;
}

int b200pose_net_set_tensor(b200pose_net* net, int index, const float* host_data, long count) {
    if (!net || !host_data) return fail("set_tensor: null pointer");
    long dims[4];
    const int nd = b200pose_net_tensor_shape(index, dims);
    if (nd < 0) return fail("tensor index %d out of range", index);
    long expect = 1;
    for (int i = 0; i < nd; ++i) expect *= dims[i];
    if (count != expect) return fail("tensor %d: got %ld elements, expected %ld", index, count, expect);
    std::vector<float>& dst = (index % 2 == 0) ? net->host_w[index / 2] : net->host_b[index / 2];
    dst.assign(host_data, host_data + count);
    net->have[index] = true;
    net->finalized = false;
    return 0;
}

int b200pose_net_finalize(b200pose_net* net) {
    if (!net) return fail("null net");
    CU(cudaSetDevice(net->device));
    for (int i = 0; i < B200POSE_NUM_TENSORS; ++i)
        if (!net->have[i]) return fail("state_dict tensor %d was never set", i);
    for (int i = 0; i < kNumConvs; ++i) {
        if (net->d_w[i]) cudaFree(net->d_w[i]);
        if (net->d_b[i]) cudaFree(net->d_b[i]);
        CU(cudaMalloc(&net->d_w[i], net->host_w[i].size() * 4));
        CU(cudaMalloc(&net->d_b[i], net->host_b[i].size() * 4));
        CU(cudaMemcpy(net->d_w[i], net->host_w[i].data(), net->host_w[i].size() * 4, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(net->d_b[i], net->host_b[i].data(), net->host_b[i].size() * 4, cudaMemcpyHostToDevice));
    }
    for (TcLayer& L : net->tc) { if (L.w) cudaFree(L.w); if (L.bias) cudaFree(L.bias); }
    net->tc.assign(16 + 5 * 7, TcLayer());
    for (int i = 1; i < 12; ++i) {
        const ConvSpec s = kTrunk[i];
        if (pack_tc_layer(net, net->tc[i - 1], {i}, s.cout < 128 ? s.cout : 128, false, 3, 1, kPoolAfter[i])) return 1;
    }
    for (int li = 0; li < 5; ++li) {
        const ConvSpec s = stage_layer(1, 0, li);
        if (pack_tc_layer(net, net->tc[11 + li], {conv_index(1, 0, li), conv_index(1, 1, li)}, li == 4 ? 48 : 128, false,
                          s.ks, li != 4, 0))
            return 1;
    }
    for (int st = 2; st <= 6; ++st)
        for (int li = 0; li < 7; ++li) {
            const ConvSpec s = stage_layer(st, 0, li);
            if (pack_tc_layer(net, net->tc[16 + (st - 2) * 7 + li], {conv_index(st, 0, li), conv_index(st, 1, li)},
                              li == 6 ? 48 : 128, li == 0, s.ks, li != 6, 0))
                return 1;
        }
    net->pn = net->pH = net->pW = 0;
    net->pmode = -1;
    drop_graphs(net);
    net->plan_cache.clear();      // cached plans point at the previous packed weights
    net->plan.clear(); net->plan_flops.clear();
    net->kmode = -1;
    net->finalized = true;
    return 0;
}

// Extents of a ragged call: n host (h, w) pairs, each a multiple of 8 in [8, H] x [8, W].
static int ragged_check(int n, int H, int W, const int* ext_h, const int* ext_w) {
    if (!ext_h || !ext_w) return fail("ragged: null extent array");
    if (n < 1 || n > kRaggedCap) return fail("ragged: batch %d outside [1, %d]", n, kRaggedCap);
    for (int i = 0; i < n; ++i)
        if (ext_h[i] < 8 || ext_w[i] < 8 || ext_h[i] % 8 || ext_w[i] % 8 || ext_h[i] > H || ext_w[i] > W)
            return fail("ragged: extent %d is %d x %d; extents must be multiples of 8 within the %d x %d canvas", i, ext_h[i],
                        ext_w[i], H, W);
    return 0;
}

// ext_h / ext_w (host, may be null): a ragged batch, see b200pose_net_forward_u8_ragged (uint8 input only).
static int net_forward_impl(b200pose_net* net, const void* input, int in_u8, int input_on_device, int n, int H, int W,
                            int mode, float* const* outputs, int outputs_on_device, cudaStream_t st, bool sync_host,
                            const int* ext_h = nullptr, const int* ext_w = nullptr) {
    if (!net || !net->finalized) return fail("net not finalized");
    if (n < 1 || H < 8 || W < 8 || (H % 8) || (W % 8)) return fail("input must be [n,3,H,W] with H, W multiples of 8");
    const bool ragged = ext_h != nullptr || ext_w != nullptr;
    if (ragged && !in_u8) return fail("ragged batches take uint8 frames");
    if (ragged && ragged_check(n, H, W, ext_h, ext_w)) return 1;
    CU(cudaSetDevice(net->device));
    if (ragged) {
        // stream-ordered after the previous call's launches, which may still read the extent array
        CU(net->ext.ensure(kRaggedCap));
        std::vector<int2> e(n);
        for (int i = 0; i < n; ++i) e[i] = make_int2(ext_h[i], ext_w[i]);
        CU(cudaMemcpyAsync(net->ext.p, e.data(), n * sizeof(int2), cudaMemcpyHostToDevice, st));
    }
    const int2* d_ext = ragged ? net->ext.p : nullptr;
    const void* d_in = input;
    const size_t elems = (size_t)n * 3 * H * W;
    if (!input_on_device) {
        if (in_u8) {
            CU(net->in_stage_u8.ensure(elems));
            CU(cudaMemcpyAsync(net->in_stage_u8.p, input, elems, cudaMemcpyHostToDevice, st));
            d_in = net->in_stage_u8.p;
        } else {
            CU(net->in_stage.ensure(elems));
            CU(cudaMemcpyAsync(net->in_stage.p, input, elems * 4, cudaMemcpyHostToDevice, st));
            d_in = net->in_stage.p;
        }
    }
    int rc;
    if (mode == B200POSE_MODE_FP32) {
        if (in_u8) {   // parity mode: materialise rtpose_preprocess, then the fp32 path
            CU(net->f_u8.ensure(elems));
            CU(u8hwc_to_f32nchw_launch(static_cast<const unsigned char*>(d_in), net->f_u8.p, n, H, W, net->preprocess, st,
                                       d_ext));
            ++g_launches;
            rc = forward_fp32(net, net->f_u8.p, n, H, W, st, d_ext);
        } else rc = forward_fp32(net, static_cast<const float*>(d_in), n, H, W, st);
    } else rc = forward_bf16(net, d_in, in_u8 ? net->preprocess : 0, n, H, W, st, mode == B200POSE_MODE_BF16X3, ragged);
    if (rc) return rc;
    net->last_in = d_in;
    net->last_in_u8 = (mode == B200POSE_MODE_FP32) ? 0 : (in_u8 ? net->preprocess : 0);
    net->pn = n; net->pH = H; net->pW = W;
    if (outputs) {
        const size_t px8 = (size_t)n * (H / 8) * (W / 8);
        for (int i = 0; i < 12; ++i)
            if (outputs[i])
                CU(cudaMemcpyAsync(outputs[i], net->out_f32[i].p, px8 * (i % 2 == 0 ? kPaf : kHeat) * 4,
                                   outputs_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
    }
    if (sync_host && (!input_on_device || (outputs && !outputs_on_device))) CU(cudaStreamSynchronize(st));
    return 0;
}

int b200pose_net_forward(b200pose_net* net, const float* input, int input_on_device, int n, int H, int W, int mode,
                         float* const* outputs, int outputs_on_device, void* cuda_stream) {
    return net_forward_impl(net, input, 0, input_on_device, n, H, W, mode, outputs, outputs_on_device,
                            reinterpret_cast<cudaStream_t>(cuda_stream), true);
}

int b200pose_net_forward_u8(b200pose_net* net, const unsigned char* images, int input_on_device, int n, int H, int W,
                            int mode, float* const* outputs, int outputs_on_device, void* cuda_stream) {
    return net_forward_impl(net, images, 1, input_on_device, n, H, W, mode, outputs, outputs_on_device,
                            reinterpret_cast<cudaStream_t>(cuda_stream), true);
}

int b200pose_net_forward_u8_ragged(b200pose_net* net, const unsigned char* canvas, int input_on_device, int n, int H,
                                   int W, const int* ext_h, const int* ext_w, int mode, float* const* outputs,
                                   int outputs_on_device, void* cuda_stream) {
    if (!ext_h || !ext_w) return fail("ragged: null extent array");
    return net_forward_impl(net, canvas, 1, input_on_device, n, H, W, mode, outputs, outputs_on_device,
                            reinterpret_cast<cudaStream_t>(cuda_stream), true, ext_h, ext_w);
}

int b200pose_net_set_preprocess(b200pose_net* net, int preprocess) {
    if (!net) return fail("null net");
    if (preprocess < 1 || preprocess > 4) return fail("preprocess must be 1 (rtpose), 2 (vgg), 3 (inception) or 4 (ssd)");
    net->preprocess = preprocess;
    return 0;
}

int b200pose_net_profile(b200pose_net* net, float* ms, double* flops, int cap, void* cuda_stream) {
    if (!net || net->plan.empty() || (net->pmode != B200POSE_MODE_BF16 && net->pmode != B200POSE_MODE_BF16X3)) return -1;
    if (cudaSetDevice(net->device) != cudaSuccess) return -1;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(cuda_stream);
    const int n = net->pn, H = net->pH, W = net->pW;
    const int total = (int)net->plan.size() + 1;
    if (cap < total) return -1;
    std::vector<cudaEvent_t> ev(total + 1);
    for (auto& e : ev) cudaEventCreate(&e);
    const void* d_in = net->last_in;
    DevBuf<float> tmp;
    if (!d_in) { if (tmp.ensure((size_t)n * 3 * H * W) != cudaSuccess) return -1; cudaMemsetAsync(tmp.p, 0, (size_t)n * 3 * H * W * 4, st); d_in = tmp.p; net->last_in_u8 = 0; }
    cudaEventRecord(ev[0], st);
    conv_first_launch(d_in, net->last_in_u8, net->d_w[0], net->d_b[0], net->t1.p, net->plan_split ? net->l1.p : nullptr, n, H, W,
                      st, net->pragged ? net->ext.p : nullptr);
    cudaEventRecord(ev[1], st);
    for (size_t i = 0; i < net->plan.size(); ++i) {
        conv_tc_launch(net->plan[i], net->num_sms, st);
        cudaEventRecord(ev[i + 2], st);
    }
    g_launches += total;
    if (cudaStreamSynchronize(st) != cudaSuccess) { fail("profile run failed: %s", cudaGetErrorString(cudaGetLastError())); return -1; }
    for (int i = 0; i < total; ++i) cudaEventElapsedTime(&ms[i], ev[i], ev[i + 1]);
    flops[0] = 2.0 * n * H * W * 27.0 * 64.0;
    for (size_t i = 0; i < net->plan.size(); ++i) flops[i + 1] = net->plan_flops[i];
    for (auto& e : ev) cudaEventDestroy(e);
    tmp.release();
    return total;
}

int b200pose_net_last_maps(b200pose_net* net, const float** paf, const float** heat, int* n, int* h, int* w) {
    if (!net || net->pn == 0) return fail("no forward has run");
    *paf = net->out_f32[10].p; *heat = net->out_f32[11].p;
    *n = net->pn; *h = net->pH / 8; *w = net->pW / 8;
    return 0;
}

// ------------------------------------------------------------------------------------------------ post
int b200pose_post_create(b200pose_post** out, int cuda_device, int batch_cap, int peak_cap, int human_cap) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail("b200pose: no CUDA device available (this library has no CPU fallback)");
    CU(cudaSetDevice(cuda_device));
    b200pose_post* p = new b200pose_post();
    p->device = cuda_device;
    // candidate-key pool: 6 Mi entries (48 MB) per image of the batch (capped at 2 GiB) - key slots for every (a, b) pair of the limbs that do not
    // fit shared memory plus partition scratch, i.e. ~2 M pairs per image - capped at 1 GiB; exhausting it sets a status bit (loud error in the Python layer)
    // two halves (warp slots + partition scratch / contiguous sorted lists), each with one slot per (a, b) PAIR of every
    // limb: 8 Mi pairs per image of the batch (random-weight 368x368 maps produce ~1 M), capped at 8 GiB in total
    const long pool = (long)batch_cap * (16L << 20) < (1L << 30) ? (long)batch_cap * (16L << 20) : (1L << 30);
    cudaError_t e = post_alloc(p->pb, batch_cap, peak_cap, human_cap, pool);
    if (e != cudaSuccess) { delete p; return fail("post_alloc failed: %s", cudaGetErrorString(e)); }
    CU(cudaStreamCreateWithFlags(&p->s2, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&p->ev_limbs, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&p->ev_asm, cudaEventDisableTiming));
    for (int b = 0; b < 2; ++b) {
        CU(cudaEventCreateWithFlags(&p->ev_fetch[b], cudaEventDisableTiming));
        CU(cudaHostAlloc(&p->hp_nh[b], (size_t)batch_cap * sizeof(int), cudaHostAllocDefault));
        CU(cudaHostAlloc(&p->hp_status[b], (size_t)batch_cap * sizeof(int), cudaHostAllocDefault));
        CU(cudaHostAlloc(&p->hp_counts[b], (size_t)batch_cap * 18 * sizeof(int), cudaHostAllocDefault));
        CU(cudaHostAlloc(&p->hp_humans[b], (size_t)batch_cap * human_cap * kHumanFloats * sizeof(float), cudaHostAllocMapped | cudaHostAllocPortable));   // written by assemble_kernel (same pointer on the device: unified addressing)
        CU(cudaEventCreateWithFlags(&p->ev_ld[b], cudaEventDisableTiming));
    }
    CU(cudaEventCreateWithFlags(&p->ev_maps, cudaEventDisableTiming));
    const char* ov = getenv("B200POSE_POST_OVERLAP");
    p->overlap = !(ov && ov[0] == '0');
    *out = p;
    return 0;
}

void b200pose_post_destroy(b200pose_post* p) {
    if (!p) return;
    cudaSetDevice(p->device);
    if (p->s2) cudaStreamSynchronize(p->s2);
    post_free(p->pb);
    p->d_heat.release(); p->d_paf.release();
    p->tta_in.release(); p->tta_out.release();
    p->ov_maps[0].release(); p->ov_maps[1].release();
    p->dims[0].release(); p->dims[1].release();
    if (p->ev_maps) cudaEventDestroy(p->ev_maps);
    for (int b = 0; b < 2; ++b) if (p->ev_ld[b]) cudaEventDestroy(p->ev_ld[b]);
    for (int b = 0; b < 2; ++b) {
        if (p->ev_fetch[b]) cudaEventDestroy(p->ev_fetch[b]);
        if (p->hp_nh[b]) cudaFreeHost(p->hp_nh[b]);
        if (p->hp_status[b]) cudaFreeHost(p->hp_status[b]);
        if (p->hp_counts[b]) cudaFreeHost(p->hp_counts[b]);
        if (p->hp_humans[b]) cudaFreeHost(p->hp_humans[b]);
    }
    if (p->ev_limbs) cudaEventDestroy(p->ev_limbs);
    if (p->ev_asm) cudaEventDestroy(p->ev_asm);
    if (p->s2) cudaStreamDestroy(p->s2);
    delete p;
}

// After the limbs kernel was enqueued on `st`: assembly + result copies on the second stream.
static int enqueue_assemble_and_fetch(b200pose_post* p, int n, cudaStream_t st) {
    CU(cudaEventRecord(p->ev_limbs, st));
    CU(cudaStreamWaitEvent(p->s2, p->ev_limbs, 0));
    const int b = (int)(p->runs & 1);
    // the assembly kernel writes the person rows straight into this run's pinned host slot (unified addressing): only the
    // rows that exist cross PCIe, instead of a copy of the full-capacity buffer (4.8 MB per step at batch 32)
    p->pb.humans_out = p->hp_humans[b];
    cudaError_t e = post_assemble(p->pb, n, p->s2);
    if (e != cudaSuccess) return fail("post_assemble: %s", cudaGetErrorString(e));
    ++g_launches;
    CU(cudaEventRecord(p->ev_asm, p->s2));
    const PostBuffers& pb = p->pb;
    CU(cudaMemcpyAsync(p->hp_nh[b], pb.n_humans, n * sizeof(int), cudaMemcpyDeviceToHost, p->s2));
    CU(cudaMemcpyAsync(p->hp_status[b], pb.status, n * sizeof(int), cudaMemcpyDeviceToHost, p->s2));
    CU(cudaMemcpyAsync(p->hp_counts[b], pb.counts, (size_t)n * 18 * sizeof(int), cudaMemcpyDeviceToHost, p->s2));
    CU(cudaEventRecord(p->ev_fetch[b], p->s2));
    p->slot_n[b] = n;
    p->runs += 1;
    p->h_px.clear();
    return 0;
}

// dims_hw (host, may be null): a ragged run, n low-resolution (h, w) pairs; image i's maps lie top-left in the h x w canvas
static int post_run_dev(b200pose_post* p, const float* d_heat, const float* d_paf, int layout, int n, int h, int w,
                        float thresh, cudaStream_t st, const int* dims_hw = nullptr) {
    if (n > p->pb.batch_cap) return fail("batch %d exceeds post batch_cap %d", n, p->pb.batch_cap);
    cudaStream_t ps = st;       // the stream peaks / limbs run on
    const int slot = (int)(p->runs & 1);
    const int2* d_dims = nullptr;
    if (dims_hw) {      // per run-parity slot: run i-1's kernels on the second stream may still read the other one
        CU(p->dims[slot].ensure(p->pb.batch_cap));
        if (p->have_ld[slot]) CU(cudaStreamWaitEvent(st, p->ev_ld[slot], 0));   // run i-2 is done with this slot
        CU(cudaMemcpyAsync(p->dims[slot].p, dims_hw, (size_t)n * sizeof(int2), cudaMemcpyHostToDevice, st));
        d_dims = p->dims[slot].p;
    }
    if (p->overlap) {
        // private copy of the maps (15 MB at batch 32) so that the next forward may overwrite the network's output
        // buffers while this run's post-processing is still reading; everything after the copy runs on s2
        const size_t eh = (size_t)n * 19 * h * w, ep = (size_t)n * 38 * h * w;
        CU(p->ov_maps[slot].ensure(eh + ep));
        if (p->have_ld[slot]) CU(cudaStreamWaitEvent(st, p->ev_ld[slot], 0));   // run i-2 is done with this slot
        CU(cudaMemcpyAsync(p->ov_maps[slot].p, d_heat, eh * 4, cudaMemcpyDeviceToDevice, st));
        CU(cudaMemcpyAsync(p->ov_maps[slot].p + eh, d_paf, ep * 4, cudaMemcpyDeviceToDevice, st));
        CU(cudaEventRecord(p->ev_maps, st));
        CU(cudaStreamWaitEvent(p->s2, p->ev_maps, 0));
        d_heat = p->ov_maps[slot].p;
        d_paf = p->ov_maps[slot].p + eh;
        ps = p->s2;
    }
    // the previous run's assembly (second stream) still reads the peak / connection buffers this run overwrites, and
    // its D2H copies of status / counts (enqueued after the assembly) must not race with this run's memset + peaks:
    // wait for the event recorded after those copies
    if (p->runs > 0) CU(cudaStreamWaitEvent(ps, p->ev_fetch[(p->runs - 1) & 1], 0));
    cudaError_t e;
    if (layout == 0) {
        e = post_peaks(p->pb, n, d_heat, (long)19 * h * w, (long)h * w, w, 1, h, w, thresh, ps, d_dims);
        if (e != cudaSuccess) return fail("post_peaks: %s", cudaGetErrorString(e));
        e = post_limbs(p->pb, n, d_paf, (long)38 * h * w, (long)h * w, w, 1, 3, h * 8, w, h, ps, d_dims);
    } else {
        if (d_dims) return fail("ragged runs take NCHW maps");
        e = post_peaks(p->pb, n, d_heat, (long)19 * h * w, 1, (long)w * 19, 19, h, w, thresh, ps);
        if (e != cudaSuccess) return fail("post_peaks: %s", cudaGetErrorString(e));
        e = post_limbs(p->pb, n, d_paf, (long)38 * h * w, 1, (long)w * 38, 38, 3, h * 8, w, h, ps);
    }
    if (e != cudaSuccess) return fail("post_limbs: %s", cudaGetErrorString(e));
    g_launches += 2;
    if (p->overlap) {
        CU(cudaEventRecord(p->ev_ld[slot], ps));
        p->have_ld[slot] = true;
    }
    p->hw_h = h; p->hw_w = w;
    return enqueue_assemble_and_fetch(p, n, ps);
}

int b200pose_post_run(b200pose_post* p, const float* heat, const float* paf, int on_device, int layout, int n, int h,
                      int w, float thresh, void* cuda_stream) {
    if (!p) return fail("null post");
    CU(cudaSetDevice(p->device));
    cudaStream_t st = reinterpret_cast<cudaStream_t>(cuda_stream);
    const float *dh = heat, *dp = paf;
    if (!on_device) {
        CU(p->d_heat.ensure((size_t)n * 19 * h * w));
        CU(p->d_paf.ensure((size_t)n * 38 * h * w));
        CU(cudaMemcpyAsync(p->d_heat.p, heat, (size_t)n * 19 * h * w * 4, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(p->d_paf.p, paf, (size_t)n * 38 * h * w * 4, cudaMemcpyHostToDevice, st));
        dh = p->d_heat.p; dp = p->d_paf.p;
    }
    return post_run_dev(p, dh, dp, layout, n, h, w, thresh, st);
}

long b200pose_post_last_ticket(b200pose_post* p) { return p ? p->runs - 1 : -1; }

int b200pose_post_select(b200pose_post* p, long ticket) {
    if (!p) return fail("null post");
    if (ticket < 0 || ticket >= p->runs || ticket < p->runs - 2) return fail("ticket %ld is not one of the last two runs", ticket);
    CU(cudaSetDevice(p->device));
    CU(cudaEventSynchronize(p->ev_fetch[ticket & 1]));
    p->cur = (int)(ticket & 1);
    p->cur_ticket = ticket;
    return 0;
}

int b200pose_post_sync(b200pose_post* p) {
    if (!p) return fail("null post");
    if (p->runs == 0) return fail("no run submitted");
    return b200pose_post_select(p, p->runs - 1);
}

int b200pose_post_status_accum(b200pose_post* p, int reset) {
    // OR of the status words of every image of every run since the last reset: lets a caller that keeps runs in flight
    // (and only reads some of them back) prove that NO run overflowed a capacity
    if (!p) return -1;
    if (cudaSetDevice(p->device) != cudaSuccess) return -1;
    if (cudaStreamSynchronize(p->s2) != cudaSuccess) return -1;
    std::vector<int> h(p->pb.batch_cap);
    if (cudaMemcpy(h.data(), p->pb.status_acc, h.size() * sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    if (reset && cudaMemset(p->pb.status_acc, 0, h.size() * sizeof(int)) != cudaSuccess) return -1;
    int acc = 0;
    for (int v : h) acc |= v;
    return acc;
}

int b200pose_post_debug_sort(b200pose_post* p, const unsigned long long* keys, int n, unsigned long long* out) {
    if (!p || !keys || !out) return fail("debug_sort: null pointer");
    CU(cudaSetDevice(p->device));
    CU(cudaStreamSynchronize(p->s2));
    cudaError_t e = post_debug_sort(p->pb, keys, n, out, nullptr);
    if (e != cudaSuccess) return fail("post_debug_sort: %s", cudaGetErrorString(e));
    g_launches += 2;
    return 0;
}

int b200pose_post_debug(b200pose_post* p, unsigned long long* out, int n, int reset) {
    if (!p || n > 16) return -1;
    if (cudaMemcpy(out, p->pb.dbg, n * sizeof(unsigned long long), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    if (reset) cudaMemset(p->pb.dbg, 0, 16 * sizeof(unsigned long long));
    return 0;
}
static int post_ready(b200pose_post* p, int img) {
    if (!p) return 0;
    if (p->cur_ticket < 0 && b200pose_post_sync(p)) return 0;
    return img >= 0 && img < p->slot_n[p->cur];
}
int b200pose_post_num_humans(b200pose_post* p, int img) { return post_ready(p, img) ? p->hp_nh[p->cur][img] : -1; }
int b200pose_post_status(b200pose_post* p, int img) { return post_ready(p, img) ? p->hp_status[p->cur][img] : -1; }
int b200pose_post_get_humans(b200pose_post* p, int img, float* out, int max_humans) {
    if (!post_ready(p, img)) return -1;
    const int n = p->hp_nh[p->cur][img] < max_humans ? p->hp_nh[p->cur][img] : max_humans;
    memcpy(out, p->hp_humans[p->cur] + (size_t)img * p->pb.human_cap * kHumanFloats, (size_t)n * kHumanFloats * sizeof(float));
    return n;
}
int b200pose_post_get_peaks(b200pose_post* p, int img, float* out, int max_peaks) {
    // valid for the LATEST run only (reads the device peak arrays, which the next run overwrites)
    if (!p || p->runs == 0 || b200pose_post_select(p, p->runs - 1)) return -1;
    const int last_n = p->slot_n[p->cur];
    if (img < 0 || img >= last_n) return -1;
    const PostBuffers& pb = p->pb;
    const size_t per = (size_t)18 * pb.peak_cap;
    if (p->h_px.empty()) {
        const size_t tot = per * last_n;
        p->h_px.resize(tot); p->h_py.resize(tot); p->h_px_s.resize(tot);
        if (cudaMemcpy(p->h_px.data(), pb.peak_x, tot * 4, cudaMemcpyDeviceToHost) != cudaSuccess ||
            cudaMemcpy(p->h_py.data(), pb.peak_y, tot * 4, cudaMemcpyDeviceToHost) != cudaSuccess ||
            cudaMemcpy(p->h_px_s.data(), pb.peak_s, tot * 4, cudaMemcpyDeviceToHost) != cudaSuccess) {
            fail("peak copy failed");
            return -1;
        }
    }
    int k = 0;
    for (int part = 0; part < 18; ++part) {
        const int c = p->hp_counts[p->cur][(size_t)img * 18 + part];
        for (int i = 0; i < c && k < max_peaks; ++i, ++k) {
            const size_t o = (size_t)img * per + (size_t)part * pb.peak_cap + i;
            out[5 * k + 0] = (float)p->h_px[o];
            out[5 * k + 1] = (float)p->h_py[o];
            out[5 * k + 2] = p->h_px_s[o];
            out[5 * k + 3] = (float)k;
            out[5 * k + 4] = (float)part;
        }
    }
    return k;
}

static int infer_impl(b200pose_net* net, b200pose_post* post, const void* input, int in_u8, int input_on_device, int n,
                      int H, int W, int mode, float thresh, void* cuda_stream) {
    if (!net || !post) return fail("null handle");
    if (net->device != post->device) return fail("net and post live on different devices");
    // host input is staged asynchronously: the caller keeps it alive until b200pose_post_sync()
    int rc = net_forward_impl(net, input, in_u8, input_on_device, n, H, W, mode, nullptr, 1,
                              reinterpret_cast<cudaStream_t>(cuda_stream), false);
    if (rc) return rc;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(cuda_stream);
    return post_run_dev(post, net->out_f32[11].p, net->out_f32[10].p, 0, n, H / 8, W / 8, thresh, st);
}

int b200pose_infer(b200pose_net* net, b200pose_post* post, const float* input, int input_on_device, int n, int H, int W,
                   int mode, float thresh, void* cuda_stream) {
    return infer_impl(net, post, input, 0, input_on_device, n, H, W, mode, thresh, cuda_stream);
}
int b200pose_infer_u8(b200pose_net* net, b200pose_post* post, const unsigned char* images, int input_on_device, int n,
                      int H, int W, int mode, float thresh, void* cuda_stream) {
    return infer_impl(net, post, images, 1, input_on_device, n, H, W, mode, thresh, cuda_stream);
}

// ------------------------------------------------------------------------------------------------ flip TTA
static int flip_merge_dev(const float* nh, const float* fh, const float* np_, const float* fp, int layout, int n, int h,
                          int w, float* oh, float* op, cudaStream_t st) {
    cudaError_t e;
    if (layout == 0) {
        e = tta_flip_merge(nh, fh, oh, n, kHeat, h, w, (long)h * w, w, 1, st);
        if (e == cudaSuccess) e = tta_flip_merge(np_, fp, op, n, kPaf, h, w, (long)h * w, w, 1, st);
    } else {
        e = tta_flip_merge(nh, fh, oh, n, kHeat, h, w, 1, (long)w * kHeat, kHeat, st);
        if (e == cudaSuccess) e = tta_flip_merge(np_, fp, op, n, kPaf, h, w, 1, (long)w * kPaf, kPaf, st);
    }
    if (e != cudaSuccess) return fail("tta_flip_merge: %s", cudaGetErrorString(e));
    g_launches += 2;
    return 0;
}

int b200pose_flip_merge(b200pose_post* p, const float* normal_heat, const float* flipped_heat, const float* normal_paf,
                        const float* flipped_paf, int on_device, int layout, int n, int h, int w, float* out_heat,
                        float* out_paf, void* cuda_stream) {
    if (!p) return fail("null post");
    if (n < 1 || h < 1 || w < 1 || (layout != 0 && layout != 1)) return fail("flip_merge: bad shape / layout");
    if (!normal_heat || !flipped_heat || !normal_paf || !flipped_paf || !out_heat || !out_paf) return fail("flip_merge: null pointer");
    CU(cudaSetDevice(p->device));
    cudaStream_t st = reinterpret_cast<cudaStream_t>(cuda_stream);
    if (on_device)
        return flip_merge_dev(normal_heat, flipped_heat, normal_paf, flipped_paf, layout, n, h, w, out_heat, out_paf, st);
    const size_t eh = (size_t)n * kHeat * h * w, ep = (size_t)n * kPaf * h * w;
    CU(p->tta_in.ensure(2 * (eh + ep)));
    CU(p->tta_out.ensure(eh + ep));
    float *d_nh = p->tta_in.p, *d_fh = d_nh + eh, *d_np = d_fh + eh, *d_fp = d_np + ep;
    float *d_oh = p->tta_out.p, *d_op = d_oh + eh;
    CU(cudaMemcpyAsync(d_nh, normal_heat, eh * 4, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_fh, flipped_heat, eh * 4, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_np, normal_paf, ep * 4, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_fp, flipped_paf, ep * 4, cudaMemcpyHostToDevice, st));
    if (int rc = flip_merge_dev(d_nh, d_fh, d_np, d_fp, layout, n, h, w, d_oh, d_op, st)) return rc;
    CU(cudaMemcpyAsync(out_heat, d_oh, eh * 4, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(out_paf, d_op, ep * 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return 0;
}

static int infer_flip_impl(b200pose_net* net, b200pose_post* post, const void* input, int in_u8, int input_on_device,
                           int n, int H, int W, int mode, float thresh, void* cuda_stream) {
    if (!net || !post) return fail("null handle");
    if (!net->finalized) return fail("net not finalized");
    if (net->device != post->device) return fail("net and post live on different devices");
    if (n < 1 || H < 8 || W < 8 || (H % 8) || (W % 8)) return fail("input must be [n,3,H,W] with H, W multiples of 8");
    if (n > post->pb.batch_cap) return fail("batch %d exceeds post batch_cap %d", n, post->pb.batch_cap);
    CU(cudaSetDevice(net->device));
    cudaStream_t st = reinterpret_cast<cudaStream_t>(cuda_stream);
    // the 2n batch [frames | mirrored frames] is assembled in the net's staging buffer
    const size_t elems = (size_t)n * 3 * H * W;
    const cudaMemcpyKind kind = input_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    const void* d_batch;
    cudaError_t e;
    if (in_u8) {
        CU(net->in_stage_u8.ensure(2 * elems));
        CU(cudaMemcpyAsync(net->in_stage_u8.p, input, elems, kind, st));
        e = tta_mirror_u8hwc(net->in_stage_u8.p, net->in_stage_u8.p + elems, n, H, W, st);
        d_batch = net->in_stage_u8.p;
    } else {
        CU(net->in_stage.ensure(2 * elems));
        CU(cudaMemcpyAsync(net->in_stage.p, input, elems * 4, kind, st));
        e = tta_mirror_f32(net->in_stage.p, net->in_stage.p + elems, (long)n * 3, H, W, st);
        d_batch = net->in_stage.p;
    }
    if (e != cudaSuccess) return fail("tta_mirror: %s", cudaGetErrorString(e));
    ++g_launches;
    int rc = net_forward_impl(net, d_batch, in_u8, 1, 2 * n, H, W, mode, nullptr, 1, st, false);
    if (rc) return rc;
    const int h = H / 8, w = W / 8;
    const size_t eh = (size_t)n * kHeat * h * w, ep = (size_t)n * kPaf * h * w;
    CU(post->d_heat.ensure(eh));
    CU(post->d_paf.ensure(ep));
    rc = flip_merge_dev(net->out_f32[11].p, net->out_f32[11].p + eh, net->out_f32[10].p, net->out_f32[10].p + ep, 0, n, h,
                        w, post->d_heat.p, post->d_paf.p, st);
    if (rc) return rc;
    return post_run_dev(post, post->d_heat.p, post->d_paf.p, 0, n, h, w, thresh, st);
}

int b200pose_infer_flip(b200pose_net* net, b200pose_post* post, const float* input, int input_on_device, int n, int H,
                        int W, int mode, float thresh, void* cuda_stream) {
    return infer_flip_impl(net, post, input, 0, input_on_device, n, H, W, mode, thresh, cuda_stream);
}
int b200pose_infer_u8_flip(b200pose_net* net, b200pose_post* post, const unsigned char* images, int input_on_device,
                           int n, int H, int W, int mode, float thresh, void* cuda_stream) {
    return infer_flip_impl(net, post, images, 1, input_on_device, n, H, W, mode, thresh, cuda_stream);
}

// ------------------------------------------------------------------------------------------------ crop_with_factor
static int crop_check(int n, int src_h, int src_w, int dest_size, int factor, CropGeom* g) {
    if (n < 1 || src_h < 1 || src_w < 1 || dest_size < 1) return fail("crop_with_factor: bad shape");
    if (factor < 8 || factor % 8) return fail("crop_with_factor: factor must be a multiple of 8 (the network's stride)");
    *g = crop_geometry(src_h, src_w, dest_size, factor);
    if (g->res_h < 1 || g->res_w < 1) return fail("crop_with_factor: the resized frame would be empty");
    if ((long)g->pad_h * g->pad_w > (1L << 28)) return fail("crop_with_factor: resized frame too large");
    return 0;
}

int b200pose_crop_geometry(int src_h, int src_w, int dest_size, int factor, double* im_scale, int* res_h, int* res_w,
                           int* pad_h, int* pad_w) {
    CropGeom g;
    if (int rc = crop_check(1, src_h, src_w, dest_size, factor, &g)) return rc;
    if (im_scale) *im_scale = g.im_scale;
    if (res_h) *res_h = g.res_h;
    if (res_w) *res_w = g.res_w;
    if (pad_h) *pad_h = g.pad_h;
    if (pad_w) *pad_w = g.pad_w;
    return 0;
}

int b200pose_net_crop_with_factor(b200pose_net* net, const unsigned char* images, int images_on_device, int n, int src_h,
                                  int src_w, int dest_size, int factor, unsigned char* out, int out_on_device,
                                  void* cuda_stream) {
    if (!net) return fail("null net");
    if (!images || !out) return fail("crop_with_factor: null pointer");
    CropGeom g;
    if (int rc = crop_check(n, src_h, src_w, dest_size, factor, &g)) return rc;
    CU(cudaSetDevice(net->device));
    cudaStream_t st = reinterpret_cast<cudaStream_t>(cuda_stream);
    const size_t raw = (size_t)n * src_h * src_w * 3, outb = (size_t)n * g.pad_h * g.pad_w * 3;
    const unsigned char* d_in = images;
    if (!images_on_device) {
        CU(net->raw_stage.ensure(raw));
        CU(cudaMemcpyAsync(net->raw_stage.p, images, raw, cudaMemcpyHostToDevice, st));
        d_in = net->raw_stage.p;
    }
    unsigned char* d_out = out;
    if (!out_on_device) {
        CU(net->in_stage_u8.ensure(outb));
        d_out = net->in_stage_u8.p;
    }
    cudaError_t e = crop_with_factor_launch(d_in, d_out, n, src_h, src_w, g, st);
    if (e != cudaSuccess) return fail("crop_with_factor_launch: %s", cudaGetErrorString(e));
    ++g_launches;
    if (!out_on_device) CU(cudaMemcpyAsync(out, d_out, outb, cudaMemcpyDeviceToHost, st));
    if (!images_on_device || !out_on_device) CU(cudaStreamSynchronize(st));
    return 0;
}

int b200pose_infer_raw_u8(b200pose_net* net, b200pose_post* post, const unsigned char* images, int input_on_device, int n,
                          int src_h, int src_w, int dest_size, int factor, int mode, float thresh, int flip,
                          void* cuda_stream) {
    if (!net || !post) return fail("null handle");
    if (!net->finalized) return fail("net not finalized");
    if (net->device != post->device) return fail("net and post live on different devices");
    if (!images) return fail("infer_raw: null pointer");
    if (n > post->pb.batch_cap) return fail("batch %d exceeds post batch_cap %d", n, post->pb.batch_cap);
    CropGeom g;
    if (int rc = crop_check(n, src_h, src_w, dest_size, factor, &g)) return rc;
    CU(cudaSetDevice(net->device));
    cudaStream_t st = reinterpret_cast<cudaStream_t>(cuda_stream);
    const int nimg = flip ? 2 * n : n, H = g.pad_h, W = g.pad_w;
    const size_t raw = (size_t)n * src_h * src_w * 3;
    // the caller keeps a host input alive until b200pose_post_sync(), as for b200pose_infer
    const unsigned char* d_raw = images;
    if (!input_on_device || flip) {
        CU(net->raw_stage.ensure(raw * (flip ? 2 : 1)));
        CU(cudaMemcpyAsync(net->raw_stage.p, images, raw, input_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
        d_raw = net->raw_stage.p;
    }
    cudaError_t e;
    if (flip) {   // mirrored RAW frames: the padding of both orientations ends up on the right, as for the reference
        e = tta_mirror_u8hwc(net->raw_stage.p, net->raw_stage.p + raw, n, src_h, src_w, st);
        if (e != cudaSuccess) return fail("tta_mirror: %s", cudaGetErrorString(e));
        ++g_launches;
    }
    CU(net->in_stage_u8.ensure((size_t)nimg * H * W * 3));
    e = crop_with_factor_launch(d_raw, net->in_stage_u8.p, nimg, src_h, src_w, g, st);
    if (e != cudaSuccess) return fail("crop_with_factor_launch: %s", cudaGetErrorString(e));
    ++g_launches;
    int rc = net_forward_impl(net, net->in_stage_u8.p, 1, 1, nimg, H, W, mode, nullptr, 1, st, false);
    if (rc) return rc;
    const int h = H / 8, w = W / 8;
    if (!flip) return post_run_dev(post, net->out_f32[11].p, net->out_f32[10].p, 0, n, h, w, thresh, st);
    const size_t eh = (size_t)n * kHeat * h * w, ep = (size_t)n * kPaf * h * w;
    CU(post->d_heat.ensure(eh));
    CU(post->d_paf.ensure(ep));
    rc = flip_merge_dev(net->out_f32[11].p, net->out_f32[11].p + eh, net->out_f32[10].p, net->out_f32[10].p + ep, 0, n, h,
                        w, post->d_heat.p, post->d_paf.p, st);
    if (rc) return rc;
    return post_run_dev(post, post->d_heat.p, post->d_paf.p, 0, n, h, w, thresh, st);
}

// Per-frame geometry of a ragged batch of raw frames packed back to back: crop_with_factor of each frame's own size,
// its byte offset in the packed input, and the canvas (largest padded height x largest padded width).
static int ragged_layout(int n, const int* src_h, const int* src_w, int dest_size, int factor, RaggedCrop* fr,
                         int* canvas_h, int* canvas_w) {
    if (!src_h || !src_w) return fail("ragged layout: null pointer");
    if (n < 1) return fail("ragged layout: no frames");
    int H = 0, W = 0;
    long off = 0;
    for (int i = 0; i < n; ++i) {
        if (int rc = crop_check(1, src_h[i], src_w[i], dest_size, factor, &fr[i].g)) {
            fail("ragged layout: frame %d (%d x %d): %s", i, src_h[i], src_w[i], g_err.c_str());
            return rc;
        }
        fr[i].src_off = off; fr[i].src_h = src_h[i]; fr[i].src_w = src_w[i];
        off += (long)src_h[i] * src_w[i] * 3;
        H = H > fr[i].g.pad_h ? H : fr[i].g.pad_h;
        W = W > fr[i].g.pad_w ? W : fr[i].g.pad_w;
    }
    if ((long)H * W > (1L << 28)) return fail("ragged layout: canvas %d x %d too large", H, W);
    *canvas_h = H;
    *canvas_w = W;
    return 0;
}

int b200pose_ragged_layout(int n, const int* src_h, const int* src_w, int dest_size, int factor, long* src_off,
                           int* pad_h, int* pad_w, int* canvas_h, int* canvas_w) {
    if (!src_off || !pad_h || !pad_w || !canvas_h || !canvas_w) return fail("ragged layout: null pointer");
    std::vector<RaggedCrop> fr(n > 0 ? n : 0);
    if (int rc = ragged_layout(n, src_h, src_w, dest_size, factor, fr.data(), canvas_h, canvas_w)) return rc;
    for (int i = 0; i < n; ++i) { src_off[i] = fr[i].src_off; pad_h[i] = fr[i].g.pad_h; pad_w[i] = fr[i].g.pad_w; }
    return 0;
}

int b200pose_infer_raw_u8_ragged(b200pose_net* net, b200pose_post* post, const unsigned char* frames,
                                 int input_on_device, int n, const int* src_h, const int* src_w, int dest_size,
                                 int factor, int mode, float thresh, void* cuda_stream) {
    if (!net || !post) return fail("null handle");
    if (!net->finalized) return fail("net not finalized");
    if (net->device != post->device) return fail("net and post live on different devices");
    if (!frames || !src_h || !src_w) return fail("infer_raw_ragged: null pointer");
    if (n < 1) return fail("infer_raw_ragged: no frames");
    if (n > post->pb.batch_cap) return fail("batch %d exceeds post batch_cap %d", n, post->pb.batch_cap);
    std::vector<RaggedCrop> fr(n);
    std::vector<int> ext_h(n), ext_w(n), dims(2 * n);
    int H = 0, W = 0;
    if (int rc = ragged_layout(n, src_h, src_w, dest_size, factor, fr.data(), &H, &W)) return rc;
    for (int i = 0; i < n; ++i) {
        ext_h[i] = fr[i].g.pad_h; ext_w[i] = fr[i].g.pad_w;
        dims[2 * i] = fr[i].g.pad_h / 8; dims[2 * i + 1] = fr[i].g.pad_w / 8;
    }
    const long off = fr[n - 1].src_off + (long)src_h[n - 1] * src_w[n - 1] * 3;     // bytes of the packed frames
    CU(cudaSetDevice(net->device));
    cudaStream_t st = reinterpret_cast<cudaStream_t>(cuda_stream);
    // the caller keeps a host input alive until b200pose_post_sync(), as for b200pose_infer_raw_u8
    const unsigned char* d_raw = frames;
    if (!input_on_device) {
        CU(net->raw_stage.ensure(off));
        CU(cudaMemcpyAsync(net->raw_stage.p, frames, off, cudaMemcpyHostToDevice, st));
        d_raw = net->raw_stage.p;
    }
    CU(net->rcrop.ensure(n));
    CU(cudaMemcpyAsync(net->rcrop.p, fr.data(), n * sizeof(RaggedCrop), cudaMemcpyHostToDevice, st));
    CU(net->in_stage_u8.ensure((size_t)n * H * W * 3));
    cudaError_t e = crop_with_factor_ragged_launch(d_raw, net->in_stage_u8.p, n, net->rcrop.p, H, W, st);
    if (e != cudaSuccess) return fail("crop_with_factor_ragged_launch: %s", cudaGetErrorString(e));
    ++g_launches;
    int rc = net_forward_impl(net, net->in_stage_u8.p, 1, 1, n, H, W, mode, nullptr, 1, st, false, ext_h.data(), ext_w.data());
    if (rc) return rc;
    return post_run_dev(post, net->out_f32[11].p, net->out_f32[10].p, 0, n, H / 8, W / 8, thresh, st, dims.data());
}

int b200pose_infer_raw_u8_multiscale(b200pose_net* net, b200pose_post* post, const unsigned char* images,
                                     int input_on_device, int n, int src_h, int src_w, int base_size, int factor,
                                     const double* scales, int n_scales, int mode, float thresh, int flip,
                                     void* cuda_stream) {
    if (!net || !post) return fail("null handle");
    if (!net->finalized) return fail("net not finalized");
    if (net->device != post->device) return fail("net and post live on different devices");
    if (!images || !scales || n_scales < 1 || n_scales > 16) return fail("infer_multiscale: bad arguments");
    if (n > post->pb.batch_cap) return fail("batch %d exceeds post batch_cap %d", n, post->pb.batch_cap);
    CropGeom base;
    if (int rc = crop_check(n, src_h, src_w, base_size, factor, &base)) return rc;
    CU(cudaSetDevice(net->device));
    cudaStream_t st = reinterpret_cast<cudaStream_t>(cuda_stream);
    const int nimg = flip ? 2 * n : n;
    const size_t raw = (size_t)n * src_h * src_w * 3;
    const unsigned char* d_raw = images;
    if (!input_on_device || flip) {
        CU(net->raw_stage.ensure(raw * (flip ? 2 : 1)));
        CU(cudaMemcpyAsync(net->raw_stage.p, images, raw, input_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
        d_raw = net->raw_stage.p;
    }
    cudaError_t e;
    if (flip) {
        e = tta_mirror_u8hwc(net->raw_stage.p, net->raw_stage.p + raw, n, src_h, src_w, st);
        if (e != cudaSuccess) return fail("tta_mirror: %s", cudaGetErrorString(e));
        ++g_launches;
    }
    const int h1 = base.pad_h / 8, w1 = base.pad_w / 8;
    CU(post->d_heat.ensure((size_t)n * kHeat * h1 * w1));
    CU(post->d_paf.ensure((size_t)n * kPaf * h1 * w1));
    for (int k = 0; k < n_scales; ++k) {
        const int dest = (int)((double)base_size * scales[k]);       // Python: int(base_size * s)
        CropGeom g;
        if (int rc = crop_check(n, src_h, src_w, dest, factor, &g)) return rc;
        const int H = g.pad_h, W = g.pad_w, h = H / 8, w = W / 8;
        CU(net->in_stage_u8.ensure((size_t)nimg * H * W * 3));
        e = crop_with_factor_launch(d_raw, net->in_stage_u8.p, nimg, src_h, src_w, g, st);
        if (e != cudaSuccess) return fail("crop_with_factor_launch: %s", cudaGetErrorString(e));
        ++g_launches;
        if (int rc = net_forward_impl(net, net->in_stage_u8.p, 1, 1, nimg, H, W, mode, nullptr, 1, st, false)) return rc;
        const size_t eh = (size_t)n * kHeat * h * w, ep = (size_t)n * kPaf * h * w;
        const float *s_heat = net->out_f32[11].p, *s_paf = net->out_f32[10].p;
        if (flip) {
            CU(post->tta_out.ensure(eh + ep));
            if (int rc = flip_merge_dev(s_heat, s_heat + eh, s_paf, s_paf + ep, 0, n, h, w, post->tta_out.p,
                                        post->tta_out.p + eh, st))
                return rc;
            s_heat = post->tta_out.p;
            s_paf = post->tta_out.p + eh;
        }
        const float div = (k == n_scales - 1) ? (float)n_scales : 0.f;
        e = resize_cubic_accum_launch(s_heat, post->d_heat.p, (long)n * kHeat, h, w, h1, w1, k == 0, div, st);
        if (e == cudaSuccess)
            e = resize_cubic_accum_launch(s_paf, post->d_paf.p, (long)n * kPaf, h, w, h1, w1, k == 0, div, st);
        if (e != cudaSuccess) return fail("resize_cubic_accum_launch: %s", cudaGetErrorString(e));
        g_launches += 2;
    }
    return post_run_dev(post, post->d_heat.p, post->d_paf.p, 0, n, h1, w1, thresh, st);
}

// ------------------------------------------------------------------------------------------------ legacy pafprocess
namespace {
std::mutex g_legacy_mu;
b200pose_post* g_legacy = nullptr;
std::vector<float> g_leg_humans;       // [nh][73]
std::vector<float> g_leg_peaks;        // by id: x, y, score
int g_leg_nh = 0;
}  // namespace

int process_paf(int p1, int p2, int p3, float* peaks, int h1, int h2, int h3, float* heatmap, int f1, int f2, int f3,
                float* pafmap) {
    (void)h2; (void)h3; (void)heatmap;
    std::lock_guard<std::mutex> lk(g_legacy_mu);
    g_leg_nh = 0;
    if (p3 != 5) return fail("process_paf: peaks must be [p1,p2,5]");
    if (f3 != 38) return fail("process_paf: pafmap must have 38 channels");
    const int P = p1 * p2;
    int dev = 0;
    cudaGetDevice(&dev);
    const int cap = 2048;
    if (!g_legacy) {
        if (b200pose_post_create(&g_legacy, dev, 1, cap, 4096)) return 2;
    }
    b200pose_post* p = g_legacy;
    CU(cudaSetDevice(p->device));
    // bucket by part (pafprocess.cpp:24-43); ids follow input order, which equals part order for the array
    // paf_to_pose_cpp builds (we require that order, the reference silently mis-indexes otherwise)
    std::vector<int> counts(18, 0), hx((size_t)18 * cap), hy((size_t)18 * cap);
    std::vector<float> hs((size_t)18 * cap);
    int prev_part = 0;
    g_leg_peaks.assign((size_t)P * 3, 0.f);
    for (int i = 0; i < P; ++i) {
        const float* r = peaks + (size_t)i * 5;
        const int part = (int)r[4];
        if (part < 0 || part >= 18) return fail("process_paf: part id %d out of range", part);
        if (part < prev_part) return fail("process_paf: peaks must be ordered by part");
        prev_part = part;
        if (counts[part] >= cap) return fail("process_paf: more than %d peaks for part %d", cap, part);
        const size_t o = (size_t)part * cap + counts[part]++;
        hx[o] = (int)r[0]; hy[o] = (int)r[1]; hs[o] = r[2];
        g_leg_peaks[3 * i] = (float)(int)r[0]; g_leg_peaks[3 * i + 1] = (float)(int)r[1]; g_leg_peaks[3 * i + 2] = r[2];
    }
    const PostBuffers& pb = p->pb;
    cudaStream_t st = nullptr;
    if (p->runs > 0) CU(cudaStreamWaitEvent(st, p->ev_fetch[(p->runs - 1) & 1], 0));   // previous call's second-stream work
    CU(cudaMemsetAsync(pb.status, 0, sizeof(int), st));
    CU(cudaMemcpyAsync(pb.counts, counts.data(), 18 * sizeof(int), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(pb.peak_x, hx.data(), hx.size() * 4, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(pb.peak_y, hy.data(), hy.size() * 4, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(pb.peak_s, hs.data(), hs.size() * 4, cudaMemcpyHostToDevice, st));
    CU(p->d_paf.ensure((size_t)f1 * f2 * f3));
    CU(cudaMemcpyAsync(p->d_paf.p, pafmap, (size_t)f1 * f2 * f3 * 4, cudaMemcpyHostToDevice, st));
    cudaError_t e = post_limbs(pb, 1, p->d_paf.p, 0, 1, (long)f2 * f3, f3, 0, h1, f2, f1, st);
    if (e != cudaSuccess) return fail("post_limbs: %s", cudaGetErrorString(e));
    ++g_launches;
    if (enqueue_assemble_and_fetch(p, 1, st)) return 3;
    if (b200pose_post_sync(p)) return 3;
    if (p->hp_status[p->cur][0] & 0xff & ~16) return fail("process_paf: capacity exceeded (status %d)", p->hp_status[p->cur][0]);
    g_leg_nh = p->hp_nh[p->cur][0];
    g_leg_humans.assign(p->hp_humans[p->cur], p->hp_humans[p->cur] + (size_t)g_leg_nh * kHumanFloats);
    return 0;
}
// The reference's getters index its vectors unchecked (pafprocess.cpp:196-218); out-of-range arguments return -1 / 0 here.
static bool leg_human_ok(int human_id) { return human_id >= 0 && human_id < g_leg_nh; }
static bool leg_cid_ok(int cid) { return cid >= 0 && (size_t)cid * 3 + 2 < g_leg_peaks.size(); }
int get_num_humans(void) { return g_leg_nh; }
int get_part_cid(int human_id, int part_id) {
    if (!leg_human_ok(human_id) || part_id < 0 || part_id >= 18) return -1;
    return (int)g_leg_humans[(size_t)human_id * kHumanFloats + 1 + 4 * part_id + 3];
}
float get_score(int human_id) { return leg_human_ok(human_id) ? g_leg_humans[(size_t)human_id * kHumanFloats] : 0.f; }
int get_part_x(int cid) { return leg_cid_ok(cid) ? (int)g_leg_peaks[3 * (size_t)cid] : -1; }
int get_part_y(int cid) { return leg_cid_ok(cid) ? (int)g_leg_peaks[3 * (size_t)cid + 1] : -1; }
float get_part_score(int cid) { return leg_cid_ok(cid) ? g_leg_peaks[3 * (size_t)cid + 2] : 0.f; }

}  // extern "C"
