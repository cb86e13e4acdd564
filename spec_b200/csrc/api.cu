// C ABI of libspecb200 (declared in include/specb200.h): handles, weight packing, the trunk op
// interpreter and the tail orchestration.  Host code only enqueues kernels on the caller's stream.
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <string.h>
#include <stdlib.h>
#include <string>
#include <vector>
#include <algorithm>

#include <nvtx3/nvToolsExt.h>

#include "../../include/specb200.h"
#include "internal.h"
#include "tail.h"

namespace sb {

NvtxRange::NvtxRange(const char* name) { nvtxRangePushA(name); }
NvtxRange::~NvtxRange() { nvtxRangePop(); }

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
bool check_cuda(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return true;
    g_err = std::string(what) + ": " + cudaGetErrorString(e);
    return false;
}

// Per-op profiling (specb200_trunk_profile) times every kernel ALONE between two events; the programmatic edges are suspended
// there so that a kernel's set-up is inside its own interval, as it is for any kernel timed on its own.
static thread_local bool g_pdl_suspended = false;
bool pdl_enabled() {
    static const bool on = [] { const char* e = getenv("SPECB200_PDL"); return !(e && e[0] == '0'); }();
    return on && !g_pdl_suspended;
}

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
static inline int prec_elem(int prec) { return prec == PREC_F32 ? 4 : 2; }

struct BufShape { int H = 0, W = 0; };

}  // namespace sb

using namespace sb;

// =============================================================================================== trunk
struct specb200_trunk {
    std::vector<specb200_op_t> ops;
    std::vector<int> buf_ch;
    std::vector<ConvWeights> w;
    std::vector<ConvWeights> w_plain;       // pair slots only: the plain [32][32][3][3] packing for odd widths
    std::vector<int> wslot_cin;      // stored (padded) Cin of the op using the slot
    std::vector<int> wslot_pair;     // slot belongs to a pixel-pair conv (weights expanded to 64 x 64)
    int out_buf = 0;
    int prec = PREC_BF16;
    int chunk = 0;
    int stem7_slot = -1;             // >= 0: op 0 is the ResNet 7x7/2 stem and runs in conv_stem7_kernel (reads the NCHW image)
    // whole-bottleneck fusion (conv_bneck.cu): fuse_first[i] = index of the first op of the group op i belongs to (-1: none);
    // a group is [downsample?] conv1 conv2 conv3 with 64 mid channels, 256 outputs, stride 1
    struct FuseGroup { int first = -1, last = -1, ds = -1, c1 = -1, c2 = -1, c3 = -1; };
    std::vector<FuseGroup> groups;
    std::vector<int> op_group;       // per op: index into groups or -1
    int64_t last_launches = 0;
    std::vector<cudaEvent_t> prof_ev;        // non-empty only inside specb200_trunk_profile
    size_t prof_n = 0;
    // cached plan
    int plan_h = -1, plan_w = -1;
    std::vector<BufShape> op_src, op_dst;    // per-op spatial dims
    std::vector<size_t> buf_elems;           // per-buffer max H*W*C (per image)
    int out_h = 0, out_w = 0;
};

static bool trunk_plan(specb200_trunk* t, int h, int w) {
    if (t->plan_h == h && t->plan_w == w) return true;
    const int nb = static_cast<int>(t->buf_ch.size());
    std::vector<BufShape> cur(nb);
    t->op_src.assign(t->ops.size(), BufShape());
    t->op_dst.assign(t->ops.size(), BufShape());
    t->buf_elems.assign(nb, 0);
    cur[0].H = h; cur[0].W = w;
    t->buf_elems[0] = static_cast<size_t>(h) * w * t->buf_ch[0];
    for (size_t i = 0; i < t->ops.size(); ++i) {
        const specb200_op_t& o = t->ops[i];
        if (o.src < 0 || o.src >= nb || o.dst < 0 || o.dst >= nb || o.src2 >= nb) { set_error("trunk: bad buffer id"); return false; }
        const BufShape s = cur[o.src];
        if (s.H <= 0) { set_error("trunk: op " + std::to_string(i) + " reads an undefined buffer"); return false; }
        BufShape d;
        switch (o.type) {
            case SPECB200_OP_CONV:
                d.H = (s.H + 2 * o.pad - o.kh) / o.stride + 1;
                d.W = (s.W + 2 * o.pad - o.kw) / o.stride + 1;
                if (o.src2 >= 0 && (cur[o.src2].H != d.H || cur[o.src2].W != d.W)) { set_error("trunk: residual shape mismatch at op " + std::to_string(i)); return false; }
                if (o.cin != t->buf_ch[o.src]) { set_error("trunk: conv cin != source buffer channels at op " + std::to_string(i)); return false; }
                break;
            case SPECB200_OP_MAXPOOL:
                d.H = (s.H + 2 - 3) / 2 + 1; d.W = (s.W + 2 - 3) / 2 + 1; break;
            case SPECB200_OP_UPADD:
                d = cur[o.dst];
                if (d.H != (s.H << o.shift) || d.W != (s.W << o.shift)) { set_error("trunk: upadd shape mismatch at op " + std::to_string(i)); return false; }
                break;
            case SPECB200_OP_BILINEAR:
                if (o.src2 < 0) { set_error("trunk: bilinear needs a size reference"); return false; }
                d = cur[o.src2]; break;
            case SPECB200_OP_COPY:
                d = s; break;
            default: set_error("trunk: unknown op type"); return false;
        }
        if (d.H <= 0 || d.W <= 0) { set_error("trunk: input too small"); return false; }
        if (o.dst_coff > 0 && (cur[o.dst].H != 0) && (cur[o.dst].H != d.H || cur[o.dst].W != d.W) && o.type != SPECB200_OP_UPADD) {
            // concat writers must agree on the spatial size; the first writer defines it
        }
        t->op_src[i] = s; t->op_dst[i] = d;
        cur[o.dst] = d;
        t->buf_elems[o.dst] = std::max(t->buf_elems[o.dst], static_cast<size_t>(d.H) * d.W * t->buf_ch[o.dst]);
    }
    t->out_h = cur[t->out_buf].H; t->out_w = cur[t->out_buf].W;
    t->plan_h = h; t->plan_w = w;
    return true;
}

// Finds [downsample 1x1 (X -> 256)]? conv1 1x1 (X -> 64, ReLU), conv2 3x3/1 (64 -> 64, ReLU), conv3 1x1 (64 -> 256, + residual,
// ReLU) runs whose intermediates are read by nobody else: those run as ONE bottleneck64_kernel launch in the 16-bit modes.
static void trunk_find_bottlenecks(specb200_trunk* t) {
    const int n = static_cast<int>(t->ops.size());
    t->op_group.assign(n, -1);
    t->groups.clear();
    if (t->prec == PREC_F32) return;
    auto is_conv = [&](int i, int cin, int cout, int k, int relu) {
        if (i < 0 || i >= n) return false;
        const specb200_op_t& o = t->ops[i];
        return o.type == SPECB200_OP_CONV && o.cin == cin && o.cout == cout && o.kh == k && o.kw == k && o.stride == 1 && o.pad == k / 2 &&
               o.relu == relu && o.dst_coff == 0 && o.pair == 0 && t->buf_ch[o.src] == cin && t->buf_ch[o.dst] == cout && o.src != 0;
    };
    // buffer `b`, defined by op `def`, is read only by the ops in `allowed` until it is redefined
    auto private_buf = [&](int b, int def, std::initializer_list<int> allowed) {
        for (int j = def + 1; j < n; ++j) {
            const specb200_op_t& o = t->ops[j];
            bool reads = (o.src == b) || (o.src2 == b) || (o.type == SPECB200_OP_UPADD && o.dst == b);
            bool ok = false;
            for (int a : allowed) ok = ok || a == j;
            if (reads && !ok) return false;
            if (o.dst == b && o.type != SPECB200_OP_UPADD) return true;      // redefined: later readers see the new tensor
        }
        return b != t->out_buf;
    };
    for (int i = 0; i + 2 < n; ++i) {
        if (t->op_group[i] >= 0) continue;
        for (int cin : {256, 64}) {
            if (!is_conv(i, cin, 64, 1, 1) || !is_conv(i + 1, 64, 64, 3, 1) || !is_conv(i + 2, 64, 256, 1, 1)) continue;
            const specb200_op_t &c1 = t->ops[i], &c2 = t->ops[i + 1], &c3 = t->ops[i + 2];
            if (c1.src2 >= 0 || c2.src2 >= 0 || c2.src != c1.dst || c3.src != c2.dst || c3.src2 < 0) continue;
            specb200_trunk::FuseGroup g;
            g.c1 = i; g.c2 = i + 1; g.c3 = i + 2; g.first = i; g.last = i + 2;
            if (cin == 256) {
                if (c3.src2 != c1.src) continue;                               // identity residual = the block input
            } else {
                if (i == 0 || !is_conv(i - 1, 64, 256, 1, 0) || t->op_group[i - 1] >= 0) continue;
                const specb200_op_t& d = t->ops[i - 1];
                if (d.src != c1.src || d.src2 >= 0 || c3.src2 != d.dst || !private_buf(d.dst, i - 1, {i + 2})) continue;
                g.ds = i - 1; g.first = i - 1;
            }
            if (!private_buf(c1.dst, i, {i + 1}) || !private_buf(c2.dst, i + 1, {i + 2})) continue;
            if (c3.dst == c1.src || c3.dst == c1.dst || c3.dst == c2.dst) continue;
            const int gi = static_cast<int>(t->groups.size());
            t->groups.push_back(g);
            for (int j = g.first; j <= g.last; ++j) t->op_group[j] = gi;
            break;
        }
    }
}

extern "C" const char* specb200_last_error(void) { return g_err.c_str(); }
extern "C" int specb200_abi_version(void) { return SPECB200_ABI_VERSION; }

extern "C" int specb200_device_check(void) {
    // cudaGetDeviceProperties takes milliseconds and serialises on driver locks (it stalled for 7..33 ms when an nvidia-smi
    // poller was running -- bench.py's first timed step, round 2): ask once per device, with the two cheap attribute queries
    static int cached[64] = {};                    // 0 unknown, 1 ok, 2 wrong architecture
    int dev = 0;
    if (!check_cuda(cudaGetDevice(&dev), "cudaGetDevice")) return 1;
    const int slot = dev & 63;
    if (cached[slot] == 0) {
        int major = 0, minor = 0;
        if (!check_cuda(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev), "cudaDeviceGetAttribute")) return 1;
        if (!check_cuda(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev), "cudaDeviceGetAttribute")) return 1;
        cached[slot] = (major == 10) ? 1 : 2;
        if (major != 10) set_error("libspecb200 requires an sm_100 (B200) device, found sm_" + std::to_string(major) + std::to_string(minor));
    }
    if (cached[slot] == 2) { set_error("libspecb200 requires an sm_100 (B200) device"); return 2; }
    return 0;
}

extern "C" int specb200_trunk_create(specb200_trunk_t** out, const specb200_op_t* ops, int32_t n_ops,
                                     const int32_t* buf_channels, int32_t n_bufs, int32_t n_wslots, int32_t out_buf,
                                     int32_t precision) {
    if (!out || !ops || !buf_channels || n_ops <= 0 || n_bufs <= 0 || out_buf < 0 || out_buf >= n_bufs) { set_error("trunk_create: bad arguments"); return 1; }
    if (precision < 0 || precision > 2) { set_error("trunk_create: bad precision"); return 1; }
    specb200_trunk* t = new specb200_trunk();
    t->ops.assign(ops, ops + n_ops);
    t->buf_ch.assign(buf_channels, buf_channels + n_bufs);
    t->w.resize(n_wslots);
    t->w_plain.resize(n_wslots);
    t->wslot_cin.assign(n_wslots, 0);
    t->wslot_pair.assign(n_wslots, 0);
    t->out_buf = out_buf;
    t->prec = precision;
    for (const auto& o : t->ops) {
        if (o.type == SPECB200_OP_CONV) {
            if (o.wslot < 0 || o.wslot >= n_wslots) { set_error("trunk_create: bad wslot"); delete t; return 1; }
            t->wslot_cin[o.wslot] = o.cin;
            const bool pair_ok = o.pair && t->prec != PREC_F32 && o.cin == 32 && o.cout == 32 && o.kh == 3 &&
                                 o.kw == 3 && o.stride == 1 && o.pad == 1 && o.dst_coff == 0 && t->buf_ch[o.src] == 32 &&
                                 t->buf_ch[o.dst] == 32 && (o.src2 < 0 || t->buf_ch[o.src2] == 32);
            t->wslot_pair[o.wslot] = pair_ok ? 1 : 0;
        }
    }
    {   // ResNet stem: dedicated kernel when op 0 is conv 7x7/2 pad 3 -> 64 (+ReLU) on the image and nothing else reads it
        const specb200_op_t& o = t->ops[0];
        bool ok = t->prec != PREC_F32 && o.type == SPECB200_OP_CONV && o.src == 0 && o.kh == 7 && o.kw == 7 && o.stride == 2 &&
                  o.pad == 3 && o.cout == 64 && o.relu && o.src2 < 0 && o.dst_coff == 0 && t->buf_ch[o.dst] == 64;
        for (size_t i = 1; i < t->ops.size() && ok; ++i) ok = t->ops[i].src != 0 && t->ops[i].src2 != 0;
        if (ok) t->stem7_slot = o.wslot;
    }
    trunk_find_bottlenecks(t);
    *out = t;
    return 0;
}

static void free_weights(ConvWeights& w) {
    if (w.w_tc) cudaFree(w.w_tc);
    if (w.w_f32) cudaFree(w.w_f32);
    if (w.bias) cudaFree(w.bias);
    w = ConvWeights();
}

// Packs one conv (BN already folded) into `w` for the precision / kernel family of the trunk.
static bool pack_conv(specb200_trunk* t, ConvWeights& w, bool stem7, const float* w_host, const float* b_host, int cout, int cin, int cin_s,
                      int kh, int kw) {
    if (cin_s < cin) { set_error("set_conv: weight cin exceeds the op's cin"); return false; }
    free_weights(w);
    w.cout = cout; w.cin = cin_s; w.kh = kh; w.kw = kw;
    w.K = kh * kw * cin_s;
    if (!check_cuda(cudaMalloc(&w.bias, sizeof(float) * cout), "cudaMalloc bias")) return false;
    if (!check_cuda(cudaMemcpy(w.bias, b_host, sizeof(float) * cout, cudaMemcpyHostToDevice), "bias upload")) return false;
    w.bias_host.assign(b_host, b_host + cout);
    auto to16 = [&](float v) {
        uint16_t bits;
        if (t->prec == PREC_BF16) { __nv_bfloat16 h = __float2bfloat16_rn(v); memcpy(&bits, &h, 2); }
        else { __half h = __float2half_rn(v); memcpy(&bits, &h, 2); }
        return bits;
    };
    if (t->prec == PREC_F32) {
        std::vector<float> pk(static_cast<size_t>(w.K) * cout, 0.f);
        for (int o = 0; o < cout; ++o)
            for (int c = 0; c < cin; ++c)
                for (int y = 0; y < kh; ++y)
                    for (int x = 0; x < kw; ++x)
                        pk[(static_cast<size_t>(y * kw + x) * cin_s + c) * cout + o] = w_host[((static_cast<size_t>(o) * cin + c) * kh + y) * kw + x];
        if (!check_cuda(cudaMalloc(&w.w_f32, pk.size() * sizeof(float)), "cudaMalloc w_f32")) return false;
        if (!check_cuda(cudaMemcpy(w.w_f32, pk.data(), pk.size() * sizeof(float), cudaMemcpyHostToDevice), "w upload")) return false;
    } else if (stem7) {
        if (cin != 3 || cout != 64 || kh != 7 || kw != 7) { set_error("set_conv: stem weights must be [64][3][7][7]"); return false; }
        w.stem7 = true; w.block_n = 64; w.cout_pad = 64; w.K = 168; w.K_pad = 192;
        std::vector<uint16_t> pk(static_cast<size_t>(64) * 192, 0);
        for (int o = 0; o < 64; ++o)
            for (int c = 0; c < 3; ++c)
                for (int y = 0; y < 7; ++y)
                    for (int x = 0; x < 7; ++x)
                        pk[static_cast<size_t>(o) * 192 + (c * 7 + y) * 8 + x] = to16(w_host[((static_cast<size_t>(o) * 3 + c) * 7 + y) * 7 + x]);
        if (!check_cuda(cudaMalloc(&w.w_tc, pk.size() * 2), "cudaMalloc w_tc")) return false;
        if (!check_cuda(cudaMemcpy(w.w_tc, pk.data(), pk.size() * 2, cudaMemcpyHostToDevice), "w upload")) return false;
        if (!conv_tc_make_weight_tmap(w)) return false;
    } else {
        w.block_n = conv_tc_pick_block_n(cout, kh * kw * cin_s);
        if (cin_s == 4) {                           // stem layout: K index = (y*kwp + x)*4 + c
            w.kwp = 1;
            while (w.kwp < kw) w.kwp <<= 1;
            w.K = kh * w.kwp * 4;
        }
        const int kw_eff = w.kwp > 0 ? w.kwp : kw;
        w.K_pad = static_cast<int>(align_up(w.K, 64));
        w.cout_pad = static_cast<int>(align_up(cout, w.block_n));
        std::vector<uint16_t> pk(static_cast<size_t>(w.cout_pad) * w.K_pad, 0);
        for (int o = 0; o < cout; ++o)
            for (int c = 0; c < cin; ++c)
                for (int y = 0; y < kh; ++y)
                    for (int x = 0; x < kw; ++x)
                        pk[static_cast<size_t>(o) * w.K_pad + static_cast<size_t>(y * kw_eff + x) * cin_s + c] =
                            to16(w_host[((static_cast<size_t>(o) * cin + c) * kh + y) * kw + x]);
        if (!check_cuda(cudaMalloc(&w.w_tc, pk.size() * 2), "cudaMalloc w_tc")) return false;
        if (!check_cuda(cudaMemcpy(w.w_tc, pk.data(), pk.size() * 2, cudaMemcpyHostToDevice), "w upload")) return false;
        if (!conv_tc_make_weight_tmap(w)) return false;
    }
    return true;
}

extern "C" int specb200_trunk_set_conv(specb200_trunk_t* t, int32_t wslot, const float* w_host, const float* b_host,
                                       int32_t cout, int32_t cin, int32_t kh, int32_t kw) {
    if (!t || wslot < 0 || wslot >= static_cast<int>(t->w.size()) || !w_host || !b_host) { set_error("set_conv: bad arguments"); return 1; }
    const int cin_s = t->wslot_cin[wslot];           // stored Cin (>= cin, zero padded)
    if (t->wslot_pair[wslot]) {
        // Pixel-pair view: [H][W][32] == [H][W/2][64].  Output pixel x = 2X + po reads input x + dx = 2(X + s) + pi with
        // s = floor((po + dx) / 2), pi = (po + dx) mod 2, so the 32->32 3x3 conv is a 64->64 3x3 conv on the half-width
        // grid whose weights are W2[po*32+co][pi*32+ci][kh][s+1] = w[co][ci][kh][dx+1] (half of them structurally zero).
        // The view needs an even width: the plain [32][32][3][3] packing is kept beside it for odd widths (gather kernel).
        if (cin != 32 || cout != 32 || kh != 3 || kw != 3) { set_error("set_conv: pair slot expects [32][32][3][3]"); return 1; }
        if (!pack_conv(t, t->w_plain[wslot], false, w_host, b_host, cout, cin, cin_s, kh, kw)) return 1;
        std::vector<float> pair_w(static_cast<size_t>(64) * 64 * 9, 0.f), pair_b(64);
        for (int po = 0; po < 2; ++po)
            for (int co = 0; co < 32; ++co) {
                pair_b[po * 32 + co] = b_host[co];
                for (int ci = 0; ci < 32; ++ci)
                    for (int y = 0; y < 3; ++y)
                        for (int dx = -1; dx <= 1; ++dx) {
                            const int q = po + dx;
                            const int sft = (q < 0) ? -1 : (q >= 2 ? 1 : 0);
                            const int pi = q - 2 * sft;
                            pair_w[((static_cast<size_t>(po * 32 + co) * 64 + pi * 32 + ci) * 3 + y) * 3 + (sft + 1)] =
                                w_host[((static_cast<size_t>(co) * 32 + ci) * 3 + y) * 3 + (dx + 1)];
                        }
            }
        return pack_conv(t, t->w[wslot], false, pair_w.data(), pair_b.data(), 64, 64, 64, 3, 3) ? 0 : 1;
    }
    return pack_conv(t, t->w[wslot], t->prec != PREC_F32 && wslot == t->stem7_slot, w_host, b_host, cout, cin, cin_s, kh, kw) ? 0 : 1;
}

extern "C" int specb200_trunk_set_chunk(specb200_trunk_t* t, int32_t chunk) {
    if (!t || chunk < 0) { set_error("set_chunk: bad arguments"); return 1; }
    t->chunk = chunk;
    return 0;
}

extern "C" int specb200_trunk_out_shape(specb200_trunk_t* t, int32_t h, int32_t w, int32_t* c_out, int32_t* h_out, int32_t* w_out) {
    if (!t) { set_error("out_shape: null handle"); return 1; }
    if (!trunk_plan(t, h, w)) return 1;
    if (c_out) *c_out = t->buf_ch[t->out_buf];
    if (h_out) *h_out = t->out_h;
    if (w_out) *w_out = t->out_w;
    return 0;
}

static int trunk_eff_batch(const specb200_trunk* t, int batch) { return (t->chunk > 0 && t->chunk < batch) ? t->chunk : batch; }

extern "C" int64_t specb200_trunk_workspace_bytes(specb200_trunk_t* t, int32_t batch, int32_t h, int32_t w) {
    if (!t || batch <= 0) { set_error("workspace_bytes: bad arguments"); return -1; }
    if (!trunk_plan(t, h, w)) return -1;
    const int eb = trunk_eff_batch(t, batch);
    size_t total = 0;
    for (size_t i = 0; i < t->buf_elems.size(); ++i) total += align_up(t->buf_elems[i] * eb * prec_elem(t->prec), 1024);
    return static_cast<int64_t>(total + 1024);
}

static int trunk_forward_impl(specb200_trunk_t* t, const float* images, int32_t batch, int32_t h, int32_t w,
                              void* workspace, int64_t workspace_bytes, float* pooled_out, int32_t pooled_ld,
                              float* feat_out, void* stream, int stop_op) {
    if (!t || !images || !workspace || batch <= 0) { set_error("trunk_forward: bad arguments"); return 1; }
    NvtxRange nvtx_trunk("specb200:trunk (backbone convs + pool)");
    if (!trunk_plan(t, h, w)) return 1;
    if (workspace_bytes < specb200_trunk_workspace_bytes(t, batch, h, w)) { set_error("trunk_forward: workspace too small"); return 1; }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int eb = trunk_eff_batch(t, batch);
    const int es = prec_elem(t->prec);
    // carve buffers
    std::vector<uint8_t*> buf(t->buf_ch.size());
    {
        uint8_t* p = reinterpret_cast<uint8_t*>(align_up(reinterpret_cast<size_t>(workspace), 1024));
        for (size_t i = 0; i < buf.size(); ++i) { buf[i] = p; p += align_up(t->buf_elems[i] * eb * es, 1024); }
    }
    int64_t launches = 0;
    const int C_out = t->buf_ch[t->out_buf];
    auto mark = [&]() { if (!t->prof_ev.empty() && t->prof_n < t->prof_ev.size()) cudaEventRecord(t->prof_ev[t->prof_n++], s); };
    for (int b0 = 0; b0 < batch; b0 += eb) {
        const int nb = std::min(eb, batch - b0);
        mark();
        if (t->stem7_slot < 0) {
            if (!images_to_nhwc_launch(images + static_cast<size_t>(b0) * 3 * h * w, buf[0], nb, h, w, t->buf_ch[0], t->prec, s)) return 1;
            ++launches;
        }
        mark();
        for (size_t i = 0; i < t->ops.size(); ++i) {
            const specb200_op_t& o = t->ops[i];
            const BufShape sS = t->op_src[i], dS = t->op_dst[i];
            if (t->op_group[i] >= 0 && static_cast<int>(i) == t->groups[t->op_group[i]].first) {
                // whole bottleneck in one launch (not when a debug read-out stops inside the group)
                const specb200_trunk::FuseGroup& g = t->groups[t->op_group[i]];
                const specb200_op_t& c1 = t->ops[g.c1];
                BottleneckArgs ba;
                ba.x = buf[c1.src]; ba.out = buf[t->ops[g.c3].dst];
                ba.N = nb; ba.H = t->op_src[g.c1].H; ba.W = t->op_src[g.c1].W; ba.Cin = c1.cin;
                ba.w1 = &t->w[c1.wslot]; ba.w2 = &t->w[t->ops[g.c2].wslot]; ba.w3 = &t->w[t->ops[g.c3].wslot];
                ba.wd = g.ds >= 0 ? &t->w[t->ops[g.ds].wslot] : nullptr;
                if ((stop_op < 0 || stop_op >= g.last) && bottleneck_applicable(ba)) {
                    if (!bottleneck_launch(ba, t->prec, s)) return 1;
                    ++launches;
                    for (int j = g.first; j <= g.last; ++j) mark();       // profile: the group's time lands on its first op
                    i = static_cast<size_t>(g.last);
                    if (static_cast<int>(i) == stop_op) break;
                    continue;
                }
            }
            if (i == 0 && t->stem7_slot >= 0) {
                const ConvWeights& cw = t->w[o.wslot];
                if (cw.bias == nullptr) { set_error("trunk_forward: stem weights not set"); return 1; }
                if (!conv_stem7_launch(images + static_cast<size_t>(b0) * 3 * h * w, buf[o.dst], cw, nb, sS.H, sS.W, dS.H, dS.W, t->prec, s)) return 1;
                ++launches;
                mark();
                if (stop_op == 0) break;
                continue;
            }
            switch (o.type) {
                case SPECB200_OP_CONV: {
                    // the pixel-pair view needs an even width; odd widths take the plain packing (gather kernel)
                    const bool pair = t->wslot_pair[o.wslot] != 0 && !((sS.W & 1) || (dS.W & 1));
                    const ConvWeights& cw = (t->wslot_pair[o.wslot] != 0 && !pair) ? t->w_plain[o.wslot] : t->w[o.wslot];
                    if (cw.bias == nullptr) { set_error("trunk_forward: conv weights for slot " + std::to_string(o.wslot) + " not set"); return 1; }
                    if (cw.cout != (pair ? 64 : o.cout) || cw.kh != o.kh || cw.kw != o.kw) { set_error("trunk_forward: weight shape mismatch at op " + std::to_string(i)); return 1; }
                    ConvParams p;
                    p.in = buf[o.src]; p.out = buf[o.dst]; p.res = o.src2 >= 0 ? buf[o.src2] : nullptr; p.bias = cw.bias;
                    p.N = nb; p.H = sS.H; p.W = sS.W; p.Cin = o.cin; p.Ho = dS.H; p.Wo = dS.W; p.Cout = o.cout;
                    p.kh = o.kh; p.kw = o.kw; p.stride = o.stride; p.pad = o.pad;
                    p.K = cw.K; p.kwp = cw.kwp;
                    const long long M = static_cast<long long>(nb) * dS.H * dS.W;
                    if (M > 0x7fffffffLL) { set_error("trunk_forward: batch too large"); return 1; }
                    p.M = static_cast<int>(M);
                    p.out_ld = t->buf_ch[o.dst]; p.out_coff = o.dst_coff;
                    p.res_ld = o.src2 >= 0 ? t->buf_ch[o.src2] : 0;
                    p.relu = o.relu;
                    if (pair) { p.W /= 2; p.Wo /= 2; p.M /= 2; p.Cin = 64; p.Cout = 64; p.out_ld = 64; p.res_ld = o.src2 >= 0 ? 64 : 0; }
                    const bool ok = (t->prec == PREC_F32) ? conv_f32_launch(p, cw, s)
                                    : (conv_halo_applicable(p, cw) ? conv_halo_launch(p, cw, t->prec, s) : conv_tc_launch(p, cw, t->prec, s));
                    if (!ok) return 1;
                    break;
                }
                case SPECB200_OP_MAXPOOL: {
                    // is the pooled tensor the output of a conv + ReLU (>= 0)?  the last writer of o.src before this op decides
                    bool nonneg = false;
                    for (int j = static_cast<int>(i) - 1; j >= 0; --j)
                        if (t->ops[j].dst == o.src) { nonneg = t->ops[j].type == SPECB200_OP_CONV && t->ops[j].relu != 0 && t->ops[j].dst_coff == 0; break; }
                    if (!maxpool3x3s2_launch(buf[o.src], buf[o.dst], nb, sS.H, sS.W, t->buf_ch[o.src], dS.H, dS.W, t->prec, s, nonneg)) return 1;
                    break;
                }
                case SPECB200_OP_UPADD:
                    if (!upsample_add_launch(buf[o.src], buf[o.dst], nb, dS.H, dS.W, t->buf_ch[o.dst], o.shift, o.relu, t->prec, s)) return 1;
                    break;
                case SPECB200_OP_BILINEAR:
                    if (!bilinear_launch(buf[o.src], buf[o.dst], nb, sS.H, sS.W, t->buf_ch[o.src], dS.H, dS.W, t->buf_ch[o.dst], o.dst_coff, t->prec, s)) return 1;
                    break;
                case SPECB200_OP_COPY:
                    if (!copy_channels_launch(buf[o.src], buf[o.dst], nb * sS.H * sS.W, t->buf_ch[o.src], t->buf_ch[o.dst], o.dst_coff, t->prec, s)) return 1;
                    break;
                default: set_error("trunk_forward: unknown op"); return 1;
            }
            ++launches;
            mark();
            if (static_cast<int>(i) == stop_op) break;
        }
        if (stop_op >= 0) {                                   // debug read-out of an intermediate activation (whole batch at once)
            const specb200_op_t& o = t->ops[stop_op];
            const BufShape dS = t->op_dst[stop_op];
            if (!nhwc_to_nchw_f32_launch(buf[o.dst], feat_out, nb, dS.H, dS.W, t->buf_ch[o.dst], t->prec, s)) return 1;
            break;
        }
        if (pooled_out) {
            if (!avgpool_launch(buf[t->out_buf], pooled_out + static_cast<size_t>(b0) * pooled_ld, pooled_ld, nb, t->out_h * t->out_w, C_out, t->prec, s)) return 1;
            ++launches;
        }
        mark();
        if (feat_out) {
            if (!nhwc_to_nchw_f32_launch(buf[t->out_buf], feat_out + static_cast<size_t>(b0) * C_out * t->out_h * t->out_w, nb, t->out_h, t->out_w, C_out, t->prec, s)) return 1;
            ++launches;
        }
    }
    t->last_launches = launches;
    return 0;
}

extern "C" int specb200_trunk_forward(specb200_trunk_t* t, const float* images, int32_t batch, int32_t h, int32_t w,
                                      void* workspace, int64_t workspace_bytes, float* pooled_out, int32_t pooled_ld,
                                      float* feat_out, void* stream) {
    return trunk_forward_impl(t, images, batch, h, w, workspace, workspace_bytes, pooled_out, pooled_ld, feat_out, stream, -1);
}

extern "C" int specb200_trunk_forward_until(specb200_trunk_t* t, const float* images, int32_t batch, int32_t h, int32_t w,
                                            void* workspace, int64_t workspace_bytes, int32_t stop_op, int32_t* c_out, int32_t* h_out,
                                            int32_t* w_out, float* act_out, void* stream) {
    if (!t || stop_op < 0 || stop_op >= static_cast<int>(t->ops.size())) { set_error("trunk_forward_until: bad op index"); return 1; }
    if (!trunk_plan(t, h, w)) return 1;
    if (t->chunk > 0 && t->chunk < batch) { set_error("trunk_forward_until: not with batch chunking"); return 1; }
    if (c_out) *c_out = t->buf_ch[t->ops[stop_op].dst];
    if (h_out) *h_out = t->op_dst[stop_op].H;
    if (w_out) *w_out = t->op_dst[stop_op].W;
    if (!act_out) return 0;                                   // shape query only
    return trunk_forward_impl(t, images, batch, h, w, workspace, workspace_bytes, nullptr, 0, act_out, stream, stop_op);
}

extern "C" int64_t specb200_trunk_last_launches(specb200_trunk_t* t) { return t ? t->last_launches : 0; }

extern "C" int32_t specb200_trunk_num_ops(specb200_trunk_t* t) { return t ? static_cast<int32_t>(t->ops.size()) : 0; }
extern "C" int32_t specb200_trunk_num_fused_bottlenecks(specb200_trunk_t* t) { return t ? static_cast<int32_t>(t->groups.size()) : 0; }
extern "C" int32_t specb200_trunk_fused_group_first_op(specb200_trunk_t* t, int32_t op) {
    if (!t || op < 0 || op >= static_cast<int32_t>(t->op_group.size()) || t->op_group[op] < 0) return -1;
    return t->groups[t->op_group[op]].first;
}

extern "C" int specb200_trunk_profile(specb200_trunk_t* t, const float* images, int32_t batch, int32_t h, int32_t w,
                                      void* workspace, int64_t workspace_bytes, float* pooled_out, int32_t pooled_ld,
                                      float* op_ms_host, void* stream) {
    if (!t || !op_ms_host) { set_error("trunk_profile: bad arguments"); return 1; }
    const int eb = trunk_eff_batch(t, batch);
    const size_t per_chunk = t->ops.size() + 3;                // start, after image conversion, after each op, after pool
    const size_t chunks = (batch + eb - 1) / eb;
    t->prof_ev.resize(per_chunk * chunks);
    for (auto& e : t->prof_ev) if (!check_cuda(cudaEventCreate(&e), "cudaEventCreate")) return 1;
    t->prof_n = 0;
    g_pdl_suspended = true;
    int rc = specb200_trunk_forward(t, images, batch, h, w, workspace, workspace_bytes, pooled_out, pooled_ld, nullptr, stream);
    g_pdl_suspended = false;
    if (rc == 0 && !check_cuda(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)), "sync")) rc = 1;
    if (rc == 0) {
        for (size_t i = 0; i + 1 < per_chunk; ++i) op_ms_host[i] = 0.f;
        for (size_t c = 0; c < chunks; ++c)
            for (size_t i = 0; i + 1 < per_chunk; ++i) {
                float ms = 0.f;
                cudaEventElapsedTime(&ms, t->prof_ev[c * per_chunk + i], t->prof_ev[c * per_chunk + i + 1]);
                op_ms_host[i] += ms;
            }
    }
    for (auto& e : t->prof_ev) cudaEventDestroy(e);
    t->prof_ev.clear();
    t->prof_n = 0;
    return rc;
}

extern "C" void specb200_trunk_destroy(specb200_trunk_t* t) {
    if (!t) return;
    for (auto& w : t->w) free_weights(w);
    for (auto& w : t->w_plain) free_weights(w);
    delete t;
}

// =============================================================================================== camcalib tail
struct CamLinear { float* w = nullptr; float* b = nullptr; int out = 0, in = 0; };
struct specb200_camtail {
    int in_features = 0, num_out = 0;
    std::vector<CamLinear> heads[3];
    bool fused = false;                 // single-layer heads concatenated into one [3*num_out][in] GEMM
    float* wcat = nullptr; float* bcat = nullptr;
    int max_hidden = 0;
    unsigned* red_counters = nullptr;   // split-K arrival counters of the fused GEMM (library-owned: they must start at zero)
};
constexpr int CAM_RED_COUNTERS = 4096, CAM_RED_SLICES = 8;

extern "C" int specb200_camtail_create(specb200_camtail_t** out, int32_t in_features, int32_t num_out) {
    if (!out || in_features <= 0 || num_out <= 0) { set_error("camtail_create: bad arguments"); return 1; }
    specb200_camtail* t = new specb200_camtail();
    t->in_features = in_features; t->num_out = num_out;
    *out = t;
    return 0;
}

extern "C" int specb200_camtail_add_linear(specb200_camtail_t* t, int32_t which, const float* w_host, const float* b_host,
                                           int32_t out_features, int32_t in_features) {
    if (!t || which < 0 || which > 2 || !w_host || !b_host) { set_error("camtail_add_linear: bad arguments"); return 1; }
    const int expect_in = t->heads[which].empty() ? t->in_features : t->heads[which].back().out;
    if (in_features != expect_in) { set_error("camtail_add_linear: in_features does not chain"); return 1; }
    CamLinear l; l.out = out_features; l.in = in_features;
    if (!check_cuda(cudaMalloc(&l.w, sizeof(float) * out_features * in_features), "cudaMalloc")) return 1;
    if (!check_cuda(cudaMalloc(&l.b, sizeof(float) * out_features), "cudaMalloc")) return 1;
    if (!check_cuda(cudaMemcpy(l.w, w_host, sizeof(float) * out_features * in_features, cudaMemcpyHostToDevice), "upload")) return 1;
    if (!check_cuda(cudaMemcpy(l.b, b_host, sizeof(float) * out_features, cudaMemcpyHostToDevice), "upload")) return 1;
    t->heads[which].push_back(l);
    return 0;
}

extern "C" int specb200_camtail_finalize(specb200_camtail_t* t) {
    if (!t) { set_error("camtail_finalize: null"); return 1; }
    for (int h = 0; h < 3; ++h) {
        if (t->heads[h].empty() || t->heads[h].back().out != t->num_out) { set_error("camtail_finalize: head incomplete"); return 1; }
        for (size_t i = 0; i + 1 < t->heads[h].size(); ++i) t->max_hidden = std::max(t->max_hidden, t->heads[h][i].out);
    }
    if (t->heads[0].size() == 1 && t->heads[1].size() == 1 && t->heads[2].size() == 1) {
        const size_t wsz = static_cast<size_t>(t->num_out) * t->in_features;
        if (!check_cuda(cudaMalloc(&t->wcat, sizeof(float) * 3 * wsz), "cudaMalloc")) return 1;
        if (!check_cuda(cudaMalloc(&t->bcat, sizeof(float) * 3 * t->num_out), "cudaMalloc")) return 1;
        for (int h = 0; h < 3; ++h) {
            if (!check_cuda(cudaMemcpy(t->wcat + h * wsz, t->heads[h][0].w, sizeof(float) * wsz, cudaMemcpyDeviceToDevice), "copy")) return 1;
            if (!check_cuda(cudaMemcpy(t->bcat + h * t->num_out, t->heads[h][0].b, sizeof(float) * t->num_out, cudaMemcpyDeviceToDevice), "copy")) return 1;
        }
        if (!check_cuda(cudaMalloc(&t->red_counters, sizeof(unsigned) * CAM_RED_COUNTERS), "cudaMalloc") ||
            !check_cuda(cudaMemset(t->red_counters, 0, sizeof(unsigned) * CAM_RED_COUNTERS), "cudaMemset")) return 1;
        t->fused = true;
    }
    return 0;
}

extern "C" int64_t specb200_camtail_workspace_bytes(specb200_camtail_t* t, int32_t batch) {
    if (!t || batch <= 0) { set_error("camtail_workspace_bytes: bad arguments"); return -1; }
    if (t->fused)        // split-K partial sums of the one concatenated GEMM
        return static_cast<int64_t>(align_up(static_cast<size_t>(CAM_RED_SLICES) * batch * 3 * t->num_out * sizeof(float), 256) + 256);
    return static_cast<int64_t>(2 * align_up(static_cast<size_t>(batch) * std::max(t->max_hidden, 4) * sizeof(float), 256) + 256);
}

extern "C" int specb200_camtail_forward(specb200_camtail_t* t, const float* pooled, int32_t pooled_ld, int32_t batch,
                                        void* workspace, int64_t workspace_bytes, float* logits_out, void* stream) {
    if (!t || !pooled || !logits_out || batch <= 0) { set_error("camtail_forward: bad arguments"); return 1; }
    NvtxRange nvtx_cam("specb200:camcalib_fc");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int ldo = 3 * t->num_out;
    if (!workspace || workspace_bytes < specb200_camtail_workspace_bytes(t, batch)) { set_error("camtail_forward: workspace too small"); return 1; }
    if (t->fused) {
        LinearRedWs red;
        red.partial = reinterpret_cast<float*>(align_up(reinterpret_cast<size_t>(workspace), 256));
        red.partial_floats = static_cast<size_t>(CAM_RED_SLICES) * batch * ldo;
        red.counters = t->red_counters; red.n_counters = CAM_RED_COUNTERS;
        return linear_f32_launch(pooled, pooled_ld, t->wcat, t->in_features, t->bcat, nullptr, 0, logits_out, ldo, batch, ldo, t->in_features, s,
                                 1, 0, nullptr, &red) ? 0 : 1;
    }
    float* tmp[2];
    tmp[0] = reinterpret_cast<float*>(align_up(reinterpret_cast<size_t>(workspace), 256));
    tmp[1] = tmp[0] + align_up(static_cast<size_t>(batch) * t->max_hidden, 64);
    for (int h = 0; h < 3; ++h) {
        const float* cur = pooled; int ld = pooled_ld;
        for (size_t i = 0; i < t->heads[h].size(); ++i) {
            const CamLinear& l = t->heads[h][i];
            const bool last = (i + 1 == t->heads[h].size());
            float* dst = last ? logits_out + h * t->num_out : tmp[i & 1];
            const int dld = last ? ldo : l.out;
            if (!linear_f32_launch(cur, ld, l.w, l.in, l.b, nullptr, 0, dst, dld, batch, l.out, l.in, s)) return 1;
            cur = dst; ld = dld;
        }
    }
    return 0;
}

extern "C" int specb200_camcalib_decode(const float* logits, int32_t logits_ld, int32_t num_out, int32_t batch,
                                        const float* img_h, const float* img_w, float* angles_out, float* rotmat_out,
                                        float* intr_out, float* fpix_out, void* stream) {
    if (!logits || !angles_out || batch <= 0) { set_error("camcalib_decode: bad arguments"); return 1; }
    NvtxRange nvtx_dec("specb200:camcalib_decode (softargmax, f_pix, R, K)");
    if (rotmat_out && (!img_h || !img_w || !intr_out)) { set_error("camcalib_decode: img_h/img_w/intrinsics required with rotmat"); return 1; }
    return camcalib_decode_launch(logits, logits_ld, num_out, img_h, img_w, angles_out, rotmat_out, intr_out, fpix_out, batch,
                                  static_cast<cudaStream_t>(stream)) ? 0 : 1;
}

extern "C" void specb200_camtail_destroy(specb200_camtail_t* t) {
    if (!t) return;
    for (int h = 0; h < 3; ++h) for (auto& l : t->heads[h]) { cudaFree(l.w); cudaFree(l.b); }
    if (t->wcat) cudaFree(t->wcat);
    if (t->bcat) cudaFree(t->bcat);
    if (t->red_counters) cudaFree(t->red_counters);
    delete t;
}

// =============================================================================================== HMR tail
// SMPL constants on the device (packed by pack_smpl below)
struct SmplConsts { float *Vt = nullptr, *Sd = nullptr, *Pd = nullptr, *Wl = nullptr, *Jt = nullptr, *Js = nullptr; };

struct specb200_hmrtail {
    int C = 0, use_cam_feats = 0, use_cam = 0, ldx = 0, kin = 0;
    float focal = 5000.f, img_res = 224.f;
    float *Fx = nullptr, *c0 = nullptr, *AsT = nullptr, *init157 = nullptr;   // folded head (see tail.cu)
    SmplConsts smpl;
    float* Jx = nullptr;
    int64_t last_launches = 0;
};

static bool upload(float** dst, const std::vector<float>& v) {
    if (!check_cuda(cudaMalloc(dst, v.size() * sizeof(float)), "cudaMalloc")) return false;
    return check_cuda(cudaMemcpy(*dst, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice), "upload");
}

// SMPL constants shared by the HMR tail and the body model: validated kinematic tree, coordinate-planar repack over a padded
// vertex axis (coalesced over vertices) and the rest-joint regression folded through the shape basis.  The integer tables
// (c_parents is fixed; c_joint_map / c_vertex_ids belong to the HMR tail) are not touched here, so handles of any number of
// SMPL models (neutral / male / female) coexist.
static void free_smpl(SmplConsts& c) {
    float* ptrs[] = {c.Vt, c.Sd, c.Pd, c.Wl, c.Jt, c.Js};
    for (float* p : ptrs) if (p) cudaFree(p);
    c = SmplConsts();
}

static bool check_parents(const int32_t* parents, const char* who) {
    static const int std_parents[24] = {-1, 0, 0, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 9, 9, 12, 13, 14, 16, 17, 18, 19, 20, 21};
    for (int i = 0; i < 24; ++i) if (parents[i] != std_parents[i]) { set_error(std::string(who) + ": unexpected SMPL kinematic tree"); return false; }
    return true;
}

static bool pack_smpl(SmplConsts& out, const float* v_template, const float* shapedirs, const float* posedirs, const float* J_regressor,
                      const float* lbs_weights) {
    const int NV = SMPL_NV, VP = SMPL_VP;
    std::vector<float> Vt(3 * static_cast<size_t>(VP), 0.f), Sd(30 * static_cast<size_t>(VP), 0.f), Pd(207 * 3 * static_cast<size_t>(VP), 0.f),
        Wl(24 * static_cast<size_t>(VP), 0.f);
    for (int v = 0; v < NV; ++v) {
        for (int c = 0; c < 3; ++c) {
            Vt[static_cast<size_t>(c) * VP + v] = v_template[v * 3 + c];
            for (int l = 0; l < 10; ++l) Sd[(static_cast<size_t>(l) * 3 + c) * VP + v] = shapedirs[(static_cast<size_t>(v) * 3 + c) * 10 + l];
        }
        for (int j = 0; j < 24; ++j) Wl[static_cast<size_t>(j) * VP + v] = lbs_weights[static_cast<size_t>(v) * 24 + j];
    }
    for (int k = 0; k < 207; ++k)
        for (int v = 0; v < NV; ++v)
            for (int c = 0; c < 3; ++c)
                Pd[(static_cast<size_t>(k) * 3 + c) * VP + v] = posedirs[static_cast<size_t>(k) * (NV * 3) + v * 3 + c];
    // rest-joint regression folded through the shape basis (fp64 on the host):
    //   J = Jreg (T + S beta) = (Jreg T) + (Jreg S) beta
    std::vector<float> Jt(72), Js(720);
    for (int j = 0; j < 24; ++j)
        for (int c = 0; c < 3; ++c) {
            double a = 0.0;
            for (int v = 0; v < NV; ++v) a += static_cast<double>(J_regressor[static_cast<size_t>(j) * NV + v]) * v_template[v * 3 + c];
            Jt[j * 3 + c] = static_cast<float>(a);
            for (int l = 0; l < 10; ++l) {
                double s = 0.0;
                for (int v = 0; v < NV; ++v) s += static_cast<double>(J_regressor[static_cast<size_t>(j) * NV + v]) * shapedirs[(static_cast<size_t>(v) * 3 + c) * 10 + l];
                Js[(j * 3 + c) * 10 + l] = static_cast<float>(s);
            }
        }
    return upload(&out.Vt, Vt) && upload(&out.Sd, Sd) && upload(&out.Pd, Pd) && upload(&out.Wl, Wl) && upload(&out.Jt, Jt) && upload(&out.Js, Js);
}

extern "C" int specb200_hmrtail_create(specb200_hmrtail_t** out, const specb200_hmr_params_t* p) {
    if (!out || !p) { set_error("hmrtail_create: bad arguments"); return 1; }
    const float* req[] = {p->fc1_w, p->fc1_b, p->fc2_w, p->fc2_b, p->decpose_w, p->decpose_b, p->decshape_w, p->decshape_b,
                          p->deccam_w, p->deccam_b, p->init_pose, p->init_shape, p->init_cam, p->v_template, p->shapedirs,
                          p->posedirs, p->J_regressor, p->lbs_weights, p->J_regressor_extra};
    for (const float* q : req) if (!q) { set_error("hmrtail_create: null parameter pointer"); return 1; }
    if (!p->parents || !p->joint_map || !p->vertex_ids) { set_error("hmrtail_create: null index table"); return 1; }
    if (!check_parents(p->parents, "hmrtail_create")) return 1;
    for (int i = 0; i < 49; ++i) if (p->joint_map[i] < 0 || p->joint_map[i] >= 54) { set_error("hmrtail_create: joint_map out of range"); return 1; }
    for (int i = 0; i < 21; ++i) if (p->vertex_ids[i] < 0 || p->vertex_ids[i] >= SMPL_NV) { set_error("hmrtail_create: vertex id out of range"); return 1; }
    if ((p->in_features % 4) != 0) { set_error("hmrtail_create: in_features must be a multiple of 4"); return 1; }
    specb200_hmrtail* t = new specb200_hmrtail();
    t->C = p->in_features; t->use_cam_feats = p->use_cam_feats; t->use_cam = p->use_cam;
    t->focal = p->focal_length; t->img_res = p->img_res;
    t->kin = t->C + 157 + (t->use_cam_feats ? 7 : 0);        // fc1 in_features
    t->ldx = static_cast<int>(align_up(t->kin, 4));
    const int NV = SMPL_NV, VP = SMPL_VP;
    bool ok = true;
    {   // fold the affine head in fp64:  P = D W2 ; Q = P W1 ; c0 = P b1 + D b2 + bd
        const int kin = t->kin, C = t->C, ns = kin - C;
        std::vector<double> D(static_cast<size_t>(157) * 1024), bd(157);
        for (int i = 0; i < 144 * 1024; ++i) D[i] = p->decpose_w[i];
        for (int i = 0; i < 10 * 1024; ++i) D[144 * 1024 + i] = p->decshape_w[i];
        for (int i = 0; i < 3 * 1024; ++i) D[154 * 1024 + i] = p->deccam_w[i];
        for (int i = 0; i < 144; ++i) bd[i] = p->decpose_b[i];
        for (int i = 0; i < 10; ++i) bd[144 + i] = p->decshape_b[i];
        for (int i = 0; i < 3; ++i) bd[154 + i] = p->deccam_b[i];
        std::vector<double> P(static_cast<size_t>(157) * 1024, 0.0);
        for (int i = 0; i < 157; ++i)
            for (int k = 0; k < 1024; ++k) {
                const double d = D[static_cast<size_t>(i) * 1024 + k];
                const float* w2 = p->fc2_w + static_cast<size_t>(k) * 1024;
                double* pr = &P[static_cast<size_t>(i) * 1024];
                for (int j = 0; j < 1024; ++j) pr[j] += d * w2[j];
            }
        std::vector<double> Q(static_cast<size_t>(157) * kin, 0.0);
        std::vector<float> c0(160, 0.f);
        for (int i = 0; i < 157; ++i) {
            double c = bd[i];
            for (int k = 0; k < 1024; ++k) {
                const double pv = P[static_cast<size_t>(i) * 1024 + k];
                c += pv * p->fc1_b[k] + D[static_cast<size_t>(i) * 1024 + k] * p->fc2_b[k];
                const float* w1 = p->fc1_w + static_cast<size_t>(k) * kin;
                double* qr = &Q[static_cast<size_t>(i) * kin];
                for (int j = 0; j < kin; ++j) qr[j] += pv * w1[j];
            }
            c0[i] = static_cast<float>(c);
        }
        std::vector<float> Fx(static_cast<size_t>(157) * C), AsT(static_cast<size_t>(164) * 160, 0.f), init(157);
        for (int i = 0; i < 157; ++i) {
            for (int j = 0; j < C; ++j) Fx[static_cast<size_t>(i) * C + j] = static_cast<float>(Q[static_cast<size_t>(i) * kin + j]);
            for (int k = 0; k < ns; ++k) AsT[static_cast<size_t>(k) * 160 + i] = static_cast<float>(Q[static_cast<size_t>(i) * kin + C + k]);
        }
        memcpy(&init[0], p->init_pose, sizeof(float) * 144); memcpy(&init[144], p->init_shape, sizeof(float) * 10); memcpy(&init[154], p->init_cam, sizeof(float) * 3);
        ok = ok && upload(&t->Fx, Fx) && upload(&t->c0, c0) && upload(&t->AsT, AsT) && upload(&t->init157, init);
    }
    {   // SMPL constants (shared packing) + the 9 extra-joint regressor rows, coordinate-planar like the rest
        ok = ok && pack_smpl(t->smpl, p->v_template, p->shapedirs, p->posedirs, p->J_regressor, p->lbs_weights);
        std::vector<float> Jx(9 * static_cast<size_t>(VP), 0.f);
        for (int v = 0; v < NV; ++v)
            for (int q = 0; q < 9; ++q) Jx[static_cast<size_t>(q) * VP + v] = p->J_regressor_extra[static_cast<size_t>(q) * NV + v];
        ok = ok && upload(&t->Jx, Jx);
    }
    ok = ok && tail_upload_tables(p->joint_map, p->vertex_ids);
    if (!ok) { specb200_hmrtail_destroy(t); return 1; }
    *out = t;
    return 0;
}

namespace {
constexpr int HEAD_KSPLIT = 8;     // split-K slices of the G GEMM (N = 157 alone would fill only 24 CTAs)
struct HmrWs { float *X, *G, *pf, *A, *Jp, *ej; size_t total; };
HmrWs hmr_carve(const specb200_hmrtail* t, int B, void* base) {
    HmrWs w;
    size_t off = 0;
    auto take = [&](size_t nfloat) { float* p = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(base) + off); off += align_up(nfloat * sizeof(float), 256); return p; };
    w.X = take(static_cast<size_t>(B) * t->ldx);
    w.G = take(static_cast<size_t>(B) * 160 * HEAD_KSPLIT);
    w.pf = take(static_cast<size_t>(B) * PF_LD);
    w.A = take(static_cast<size_t>(B) * 288);
    w.Jp = take(static_cast<size_t>(B) * 72);
    w.ej = take(static_cast<size_t>(B) * 4 * 27);
    w.total = off;
    return w;
}
}  // namespace

extern "C" int64_t specb200_hmrtail_workspace_bytes(specb200_hmrtail_t* t, int32_t batch) {
    if (!t || batch <= 0) { set_error("hmrtail_workspace_bytes: bad arguments"); return -1; }
    return static_cast<int64_t>(hmr_carve(t, batch, nullptr).total);
}
extern "C" int32_t specb200_hmrtail_x_ld(specb200_hmrtail_t* t) { return t ? t->ldx : 0; }

extern "C" int specb200_hmrtail_forward(specb200_hmrtail_t* t, int32_t B, void* workspace, int64_t workspace_bytes,
                                        const float* cam_rotmat, const float* cam_intr, const float* bbox_scale,
                                        const float* bbox_center, const float* img_w, const float* img_h,
                                        const specb200_hmr_outputs_t* o, void* stream) {
    if (!t || !workspace || !o || B <= 0) { set_error("hmrtail_forward: bad arguments"); return 1; }
    if ((reinterpret_cast<size_t>(workspace) & 255) != 0) { set_error("hmrtail_forward: workspace must be 256-byte aligned"); return 1; }
    if (workspace_bytes < specb200_hmrtail_workspace_bytes(t, B)) { set_error("hmrtail_forward: workspace too small"); return 1; }
    if ((t->use_cam_feats || t->use_cam) && (!cam_rotmat || !cam_intr || !img_h)) { set_error("hmrtail_forward: camera inputs required"); return 1; }
    if (t->use_cam && (!bbox_scale || !bbox_center || !img_w)) { set_error("hmrtail_forward: bbox inputs required"); return 1; }
    if (!o->smpl_vertices || !o->smpl_joints3d || !o->smpl_joints2d || !o->pred_cam_t || !o->pred_pose || !o->pred_cam || !o->pred_shape || !o->pred_pose_6d) {
        set_error("hmrtail_forward: null output pointer"); return 1;
    }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    NvtxRange nvtx_tail("specb200:hmr_tail (head x3, rot6d, SMPL LBS, joints, projection)");
    const HmrWs w = hmr_carve(t, B, workspace);
    const int C = t->C, ldx = t->ldx;
    int64_t n = 0;
    // G = xf (D W2 W1[:, :C])^T + c0 : the only GEMM of the folded head
    int ks_used = HEAD_KSPLIT;                                // e.g. C = 100 yields 7 slices, not 8: sum what was written
    if (!linear_f32_launch(w.X, ldx, t->Fx, C, t->c0, nullptr, 0, w.G, 160, B, 157, C, s, HEAD_KSPLIT, static_cast<size_t>(B) * 160, &ks_used)) return 1; ++n;
    if (!head_iter_launch(w.X, ldx, C, w.G, ks_used, t->AsT, t->init157, cam_rotmat, cam_intr, img_h, t->use_cam_feats, B, s)) return 1; ++n;
    if (!smpl_prep_launch(w.X, ldx, C, t->smpl.Jt, t->smpl.Js, w.pf, w.A, w.Jp, o->pred_pose, o->ld_pose, o->pred_pose_6d, o->ld_pose_6d,
                          o->pred_shape, o->ld_shape, o->pred_cam, o->ld_cam, B, s)) return 1; ++n;
    if (!smpl_verts_launch(t->smpl.Vt, t->smpl.Sd, t->smpl.Pd, t->smpl.Wl, w.X, ldx, C, w.pf, w.A, o->smpl_vertices, o->ld_vertices, B, s)) return 1; ++n;
    if (!smpl_joints_launch(o->smpl_vertices, o->ld_vertices, w.Jp, t->Jx, w.ej, w.X, ldx, C, cam_rotmat, cam_intr, bbox_scale, bbox_center,
                            img_w, img_h, o->smpl_joints3d, o->ld_joints3d, o->smpl_joints2d, o->ld_joints2d, o->pred_cam_t, o->ld_cam_t,
                            t->use_cam, t->focal, t->img_res, B, s)) return 1; n += 2;      // extra-joint regression + joints/projection
    t->last_launches = n;
    return 0;
}

extern "C" int64_t specb200_hmrtail_last_launches(specb200_hmrtail_t* t) { return t ? t->last_launches : 0; }

extern "C" void specb200_hmrtail_destroy(specb200_hmrtail_t* t) {
    if (!t) return;
    float* ptrs[] = {t->Fx, t->c0, t->AsT, t->init157, t->Jx};
    for (float* p : ptrs) if (p) cudaFree(p);
    free_smpl(t->smpl);
    delete t;
}

// =============================================================================================== SMPL body model
struct specb200_body {
    SmplConsts smpl;
    float* JT24 = nullptr;        // J_regressor transposed, [6890][24] (regress_joints)
};

extern "C" int specb200_body_create(specb200_body_t** out, const float* v_template, const float* shapedirs, const float* posedirs,
                                    const float* J_regressor, const float* lbs_weights, const int32_t* parents) {
    if (!out || !v_template || !shapedirs || !posedirs || !J_regressor || !lbs_weights || !parents) { set_error("body_create: bad arguments"); return 1; }
    if (!check_parents(parents, "body_create")) return 1;
    specb200_body* t = new specb200_body();
    bool ok = pack_smpl(t->smpl, v_template, shapedirs, posedirs, J_regressor, lbs_weights);
    std::vector<float> JT(static_cast<size_t>(SMPL_NV) * 24);
    for (int j = 0; j < 24; ++j)
        for (int v = 0; v < SMPL_NV; ++v) JT[static_cast<size_t>(v) * 24 + j] = J_regressor[static_cast<size_t>(j) * SMPL_NV + v];
    ok = ok && upload(&t->JT24, JT);
    if (!ok) { specb200_body_destroy(t); return 1; }
    *out = t;
    return 0;
}

namespace {
struct BodyWs { float *X, *pf, *A; size_t total; };
BodyWs body_carve(int B, void* base) {
    BodyWs w;
    size_t off = 0;
    auto take = [&](size_t nfloat) { float* p = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(base) + off); off += align_up(nfloat * sizeof(float), 256); return p; };
    w.X = take(static_cast<size_t>(B) * BODY_XLD);
    w.pf = take(static_cast<size_t>(B) * PF_LD);
    w.A = take(static_cast<size_t>(B) * 288);
    w.total = off;
    return w;
}
}  // namespace

extern "C" int64_t specb200_body_workspace_bytes(specb200_body_t* t, int32_t batch) {
    if (!t || batch <= 0) { set_error("body_workspace_bytes: bad arguments"); return -1; }
    return static_cast<int64_t>(body_carve(batch, nullptr).total);
}

extern "C" int specb200_body_forward(specb200_body_t* t, int32_t B, const float* betas, const float* pose, int32_t pose_kind,
                                     void* workspace, int64_t workspace_bytes, float* verts, int64_t ld_verts, float* joints24,
                                     int64_t ld_joints24, void* stream) {
    if (!t || B <= 0 || !betas || !pose || !workspace || !verts || !joints24) { set_error("body_forward: bad arguments"); return 1; }
    if (pose_kind != 0 && pose_kind != 1) { set_error("body_forward: pose_kind must be 0 (axis-angle) or 1 (rotation matrices)"); return 1; }
    if ((reinterpret_cast<size_t>(workspace) & 255) != 0) { set_error("body_forward: workspace must be 256-byte aligned"); return 1; }
    if (workspace_bytes < specb200_body_workspace_bytes(t, B)) { set_error("body_forward: workspace too small"); return 1; }
    if (ld_verts < SMPL_NV * 3 || ld_joints24 < 72) { set_error("body_forward: output strides too small"); return 1; }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    NvtxRange nvtx_body("specb200:body_model (rodrigues, SMPL LBS)");
    const BodyWs w = body_carve(B, workspace);
    if (!body_prep_launch(betas, pose, pose_kind, t->smpl.Jt, t->smpl.Js, w.X, w.pf, w.A, joints24, ld_joints24, B, s)) return 1;
    return smpl_verts_launch(t->smpl.Vt, t->smpl.Sd, t->smpl.Pd, t->smpl.Wl, w.X, BODY_XLD, 0, w.pf, w.A, verts, ld_verts, B, s) ? 0 : 1;
}

extern "C" int specb200_body_regress_joints(specb200_body_t* t, int32_t B, const float* verts, int64_t ld_verts, const float* rot,
                                            float* joints24, void* stream) {
    if (!t || B <= 0 || !verts || !joints24 || ld_verts < SMPL_NV * 3) { set_error("body_regress_joints: bad arguments"); return 1; }
    return regress_joints24_launch(t->JT24, B, verts, ld_verts, rot, joints24, static_cast<cudaStream_t>(stream)) ? 0 : 1;
}

extern "C" void specb200_body_destroy(specb200_body_t* t) {
    if (!t) return;
    free_smpl(t->smpl);
    if (t->JT24) cudaFree(t->JT24);
    delete t;
}

// =============================================================================================== standalone
extern "C" int specb200_linear_f32(const float* a, int32_t lda, const float* w, int32_t ldw, const float* bias, float* out,
                                   int32_t ldo, int32_t m, int32_t n, int32_t k, void* stream) {
    return linear_f32_launch(a, lda, w, ldw, bias, nullptr, 0, out, ldo, m, n, k, static_cast<cudaStream_t>(stream)) ? 0 : 1;
}

// =============================================================================================== eval metrics
struct specb200_eval { float* JT = nullptr; int* map = nullptr; int n_map = 14; };

extern "C" int specb200_eval_create_mapped(specb200_eval_t** out, const float* J_host, const int32_t* map_host, int32_t n_map) {
    if (!out || !J_host || !map_host) { set_error("eval_create: bad arguments"); return 1; }
    if (n_map != 14 && n_map != 17) { set_error("eval_create: the joint mapper must have 14 or 17 entries"); return 1; }
    for (int i = 0; i < n_map; ++i) if (map_host[i] < 0 || map_host[i] >= 17) { set_error("eval_create: joint mapper out of range"); return 1; }
    specb200_eval* t = new specb200_eval();
    t->n_map = n_map;
    std::vector<float> JT(static_cast<size_t>(SMPL_NV) * 20, 0.f);
    for (int j = 0; j < 17; ++j)
        for (int v = 0; v < SMPL_NV; ++v) JT[static_cast<size_t>(v) * 20 + j] = J_host[static_cast<size_t>(j) * SMPL_NV + v];
    bool ok = upload(&t->JT, JT);
    ok = ok && check_cuda(cudaMalloc(&t->map, n_map * sizeof(int)), "cudaMalloc") &&
         check_cuda(cudaMemcpy(t->map, map_host, n_map * sizeof(int), cudaMemcpyHostToDevice), "upload");
    if (!ok) { specb200_eval_destroy(t); return 1; }
    *out = t;
    return 0;
}
extern "C" int specb200_eval_create(specb200_eval_t** out, const float* J_host, const int32_t* map_host) {
    return specb200_eval_create_mapped(out, J_host, map_host, 14);
}
extern "C" int64_t specb200_eval_workspace_bytes(specb200_eval_t* t, int32_t batch) {
    if (!t || batch <= 0) { set_error("eval_workspace_bytes: bad arguments"); return -1; }
    return static_cast<int64_t>(sizeof(float)) * (static_cast<int64_t>(2) * batch * 51 + static_cast<int64_t>(2) * batch * 3) + 256;
}
extern "C" int specb200_eval_forward_ex(specb200_eval_t* t, int32_t B, const float* pred_verts, int64_t ld_pred, const float* pred_rot,
                                        const float* gt_kp, const float* gt_verts, int64_t ld_gt, const float* gt_rot, int32_t center_v2v,
                                        void* ws, int64_t ws_bytes, float* mpjpe, float* pampjpe, float* v2v, float* pred_kp,
                                        float* mpjpe_pj, float* pampjpe_pj, int32_t n_map, void* stream) {
    if (!t || B <= 0 || !pred_verts || !ws || !mpjpe || !pampjpe) { set_error("eval_forward: bad arguments"); return 1; }
    if (n_map != t->n_map) {
        set_error("eval_forward: the handle evaluates " + std::to_string(t->n_map) + " joints, the caller passed " + std::to_string(n_map));
        return 1;
    }
    if (ws_bytes < specb200_eval_workspace_bytes(t, B)) { set_error("eval_forward: workspace too small"); return 1; }
    float* w = reinterpret_cast<float*>(align_up(reinterpret_cast<size_t>(ws), 16));
    return eval_launch(t->JT, t->map, t->n_map, B, pred_verts, ld_pred, pred_rot, gt_kp, gt_verts, ld_gt, gt_rot, center_v2v, w, mpjpe,
                       pampjpe, v2v, pred_kp, mpjpe_pj, pampjpe_pj, static_cast<cudaStream_t>(stream)) ? 0 : 1;
}
extern "C" int specb200_eval_forward(specb200_eval_t* t, int32_t B, const float* pred_verts, int64_t ld_pred, const float* gt_kp14,
                                     const float* gt_verts, int64_t ld_gt, int32_t center_v2v, void* ws, int64_t ws_bytes,
                                     float* mpjpe, float* pampjpe, float* v2v, float* pred_kp14, void* stream) {
    return specb200_eval_forward_ex(t, B, pred_verts, ld_pred, nullptr, gt_kp14, gt_verts, ld_gt, nullptr, center_v2v, ws, ws_bytes,
                                    mpjpe, pampjpe, v2v, pred_kp14, nullptr, nullptr, 14, stream);
}
extern "C" int specb200_eval_joint_errors(int32_t B, int32_t n, const float* pred, const float* gt, const float* rot_pred,
                                          const float* rot_gt, int32_t center, float* mpjpe, float* pampjpe, float* mpjpe_pj,
                                          float* pampjpe_pj, void* stream) {
    if (B <= 0 || !pred || !gt || !mpjpe || !pampjpe) { set_error("eval_joint_errors: bad arguments"); return 1; }
    return joint_errors_launch(n, B, pred, gt, rot_pred, rot_gt, center, mpjpe, pampjpe, mpjpe_pj, pampjpe_pj,
                               static_cast<cudaStream_t>(stream)) ? 0 : 1;
}
extern "C" void specb200_eval_destroy(specb200_eval_t* t) {
    if (!t) return;
    if (t->JT) cudaFree(t->JT);
    if (t->map) cudaFree(t->map);
    delete t;
}
