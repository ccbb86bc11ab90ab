// VAE decoder handle: repacked fp16 parameters keyed by the reference's state_dict names and the decode schedule.
//   reference: models/vae3d_dib.py:437-440 (VAE.decode), :369-387 (Decoder.forward), :220-226 (MidBlock),
//              :259-267 (UpBlock), :128-145 (ResnetBlock), :34-48 (VolumeAttention)
// Activations are channels-last fp16 [P, S^3, C]; every primitive is independent (GroupNorm statistics are
// per primitive), so the whole decoder is a batch of P tiny volumes.
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "kernels.cuh"

namespace tpx {
int launch_pack_conv3(const void* src, int dtype, __half* dst, int Cout, int Cin, int transposed, cudaStream_t st, int CinP = 0);
int launch_pack_convt2(const void* src, int dtype, __half* dst, int Cin, int Cout, cudaStream_t st);
}  // namespace tpx
using namespace tpx;

struct VaeRes {
    int cin, cout;
    __half *n1g, *n1b, *W1, *b1, *n2g, *n2b, *W2, *b2, *Wsc, *bsc;  // Wsc null when cin == cout
};

struct tpx_vae {
    int C0, C1, Cout, heads;
    __half* store = nullptr;
    size_t store_halves = 0;
    __half *w_pq, *b_pq, *Win, *bin;
    VaeRes res[6];                           // mid0, mid1, up0.0, up0.1, up1.0, up1.1
    __half *ang, *anb, *Wqkv, *Wap, *bap;    // mid attention
    __half *Wup, *bup;                       // [8*C0, C0], [8*C0]
    __half *nog, *nob, *Wout, *bout;         // norm_out, conv_out (padded to 16 rows)
    std::vector<std::string> required;
    std::vector<uint8_t> seen;
    bool finalized = false;
};

namespace {
const char* kResPrefix[6] = {"decoder.mid_block.nets.0.", "decoder.mid_block.nets.1.", "decoder.up_blocks.0.nets.0.", "decoder.up_blocks.0.nets.1.",
                             "decoder.up_blocks.1.nets.0.", "decoder.up_blocks.1.nets.1."};

struct HCarver {
    __half* base;
    size_t off = 0;
    __half* take(size_t n) {
        __half* p = base == nullptr ? nullptr : base + off;
        off += (n + 63) & ~static_cast<size_t>(63);   // 128-B slots (TMA operands need 16-B alignment)
        return p;
    }
};

void carve(tpx_vae* h, __half* base) {
    HCarver c{base};
    const size_t C0 = h->C0, C1 = h->C1;
    h->w_pq = c.take(8); h->b_pq = c.take(8);
    h->Win = c.take(C0 * 27); h->bin = c.take(C0);
    for (int i = 0; i < 6; ++i) {
        VaeRes& r = h->res[i];
        r.cin = i < 4 ? h->C0 : (i == 4 ? h->C0 : h->C1);
        r.cout = i < 4 ? h->C0 : h->C1;
        r.n1g = c.take(r.cin); r.n1b = c.take(r.cin);
        r.W1 = c.take(static_cast<size_t>(r.cout) * 27 * r.cin); r.b1 = c.take(r.cout);
        r.n2g = c.take(r.cout); r.n2b = c.take(r.cout);
        r.W2 = c.take(static_cast<size_t>(r.cout) * 27 * r.cout); r.b2 = c.take(r.cout);
        if (r.cin != r.cout) { r.Wsc = c.take(static_cast<size_t>(r.cout) * r.cin); r.bsc = c.take(r.cout); }
        else { r.Wsc = nullptr; r.bsc = nullptr; }
    }
    h->ang = c.take(C0); h->anb = c.take(C0);
    h->Wqkv = c.take(3 * C0 * C0); h->Wap = c.take(C0 * C0); h->bap = c.take(C0);
    h->Wup = c.take(8 * C0 * C0); h->bup = c.take(8 * C0);
    h->nog = c.take(C1); h->nob = c.take(C1);
    h->Wout = c.take(16 * 27 * C1); h->bout = c.take(16);
    h->store_halves = c.off;
}

enum SlotKind { SK_PLAIN, SK_CONV3, SK_CONV3_T, SK_CONVT2, SK_BIAS_REP8 };
struct VSlot {
    __half* ptr;
    SlotKind kind;
    std::vector<int64_t> shape;
    int a, b;  // conv dims (Cout, Cin) or (Cin, Cout)
};

bool find_vslot(tpx_vae* h, const std::string& key, VSlot* s) {
    const int64_t C0 = h->C0, C1 = h->C1;
    auto plain = [&](__half* p, std::vector<int64_t> shp) { *s = VSlot{p, SK_PLAIN, shp, 0, 0}; return true; };
    if (key == "post_quant_conv.weight") return plain(h->w_pq, {1, 1, 1, 1, 1});
    if (key == "post_quant_conv.bias") return plain(h->b_pq, {1});
    if (key == "decoder.conv_in.weight") return plain(h->Win, {C0, 1, 3, 3, 3});
    if (key == "decoder.conv_in.bias") return plain(h->bin, {C0});
    if (key == "decoder.norm_out.weight") return plain(h->nog, {C1});
    if (key == "decoder.norm_out.bias") return plain(h->nob, {C1});
    if (key == "decoder.conv_out.weight") { *s = VSlot{h->Wout, SK_CONV3_T, {C1, h->Cout, 3, 3, 3}, h->Cout, static_cast<int>(C1)}; return true; }
    if (key == "decoder.conv_out.bias") return plain(h->bout, {h->Cout});
    if (key == "decoder.up_blocks.0.upsample.weight") { *s = VSlot{h->Wup, SK_CONVT2, {C0, C0, 2, 2, 2}, static_cast<int>(C0), static_cast<int>(C0)}; return true; }
    if (key == "decoder.up_blocks.0.upsample.bias") { *s = VSlot{h->bup, SK_BIAS_REP8, {C0}, static_cast<int>(C0), 0}; return true; }
    const std::string a = "decoder.mid_block.attns.0.";
    if (key == a + "norm.weight") return plain(h->ang, {C0});
    if (key == a + "norm.bias") return plain(h->anb, {C0});
    if (key == a + "attn.qkv.weight") return plain(h->Wqkv, {3 * C0, C0});
    if (key == a + "attn.proj.weight") return plain(h->Wap, {C0, C0});
    if (key == a + "attn.proj.bias") return plain(h->bap, {C0});
    for (int i = 0; i < 6; ++i) {
        const std::string p = kResPrefix[i];
        if (key.rfind(p, 0) != 0) continue;
        VaeRes& r = h->res[i];
        const std::string t = key.substr(p.size());
        if (t == "norm1.weight") return plain(r.n1g, {r.cin});
        if (t == "norm1.bias") return plain(r.n1b, {r.cin});
        if (t == "norm2.weight") return plain(r.n2g, {r.cout});
        if (t == "norm2.bias") return plain(r.n2b, {r.cout});
        if (t == "conv1.weight") { *s = VSlot{r.W1, SK_CONV3, {r.cout, r.cin, 3, 3, 3}, r.cout, r.cin}; return true; }
        if (t == "conv1.bias") return plain(r.b1, {r.cout});
        if (t == "conv2.weight") { *s = VSlot{r.W2, SK_CONV3, {r.cout, r.cout, 3, 3, 3}, r.cout, r.cout}; return true; }
        if (t == "conv2.bias") return plain(r.b2, {r.cout});
        if (r.Wsc != nullptr && t == "shortcut.weight") return plain(r.Wsc, {r.cout, r.cin, 1, 1, 1});
        if (r.Wsc != nullptr && t == "shortcut.bias") return plain(r.bsc, {r.cout});
        return false;
    }
    return false;
}

__global__ void rep8_kernel(const __half* __restrict__ src, __half* __restrict__ dst, int C) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 8 * C) dst[i] = src[i % C];
}

struct VaeWs {
    __half *X, *T1, *T2, *X2, *Q, *K, *V, *U, *G, *sa, *sb, *sc, *sd;
    size_t total;
};
VaeWs carve_vws(const tpx_vae* h, int P, uint8_t* base) {
    VaeWs w;
    size_t off = 0;
    auto take = [&](size_t halves) { uint8_t* p = base == nullptr ? nullptr : base + off; off += (halves * 2 + 1023) & ~static_cast<size_t>(1023); return reinterpret_cast<__half*>(p); };
    const size_t S4 = static_cast<size_t>(P) * 64 * h->C0, S8 = static_cast<size_t>(P) * 512 * h->C0, s8 = static_cast<size_t>(P) * 512 * h->C1;
    w.X = take(S4); w.T1 = take(S4); w.T2 = take(S4); w.X2 = take(S4); w.Q = take(S4); w.K = take(S4); w.V = take(S4);
    w.U = take(S8); w.G = take(S8);
    w.sa = take(s8); w.sb = take(s8); w.sc = take(s8); w.sd = take(s8);
    w.total = off;
    return w;
}

int conv3(const __half* x, const __half* W, const __half* bias, const __half* resid, float alpha, __half* out, float* out32, int n_valid, int P, int S,
          int C, int Cout, int epi, cudaStream_t st) {
    // 8^3 layers with narrow outputs: the input block is staged once per output tile (conv_halo.cu) instead of once per tap
    if (conv3_halo_supported(S, C, Cout, epi)) return launch_conv3_halo(x, W, bias, resid, alpha, out, out32, n_valid, P, C, Cout, epi, st);
    GemmProblem p{};
    p.A = x; p.a_mode = AMODE_CONV3; p.conv_S = S; p.conv_C = C; p.W = W;
    p.M = P * S * S * S; p.N = Cout; p.K = 27 * C; p.BN = Cout; p.epi = epi;
    GemmArgs a{};
    a.bias = bias; a.post_scale = 1.0f; a.out0 = out; a.ldo = Cout; a.resid = resid; a.alpha = alpha; a.out32 = out32; a.n_valid = n_valid;
    a.S3 = S * S * S;
    p.args = a;
    return launch_gemm(p, st);
}

// ResnetBlock (vae3d_dib.py:128-145) on a channels-last [P, S^3, cin] volume -> out [P, S^3, cout]:
// GN+SiLU -> conv1 -> GN+SiLU -> conv2 with (x + shortcut(x)) * sqrt(1/2) in its epilogue; the 1x1 shortcut (cin != cout) goes to `sc`.
int res_block(const VaeRes& r, int P, int S, const __half* x, __half* out, __half* t1, __half* t2, __half* sc, cudaStream_t st) {
    const int S3 = S * S * S;
    const float eps = 1e-5f;
    int rc;
    if ((rc = launch_groupnorm_silu(x, r.n1g, r.n1b, P, S3, r.cin, r.cin < 32 ? r.cin : 32, eps, 1, t1, st)) != TPX_OK) return rc;
    if ((rc = conv3(t1, r.W1, r.b1, nullptr, 1.f, t2, nullptr, 0, P, S, r.cin, r.cout, EPI_STORE, st)) != TPX_OK) return rc;
    if ((rc = launch_groupnorm_silu(t2, r.n2g, r.n2b, P, S3, r.cout, r.cout < 32 ? r.cout : 32, eps, 1, t1, st)) != TPX_OK) return rc;
    const __half* resid = x;
    if (r.Wsc != nullptr) {
        GemmProblem p{};
        p.A = x; p.a_mode = AMODE_LINEAR; p.lda = r.cin; p.W = r.Wsc; p.M = P * S3; p.N = r.cout; p.K = r.cin; p.BN = r.cout; p.epi = EPI_STORE;
        GemmArgs a{};
        a.bias = r.bsc; a.post_scale = 1.0f; a.out0 = sc; a.ldo = r.cout;
        p.args = a;
        if ((rc = launch_gemm(p, st)) != TPX_OK) return rc;
        resid = sc;
    }
    return conv3(t1, r.W2, r.b2, resid, sqrtf(0.5f), out, nullptr, 0, P, S, r.cout, r.cout, EPI_RESID_SCALE, st);
}

// VolumeAttention (vae3d_dib.py:34-48) at 4^3 x C: GN -> qkv -> 64-token attention per primitive -> proj, (x + res) * sqrt(1/2)
int mid_attention(const __half* gamma, const __half* beta, const __half* Wqkv, const __half* Wproj, const __half* bproj, int heads, int P, int C,
                  const __half* x, __half* out, __half* t1, __half* t2, __half* q, __half* k, __half* v, cudaStream_t st) {
    int rc;
    if ((rc = launch_groupnorm_silu(x, gamma, beta, P, 64, C, 32, 1e-5f, 0, t1, st)) != TPX_OK) return rc;
    GemmProblem p{};
    p.A = t1; p.a_mode = AMODE_LINEAR; p.lda = C; p.W = Wqkv; p.M = P * 64; p.N = 3 * C; p.K = C; p.BN = 256; p.epi = EPI_HEADS;
    GemmArgs a{};
    a.post_scale = 1.0f; a.out0 = q; a.out1 = k; a.out2 = v; a.split_cols = C; a.Dh = 32; a.DhP = 32; a.H = heads; a.Nseq = 64;
    p.args = a;
    if ((rc = launch_gemm(p, st)) != TPX_OK) return rc;
    if ((rc = launch_attention(q, k, v, t2, P, heads, 64, 64, 32, 32, 1.0f / sqrtf(32.f), st)) != TPX_OK) return rc;
    GemmProblem pr{};
    pr.A = t2; pr.a_mode = AMODE_LINEAR; pr.lda = C; pr.W = Wproj; pr.M = P * 64; pr.N = C; pr.K = C; pr.BN = 256; pr.epi = EPI_RESID_SCALE;
    GemmArgs b{};
    b.bias = bproj; b.post_scale = 1.0f; b.out0 = out; b.ldo = C; b.resid = x; b.alpha = sqrtf(0.5f);
    pr.args = b;
    return launch_gemm(pr, st);
}

// ---- encoder ------------------------------------------------------------------------------------------------------------------------
// Its own handle and parameter store: the decoder handle, its workspace and its key contract are untouched by it.
//   reference: models/vae3d_dib.py:270-327 (Encoder), :147-184 (DownBlock), :428-435 (quant_conv, VAE.encode)
const char* kEncResPrefix[6] = {"encoder.down_blocks.0.nets.0.", "encoder.down_blocks.0.nets.1.", "encoder.down_blocks.1.nets.0.",
                                "encoder.down_blocks.1.nets.1.", "encoder.mid_block.nets.0.", "encoder.mid_block.nets.1."};
}  // namespace

struct tpx_vae_encoder {
    int Cin, L, C0, C1, heads;                // in_channels, latent_channels, down_channels (C0, C1), attention heads
    __half* store = nullptr;
    size_t store_halves = 0;
    __half *Win, *bin;                        // conv_in [C0, 27*C0]: input channels zero-padded to C0
    VaeRes res[6];                            // down0.0, down0.1 (C0 at 8^3), down1.0 (C0 -> C1), down1.1, mid0, mid1 (C1 at 4^3)
    __half *Wds, *bds;                        // down_blocks.0.downsample, stride 2
    __half *ang, *anb, *Wqkv, *Wap, *bap;     // mid attention
    __half *nog, *nob, *Wout, *bout;          // norm_out, conv_out (2L rows, padded to 16)
    __half* mix;                              // quant_conv weight [2L, 2L] then bias [2L]
    std::vector<std::string> required;
    std::vector<uint8_t> seen;
    bool finalized = false;
};

namespace {
void carve_enc(tpx_vae_encoder* h, __half* base) {
    HCarver c{base};
    const size_t C0 = h->C0, C1 = h->C1, L2 = 2 * h->L;
    h->Win = c.take(C0 * 27 * C0); h->bin = c.take(C0);
    for (int i = 0; i < 6; ++i) {
        VaeRes& r = h->res[i];
        r.cin = i < 3 ? h->C0 : h->C1;
        r.cout = i < 2 ? h->C0 : h->C1;
        r.n1g = c.take(r.cin); r.n1b = c.take(r.cin);
        r.W1 = c.take(static_cast<size_t>(r.cout) * 27 * r.cin); r.b1 = c.take(r.cout);
        r.n2g = c.take(r.cout); r.n2b = c.take(r.cout);
        r.W2 = c.take(static_cast<size_t>(r.cout) * 27 * r.cout); r.b2 = c.take(r.cout);
        if (r.cin != r.cout) { r.Wsc = c.take(static_cast<size_t>(r.cout) * r.cin); r.bsc = c.take(r.cout); }
        else { r.Wsc = nullptr; r.bsc = nullptr; }
    }
    h->Wds = c.take(C0 * 27 * C0); h->bds = c.take(C0);
    h->ang = c.take(C1); h->anb = c.take(C1);
    h->Wqkv = c.take(3 * C1 * C1); h->Wap = c.take(C1 * C1); h->bap = c.take(C1);
    h->nog = c.take(C1); h->nob = c.take(C1);
    h->Wout = c.take(16 * 27 * C1); h->bout = c.take(16);
    h->mix = c.take(L2 * L2 + L2);
    h->store_halves = c.off;
}

enum { EK_PLAIN, EK_CONV3, EK_CONV3_PADIN };
struct ESlot {
    __half* ptr;
    int kind;
    std::vector<int64_t> shape;
};

bool find_eslot(tpx_vae_encoder* h, const std::string& key, ESlot* s) {
    const int64_t C0 = h->C0, C1 = h->C1, L2 = 2 * h->L;
    auto plain = [&](__half* p, std::vector<int64_t> shp) { *s = ESlot{p, EK_PLAIN, shp}; return true; };
    auto conv = [&](__half* p, int64_t co, int64_t ci) { *s = ESlot{p, EK_CONV3, {co, ci, 3, 3, 3}}; return true; };
    if (key == "quant_conv.weight") return plain(h->mix, {L2, L2, 1, 1, 1});
    if (key == "quant_conv.bias") return plain(h->mix + L2 * L2, {L2});
    if (key == "encoder.conv_in.weight") { *s = ESlot{h->Win, EK_CONV3_PADIN, {C0, h->Cin, 3, 3, 3}}; return true; }
    if (key == "encoder.conv_in.bias") return plain(h->bin, {C0});
    if (key == "encoder.down_blocks.0.downsample.weight") return conv(h->Wds, C0, C0);
    if (key == "encoder.down_blocks.0.downsample.bias") return plain(h->bds, {C0});
    if (key == "encoder.norm_out.weight") return plain(h->nog, {C1});
    if (key == "encoder.norm_out.bias") return plain(h->nob, {C1});
    if (key == "encoder.conv_out.weight") return conv(h->Wout, L2, C1);     // rows >= 2L stay zero
    if (key == "encoder.conv_out.bias") return plain(h->bout, {L2});
    const std::string a = "encoder.mid_block.attns.0.";
    if (key == a + "norm.weight") return plain(h->ang, {C1});
    if (key == a + "norm.bias") return plain(h->anb, {C1});
    if (key == a + "attn.qkv.weight") return plain(h->Wqkv, {3 * C1, C1});
    if (key == a + "attn.proj.weight") return plain(h->Wap, {C1, C1});
    if (key == a + "attn.proj.bias") return plain(h->bap, {C1});
    for (int i = 0; i < 6; ++i) {
        const std::string p = kEncResPrefix[i];
        if (key.rfind(p, 0) != 0) continue;
        VaeRes& r = h->res[i];
        const std::string t = key.substr(p.size());
        if (t == "norm1.weight") return plain(r.n1g, {r.cin});
        if (t == "norm1.bias") return plain(r.n1b, {r.cin});
        if (t == "norm2.weight") return plain(r.n2g, {r.cout});
        if (t == "norm2.bias") return plain(r.n2b, {r.cout});
        if (t == "conv1.weight") return conv(r.W1, r.cout, r.cin);
        if (t == "conv1.bias") return plain(r.b1, {r.cout});
        if (t == "conv2.weight") return conv(r.W2, r.cout, r.cout);
        if (t == "conv2.bias") return plain(r.b2, {r.cout});
        if (r.Wsc != nullptr && t == "shortcut.weight") return plain(r.Wsc, {r.cout, r.cin, 1, 1, 1});
        if (r.Wsc != nullptr && t == "shortcut.bias") return plain(r.bsc, {r.cout});
        return false;
    }
    return false;
}

struct EncWs {
    __half *e0, *e1, *e2, *e3;              // [P, 8^3, C0]
    __half* d0;                              // [P, 4^3, C0]
    __half *X, *X2, *T1, *T2, *SC, *Q, *K, *V; // [P, 4^3, C1]
    size_t total;
};
EncWs carve_ews(const tpx_vae_encoder* h, int P, uint8_t* base) {
    EncWs w;
    size_t off = 0;
    auto take = [&](size_t halves) { uint8_t* p = base == nullptr ? nullptr : base + off; off += (halves * 2 + 1023) & ~static_cast<size_t>(1023); return reinterpret_cast<__half*>(p); };
    const size_t S8 = static_cast<size_t>(P) * 512 * h->C0, s4 = static_cast<size_t>(P) * 64 * h->C0, S4 = static_cast<size_t>(P) * 64 * h->C1;
    w.e0 = take(S8); w.e1 = take(S8); w.e2 = take(S8); w.e3 = take(S8);
    w.d0 = take(s4);
    w.X = take(S4); w.X2 = take(S4); w.T1 = take(S4); w.T2 = take(S4); w.SC = take(S4); w.Q = take(S4); w.K = take(S4); w.V = take(S4);
    w.total = off;
    return w;
}

// Stage checkpoints of the schedule (tpx_vae_encode_stage): the channels-last fp16 activation after it
enum { ES_FULL = 0, ES_CONV_IN = 1, ES_DOWN0 = 2, ES_DOWN1 = 3, ES_MID = 4 };

int encode_impl(tpx_vae_encoder* h, const void* x, int x_dtype, void* params, int params_dtype, int P, void* ws, size_t ws_bytes, int stage,
                void* stage_out, cudaStream_t st) {
    TPX_CHECK(h != nullptr && x != nullptr && ws != nullptr && (params != nullptr || stage_out != nullptr), TPX_ERR_ARG, "vae_encode: null argument");
    TPX_CHECK(h->finalized, TPX_ERR_STATE, "vae_encode: weights not finalized (set every encoder key first)");
    TPX_CHECK(P > 0, TPX_ERR_SHAPE, "vae_encode: empty batch");
    TPX_CHECK(ws_bytes >= tpx_vae_encoder_workspace_bytes(h, P), TPX_ERR_ARG, "vae_encode: workspace too small (%zu < %zu)", ws_bytes,
              tpx_vae_encoder_workspace_bytes(h, P));
    TPX_CHECK((reinterpret_cast<uintptr_t>(ws) & 255) == 0, TPX_ERR_ARG, "vae_encode: workspace must be 256-B aligned");
    TPX_CHECK(x_dtype == TPX_DTYPE_F32 || x_dtype == TPX_DTYPE_F16, TPX_ERR_ARG, "vae_encode: bad input dtype %d", x_dtype);
    TPX_CHECK(stage != ES_FULL || params_dtype == TPX_DTYPE_F32 || params_dtype == TPX_DTYPE_F16, TPX_ERR_ARG, "vae_encode: bad output dtype %d",
              params_dtype);
    int rc = tpx_device_check();
    if (rc != TPX_OK) return rc;
    EncWs w = carve_ews(h, P, static_cast<uint8_t*>(ws));
    const int C0 = h->C0, C1 = h->C1;
    auto emit = [&](const __half* act, size_t halves) -> int {
        TPX_CUDA(cudaMemcpyAsync(stage_out, act, halves * 2, cudaMemcpyDeviceToDevice, st));
        return TPX_OK;
    };
#define TPX_RC(call) do { rc = (call); if (rc != TPX_OK) return rc; } while (0)
    // conv_in Cin -> C0 at 8^3: zero-padded channels-last input through the 32-channel halo convolution
    TPX_RC(launch_vae_pack_input(x, x_dtype, P, h->Cin, C0, w.e0, st));
    TPX_RC(conv3(w.e0, h->Win, h->bin, nullptr, 1.f, w.e1, nullptr, 0, P, 8, C0, C0, EPI_STORE, st));
    if (stage == ES_CONV_IN) return emit(w.e1, static_cast<size_t>(P) * 512 * C0);
    // down_blocks.0: two ResnetBlocks C0 at 8^3, then the stride-2 convolution 8^3 -> 4^3
    TPX_RC(res_block(h->res[0], P, 8, w.e1, w.e0, w.e2, w.e3, nullptr, st));
    TPX_RC(res_block(h->res[1], P, 8, w.e0, w.e1, w.e2, w.e3, nullptr, st));
    {
        GemmProblem p{};
        p.A = w.e1; p.a_mode = AMODE_CONV3_S2; p.conv_S = 8; p.conv_C = C0; p.W = h->Wds;
        p.M = P * 64; p.N = C0; p.K = 27 * C0; p.BN = C0; p.epi = EPI_STORE;
        GemmArgs a{};
        a.bias = h->bds; a.post_scale = 1.0f; a.out0 = w.d0; a.ldo = C0; a.S3 = 64;
        p.args = a;
        TPX_RC(launch_gemm(p, st));
    }
    if (stage == ES_DOWN0) return emit(w.d0, static_cast<size_t>(P) * 64 * C0);
    // down_blocks.1: ResnetBlock C0 -> C1 (1x1 shortcut on its input), ResnetBlock C1, at 4^3
    TPX_RC(res_block(h->res[2], P, 4, w.d0, w.X, w.T1, w.T2, w.SC, st));
    TPX_RC(res_block(h->res[3], P, 4, w.X, w.X2, w.T1, w.T2, nullptr, st));
    if (stage == ES_DOWN1) return emit(w.X2, static_cast<size_t>(P) * 64 * C1);
    // mid_block (vae3d_dib.py:220-226): the decoder's blocks at the same shape
    TPX_RC(res_block(h->res[4], P, 4, w.X2, w.X, w.T1, w.T2, nullptr, st));
    TPX_RC(mid_attention(h->ang, h->anb, h->Wqkv, h->Wap, h->bap, h->heads, P, C1, w.X, w.X2, w.T1, w.T2, w.Q, w.K, w.V, st));
    TPX_RC(res_block(h->res[5], P, 4, w.X2, w.X, w.T1, w.T2, nullptr, st));
    if (stage == ES_MID) return emit(w.X, static_cast<size_t>(P) * 64 * C1);
    // norm_out + SiLU, conv_out C1 -> 2L with quant_conv (1x1, 2L -> 2L) in its epilogue -> parameters NCDHW [P, 2L, 4, 4, 4]
    TPX_RC(launch_groupnorm_silu(w.X, h->nog, h->nob, P, 64, C1, 32, 1e-5f, 1, w.T1, st));
    {
        GemmProblem p{};
        p.A = w.T1; p.a_mode = AMODE_CONV3; p.conv_S = 4; p.conv_C = C1; p.W = h->Wout;
        p.M = P * 64; p.N = 16; p.K = 27 * C1; p.BN = 16; p.epi = EPI_NCDHW_MIX;
        GemmArgs a{};
        a.bias = h->bout; a.post_scale = 1.0f; a.mix = h->mix; a.n_valid = 2 * h->L; a.S3 = 64;
        a.out0 = params_dtype == TPX_DTYPE_F16 ? static_cast<__half*>(params) : nullptr;
        a.out32 = params_dtype == TPX_DTYPE_F32 ? static_cast<float*>(params) : nullptr;
        p.args = a;
        TPX_RC(launch_gemm(p, st));
    }
#undef TPX_RC
    return TPX_OK;
}
}  // namespace

extern "C" {

int tpx_vae_create(const tpx_vae_config* c, tpx_vae** out) {
    TPX_CHECK(c != nullptr && out != nullptr, TPX_ERR_ARG, "vae_create: null argument");
    TPX_CHECK(c->latent_channels == 1, TPX_ERR_SHAPE, "vae_create: latent_channels %d unsupported (kernel set covers the shipped config: 1)", c->latent_channels);
    TPX_CHECK(c->ch_mid == 256 && c->ch_out == 32 && c->out_channels >= 1 && c->out_channels <= 16, TPX_ERR_SHAPE,
              "vae_create: up_channels (%d,%d)/out %d unsupported (kernel set covers the shipped config: (256,32)/6)", c->ch_mid, c->ch_out, c->out_channels);
    TPX_CHECK(c->attn_heads > 0 && c->ch_mid % c->attn_heads == 0 && (c->ch_mid / c->attn_heads) == 32, TPX_ERR_SHAPE, "vae_create: attention head dim must be 32");
    int rc = tpx_device_check();
    if (rc != TPX_OK) return rc;
    tpx_vae* h = new tpx_vae();
    h->C0 = c->ch_mid; h->C1 = c->ch_out; h->Cout = c->out_channels; h->heads = c->attn_heads;
    carve(h, nullptr);
    cudaError_t e = cudaMalloc(&h->store, h->store_halves * 2);
    if (e != cudaSuccess) { delete h; return cuda_fail(e, "cudaMalloc(vae parameter store)"); }
    e = cudaMemset(h->store, 0, h->store_halves * 2);
    if (e != cudaSuccess) { cudaFree(h->store); delete h; return cuda_fail(e, "cudaMemset(vae parameter store)"); }
    carve(h, h->store);
    auto& r = h->required;
    for (const char* k : {"post_quant_conv.weight", "post_quant_conv.bias", "decoder.conv_in.weight", "decoder.conv_in.bias", "decoder.norm_out.weight",
                          "decoder.norm_out.bias", "decoder.conv_out.weight", "decoder.conv_out.bias", "decoder.up_blocks.0.upsample.weight",
                          "decoder.up_blocks.0.upsample.bias", "decoder.mid_block.attns.0.norm.weight", "decoder.mid_block.attns.0.norm.bias",
                          "decoder.mid_block.attns.0.attn.qkv.weight", "decoder.mid_block.attns.0.attn.proj.weight",
                          "decoder.mid_block.attns.0.attn.proj.bias"})
        r.emplace_back(k);
    for (int i = 0; i < 6; ++i) {
        for (const char* k : {"norm1.weight", "norm1.bias", "conv1.weight", "conv1.bias", "norm2.weight", "norm2.bias", "conv2.weight", "conv2.bias"})
            r.emplace_back(std::string(kResPrefix[i]) + k);
        if (h->res[i].Wsc != nullptr) { r.emplace_back(std::string(kResPrefix[i]) + "shortcut.weight"); r.emplace_back(std::string(kResPrefix[i]) + "shortcut.bias"); }
    }
    h->seen.assign(r.size(), 0);
    *out = h;
    return TPX_OK;
}

void tpx_vae_destroy(tpx_vae* h) {
    if (h == nullptr) return;
    if (h->store != nullptr) cudaFree(h->store);
    delete h;
}

int tpx_vae_set_weight(tpx_vae* h, const char* ref_key, const void* dev_ptr, int dtype, const int64_t* shape, int ndim, void* stream) {
    TPX_CHECK(h != nullptr && ref_key != nullptr && dev_ptr != nullptr && shape != nullptr, TPX_ERR_ARG, "vae_set_weight: null argument");
    const std::string key(ref_key);
    if (key.rfind("encoder.", 0) == 0 || key.rfind("quant_conv.", 0) == 0) return 1;  // not on the decode path
    VSlot s;
    if (!find_vslot(h, key, &s)) { set_error("vae_set_weight: unexpected key '%s'", ref_key); return TPX_ERR_KEY; }
    bool ok = ndim == static_cast<int>(s.shape.size());
    long long n = 1;
    for (int i = 0; ok && i < ndim; ++i) { ok = shape[i] == s.shape[i]; n *= shape[i]; }
    TPX_CHECK(ok, TPX_ERR_SHAPE, "vae_set_weight: size mismatch for %s", ref_key);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int rc = TPX_OK;
    switch (s.kind) {
        case SK_PLAIN: rc = launch_to_half(dev_ptr, dtype, s.ptr, n, st); break;
        case SK_CONV3: rc = launch_pack_conv3(dev_ptr, dtype, s.ptr, s.a, s.b, 0, st); break;
        case SK_CONV3_T: rc = launch_pack_conv3(dev_ptr, dtype, s.ptr, s.a, s.b, 1, st); break;   // rows >= Cout stay zero
        case SK_CONVT2: rc = launch_pack_convt2(dev_ptr, dtype, s.ptr, s.a, s.b, st); break;
        case SK_BIAS_REP8: {
            rc = launch_to_half(dev_ptr, dtype, s.ptr, n, st);   // first C entries, then replicated for the 8 output offsets
            if (rc == TPX_OK) { rep8_kernel<<<(8 * s.a + 255) / 256, 256, 0, st>>>(s.ptr, s.ptr, s.a); rc = cudaGetLastError() == cudaSuccess ? TPX_OK : TPX_ERR_CUDA; }
            break;
        }
    }
    if (rc != TPX_OK) return rc;
    for (size_t i = 0; i < h->required.size(); ++i)
        if (h->required[i] == key) h->seen[i] = 1;
    h->finalized = false;
    return TPX_OK;
}

int tpx_vae_finalize(tpx_vae* h, void* stream) {
    (void)stream;
    TPX_CHECK(h != nullptr, TPX_ERR_ARG, "vae_finalize: null handle");
    for (size_t i = 0; i < h->required.size(); ++i) TPX_CHECK(h->seen[i], TPX_ERR_STATE, "vae_finalize: missing key '%s' in state_dict", h->required[i].c_str());
    h->finalized = true;
    return TPX_OK;
}

size_t tpx_vae_workspace_bytes(const tpx_vae* h, int P) {
    if (h == nullptr || P <= 0) return 0;
    return carve_vws(h, P, nullptr).total;
}

int tpx_vae_decode(tpx_vae* h, const void* z, int z_dtype, void* out, int out_dtype, int P, void* ws, size_t ws_bytes, void* stream) {
    TPX_CHECK(h != nullptr && z != nullptr && out != nullptr && ws != nullptr, TPX_ERR_ARG, "vae_decode: null argument");
    TPX_CHECK(h->finalized, TPX_ERR_STATE, "vae_decode: weights not finalized (load_state_dict first)");
    TPX_CHECK(P > 0, TPX_ERR_SHAPE, "vae_decode: empty batch");
    TPX_CHECK(ws_bytes >= tpx_vae_workspace_bytes(h, P), TPX_ERR_ARG, "vae_decode: workspace too small (%zu < %zu)", ws_bytes, tpx_vae_workspace_bytes(h, P));
    TPX_CHECK((reinterpret_cast<uintptr_t>(ws) & 255) == 0, TPX_ERR_ARG, "vae_decode: workspace must be 256-B aligned");
    TPX_CHECK(out_dtype == TPX_DTYPE_F32 || out_dtype == TPX_DTYPE_F16, TPX_ERR_ARG, "vae_decode: bad output dtype %d", out_dtype);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    VaeWs w = carve_vws(h, P, static_cast<uint8_t*>(ws));
    const int C0 = h->C0, C1 = h->C1;
    const float skip = sqrtf(0.5f);
    const float eps = 1e-5f;
    int rc;
#define TPX_RC(call) do { rc = (call); if (rc != TPX_OK) return rc; } while (0)
    TPX_RC(launch_vae_conv_in(z, z_dtype, h->w_pq, h->b_pq, h->Win, h->bin, P, C0, w.X, st));
    __half *X = w.X, *X2 = w.X2;
    auto res4 = [&](const VaeRes& r) -> int {   // ResnetBlock C0->C0 at 4^3
        const int rc2 = res_block(r, P, 4, X, X2, w.T1, w.T2, nullptr, st);
        std::swap(X, X2);
        return rc2;
    };
    TPX_RC(res4(h->res[0]));
    TPX_RC(mid_attention(h->ang, h->anb, h->Wqkv, h->Wap, h->bap, h->heads, P, C0, X, X2, w.T1, w.T2, w.Q, w.K, w.V, st));
    std::swap(X, X2);
    TPX_RC(res4(h->res[1]));
    TPX_RC(res4(h->res[2]));
    TPX_RC(res4(h->res[3]));
    {   // ConvTranspose3d(k2,s2): 8 independent 1x1 GEMMs, one per output offset (a,b,c); each writes its stride-2 sub-lattice of the
        // 8^3 volume with bulk tensor stores (full 128-B lines; the single N = 8*C0 GEMM with a per-thread scatter epilogue was store-bound)
        for (int abc = 0; abc < 8; ++abc) {
            GemmProblem p{};
            p.A = X; p.a_mode = AMODE_LINEAR; p.lda = C0; p.W = h->Wup + static_cast<size_t>(abc) * C0 * C0; p.M = P * 64; p.N = C0; p.K = C0; p.BN = 256;
            p.epi = EPI_STORE;
            GemmArgs a{};
            a.bias = h->bup + static_cast<size_t>(abc) * C0; a.post_scale = 1.0f; a.ldo = C0; a.convt_store = 1;
            a.out0 = w.U + (static_cast<size_t>((abc >> 2) * 8 + ((abc >> 1) & 1)) * 8 + (abc & 1)) * C0;
            p.args = a;
            TPX_RC(launch_gemm(p, st));
        }
    }
    {   // ResnetBlock C0 -> C1 at 8^3 with 1x1 shortcut
        const VaeRes& r = h->res[4];
        TPX_RC(launch_groupnorm_silu(w.U, r.n1g, r.n1b, P, 512, C0, 32, eps, 1, w.G, st));
        TPX_RC(conv3(w.G, r.W1, r.b1, nullptr, 1.f, w.sa, nullptr, 0, P, 8, C0, C1, EPI_STORE, st));
        TPX_RC(launch_groupnorm_silu(w.sa, r.n2g, r.n2b, P, 512, C1, 32, eps, 1, w.sb, st));
        GemmProblem p{};
        p.A = w.U; p.a_mode = AMODE_LINEAR; p.lda = C0; p.W = r.Wsc; p.M = P * 512; p.N = C1; p.K = C0; p.BN = 32; p.epi = EPI_STORE;
        GemmArgs a{};
        a.bias = r.bsc; a.post_scale = 1.0f; a.out0 = w.sc; a.ldo = C1;
        p.args = a;
        TPX_RC(launch_gemm(p, st));
        TPX_RC(conv3(w.sb, r.W2, r.b2, w.sc, skip, w.sd, nullptr, 0, P, 8, C1, C1, EPI_RESID_SCALE, st));
    }
    {   // ResnetBlock C1 -> C1 at 8^3
        const VaeRes& r = h->res[5];
        TPX_RC(launch_groupnorm_silu(w.sd, r.n1g, r.n1b, P, 512, C1, 32, eps, 1, w.sa, st));
        TPX_RC(conv3(w.sa, r.W1, r.b1, nullptr, 1.f, w.sb, nullptr, 0, P, 8, C1, C1, EPI_STORE, st));
        TPX_RC(launch_groupnorm_silu(w.sb, r.n2g, r.n2b, P, 512, C1, 32, eps, 1, w.sa, st));
        TPX_RC(conv3(w.sa, r.W2, r.b2, w.sd, skip, w.sc, nullptr, 0, P, 8, C1, C1, EPI_RESID_SCALE, st));
    }
    TPX_RC(launch_groupnorm_silu(w.sc, h->nog, h->nob, P, 512, C1, 32, eps, 1, w.sa, st));
    TPX_RC(conv3(w.sa, h->Wout, h->bout, nullptr, 1.f, out_dtype == TPX_DTYPE_F16 ? static_cast<__half*>(out) : nullptr,
                 out_dtype == TPX_DTYPE_F32 ? static_cast<float*>(out) : nullptr, h->Cout, P, 8, C1, 16, EPI_NCDHW, st));
#undef TPX_RC
    return TPX_OK;
}

int tpx_vae_encoder_create(const tpx_vae_encoder_config* c, tpx_vae_encoder** out) {
    TPX_CHECK(c != nullptr && out != nullptr, TPX_ERR_ARG, "vae_encoder_create: null argument");
    TPX_CHECK(c->latent_channels == 1, TPX_ERR_SHAPE, "vae_encoder_create: latent_channels %d unsupported (kernel set covers the shipped config: 1)",
              c->latent_channels);
    TPX_CHECK(c->in_channels >= 1 && c->in_channels <= 16, TPX_ERR_SHAPE, "vae_encoder_create: in_channels %d unsupported (1..16)", c->in_channels);
    TPX_CHECK(c->ch0 == 32 && c->ch1 == 256, TPX_ERR_SHAPE, "vae_encoder_create: down_channels (%d,%d) unsupported (kernel set covers the shipped config: (32,256))",
              c->ch0, c->ch1);
    TPX_CHECK(c->attn_heads > 0 && c->ch1 % c->attn_heads == 0 && (c->ch1 / c->attn_heads) == 32, TPX_ERR_SHAPE, "vae_encoder_create: attention head dim must be 32");
    int rc = tpx_device_check();
    if (rc != TPX_OK) return rc;
    tpx_vae_encoder* h = new tpx_vae_encoder();
    h->Cin = c->in_channels; h->L = c->latent_channels; h->C0 = c->ch0; h->C1 = c->ch1; h->heads = c->attn_heads;
    carve_enc(h, nullptr);
    cudaError_t e = cudaMalloc(&h->store, h->store_halves * 2);
    if (e != cudaSuccess) { delete h; return cuda_fail(e, "cudaMalloc(vae encoder parameter store)"); }
    e = cudaMemset(h->store, 0, h->store_halves * 2);
    if (e != cudaSuccess) { cudaFree(h->store); delete h; return cuda_fail(e, "cudaMemset(vae encoder parameter store)"); }
    carve_enc(h, h->store);
    auto& r = h->required;
    for (const char* k : {"encoder.conv_in.weight", "encoder.conv_in.bias", "encoder.down_blocks.0.downsample.weight", "encoder.down_blocks.0.downsample.bias",
                          "encoder.mid_block.attns.0.norm.weight", "encoder.mid_block.attns.0.norm.bias", "encoder.mid_block.attns.0.attn.qkv.weight",
                          "encoder.mid_block.attns.0.attn.proj.weight", "encoder.mid_block.attns.0.attn.proj.bias", "encoder.norm_out.weight",
                          "encoder.norm_out.bias", "encoder.conv_out.weight", "encoder.conv_out.bias", "quant_conv.weight", "quant_conv.bias"})
        r.emplace_back(k);
    for (int i = 0; i < 6; ++i) {
        for (const char* k : {"norm1.weight", "norm1.bias", "conv1.weight", "conv1.bias", "norm2.weight", "norm2.bias", "conv2.weight", "conv2.bias"})
            r.emplace_back(std::string(kEncResPrefix[i]) + k);
        if (h->res[i].Wsc != nullptr) { r.emplace_back(std::string(kEncResPrefix[i]) + "shortcut.weight"); r.emplace_back(std::string(kEncResPrefix[i]) + "shortcut.bias"); }
    }
    h->seen.assign(r.size(), 0);
    *out = h;
    return TPX_OK;
}

void tpx_vae_encoder_destroy(tpx_vae_encoder* h) {
    if (h == nullptr) return;
    if (h->store != nullptr) cudaFree(h->store);
    delete h;
}

int tpx_vae_encoder_set_weight(tpx_vae_encoder* h, const char* ref_key, const void* dev_ptr, int dtype, const int64_t* shape, int ndim, void* stream) {
    TPX_CHECK(h != nullptr && ref_key != nullptr && dev_ptr != nullptr && shape != nullptr, TPX_ERR_ARG, "vae_encoder_set_weight: null argument");
    const std::string key(ref_key);
    if (key.rfind("encoder.", 0) != 0 && key.rfind("quant_conv.", 0) != 0) return 1;   // decoder.* / post_quant_conv.*: not on the encode path
    ESlot s;
    if (!find_eslot(h, key, &s)) { set_error("vae_encoder_set_weight: unexpected key '%s'", ref_key); return TPX_ERR_KEY; }
    bool ok = ndim == static_cast<int>(s.shape.size());
    long long n = 1;
    for (int i = 0; ok && i < ndim; ++i) { ok = shape[i] == s.shape[i]; n *= shape[i]; }
    TPX_CHECK(ok, TPX_ERR_SHAPE, "vae_encoder_set_weight: size mismatch for %s", ref_key);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int rc = TPX_OK;
    switch (s.kind) {
        case EK_PLAIN: rc = launch_to_half(dev_ptr, dtype, s.ptr, n, st); break;
        case EK_CONV3: rc = launch_pack_conv3(dev_ptr, dtype, s.ptr, static_cast<int>(s.shape[0]), static_cast<int>(s.shape[1]), 0, st); break;
        case EK_CONV3_PADIN: rc = launch_pack_conv3(dev_ptr, dtype, s.ptr, static_cast<int>(s.shape[0]), static_cast<int>(s.shape[1]), 0, st, h->C0); break;
    }
    if (rc != TPX_OK) return rc;
    for (size_t i = 0; i < h->required.size(); ++i)
        if (h->required[i] == key) h->seen[i] = 1;
    h->finalized = false;
    return TPX_OK;
}

int tpx_vae_encoder_finalize(tpx_vae_encoder* h, void* stream) {
    (void)stream;
    TPX_CHECK(h != nullptr, TPX_ERR_ARG, "vae_encoder_finalize: null handle");
    for (size_t i = 0; i < h->required.size(); ++i) TPX_CHECK(h->seen[i], TPX_ERR_STATE, "vae_encoder_finalize: missing key '%s' in state_dict", h->required[i].c_str());
    h->finalized = true;
    return TPX_OK;
}

size_t tpx_vae_encoder_workspace_bytes(const tpx_vae_encoder* h, int P) {
    if (h == nullptr || P <= 0) return 0;
    return carve_ews(h, P, nullptr).total;
}

int tpx_vae_encode(tpx_vae_encoder* h, const void* x, int x_dtype, void* params, int params_dtype, int P, void* ws, size_t ws_bytes, void* stream) {
    return encode_impl(h, x, x_dtype, params, params_dtype, P, ws, ws_bytes, ES_FULL, nullptr, static_cast<cudaStream_t>(stream));
}

int tpx_vae_encode_stage(tpx_vae_encoder* h, const void* x, int x_dtype, int P, int stage, void* out, void* ws, size_t ws_bytes, void* stream) {
    TPX_CHECK(stage >= ES_CONV_IN && stage <= ES_MID, TPX_ERR_ARG, "vae_encode_stage: stage %d out of range (1..4)", stage);
    TPX_CHECK(out != nullptr, TPX_ERR_ARG, "vae_encode_stage: null output");
    return encode_impl(h, x, x_dtype, nullptr, TPX_DTYPE_F16, P, ws, ws_bytes, stage, out, static_cast<cudaStream_t>(stream));
}

int tpx_vae_posterior(const void* params, int dtype, int64_t batch, int64_t half_elems, int deterministic, void* logvar, void* std_out, void* var,
                      void* stream) {
    TPX_CHECK(batch >= 0 && half_elems >= 0, TPX_ERR_ARG, "vae_posterior: negative size");
    if (batch * half_elems == 0) return TPX_OK;
    TPX_CHECK(params != nullptr && logvar != nullptr && std_out != nullptr && var != nullptr, TPX_ERR_ARG, "vae_posterior: null argument");
    int rc = tpx_device_check();
    if (rc != TPX_OK) return rc;
    return launch_vae_posterior(params, dtype, batch, half_elems, deterministic, logvar, std_out, var, static_cast<cudaStream_t>(stream));
}

int tpx_conv3d_k3_s2(const void* x, const void* W, const void* bias, void* out, int P, int C, int Cout, void* stream) {
    TPX_CHECK(x != nullptr && W != nullptr && out != nullptr, TPX_ERR_ARG, "conv3d_k3_s2: null argument");
    TPX_CHECK(P > 0, TPX_ERR_SHAPE, "conv3d_k3_s2: empty batch");
    int rc = tpx_device_check();
    if (rc != TPX_OK) return rc;
    GemmProblem p{};
    p.A = static_cast<const __half*>(x); p.a_mode = AMODE_CONV3_S2; p.conv_S = 8; p.conv_C = C; p.W = static_cast<const __half*>(W);
    p.M = P * 64; p.N = Cout; p.K = 27 * C; p.BN = Cout; p.epi = EPI_STORE;
    GemmArgs a{};
    a.bias = static_cast<const __half*>(bias); a.post_scale = 1.0f; a.out0 = static_cast<__half*>(out); a.ldo = Cout; a.S3 = 64;
    p.args = a;
    return launch_gemm(p, static_cast<cudaStream_t>(stream));
}

int tpx_primsdf_query(const float* x, const float* srt, const float* feat, int64_t n, int K, int S, int dim_feat, int inference, float* out, void* stream) {
    if (n == 0) return TPX_OK;
    TPX_CHECK(n > 0 && x != nullptr && srt != nullptr && feat != nullptr && out != nullptr, TPX_ERR_ARG, "primsdf_query: null argument or negative n");
    return launch_primsdf_query(x, srt, feat, n, K, S, dim_feat, inference, out, static_cast<cudaStream_t>(stream));
}

int tpx_raymarch_preview(const float* tpl, const float* primpos, const float* primrot, const float* primscale, const float* campos, const float* camrot,
                         const float* focal, const float* princpt, int N, int K, int S, int H, int W, float volradius, float stepsize, float fadescale,
                         float fadeexp, float* rgba_out, void* stream) {
    TPX_CHECK(tpl != nullptr && primpos != nullptr && primrot != nullptr && primscale != nullptr && campos != nullptr && camrot != nullptr && focal != nullptr &&
                  princpt != nullptr && rgba_out != nullptr,
              TPX_ERR_ARG, "raymarch_preview: null argument");
    int rc = tpx_device_check();
    if (rc != TPX_OK) return rc;
    return launch_raymarch_preview(tpl, primpos, primrot, primscale, campos, camrot, focal, princpt, N, K, S, H, W, volradius, stepsize, fadescale, fadeexp, rgba_out,
                                   static_cast<cudaStream_t>(stream));
}

size_t tpx_primsdf_grid_bytes(int64_t cap_entries) { return cap_entries > 0 ? primsdf_grid_bytes(cap_entries) : 0; }

int tpx_primsdf_grid_build(const float* srt, int K, void* grid_ws, size_t grid_bytes, void* stream) {
    TPX_CHECK(srt != nullptr && grid_ws != nullptr, TPX_ERR_ARG, "primsdf_grid_build: null argument");
    int rc = tpx_device_check();
    if (rc != TPX_OK) return rc;
    return launch_primsdf_grid_build(srt, K, grid_ws, grid_bytes, static_cast<cudaStream_t>(stream));
}

int tpx_primsdf_query_grid(const float* x, const float* srt, const float* feat, const void* grid_ws, size_t grid_bytes, int64_t n, int K, int S, int dim_feat,
                           int inference, float* out, void* stream) {
    if (n == 0) return TPX_OK;
    TPX_CHECK(n > 0 && x != nullptr && srt != nullptr && feat != nullptr && out != nullptr && grid_ws != nullptr, TPX_ERR_ARG,
              "primsdf_query_grid: null argument or negative n");
    return launch_primsdf_query_grid(x, srt, feat, grid_ws, grid_bytes, n, K, S, dim_feat, inference, out, static_cast<cudaStream_t>(stream));
}

int tpx_groupnorm_silu(const void* x, const void* gamma, const void* beta, int P, int S3, int C, int groups, float eps, int apply_silu, void* out,
                       void* stream) {
    TPX_CHECK(x != nullptr && gamma != nullptr && beta != nullptr && out != nullptr, TPX_ERR_ARG, "groupnorm_silu: null argument");
    return launch_groupnorm_silu(static_cast<const __half*>(x), static_cast<const __half*>(gamma), static_cast<const __half*>(beta), P, S3, C, groups, eps,
                                 apply_silu, static_cast<__half*>(out), static_cast<cudaStream_t>(stream));
}

int tpx_conv3d_k3(const void* x, const void* W, const void* bias, const void* resid, float alpha, void* out, int P, int S, int C, int Cout, void* stream) {
    TPX_CHECK(x != nullptr && W != nullptr && out != nullptr, TPX_ERR_ARG, "conv3d_k3: null argument");
    int rc = tpx_device_check();
    if (rc != TPX_OK) return rc;
    const bool plain = resid == nullptr && alpha == 1.0f;
    return conv3(static_cast<const __half*>(x), static_cast<const __half*>(W), static_cast<const __half*>(bias), static_cast<const __half*>(resid), alpha,
                 static_cast<__half*>(out), nullptr, 0, P, S, C, Cout, plain ? EPI_STORE : EPI_RESID_SCALE, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
