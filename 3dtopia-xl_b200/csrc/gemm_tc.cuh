// Persistent, warp-specialised tcgen05 GEMM for sm_100a:   C[M,N] = A[M,K] * W[N,K]^T  (+ fused epilogue)
//
//   warp 0   : TMA producer  (cp.async.bulk.tensor -> 128B/64B-swizzled smem ring, mbarrier complete_tx)
//   warp 1   : MMA issuer    (one thread: tcgen05.mma cta_group::1 kind::f16, 128 x BN x 16, fp32 accum in TMEM)
//   warp 2   : TMEM allocator
//   warps 4-7: epilogue      (tcgen05.ld 32x32b, one accumulator row per thread; fused bias / GELU / gated
//                             residual / head split / conv scatter; 16-byte stores)
//   Two TMEM accumulator stages so the epilogue of tile i overlaps the MMAs of tile i+1.
//
// A-operand modes: AMODE_LINEAR (2-D tensor map over a row-major [M,K] fp16 matrix) and AMODE_CONV3 (5-D tensor
// map over a channels-last [P,S,S,S,C] fp16 volume: the 27 taps of a 3x3x3 / pad 1 convolution are 27 shifted
// box loads, the halo comes from TMA out-of-bounds zero fill — implicit GEMM with no im2col buffer).
// AMODE_CONV3_S2 is the stride-2 version over an 8^3 input (the encoder's downsample, vae3d_dib.py:168): the tensor
// map traverses x / y / z with element stride 2, so one box of 8^3 voxels delivers the 4^3 input voxels a tap reads
// for two primitives (128 rows); the tap offset is the box start (dx-1, dy-1, dz-1), the pad-1 halo the zero fill.
#pragma once
#include "tpx_common.cuh"

namespace tpx {

enum GemmEpiMode : int {
    EPI_STORE = 0,       // out0[row*ldo+col] = h( h(acc+bias) * post_scale )
    EPI_GELU = 1,        // out0 = h( gelu_tanh( h(acc+bias) ) )
    EPI_HEADS = 2,       // split columns into (which, head, d) -> out{which}[b,head,n,DhP]  (zero pad written)
    EPI_GATED = 3,       // xres[row*ldx+col] += float( h( gate[b,col] * h(acc+bias) ) )
    EPI_RESID_SCALE = 4, // out0 = h( (acc + bias + resid[row*ldo+col]) * alpha )
    EPI_CONVT2 = 5,      // k2s2 transposed conv scatter: col=(abc,co), row=(p,z,y,x)@4^3 -> channels-last 8^3
    EPI_NCDHW = 6,       // out[(p*Cout+co)*S3 + vox] = acc + bias   (fp32 or fp16 out, co < n_valid)
    EPI_NCDHW_MIX = 7,   // out[(p*n_valid+j)*S3 + vox] = sum_c mix[j,c] * h(acc_c + bias_c) + mix_bias[j]   (a 1x1 conv folded in)
};
enum GemmAMode : int { AMODE_LINEAR = 0, AMODE_CONV3 = 1, AMODE_CONV3_S2 = 2 };

struct GemmArgs {
    int M, N, num_kb;
    int conv_S, chunks_per_tap;
    const __half* bias;
    float post_scale;
    __half* out0;
    __half* out1;
    __half* out2;
    int ldo;
    int split_cols, Dh, DhP, H, Nseq;
    int vt_which_plus1, vt_ld;   // EPI_HEADS: column group (which+1) stored TRANSPOSED as [b,head,DhP,vt_ld] (keys contiguous); 0 = none
    float* xres;
    int ldx;
    const __half* gate;
    int gate_bstride, rows_per_batch, gate_batches;
    const __half* resid;
    float alpha;
    float* out32;
    int n_valid, S3;
    int convt_store;  // EPI_STORE: 1 = rows are (primitive, 4^3 voxel) and the output map is the 5-D stride-2 lattice of one (a,b,c) offset of
                      // a ConvTranspose3d(k2,s2): a warp's 32 rows are one [2 z][4 y][4 x] box (vae3d_dib.py:220-226)
    int pdl_trigger;  // 2-CTA kernel: 1 = griddepcontrol.launch_dependents after the prologue (launched with the PDL attribute)
    int heads_tma;    // EPI_HEADS: 1 = outputs leave as 24-column bulk tensor stores (launcher checked the geometry, padding is pre-zeroed)
    long long* dbg;   // timeline probe (tpx_debug_gemm_timeline): 16 int64 per CTA, nullptr in the product path
    const __half* mix;   // EPI_NCDHW_MIX: [n_valid, n_valid] channel-mix weight followed by its [n_valid] bias (n_valid <= 4)
};

template <int BN, int BK>
struct GemmCfg {
    static constexpr int BM = 128;
    static constexpr int SW = BK * 2;
    static constexpr int A_BYTES = BM * BK * 2;
    static constexpr int B_BYTES = BN * BK * 2;
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int STAGES_RAW = (192 * 1024) / STAGE_BYTES;
    static constexpr int STAGES = STAGES_RAW > 8 ? 8 : STAGES_RAW;
    static constexpr int TMEM_COLS = (2 * BN <= 32) ? 32 : (2 * BN <= 64) ? 64 : (2 * BN <= 128) ? 128 : (2 * BN <= 256) ? 256 : 512;
    // epilogue staging for the TMA stores: per epilogue warp two buffers of 32 rows x 128 B (1024-B aligned: 128-B swizzle)
    static constexpr int STAGING_BYTES = (BN % 64 == 0 || BN % 24 == 0) ? 4 * 2 * 4096 : 0;
    // dynamic shared memory is declared __align__(1024) (the kernel traps if the base is not), so no alignment slack is budgeted
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + STAGING_BYTES + 256 /*barriers*/ + 2048 /*bias + gate tile, fp32*/;
    static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
    static_assert(B_BYTES % 1024 == 0 && A_BYTES % 1024 == 0, "stage operands must stay 1024-B aligned");
    static_assert(BN % 16 == 0 && BN <= 256, "UMMA N");
};

__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}

union Pack8 {
    uint4 u;
    __half2 h2[4];
    __half h[8];
};

// ---- epilogue ---------------------------------------------------------------------------------------------------
// One thread owns one accumulator row; columns arrive in chunks of CH (32) fp32 values from TMEM.  bias (and the
// adaLN gate when it is uniform over the tile's rows) are staged once per tile in shared memory as fp32, every
// global load of a chunk is issued before the first use, and the (which, head, d) split of a column is advanced
// incrementally instead of divided out per group.
struct HeadCursor {
    int which, head, d;
    int b, n;   // batch / token of this thread's row
};

__device__ __forceinline__ float gelu_tanh_fast(float x) {
    // 0.5 x (1 + tanh(u)),  tanh(u) = 1 - 2 / (1 + e^{2u});  MUFU.EX2 + MUFU.RCP, abs error ~1e-7 (fp16 output)
    const float u = 0.7978845608028654f * (x + 0.044715f * x * x * x);
    const float e = __expf(2.0f * u);
    const float th = 1.0f - __fdividef(2.0f, 1.0f + e);
    return 0.5f * x * (1.0f + th);
}

// h(a), h(b) as floats through ONE packed conversion (F2FP.F16.F32.PACK_AB, ALU pipe); the scalar cvt.rn.f16.f32 is an XU-pipe
// instruction (16 / clk / SM, shared with MUFU) and was the bound of the GELU / gated epilogues.
__device__ __forceinline__ float2 round_h2(float a, float b) { return __half22float2(__floats2half2_rn(a, b)); }
// gelu_tanh(x) = 0.5 x (1 + tanh(u)) = x * sigmoid(2u),  u = sqrt(2/pi) (x + 0.044715 x^3):  x / (1 + 2^(-2 u log2 e)).
// Five FMA-pipe operations + MUFU.EX2 + MUFU.RCP; saturates cleanly (2^+inf -> rcp(inf) = 0, 2^-inf -> 1).
__device__ __forceinline__ float gelu_tanh_sigmoid(float x) {
    const float k0 = -2.0f * 0.7978845608028654f * 1.4426950408889634f, k1 = k0 * 0.044715f;
    const float t = x * x;
    const float arg = x * fmaf(k1, t, k0);
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(arg));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + e));
    return x * r;
}

template <int EPI, int CH>
__device__ __forceinline__ void epi_chunk(const GemmArgs& g, const float* __restrict__ sb, const float* __restrict__ sg, bool gate_in_smem, int row,
                                          bool row_ok, int col0, int c0, const uint32_t* acc, HeadCursor& hc, size_t head_row_off) {
    constexpr int NG = CH / 8;
    float v[CH];
#pragma unroll
    for (int i = 0; i < CH; i += 4) {
        const float4 b4 = *reinterpret_cast<const float4*>(sb + c0 + i);
        v[i] = __uint_as_float(acc[i]) + b4.x;
        v[i + 1] = __uint_as_float(acc[i + 1]) + b4.y;
        v[i + 2] = __uint_as_float(acc[i + 2]) + b4.z;
        v[i + 3] = __uint_as_float(acc[i + 3]) + b4.w;
    }
    bool ok[NG];
#pragma unroll
    for (int j = 0; j < NG; ++j) ok[j] = row_ok && (col0 + j * 8 < g.N);

    if constexpr (EPI == EPI_STORE || EPI == EPI_GELU) {
        __half* op = g.out0 + static_cast<size_t>(row) * g.ldo + col0;
#pragma unroll
        for (int j = 0; j < NG; ++j) {
            Pack8 o;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                float x = h2f_round(v[j * 8 + i]);
                if constexpr (EPI == EPI_GELU) x = gelu_tanh_fast(x);
                else if (g.post_scale != 1.0f) x = x * g.post_scale;
                o.h[i] = __float2half_rn(x);
            }
            if (ok[j]) *reinterpret_cast<uint4*>(op + j * 8) = o.u;
        }
    } else if constexpr (EPI == EPI_HEADS) {
#pragma unroll
        for (int j = 0; j < NG; ++j) {
            __half* base = hc.which == 0 ? g.out0 : (hc.which == 1 ? g.out1 : g.out2);
            const bool sc = g.post_scale != 1.0f && hc.which == 0;
            Pack8 o;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                float x = h2f_round(v[j * 8 + i]);
                if (sc) x = x * g.post_scale;
                o.h[i] = __float2half_rn(x);
            }
            if (hc.which + 1 == g.vt_which_plus1) {
                // transposed store for the tcgen05 attention's PV operand: [b, head, d, token] (tokens contiguous)
                __half* dst = base + (static_cast<size_t>(hc.b * g.H + hc.head) * g.DhP + hc.d) * g.vt_ld + hc.n;
                if (ok[j]) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) dst[static_cast<size_t>(i) * g.vt_ld] = o.h[i];
                    if (hc.d + 8 == g.Dh)
                        for (int p = g.Dh; p < g.DhP; ++p) dst[static_cast<size_t>(p - hc.d) * g.vt_ld] = __float2half_rn(0.f);
                }
            } else {
                __half* dst = base + head_row_off + static_cast<size_t>(hc.head) * g.Nseq * g.DhP + hc.d;
                if (ok[j]) {
                    *reinterpret_cast<uint4*>(dst) = o.u;
                    if (hc.d + 8 == g.Dh)   // last real group of this head: write the zero padding d in [Dh, DhP)
                        for (int p = g.Dh; p < g.DhP; p += 8) *reinterpret_cast<uint4*>(dst + (p - hc.d)) = make_uint4(0, 0, 0, 0);
                }
            }
            hc.d += 8;
            if (hc.d >= g.Dh) {
                hc.d = 0;
                if (++hc.head == g.H) { hc.head = 0; ++hc.which; }
            }
        }
    } else if constexpr (EPI == EPI_GATED) {
        float* xp = g.xres + static_cast<size_t>(row) * g.ldx + col0;
        float4 xr[2 * NG];
#pragma unroll
        for (int j = 0; j < NG; ++j) {
            xr[2 * j] = ok[j] ? *reinterpret_cast<const float4*>(xp + j * 8) : make_float4(0.f, 0.f, 0.f, 0.f);
            xr[2 * j + 1] = ok[j] ? *reinterpret_cast<const float4*>(xp + j * 8 + 4) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        float gt[CH];
        if (gate_in_smem) {
#pragma unroll
            for (int i = 0; i < CH; i += 4) {
                const float4 g4 = *reinterpret_cast<const float4*>(sg + c0 + i);
                gt[i] = g4.x; gt[i + 1] = g4.y; gt[i + 2] = g4.z; gt[i + 3] = g4.w;
            }
        } else {
            const int b = (row / g.rows_per_batch) % g.gate_batches;
            const __half* gp = g.gate + static_cast<size_t>(b) * g.gate_bstride + col0;
#pragma unroll
            for (int j = 0; j < NG; ++j) {
                Pack8 t;
                t.u = ok[j] ? *reinterpret_cast<const uint4*>(gp + j * 8) : make_uint4(0, 0, 0, 0);
#pragma unroll
                for (int i = 0; i < 8; ++i) gt[j * 8 + i] = __half2float(t.h[i]);
            }
        }
#pragma unroll
        for (int j = 0; j < NG; ++j) {
            float4 a = xr[2 * j], c = xr[2 * j + 1];
            a.x += h2f_round(gt[j * 8 + 0] * h2f_round(v[j * 8 + 0]));
            a.y += h2f_round(gt[j * 8 + 1] * h2f_round(v[j * 8 + 1]));
            a.z += h2f_round(gt[j * 8 + 2] * h2f_round(v[j * 8 + 2]));
            a.w += h2f_round(gt[j * 8 + 3] * h2f_round(v[j * 8 + 3]));
            c.x += h2f_round(gt[j * 8 + 4] * h2f_round(v[j * 8 + 4]));
            c.y += h2f_round(gt[j * 8 + 5] * h2f_round(v[j * 8 + 5]));
            c.z += h2f_round(gt[j * 8 + 6] * h2f_round(v[j * 8 + 6]));
            c.w += h2f_round(gt[j * 8 + 7] * h2f_round(v[j * 8 + 7]));
            if (ok[j]) {
                *reinterpret_cast<float4*>(xp + j * 8) = a;
                *reinterpret_cast<float4*>(xp + j * 8 + 4) = c;
            }
        }
    } else if constexpr (EPI == EPI_RESID_SCALE) {
        const size_t off = static_cast<size_t>(row) * g.ldo + col0;
        Pack8 rs[NG];
#pragma unroll
        for (int j = 0; j < NG; ++j) rs[j].u = (ok[j] && g.resid != nullptr) ? *reinterpret_cast<const uint4*>(g.resid + off + j * 8) : make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int j = 0; j < NG; ++j) {
            Pack8 o;
#pragma unroll
            for (int i = 0; i < 8; ++i) o.h[i] = __float2half_rn((v[j * 8 + i] + __half2float(rs[j].h[i])) * g.alpha);
            if (ok[j]) *reinterpret_cast<uint4*>(g.out0 + off + j * 8) = o.u;
        }
    } else if constexpr (EPI == EPI_CONVT2) {
        const int p = row >> 6, vox = row & 63;
        const int z = vox >> 4, y = (vox >> 2) & 3, x = vox & 3;
#pragma unroll
        for (int j = 0; j < NG; ++j) {
            const int col = col0 + j * 8;
            const int abc = col / g.split_cols;
            const int co = col - abc * g.split_cols;
            const int oz = 2 * z + (abc >> 2), oy = 2 * y + ((abc >> 1) & 1), ox = 2 * x + (abc & 1);
            Pack8 o;
#pragma unroll
            for (int i = 0; i < 8; ++i) o.h[i] = __float2half_rn(v[j * 8 + i]);
            if (ok[j]) *reinterpret_cast<uint4*>(g.out0 + (static_cast<size_t>(p) * 512 + (oz * 8 + oy) * 8 + ox) * g.split_cols + co) = o.u;
        }
    } else if constexpr (EPI == EPI_NCDHW) {
        const int p = row / g.S3, vox = row - p * g.S3;
#pragma unroll
        for (int i = 0; i < CH; ++i) {
            const int co = col0 + i;
            if (row_ok && co < g.n_valid) {
                const size_t off = (static_cast<size_t>(p) * g.n_valid + co) * g.S3 + vox;
                if (g.out32 != nullptr) g.out32[off] = v[i];
                else g.out0[off] = __float2half_rn(v[i]);
            }
        }
    } else if constexpr (EPI == EPI_NCDHW_MIX) {
        // the convolution's n_valid channels of this row round to fp16 (one rounding per layer), then the 1x1 mix runs in fp32 on them
        const int p = row / g.S3, vox = row - p * g.S3;
        const int nv = g.n_valid;
        float hc[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) hc[c] = h2f_round(v[c]);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (j >= nv) break;
            float s = __half2float(g.mix[nv * nv + j]);
#pragma unroll
            for (int c = 0; c < 4; ++c)
                if (c < nv) s = fmaf(__half2float(g.mix[j * nv + c]), hc[c], s);
            if (row_ok) {
                const size_t off = (static_cast<size_t>(p) * nv + j) * g.S3 + vox;
                if (g.out32 != nullptr) g.out32[off] = s;
                else g.out0[off] = __float2half_rn(s);
            }
        }
    }
}

// ---- epilogue through shared memory + TMA (EPI_STORE / EPI_GELU / EPI_GATED, tiles that are a multiple of 64 wide) -----------
// Each epilogue warp owns 32 accumulator rows (TMEM lanes) and walks the tile's columns in 32-column chunks; the tcgen05.ld of
// chunk k+1 is in flight while chunk k is converted.  Results go to a 32-row x 128-B staging buffer in the 128-B-swizzled layout
// (conflict-free 16-B stores) and leave as ONE bulk tensor store per 128-B row group:
//   fp16 outputs: 64 columns per store (cp.async.bulk.tensor, full 128-B lines instead of 16-B pieces per thread);
//   gated residual: 32 fp32 columns per cp.reduce.async.bulk.tensor .add — the L2 performs  x += h(gate * h(acc + b)),  so the
//   epilogue never loads the residual (one add per element per launch: deterministic; the L2 adder flushes subnormals).
// Rows >= M and columns >= N are clipped by the tensor map.
constexpr bool gemm_tma_epilogue(int epi, int bn) { return (epi == EPI_STORE || epi == EPI_GELU || epi == EPI_GATED) && bn % 64 == 0; }

// NSPLIT warps share one 32-row slab (the 2-CTA kernel runs 8 epilogue warps: NSPLIT = 2, this warp is `part`); a warp owns NBUF
// staging buffers of 4 KB.
template <int NBUF>
__device__ __forceinline__ void staging_acquire(int lane) {
    if (lane == 0) bulk_wait_read<NBUF - 1>();      // the bulk operation that last read the buffer about to be rewritten is done
    __syncwarp();
}

template <int EPI, int NCH, int NSPLIT, int NBUF>
__device__ __forceinline__ void epilogue_tma(const GemmArgs& g, const CUtensorMap* tmC, const float* __restrict__ sb, const float* __restrict__ sg,
                                             bool gate_in_smem, uint32_t taddr, uint32_t stg, uint32_t& sbuf, int row0, int n0, int lane, int part) {
    const uint32_t srow = stg + lane * 128;
    const int sw = lane & 7;
    // this warp's chunks: units of UW chunks (fp16: 2 chunks = one 128-B row of 64 columns; gated: 1 chunk = 32 fp32 columns)
    constexpr int UW = EPI == EPI_GATED ? 1 : 2;
    constexpr int NU = NCH / UW;
    constexpr int NIT = ((NU + NSPLIT - 1) / NSPLIT) * UW;      // chunk iterations of one warp (some may fall outside the tile)
    auto chunk_of = [&](int it) { return ((it / UW) * NSPLIT + part) * UW + (it % UW); };
    uint32_t r[2][32];
    if (chunk_of(0) < NCH) tmem_ld_32x32(taddr + chunk_of(0) * 32, r[0]);
#pragma unroll
    for (int it = 0; it < NIT; ++it) {
        const int k = chunk_of(it);
        if (k >= NCH) break;                        // warp-uniform
        tmem_ld_wait_dep(r[it & 1]);
        if (it + 1 < NIT && chunk_of(it + 1) < NCH) tmem_ld_32x32(taddr + chunk_of(it + 1) * 32, r[(it + 1) & 1]);
        const uint32_t* acc = r[it & 1];
        const int c0 = k * 32;
        if constexpr (EPI == EPI_GATED) {
            staging_acquire<NBUF>(lane);
            const uint32_t boff = NBUF == 1 ? 0u : (sbuf & 1) * 4096u;
            const uint32_t dst = srow + boff;
            float gt[32];
            if (gate_in_smem) {
#pragma unroll
                for (int i = 0; i < 32; i += 4) {
                    const float4 g4 = *reinterpret_cast<const float4*>(sg + c0 + i);
                    gt[i] = g4.x; gt[i + 1] = g4.y; gt[i + 2] = g4.z; gt[i + 3] = g4.w;
                }
            } else {
                const int b = ((row0 + lane) / g.rows_per_batch) % g.gate_batches;
                const __half* gp = g.gate + static_cast<size_t>(b) * g.gate_bstride + n0 + c0;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    Pack8 t;
                    t.u = (n0 + c0 + j * 8 < g.N) ? *reinterpret_cast<const uint4*>(gp + j * 8) : make_uint4(0, 0, 0, 0);
#pragma unroll
                    for (int i = 0; i < 8; ++i) gt[j * 8 + i] = __half2float(t.h[i]);
                }
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float4 b4 = *reinterpret_cast<const float4*>(sb + c0 + j * 4);
                const float2 v01 = round_h2(__uint_as_float(acc[j * 4 + 0]) + b4.x, __uint_as_float(acc[j * 4 + 1]) + b4.y);
                const float2 v23 = round_h2(__uint_as_float(acc[j * 4 + 2]) + b4.z, __uint_as_float(acc[j * 4 + 3]) + b4.w);
                const float2 o01 = round_h2(gt[j * 4 + 0] * v01.x, gt[j * 4 + 1] * v01.y);
                const float2 o23 = round_h2(gt[j * 4 + 2] * v23.x, gt[j * 4 + 3] * v23.y);
                const float o[4] = {o01.x, o01.y, o23.x, o23.y};
                asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(dst + ((j ^ sw) << 4)), "f"(o[0]), "f"(o[1]), "f"(o[2]), "f"(o[3]) : "memory");
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                tma_reduce_add_2d(tmC, stg + boff, n0 + c0, row0);
                bulk_commit();
            }
            ++sbuf;
        } else {
            if ((it & 1) == 0) staging_acquire<NBUF>(lane);
            const uint32_t boff = NBUF == 1 ? 0u : (sbuf & 1) * 4096u;
            const uint32_t dst = srow + boff;
            uint32_t pk[16];
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
                const float4 b4 = *reinterpret_cast<const float4*>(sb + c0 + i);
                float x[4] = {__uint_as_float(acc[i]) + b4.x, __uint_as_float(acc[i + 1]) + b4.y, __uint_as_float(acc[i + 2]) + b4.z,
                              __uint_as_float(acc[i + 3]) + b4.w};
                if (EPI == EPI_GELU || g.post_scale != 1.0f) {     // otherwise the pack below is the one rounding
                    const float2 r01 = round_h2(x[0], x[1]), r23 = round_h2(x[2], x[3]);
                    x[0] = r01.x; x[1] = r01.y; x[2] = r23.x; x[3] = r23.y;
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        if constexpr (EPI == EPI_GELU) x[e] = gelu_tanh_sigmoid(x[e]);
                        else x[e] *= g.post_scale;
                    }
                }
                const __half2 h0 = __floats2half2_rn(x[0], x[1]), h1 = __floats2half2_rn(x[2], x[3]);
                pk[i >> 1] = *reinterpret_cast<const uint32_t*>(&h0);
                pk[(i >> 1) + 1] = *reinterpret_cast<const uint32_t*>(&h1);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q)
                asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst + ((((it & 1) * 4 + q) ^ sw) << 4)), "r"(pk[4 * q]), "r"(pk[4 * q + 1]),
                             "r"(pk[4 * q + 2]), "r"(pk[4 * q + 3])
                             : "memory");
            if ((it & 1) == 1) {
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) {
                    if (g.convt_store != 0) tma_store_5d(tmC, stg + boff, n0 + (k - 1) * 32, 0, 0, (row0 & 63) >> 4, row0 >> 6);
                    else tma_store_2d(tmC, stg + boff, n0 + (k - 1) * 32, row0);
                    bulk_commit();
                }
                ++sbuf;
            }
        }
    }
}

// ---- EPI_HEADS through shared memory + TMA ---------------------------------------------------------------------------------------
// Column groups of 24 (= Dh / 3 for Dh = 72; every tile, head and q/k/v boundary is a multiple of 24): a warp's 32 rows x 24
// columns are one box of the destination [B*H*Nseq, DhP] matrix (rows (b, head, n0 .. n0+31), columns d0 .. d0+23), or — for the
// transposed V the tcgen05 attention reads — one 24-row x 32-token box of [B*H*DhP, vt_ld].  Needs Nseq % 32 == 0 (a 32-row slab
// never straddles a sequence), Dh % 24 == 0, and the head-dim padding columns d >= Dh already zero (the launcher's caller memsets).
constexpr int HG = 24;
template <int NG, int NSPLIT, int NBUF>
__device__ __forceinline__ void epilogue_heads_tma(const GemmArgs& g, const CUtensorMap* tmQ, const CUtensorMap* tmK, const CUtensorMap* tmV,
                                                   const float* __restrict__ sb, uint32_t taddr, uint32_t stg, uint32_t& sbuf, int row0, int n0, int lane,
                                                   int part) {
    if (row0 >= g.M) return;                        // whole slab outside the matrix (M is a multiple of 32 here)
    const int b = row0 / g.Nseq, nfirst = row0 - b * g.Nseq;
    constexpr int NIT = (NG + NSPLIT - 1) / NSPLIT;
    uint32_t r[2][24];
    if (part < NG) {
        tmem_ld_32x16_to(taddr + part * HG, r[0]);
        tmem_ld_32x8_to(taddr + part * HG + 16, r[0] + 16);
    }
#pragma unroll
    for (int it = 0; it < NIT; ++it) {
        const int k = it * NSPLIT + part;
        if (k >= NG) break;                         // warp-uniform
        tmem_ld_wait_dep24(r[it & 1]);
        if (it + 1 < NIT && k + NSPLIT < NG) {
            tmem_ld_32x16_to(taddr + (k + NSPLIT) * HG, r[(it + 1) & 1]);
            tmem_ld_32x8_to(taddr + (k + NSPLIT) * HG + 16, r[(it + 1) & 1] + 16);
        }
        const uint32_t* acc = r[it & 1];
        const int c0 = k * HG;
        const int col = n0 + c0;
        const int which = col / g.split_cols;
        const int cw = col - which * g.split_cols;
        const int head = cw / g.Dh;
        const int d0 = cw - head * g.Dh;
        const bool sc = g.post_scale != 1.0f && which == 0;
        uint32_t pk[12];
#pragma unroll
        for (int i = 0; i < HG; i += 4) {
            const float4 b4 = *reinterpret_cast<const float4*>(sb + c0 + i);
            float x[4] = {__uint_as_float(acc[i]) + b4.x, __uint_as_float(acc[i + 1]) + b4.y, __uint_as_float(acc[i + 2]) + b4.z,
                          __uint_as_float(acc[i + 3]) + b4.w};
            if (sc) {
                const float2 r01 = round_h2(x[0], x[1]), r23 = round_h2(x[2], x[3]);
                x[0] = r01.x * g.post_scale; x[1] = r01.y * g.post_scale; x[2] = r23.x * g.post_scale; x[3] = r23.y * g.post_scale;
            }
            const __half2 h0 = __floats2half2_rn(x[0], x[1]), h1 = __floats2half2_rn(x[2], x[3]);
            pk[i >> 1] = *reinterpret_cast<const uint32_t*>(&h0);
            pk[(i >> 1) + 1] = *reinterpret_cast<const uint32_t*>(&h1);
        }
        staging_acquire<NBUF>(lane);
        const uint32_t buf = stg + (NBUF == 1 ? 0u : (sbuf & 1) * 4096u);
        const bool transposed = which + 1 == g.vt_which_plus1;
        if (transposed) {
            // staging [24 d][32 tokens] fp16: lane = token
#pragma unroll
            for (int i = 0; i < 12; ++i) {
                const uint16_t lo = static_cast<uint16_t>(pk[i] & 0xFFFFu), hi = static_cast<uint16_t>(pk[i] >> 16);
                asm volatile("st.shared.b16 [%0], %1;" ::"r"(buf + (2 * i) * 64 + lane * 2), "h"(lo) : "memory");
                asm volatile("st.shared.b16 [%0], %1;" ::"r"(buf + (2 * i + 1) * 64 + lane * 2), "h"(hi) : "memory");
            }
        } else {
            // staging [32 rows][24 columns] fp16 (48-B rows: conflict-free 16-B stores)
#pragma unroll
            for (int q = 0; q < 3; ++q)
                asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(buf + lane * 48 + q * 16), "r"(pk[4 * q]), "r"(pk[4 * q + 1]), "r"(pk[4 * q + 2]),
                             "r"(pk[4 * q + 3])
                             : "memory");
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
            if (transposed) tma_store_2d(tmV, buf, nfirst, (b * g.H + head) * g.DhP + d0);
            else tma_store_2d(which == 0 ? tmQ : (which == 1 ? tmK : tmV), buf, d0, (b * g.H + head) * g.Nseq + nfirst);
            bulk_commit();
        }
        ++sbuf;
    }
}

__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, 128;" ::: "memory"); }

template <int BN, int BK, int AMODE, int EPI>
__global__ void __launch_bounds__(256, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmC,
               const __grid_constant__ CUtensorMap tmD, const __grid_constant__ CUtensorMap tmE, const GemmArgs g) {
    using Cfg = GemmCfg<BN, BK>;
    constexpr int STAGES = Cfg::STAGES;
    constexpr bool kTmaEpi = gemm_tma_epilogue(EPI, BN);
    constexpr bool kHeadsTma = EPI == EPI_HEADS && BN % HG == 0 && Cfg::STAGING_BYTES > 0;   // taken when g.heads_tma is set
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = smem_raw;
    if ((smem_u32(smem_raw) & 1023u) != 0) __trap();   // the swizzled operand / staging tiles need a 1024-B aligned base
    // layout: [operand ring][epilogue staging][barriers 256 B][bias + gate tile 2 KB]
    constexpr int OFF_BAR = STAGES * Cfg::STAGE_BYTES + Cfg::STAGING_BYTES;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* tfull_bar = empty_bar + STAGES;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
    float* s_bias = reinterpret_cast<float*>(smem + OFF_BAR + 256);
    float* s_gate = s_bias + 256;

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        if constexpr (kTmaEpi) tma_prefetch_desc(&tmC);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int s = 0; s < 2; ++s) {
            mbar_init(&tfull_bar[s], 1);
            mbar_init(&tempty_bar[s], 128);
        }
        fence_barrier_init();
        fence_proxy_async();
    }
    if (warp == 2) {
        tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // timeline probe: compiled only into the wide linear kernels it was written for — in the narrow-tile convolution kernels the MMA
    // issuer has ~64 cycles per k-block and the (never taken) probe branches cost 14 % there
    constexpr bool kProbe = AMODE == AMODE_LINEAR && BN >= 128;
    long long* const dbg = (kProbe && g.dbg != nullptr) ? g.dbg + static_cast<size_t>(blockIdx.x) * 16 : nullptr;
    const long long t_entry = dbg != nullptr ? clock64() : 0;
    pdl_launch_dependents();   // the next kernel of the stream may start its own prologue
    pdl_wait();                // ... and ours ends here: the operands written by the previous kernel are now visible
    if (dbg != nullptr && threadIdx.x == 0) {
        unsigned long long gt;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
        dbg[0] = clock64(); dbg[11] = static_cast<long long>(gt); dbg[13] = t_entry;
    }

    const int tiles_n = (g.N + BN - 1) / BN;
    const int tiles_m = (g.M + 127) / 128;
    const int num_tiles = tiles_m * tiles_n;
    const int num_kb = g.num_kb;

    if (warp == 0) {
        // warp-converged producer: every lane follows the ring, one elected lane arms the barrier and issues the TMA
        int stage = 0;
        uint32_t phase = 0;
        long long w_empty = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            const int m_blk = tile / tiles_n, n_blk = tile - m_blk * tiles_n;
            for (int kb = 0; kb < num_kb; ++kb) {
                const long long tw = dbg != nullptr ? clock64() : 0;
                mbar_wait(&empty_bar[stage], phase ^ 1);
                if (dbg != nullptr) w_empty += clock64() - tw;
                if (elect_one()) {
                    uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
                    mbar_arrive_expect_tx(&full_bar[stage], Cfg::STAGE_BYTES);
                    if constexpr (AMODE == AMODE_LINEAR) {
                        tma_load_2d(sa, &tmA, &full_bar[stage], kb * BK, m_blk * 128);
                    } else {
                        const int tap = kb / g.chunks_per_tap, chunk = kb - tap * g.chunks_per_tap;
                        const int dz = tap / 9, dy = (tap / 3) % 3, dx = tap % 3;
                        if (AMODE == AMODE_CONV3_S2 || g.conv_S == 4) {  // 128 rows = 2 primitives x 4^3 (output) voxels
                            tma_load_5d(sa, &tmA, &full_bar[stage], chunk * BK, dx - 1, dy - 1, dz - 1, m_blk * 2);
                        } else {              // S == 8: 128 rows = 2 z-slices of one primitive
                            tma_load_5d(sa, &tmA, &full_bar[stage], chunk * BK, dx - 1, dy - 1, (m_blk & 3) * 2 + dz - 1, m_blk >> 2);
                        }
                    }
                    tma_load_2d(sa + Cfg::A_BYTES, &tmB, &full_bar[stage], kb * BK, n_blk * BN);
                }
                __syncwarp();
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
        }
        if (dbg != nullptr && lane == 0) { dbg[5] = w_empty; dbg[6] = clock64(); }
    } else if (warp == 1) {
        // The whole warp runs this loop with warp-uniform control flow and one elected lane issues: descriptors and
        // the TMEM address then live in uniform registers, which keeps the tcgen05.mma issue rate high.
        constexpr uint32_t idesc = umma_idesc_f16(128, BN);
        const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
        const uint32_t smem_u = __shfl_sync(0xffffffffu, smem_u32(smem), 0);
        int stage = 0;
        uint32_t phase = 0;
        int acc = 0;
        uint32_t acc_phase = 0;
        long long w_full = 0, w_tempty = 0, t_first = 0;
        int ntile = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            long long tw = dbg != nullptr ? clock64() : 0;
            mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
            if (dbg != nullptr) w_tempty += clock64() - tw;
            tc_fence_after();
            const uint32_t tmem_d = tmem_u + acc * BN;
            for (int kb = 0; kb < num_kb; ++kb) {
                tw = dbg != nullptr ? clock64() : 0;
                mbar_wait(&full_bar[stage], phase);
                if (dbg != nullptr) { const long long tn = clock64(); w_full += tn - tw; if (ntile == 0 && kb == 0) t_first = tn; }
                tc_fence_after();
                const uint32_t a_addr = smem_u + stage * Cfg::STAGE_BYTES;
                const uint64_t adesc = umma_desc_kmajor<Cfg::SW>(a_addr);
                const uint64_t bdesc = umma_desc_kmajor<Cfg::SW>(a_addr + Cfg::A_BYTES);
                if (elect_one()) {
#pragma unroll
                    for (int k = 0; k < BK / 16; ++k) umma_f16(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
                    umma_commit(&empty_bar[stage]);   // frees the smem slot when these MMAs retire
                }
                __syncwarp();
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
            if (elect_one()) umma_commit(&tfull_bar[acc]);   // accumulator complete -> epilogue
            __syncwarp();
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            ++ntile;
        }
        if (dbg != nullptr && lane == 0) { dbg[1] = t_first; dbg[2] = clock64(); dbg[3] = w_full; dbg[4] = w_tempty; dbg[10] = ntile; }
    } else if (warp >= 4) {
        const int quad = warp & 3;
        const int et = threadIdx.x - 128;
        int acc = 0;
        uint32_t acc_phase = 0;
        const bool gate_in_smem = (EPI == EPI_GATED) && (g.rows_per_batch % 128 == 0);
        long long w_tfull = 0, t_proc = 0;
        uint32_t sbuf = 0;      // running staging-buffer index of this warp (two buffers in rotation)
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            const int m_blk = tile / tiles_n, n_blk = tile - m_blk * tiles_n;
            const int n0 = n_blk * BN;
            // stage this tile's bias (and gate) while the MMAs of the tile are still running
            epi_bar_sync();
            for (int c = et; c < BN; c += 128) {
                const int col = n0 + c;
                s_bias[c] = (g.bias != nullptr && col < g.N) ? __half2float(g.bias[col]) : 0.f;
                if constexpr (EPI == EPI_GATED) {
                    if (gate_in_smem) {
                        const int b = ((m_blk * 128) / g.rows_per_batch) % g.gate_batches;
                        s_gate[c] = col < g.N ? __half2float(g.gate[static_cast<size_t>(b) * g.gate_bstride + col]) : 0.f;
                    }
                }
            }
            epi_bar_sync();
            const int row = m_blk * 128 + quad * 32 + lane;
            const bool row_ok = row < g.M;
            HeadCursor hc{0, 0, 0, 0, 0};
            size_t head_row_off = 0;
            if constexpr (EPI == EPI_HEADS) {
                hc.which = n0 / g.split_cols;
                const int c = n0 - hc.which * g.split_cols;
                hc.head = c / g.Dh;
                hc.d = c - hc.head * g.Dh;
                hc.b = row / g.Nseq;
                hc.n = row - hc.b * g.Nseq;
                head_row_off = (static_cast<size_t>(hc.b) * g.H * g.Nseq + hc.n) * g.DhP;
            }
            const long long tw = dbg != nullptr ? clock64() : 0;
            mbar_wait(&tfull_bar[acc], acc_phase);
            const long long tp = dbg != nullptr ? clock64() : 0;
            w_tfull += tp - tw;
            tc_fence_after();
            const uint32_t taddr = tmem_base + acc * BN + (static_cast<uint32_t>(quad * 32) << 16);
            bool done = false;
            if constexpr (kHeadsTma) {
                if (g.heads_tma != 0) {
                    epilogue_heads_tma<BN / HG, 1, 2>(g, &tmC, &tmD, &tmE, s_bias, taddr, smem_u32(smem) + STAGES * Cfg::STAGE_BYTES + quad * 8192, sbuf,
                                                      m_blk * 128 + quad * 32, n0, lane, 0);
                    done = true;
                }
            }
            if constexpr (kTmaEpi) {
                epilogue_tma<EPI, BN / 32, 1, 2>(g, &tmC, s_bias, s_gate, gate_in_smem, taddr, smem_u32(smem) + STAGES * Cfg::STAGE_BYTES + quad * 8192,
                                                 sbuf, m_blk * 128 + quad * 32, n0, lane, 0);
            } else if (!done) {
                constexpr int CH = BN >= 32 ? 32 : 16;
#pragma unroll 1
                for (int c0 = 0; c0 < BN; c0 += CH) {
                    uint32_t r[32];
                    if constexpr (CH == 32) tmem_ld_32x32(taddr + c0, r);
                    else tmem_ld_32x16(taddr + c0, r);
                    tmem_ld_wait();
                    epi_chunk<EPI, CH>(g, s_bias, s_gate, gate_in_smem, row, row_ok, n0 + c0, c0, r, hc, head_row_off);
                }
            }
            tc_fence_before();
            mbar_arrive(&tempty_bar[acc]);
            if (dbg != nullptr) t_proc += clock64() - tp;
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        if constexpr (kTmaEpi || kHeadsTma) {
            if (lane == 0) bulk_wait<0>();          // every bulk store / reduce of this warp has been performed
        }
        if (dbg != nullptr && et == 0) { dbg[7] = w_tfull; dbg[8] = t_proc; dbg[9] = clock64(); }
    }
    tc_fence_before();
    __syncthreads();
    if (dbg != nullptr && threadIdx.x == 0) {
        unsigned long long gt;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        dbg[12] = static_cast<long long>(gt); dbg[14] = clock64(); dbg[15] = smid;
    }
    if (warp == 2) {
        __syncwarp();
        tc_fence_after();
        tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
    }
}

// =====================================================================================================================
// 2-CTA variant (cta_group::2): a cluster of two CTAs on one TPC computes a 256 x BN tile.  CTA r owns rows
// [m0 + 128 r, +128) (its own A tile, its own TMEM accumulator lanes) and loads HALF of the B tile (BN/2 rows of W);
// the leader's single thread issues tcgen05.mma.cta_group::2 (M = 256), the hardware reads the two B halves from both
// CTAs' shared memory.  Per SM this halves the B traffic from L2 and the B bytes written to shared memory per MMA cycle.
//   full[stage]   lives in the LEADER: both CTAs' TMA loads complete_tx on it (peer bit masked off the mbarrier address)
//   empty[stage]  one per CTA, released by a multicast tcgen05.commit from the leader
//   tfull[acc]    one per CTA (multicast commit);  tempty[acc] in the leader, 256 arrivals (both CTAs' epilogue threads)
// =====================================================================================================================
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;   // clears the CTA-rank bit of a shared::cluster address (-> even CTA of the pair)

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_load_2d_2sm(void* dst, const CUtensorMap* m, uint32_t leader_bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(m)), "r"(leader_bar), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void umma_f16_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar) {   // arrives on the same-offset barrier of BOTH CTAs
    const uint16_t mask = 3;
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
                 "h"(mask)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}

template <int BN>
struct Gemm2Cfg {
    static constexpr int BK = 64;
    static constexpr int A_BYTES = 128 * BK * 2;
    static constexpr int BH_BYTES = (BN / 2) * BK * 2;           // this CTA's half of the B tile
    static constexpr int STAGE_BYTES = A_BYTES + BH_BYTES;
    static constexpr int STAGES_RAW = (192 * 1024) / STAGE_BYTES;
    static constexpr int STAGES = STAGES_RAW > 8 ? 8 : STAGES_RAW;
    static constexpr int TMEM_COLS = (2 * BN <= 256) ? 256 : 512;
    static constexpr int STAGING_BYTES = 8 * 4096;               // eight epilogue warps, one 32-row x 128-B buffer each
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + STAGING_BYTES + 256 + 2048;
    static constexpr int THREADS = 384;                          // 4 control warps + 8 epilogue warps
    static_assert(BH_BYTES % 1024 == 0, "B half tile must stay 1024-B aligned");
    static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
};

__device__ __forceinline__ void epi2_bar_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

template <int BN, int EPI>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(384, 1)
gemm_tc2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmC,
                const __grid_constant__ CUtensorMap tmD, const __grid_constant__ CUtensorMap tmE, const GemmArgs g) {
    using Cfg = Gemm2Cfg<BN>;
    constexpr int STAGES = Cfg::STAGES;
    constexpr int BK = 64;
    constexpr bool kTmaEpi = gemm_tma_epilogue(EPI, BN);
    constexpr bool kHeadsTma = EPI == EPI_HEADS && BN % HG == 0;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = smem_raw;
    if ((smem_u32(smem_raw) & 1023u) != 0) __trap();
    constexpr int OFF_STG = STAGES * Cfg::STAGE_BYTES;
    constexpr int OFF_BAR = OFF_STG + Cfg::STAGING_BYTES;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* tfull_bar = empty_bar + STAGES;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
    float* s_bias = reinterpret_cast<float*>(smem + OFF_BAR + 256);
    float* s_gate = s_bias + 256;

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        if constexpr (kTmaEpi || kHeadsTma) tma_prefetch_desc(&tmC);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full_bar[s], 1);     // leader's producer arms it with the bytes of BOTH CTAs
            mbar_init(&empty_bar[s], 1);
        }
        for (int s = 0; s < 2; ++s) {
            mbar_init(&tfull_bar[s], 1);
            mbar_init(&tempty_bar[s], 16);  // one elected lane of each of the 8 epilogue warps of both CTAs
        }
        fence_barrier_init();
        fence_proxy_async();
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(Cfg::TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    cluster_sync_all();                     // barriers of both CTAs initialised before any remote arrive / TMA signal
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    long long* const dbg = g.dbg != nullptr ? g.dbg + static_cast<size_t>(blockIdx.x) * 16 : nullptr;
    const long long t_entry = dbg != nullptr ? clock64() : 0;
    if (g.pdl_trigger != 0) pdl_launch_dependents();
    pdl_wait();   // no-op for a normally launched grid
    if (dbg != nullptr && threadIdx.x == 0) { dbg[0] = clock64(); dbg[13] = t_entry; }

    const int tiles_n = (g.N + BN - 1) / BN;
    const int tiles_m = (g.M + 255) / 256;
    const int num_tiles = tiles_m * tiles_n;
    const int num_kb = g.num_kb;
    const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;

    if (warp == 0) {
        const uint32_t full0 = smem_u32(&full_bar[0]) & kPeerBitMask;      // the leader's barriers, from either CTA
        int stage = 0;
        uint32_t phase = 0;
        long long w_empty = 0;
        for (int tile = cluster_id; tile < num_tiles; tile += num_clusters) {
            const int m_blk = tile / tiles_n, n_blk = tile - m_blk * tiles_n;
            for (int kb = 0; kb < num_kb; ++kb) {
                const long long tw = dbg != nullptr ? clock64() : 0;
                mbar_wait(&empty_bar[stage], phase ^ 1);
                if (dbg != nullptr) w_empty += clock64() - tw;
                if (elect_one()) {
                    uint8_t* sa = smem + stage * Cfg::STAGE_BYTES;
                    if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2 * Cfg::STAGE_BYTES);
                    tma_load_2d_2sm(sa, &tmA, full0 + stage * 8, kb * BK, m_blk * 256 + static_cast<int>(rank) * 128);
                    tma_load_2d_2sm(sa + Cfg::A_BYTES, &tmB, full0 + stage * 8, kb * BK, n_blk * BN + static_cast<int>(rank) * (BN / 2));
                }
                __syncwarp();
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
        }
        if (dbg != nullptr && lane == 0) { dbg[5] = w_empty; dbg[6] = clock64(); }
    } else if (warp == 1) {
        if (leader) {
            constexpr uint32_t idesc = umma_idesc_f16(256, BN);
            const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
            const uint32_t smem_u = __shfl_sync(0xffffffffu, smem_u32(smem), 0);
            int stage = 0;
            uint32_t phase = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            long long w_full = 0, w_tempty = 0, t_first = 0;
            int ntile = 0;
            for (int tile = cluster_id; tile < num_tiles; tile += num_clusters) {
                long long tw = dbg != nullptr ? clock64() : 0;
                mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
                if (dbg != nullptr) w_tempty += clock64() - tw;
                tc_fence_after();
                const uint32_t tmem_d = tmem_u + acc * BN;
                for (int kb = 0; kb < num_kb; ++kb) {
                    tw = dbg != nullptr ? clock64() : 0;
                    mbar_wait(&full_bar[stage], phase);
                    if (dbg != nullptr) { const long long tn = clock64(); w_full += tn - tw; if (ntile == 0 && kb == 0) t_first = tn; }
                    tc_fence_after();
                    const uint32_t a_addr = smem_u + stage * Cfg::STAGE_BYTES;
                    const uint64_t adesc = umma_desc_kmajor<128>(a_addr);
                    const uint64_t bdesc = umma_desc_kmajor<128>(a_addr + Cfg::A_BYTES);
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < BK / 16; ++k) umma_f16_2sm(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
                        umma_commit_2sm(&empty_bar[stage]);
                    }
                    __syncwarp();
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                if (elect_one()) umma_commit_2sm(&tfull_bar[acc]);
                __syncwarp();
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                ++ntile;
            }
            if (dbg != nullptr && lane == 0) { dbg[1] = t_first; dbg[2] = clock64(); dbg[3] = w_full; dbg[4] = w_tempty; }
        }
    } else if (warp >= 4) {
        const int quad = warp & 3;              // TMEM lane quadrant = warp id % 4
        const int part = (warp - 4) >> 2;       // which half of the column units this warp takes
        const int et = threadIdx.x - 128;
        int acc = 0;
        uint32_t acc_phase = 0;
        const bool gate_in_smem = (EPI == EPI_GATED) && (g.rows_per_batch % 128 == 0);
        const uint32_t tempty0 = smem_u32(&tempty_bar[0]) & kPeerBitMask;
        const uint32_t stg = smem_u32(smem) + OFF_STG + (warp - 4) * 4096;
        long long w_tfull = 0, t_proc = 0;
        uint32_t sbuf = 0;
        int ntile = 0;
        for (int tile = cluster_id; tile < num_tiles; tile += num_clusters) {
            const int m_blk = tile / tiles_n, n_blk = tile - m_blk * tiles_n;
            const int n0 = n_blk * BN;
            const int row0 = m_blk * 256 + static_cast<int>(rank) * 128;
            epi2_bar_sync();
            for (int c = et; c < BN; c += 256) {
                const int col = n0 + c;
                s_bias[c] = (g.bias != nullptr && col < g.N) ? __half2float(g.bias[col]) : 0.f;
                if constexpr (EPI == EPI_GATED) {
                    if (gate_in_smem) {
                        const int b = (row0 / g.rows_per_batch) % g.gate_batches;
                        s_gate[c] = col < g.N ? __half2float(g.gate[static_cast<size_t>(b) * g.gate_bstride + col]) : 0.f;
                    }
                }
            }
            epi2_bar_sync();
            const long long tw = dbg != nullptr ? clock64() : 0;
            mbar_wait(&tfull_bar[acc], acc_phase);
            const long long tp = dbg != nullptr ? clock64() : 0;
            w_tfull += tp - tw;
            tc_fence_after();
            const uint32_t taddr = tmem_base + acc * BN + (static_cast<uint32_t>(quad * 32) << 16);
            bool done = false;
            if constexpr (kHeadsTma) {
                if (g.heads_tma != 0) {
                    epilogue_heads_tma<BN / HG, 2, 1>(g, &tmC, &tmD, &tmE, s_bias, taddr, stg, sbuf, row0 + quad * 32, n0, lane, part);
                    done = true;
                }
            }
            if constexpr (kTmaEpi) {
                epilogue_tma<EPI, BN / 32, 2, 1>(g, &tmC, s_bias, s_gate, gate_in_smem, taddr, stg, sbuf, row0 + quad * 32, n0, lane, part);
            } else if (!done) {
                // per-thread path (ragged head split / tile widths the bulk stores do not cover): this warp takes every second chunk
                const int row = row0 + quad * 32 + lane;
                const bool row_ok = row < g.M;
#pragma unroll 1
                for (int c0 = part * 32; c0 < BN; c0 += 64) {
                    HeadCursor hc{0, 0, 0, 0, 0};
                    size_t head_row_off = 0;
                    if constexpr (EPI == EPI_HEADS) {
                        hc.which = (n0 + c0) / g.split_cols;
                        const int c = (n0 + c0) - hc.which * g.split_cols;
                        hc.head = c / g.Dh;
                        hc.d = c - hc.head * g.Dh;
                        hc.b = row / g.Nseq;
                        hc.n = row - hc.b * g.Nseq;
                        head_row_off = (static_cast<size_t>(hc.b) * g.H * g.Nseq + hc.n) * g.DhP;
                    }
                    uint32_t r[32];
                    tmem_ld_32x32(taddr + c0, r);
                    tmem_ld_wait();
                    epi_chunk<EPI, 32>(g, s_bias, s_gate, gate_in_smem, row, row_ok, n0 + c0, c0, r, hc, head_row_off);
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(tempty0 + acc * 8);     // leader's tempty, from both CTAs
            if (dbg != nullptr) t_proc += clock64() - tp;
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            ++ntile;
        }
        if constexpr (kTmaEpi || kHeadsTma) {
            if (lane == 0) bulk_wait<0>();
        }
        if (dbg != nullptr && et == 0) { dbg[7] = w_tfull; dbg[8] = t_proc; dbg[9] = clock64(); dbg[10] = ntile; }
    }
    tc_fence_before();
    cluster_sync_all();                     // neither CTA may exit (or free TMEM) while its peer can still signal / read it
    if (dbg != nullptr && threadIdx.x == 0) {
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        dbg[14] = clock64(); dbg[15] = smid;
    }
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(Cfg::TMEM_COLS) : "memory");
    }
}

// ---- host side ----------------------------------------------------------------------------------------
struct GemmProblem {
    // A operand
    const __half* A;
    int a_mode;         // AMODE_*
    int lda;            // linear: row stride in elements
    int conv_S, conv_C; // conv: spatial size (4|8) and channel count of the channels-last volume; P = M / S^3
    // W operand [N, K] row-major fp16 (K-major)
    const __half* W;
    int M, N, K;
    int BN;             // tile N (128/192/256/64/32/16); BK chosen from K (64, or 32 when conv_C == 32)
    int epi;
    GemmArgs args;      // epilogue fields (M,N,num_kb filled by the launcher)
};
int launch_gemm(const GemmProblem& p, cudaStream_t stream);
int launch_gemm_2cta(const GemmProblem& p, cudaStream_t stream);   // cta_group::2 path (LINEAR, DiT epilogues, BN in {128,192,256})
int gemm_num_sms();

}  // namespace tpx
