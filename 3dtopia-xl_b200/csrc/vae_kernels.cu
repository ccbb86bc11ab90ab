// VAE-decoder kernels that are not GEMM shaped: the 1->C input convolution, GroupNorm(+SiLU) on
// channels-last fp16 volumes, and the weight repacks into the implicit-GEMM [Cout, 27*Cin] layout.
//   reference: models/vae3d_dib.py:93-145 (ResnetBlock), :344 (conv_in), :366-367 (norm_out / conv_out), :429
#include <cstdlib>

#include "kernels.cuh"

namespace tpx {

// ---------------------------------------------------------------------------------------------------------
// post_quant_conv (1x1x1, 1->1) + conv_in (3x3x3, pad 1, 1->C) : z [P,1,4,4,4] -> channels-last fp16 [P,64,C]
// One CTA per primitive, one thread per output channel; the 6^3 zero-padded latent lives in smem.
// ---------------------------------------------------------------------------------------------------------
template <typename ZT>
__global__ void __launch_bounds__(256) vae_conv_in_kernel(const ZT* __restrict__ z, const __half* __restrict__ w_pq, const __half* __restrict__ b_pq,
                                                          const __half* __restrict__ W /*[C,27]*/, const __half* __restrict__ bias, int C,
                                                          __half* __restrict__ out) {
    __shared__ float s_z[6 * 6 * 6];
    const int p = blockIdx.x;
    for (int i = threadIdx.x; i < 216; i += blockDim.x) s_z[i] = 0.f;
    __syncthreads();
    if (threadIdx.x < 64) {
        const int v = threadIdx.x;
        const float zq = h2f_round(static_cast<float>(z[static_cast<size_t>(p) * 64 + v]) * __half2float(w_pq[0]) + __half2float(b_pq[0]));
        s_z[(((v >> 4) + 1) * 6 + ((v >> 2) & 3) + 1) * 6 + (v & 3) + 1] = zq;
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float w[27];
#pragma unroll
        for (int t = 0; t < 27; ++t) w[t] = __half2float(W[c * 27 + t]);
        const float b = __half2float(bias[c]);
        for (int v = 0; v < 64; ++v) {
            const int zz = v >> 4, yy = (v >> 2) & 3, xx = v & 3;
            float acc = b;
#pragma unroll
            for (int t = 0; t < 27; ++t) acc = fmaf(w[t], s_z[((zz + t / 9) * 6 + yy + (t / 3) % 3) * 6 + xx + t % 3], acc);
            out[(static_cast<size_t>(p) * 64 + v) * C + c] = __float2half_rn(acc);
        }
    }
}

int launch_vae_conv_in(const void* z, int z_dtype, const __half* w_pq, const __half* b_pq, const __half* W, const __half* bias, int P, int C,
                       __half* out, cudaStream_t st) {
    if (P <= 0) return TPX_OK;
    ProfScope prof(PROF_VAE_MISC, st);
    if (z_dtype == TPX_DTYPE_F32) vae_conv_in_kernel<float><<<P, 256, 0, st>>>(static_cast<const float*>(z), w_pq, b_pq, W, bias, C, out);
    else if (z_dtype == TPX_DTYPE_F16) vae_conv_in_kernel<__half><<<P, 256, 0, st>>>(static_cast<const __half*>(z), w_pq, b_pq, W, bias, C, out);
    else { set_error("vae_conv_in: unsupported latent dtype %d", z_dtype); return TPX_ERR_ARG; }
    TPX_LAUNCH_CHECK();
    return TPX_OK;
}

// ---------------------------------------------------------------------------------------------------------
// GroupNorm(groups, eps, affine) [+ SiLU] on channels-last fp16 [P, S3, C]; statistics per (primitive, group)
// in fp32.  One CTA per primitive; each thread streams 16-byte channel octets (coalesced), per-channel
// partial sums meet in shared memory, then a second streaming pass normalises (the re-read hits L2).
// ---------------------------------------------------------------------------------------------------------
constexpr int GN_MAXC = 256;
// x * sigmoid(x) with MUFU.EX2 + MUFU.RCP (relative error ~2e-7, far below the fp16 rounding of the result)
__device__ __forceinline__ float silu_fast(float x) {
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-1.4426950408889634f * x));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + e));
    return x * r;
}
// RES > 0: the primitive's S3 * C / 8 octets are exactly RES per thread and stay in registers between the statistics and the
// normalisation (one read, RES loads in flight per thread: the 32 KB volumes of the 4^3 stage and of the 32-channel 8^3 stage);
// RES == 0: streaming two-pass version for larger volumes.
template <int RES>
__global__ void __launch_bounds__(256, RES > 0 ? 3 : 1) groupnorm_silu_kernel(const __half* __restrict__ x, const __half* __restrict__ gamma,
                                                             const __half* __restrict__ beta, int S3, int C, int groups, float eps, int apply_silu,
                                                             __half* __restrict__ out) {
    __shared__ float s_sum[GN_MAXC], s_sq[GN_MAXC], s_scale[GN_MAXC], s_shift[GN_MAXC];
    __shared__ float s_part[256 * 16];
    const int p = blockIdx.x;
    const int oct = C >> 3;                    // 16-byte octets per voxel
    const int total = S3 * oct;
    const uint4* xp = reinterpret_cast<const uint4*>(x + static_cast<size_t>(p) * S3 * C);
    // blockDim (256) is a multiple of oct (<= 32), so a thread always sees the same octet
    const int my_oct = threadIdx.x % oct;
    float ls[8], lq[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { ls[i] = 0.f; lq[i] = 0.f; }
    Pack8 keep[RES > 0 ? RES : 1];
    if constexpr (RES > 0) {
#pragma unroll
        for (int j = 0; j < RES; ++j) keep[j].u = xp[threadIdx.x + j * 256];
#pragma unroll
        for (int j = 0; j < RES; ++j) {
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const float f = __half2float(keep[j].h[k]);
                ls[k] += f;
                lq[k] = fmaf(f, f, lq[k]);
            }
        }
    } else {
#pragma unroll 4
        for (int i = threadIdx.x; i < total; i += blockDim.x) {
            Pack8 v;
            v.u = xp[i];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const float f = __half2float(v.h[k]);
                ls[k] += f;
                lq[k] = fmaf(f, f, lq[k]);
            }
        }
    }
    // deterministic cross-thread reduction (fixed order; run-to-run bit-identical): per-thread partials -> smem,
    // then channel c sums the partials of the 256/oct threads that own its octet.
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        s_part[threadIdx.x * 16 + k] = ls[k];
        s_part[threadIdx.x * 16 + 8 + k] = lq[k];
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const int o = c >> 3, k = c & 7;
        float a = 0.f, b = 0.f;
        for (int t = o; t < 256; t += oct) {
            a += s_part[t * 16 + k];
            b += s_part[t * 16 + 8 + k];
        }
        s_sum[c] = a;
        s_sq[c] = b;
    }
    __syncthreads();
    const int cpg = C / groups;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const int g0 = (c / cpg) * cpg;
        float gs = 0.f, gq = 0.f;
        for (int k = 0; k < cpg; ++k) { gs += s_sum[g0 + k]; gq += s_sq[g0 + k]; }
        const float n = static_cast<float>(S3 * cpg);
        const float mean = gs / n;
        const float var = fmaxf(gq / n - mean * mean, 0.f);
        const float rstd = rsqrtf(var + eps);
        const float sc = rstd * __half2float(gamma[c]);
        s_scale[c] = sc;
        s_shift[c] = __half2float(beta[c]) - mean * sc;
    }
    __syncthreads();
    float sc[8], sh[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) { sc[k] = s_scale[my_oct * 8 + k]; sh[k] = s_shift[my_oct * 8 + k]; }
    uint4* op = reinterpret_cast<uint4*>(out + static_cast<size_t>(p) * S3 * C);
    if constexpr (RES > 0) {
#pragma unroll
        for (int j = 0; j < RES; ++j) {
            Pack8 o;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                float f = fmaf(__half2float(keep[j].h[k]), sc[k], sh[k]);
                if (apply_silu) f = silu_fast(f);
                o.h[k] = __float2half_rn(f);
            }
            op[threadIdx.x + j * 256] = o.u;
        }
    } else {
#pragma unroll 4
        for (int i = threadIdx.x; i < total; i += blockDim.x) {
            Pack8 v, o;
            v.u = xp[i];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                float f = fmaf(__half2float(v.h[k]), sc[k], sh[k]);
                if (apply_silu) f = silu_fast(f);
                o.h[k] = __float2half_rn(f);
            }
            op[i] = o.u;
        }
    }
}

// Streaming version: persistent CTAs pull (primitive, channel slice) units of 32 or 64 KB through a 3-stage shared-memory ring with
// TMA (two units in flight per CTA), compute the group statistics and the normalisation on the staged copy — ONE pass over HBM
// whatever the volume size — and write the result with coalesced 16-byte stores.  A slice holds whole groups, so slices are
// independent: the 8^3 x 256-channel tensor (262 KB per primitive, 537 MB in all) no longer needs a second read.  Statistics:
// per-thread partials -> xor-shuffles across the lanes that own the same channel octet -> one 64-byte record per (warp, octet) ->
// the first `oct` threads finish the sums in a fixed order (run-to-run bit-identical) and turn them into per-channel scale / shift
// (groups of 1, 2, 4 or 8 channels never straddle an octet; no division, no global load in that serial section).
// NT = 256: two CTAs per SM for the 32 KB units, so one CTA's exponentials run under the other's reduction; NT = 512: one CTA per SM
// for the 64 KB units.  (1 024 threads per CTA measured 2x slower: three block-wide barriers per unit with 32 warps waiting.)
template <int NT>
__global__ void __launch_bounds__(NT, NT == 256 ? 2 : 1)
groupnorm_stream_kernel(const __grid_constant__ CUtensorMap tmIn, __half* __restrict__ out, const __half* __restrict__ gamma,
                        const __half* __restrict__ beta, int S3, int C, int CW, int cpg, float eps, int apply_silu, int nunits, int NS, int box_rows) {
    constexpr int NW = NT / 32;
    extern __shared__ __align__(1024) uint8_t gsm_raw[];
    uint8_t* gsm = gsm_raw + ((128u - (smem_u32(gsm_raw) & 127u)) & 127u);      // no swizzle: 128-byte alignment is enough
    __shared__ __align__(16) float s_ss[32 * 16];            // [octet][8 scales, 8 shifts]
    __shared__ float s_gamma[GN_MAXC], s_beta[GN_MAXC];
    __shared__ __align__(8) uint64_t full[8];
    for (int c = threadIdx.x; c < C; c += NT) {
        s_gamma[c] = __half2float(gamma[c]);
        s_beta[c] = __half2float(beta[c]);
    }
    const int unit_bytes = S3 * CW * 2;
    float* s_red = reinterpret_cast<float*>(gsm + static_cast<size_t>(NS) * unit_bytes);   // [warp pair][octet][8 sums, 8 sums of squares]
    const int slices = C / CW;
    const int oct = CW >> 3;                   // 16-byte octets per voxel row of the slice (power of two, <= 32)
    const int total = S3 * oct;
    const int oct_shift = 31 - __clz(oct);
    const float inv_n = 1.0f / static_cast<float>(S3 * cpg);
    const int n_my = (nunits - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int my_oct = lane & (oct - 1);       // NT and 32 are multiples of oct: a thread always sees the same 8 channels
    if (threadIdx.x == 0) {
        tma_prefetch_desc(&tmIn);
        for (int i = 0; i < NS; ++i) mbar_init(&full[i], 1);
        fence_barrier_init();
        fence_proxy_async();
    }
    __syncthreads();
    auto load_unit = [&](int i) {
        const int u = blockIdx.x + i * gridDim.x;
        const int pp = u / slices, sl = u - pp * slices, st = i % NS;
        uint8_t* dst = gsm + static_cast<size_t>(st) * unit_bytes;
        mbar_arrive_expect_tx(&full[st], unit_bytes);
        for (int r0 = 0; r0 < S3; r0 += box_rows) tma_load_2d(dst + static_cast<size_t>(r0) * CW * 2, &tmIn, &full[st], sl * CW, pp * S3 + r0);
    };
    if (threadIdx.x == 0)
        for (int i = 0; i < NS && i < n_my; ++i) load_unit(i);
    for (int i = 0; i < n_my; ++i) {
        const int st = i % NS;
        const int u = blockIdx.x + i * gridDim.x;
        const int pp = u / slices, sl = u - pp * slices;
        mbar_wait(&full[st], (i / NS) & 1);
        uint4* up = reinterpret_cast<uint4*>(gsm + static_cast<size_t>(st) * unit_bytes);
        float ls[8], lq[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) { ls[k] = 0.f; lq[k] = 0.f; }
#pragma unroll 4
        for (int j = threadIdx.x; j < total; j += NT) {
            Pack8 v;
            v.u = up[j];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const float f = __half2float(v.h[k]);
                ls[k] += f;
                lq[k] = fmaf(f, f, lq[k]);
            }
        }
        for (int off = oct; off < 32; off <<= 1) {
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                ls[k] += __shfl_xor_sync(0xffffffffu, ls[k], off);
                lq[k] += __shfl_xor_sync(0xffffffffu, lq[k], off);
            }
        }
        // upper half of the warps deposits its records, the lower half adds them to its own (halves the scratch: two CTAs per SM fit)
        if (warp >= NW / 2 && lane < oct) {
            float4* dst = reinterpret_cast<float4*>(s_red + ((warp - NW / 2) * oct + lane) * 16);
            dst[0] = make_float4(ls[0], ls[1], ls[2], ls[3]);
            dst[1] = make_float4(ls[4], ls[5], ls[6], ls[7]);
            dst[2] = make_float4(lq[0], lq[1], lq[2], lq[3]);
            dst[3] = make_float4(lq[4], lq[5], lq[6], lq[7]);
        }
        __syncthreads();
        if (warp < NW / 2 && lane < oct) {
            float4* dst = reinterpret_cast<float4*>(s_red + (warp * oct + lane) * 16);
            const float4 a0 = dst[0], a1 = dst[1], b0 = dst[2], b1 = dst[3];
            dst[0] = make_float4(ls[0] + a0.x, ls[1] + a0.y, ls[2] + a0.z, ls[3] + a0.w);
            dst[1] = make_float4(ls[4] + a1.x, ls[5] + a1.y, ls[6] + a1.z, ls[7] + a1.w);
            dst[2] = make_float4(lq[0] + b0.x, lq[1] + b0.y, lq[2] + b0.z, lq[3] + b0.w);
            dst[3] = make_float4(lq[4] + b1.x, lq[5] + b1.y, lq[6] + b1.z, lq[7] + b1.w);
        }
        __syncthreads();
        if (threadIdx.x < oct) {
            float cs[8], cq[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) { cs[k] = 0.f; cq[k] = 0.f; }
#pragma unroll
            for (int w = 0; w < NW / 2; ++w) {
                const float4* src = reinterpret_cast<const float4*>(s_red + (w * oct + threadIdx.x) * 16);
                const float4 a0 = src[0], a1 = src[1], b0 = src[2], b1 = src[3];
                cs[0] += a0.x; cs[1] += a0.y; cs[2] += a0.z; cs[3] += a0.w; cs[4] += a1.x; cs[5] += a1.y; cs[6] += a1.z; cs[7] += a1.w;
                cq[0] += b0.x; cq[1] += b0.y; cq[2] += b0.z; cq[3] += b0.w; cq[4] += b1.x; cq[5] += b1.y; cq[6] += b1.z; cq[7] += b1.w;
            }
            // group sums by butterfly (cpg in {1, 2, 4, 8}: groups never straddle the octet); every member ends up with its group's sums
            if (cpg >= 2) {
#pragma unroll
                for (int q = 0; q < 8; q += 2) {
                    const float a = cs[q] + cs[q + 1], b = cq[q] + cq[q + 1];
                    cs[q] = cs[q + 1] = a;
                    cq[q] = cq[q + 1] = b;
                }
            }
            if (cpg >= 4) {
#pragma unroll
                for (int q = 0; q < 8; ++q)
                    if ((q & 2) == 0) {
                        const float a = cs[q] + cs[q + 2], b = cq[q] + cq[q + 2];
                        cs[q] = cs[q + 2] = a;
                        cq[q] = cq[q + 2] = b;
                    }
            }
            if (cpg >= 8) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float a = cs[q] + cs[q + 4], b = cq[q] + cq[q + 4];
                    cs[q] = cs[q + 4] = a;
                    cq[q] = cq[q + 4] = b;
                }
            }
            const int c0 = sl * CW + threadIdx.x * 8;
            float scv[8], shv[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const float mean = cs[q] * inv_n;
                const float rstd = rsqrtf(fmaxf(cq[q] * inv_n - mean * mean, 0.f) + eps);
                scv[q] = rstd * s_gamma[c0 + q];
                shv[q] = s_beta[c0 + q] - mean * scv[q];
            }
            float4* dst = reinterpret_cast<float4*>(s_ss + threadIdx.x * 16);
            dst[0] = make_float4(scv[0], scv[1], scv[2], scv[3]);
            dst[1] = make_float4(scv[4], scv[5], scv[6], scv[7]);
            dst[2] = make_float4(shv[0], shv[1], shv[2], shv[3]);
            dst[3] = make_float4(shv[4], shv[5], shv[6], shv[7]);
        }
        __syncthreads();
        float sc[8], sh[8];
        {
            const float4* src = reinterpret_cast<const float4*>(s_ss + my_oct * 16);
            const float4 a0 = src[0], a1 = src[1], b0 = src[2], b1 = src[3];
            sc[0] = a0.x; sc[1] = a0.y; sc[2] = a0.z; sc[3] = a0.w; sc[4] = a1.x; sc[5] = a1.y; sc[6] = a1.z; sc[7] = a1.w;
            sh[0] = b0.x; sh[1] = b0.y; sh[2] = b0.z; sh[3] = b0.w; sh[4] = b1.x; sh[5] = b1.y; sh[6] = b1.z; sh[7] = b1.w;
        }
        // results leave through plain 16-byte stores (consecutive threads, consecutive octets of a row: coalesced), so the stage is
        // free for the next TMA load as soon as every thread has read it: NS - 1 units stay in flight per CTA
        uint4* op = reinterpret_cast<uint4*>(out + (static_cast<size_t>(pp) * S3 * C + static_cast<size_t>(sl) * CW));
        const int row_oct = C >> 3;
#pragma unroll 4
        for (int j = threadIdx.x; j < total; j += NT) {
            Pack8 v, o;
            v.u = up[j];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                float f = fmaf(__half2float(v.h[k]), sc[k], sh[k]);
                if (apply_silu) f = silu_fast(f);
                o.h[k] = __float2half_rn(f);
            }
            const int row = j >> oct_shift;
            op[static_cast<size_t>(row) * row_oct + (j & (oct - 1))] = o.u;
        }
        __syncthreads();                       // every thread is done with this stage
        if (threadIdx.x == 0 && i + NS < n_my) load_unit(i + NS);
    }
}

int launch_groupnorm_silu(const __half* x, const __half* gamma, const __half* beta, int P, int S3, int C, int groups, float eps, int apply_silu,
                          __half* out, cudaStream_t st) {
    TPX_CHECK(C % 8 == 0 && C <= GN_MAXC && 256 % (C / 8) == 0 && groups > 0 && C % groups == 0, TPX_ERR_SHAPE,
              "groupnorm: channels %d / groups %d unsupported (C%%8==0, C<=%d, C/8 | 256)", C, groups, GN_MAXC);
    if (P <= 0) return TPX_OK;
    ProfScope prof(PROF_GROUPNORM, st);
    // streaming path: units of 32 KB (whole primitive) or 64 KB (64-channel slice of a larger primitive)
    static const bool stream_on = !(getenv("TPX_GN_STREAM") != nullptr && getenv("TPX_GN_STREAM")[0] == '0');
    const int cpg = C / groups;
    int CW = 0;
    if (static_cast<long long>(S3) * C * 2 == 32768) CW = C;
    else if (C % 64 == 0 && static_cast<long long>(S3) * 128 == 65536) CW = 64;
    const bool cpg_ok = cpg == 1 || cpg == 2 || cpg == 4 || cpg == 8;
    if (stream_on && CW > 0 && cpg_ok && (CW & (CW - 1)) == 0 && CW >= 8 && (S3 <= 256 || S3 % 256 == 0)) {
        const int unit_bytes = S3 * CW * 2;
        const bool big = unit_bytes > 32768;
        const int NT = big ? 512 : 256;
        const int NS = 3;
        const int box_rows = S3 < 256 ? S3 : 256;
        const long long dims[2] = {C, static_cast<long long>(P) * S3};
        const long long strides[1] = {2LL * C};
        const int box[2] = {CW, box_rows};
        CUtensorMap tmi;
        // no L2 promotion beyond the row segment a unit really reads (a 256-byte promotion would fetch the neighbouring slices too)
        int rc = make_tensor_map_nd(x, 2, dims, strides, box, 0, &tmi, CW * 2);
        if (rc != TPX_OK) return rc;
        const int nunits = P * (C / CW);
        const int smem = NS * unit_bytes + (NT / 64) * (CW / 8) * 64 + 128;
        static bool attr_set = false;
        if (!attr_set) {
            TPX_CUDA(cudaFuncSetAttribute(groupnorm_stream_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, 3 * 32768 + 8192 + 128));
            TPX_CUDA(cudaFuncSetAttribute(groupnorm_stream_kernel<512>, cudaFuncAttributeMaxDynamicSharedMemorySize, 3 * 65536 + 8192 + 128));
            attr_set = true;
        }
        if (big) {
            const int grid = nunits < 148 ? nunits : 148;
            groupnorm_stream_kernel<512><<<grid, 512, smem, st>>>(tmi, out, gamma, beta, S3, C, CW, cpg, eps, apply_silu, nunits, NS, box_rows);
        } else {
            const int grid = nunits < 296 ? nunits : 296;      // two CTAs per SM: one's exponentials run under the other's reduction
            groupnorm_stream_kernel<256><<<grid, 256, smem, st>>>(tmi, out, gamma, beta, S3, C, CW, cpg, eps, apply_silu, nunits, NS, box_rows);
        }
        TPX_LAUNCH_CHECK();
        return TPX_OK;
    }
    if (S3 * (C / 8) == 8 * 256) groupnorm_silu_kernel<8><<<P, 256, 0, st>>>(x, gamma, beta, S3, C, groups, eps, apply_silu, out);
    else groupnorm_silu_kernel<0><<<P, 256, 0, st>>>(x, gamma, beta, S3, C, groups, eps, apply_silu, out);
    TPX_LAUNCH_CHECK();
    return TPX_OK;
}

// ---------------------------------------------------------------------------------------------------------
// VAE encoder input: x [P, Cin, 8, 8, 8] NCDHW (fp32 / fp16) -> channels-last fp16 [P, 512, CP], channels Cin..CP-1 zero, so the
// 6-channel conv_in runs on the 32-channel halo convolution (its packed weights have zero columns there).  One thread per voxel:
// the Cin loads are coalesced across the warp's voxels, the CP-channel row leaves as 16-byte stores.
// ---------------------------------------------------------------------------------------------------------
template <typename T, int CP>
__global__ void __launch_bounds__(256) vae_pack_input_kernel(const T* __restrict__ x, int P, int Cin, __half* __restrict__ out) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= static_cast<long long>(P) * 512) return;
    const long long p = i >> 9;
    const int vox = static_cast<int>(i & 511);
    const T* src = x + p * Cin * 512 + vox;
    uint4* dst = reinterpret_cast<uint4*>(out + i * CP);
#pragma unroll
    for (int o = 0; o < CP / 8; ++o) {
        Pack8 v;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int c = o * 8 + k;
            v.h[k] = c < Cin ? __float2half_rn(static_cast<float>(src[static_cast<long long>(c) * 512])) : __float2half_rn(0.f);
        }
        dst[o] = v.u;
    }
}

int launch_vae_pack_input(const void* x, int dtype, int P, int Cin, int CP, __half* out, cudaStream_t st) {
    TPX_CHECK(CP == 32 && Cin >= 1 && Cin <= CP, TPX_ERR_SHAPE, "vae_pack_input: %d input channels into %d unsupported", Cin, CP);
    if (P <= 0) return TPX_OK;
    ProfScope prof(PROF_VAE_MISC, st);
    const unsigned grid = static_cast<unsigned>((static_cast<long long>(P) * 512 + 255) / 256);
    if (dtype == TPX_DTYPE_F32) vae_pack_input_kernel<float, 32><<<grid, 256, 0, st>>>(static_cast<const float*>(x), P, Cin, out);
    else if (dtype == TPX_DTYPE_F16) vae_pack_input_kernel<__half, 32><<<grid, 256, 0, st>>>(static_cast<const __half*>(x), P, Cin, out);
    else { set_error("vae_pack_input: unsupported input dtype %d", dtype); return TPX_ERR_ARG; }
    TPX_LAUNCH_CHECK();
    return TPX_OK;
}

// ---------------------------------------------------------------------------------------------------------
// DiagonalGaussianDistribution fields (vae3d_dib.py:51-60) in the parameters' dtype, the reference's operation order:
// logvar = clamp(params[:, half:], -30, 20); std = exp(0.5 * logvar); var = exp(logvar) — each op rounded to T as torch does;
// deterministic: std = var = 0.  params [B, 2 * half] (the mean is the first half, a view on the host side).
// ---------------------------------------------------------------------------------------------------------
template <typename T>
__global__ void vae_posterior_kernel(const T* __restrict__ params, long long B, long long half, int deterministic, T* __restrict__ logvar,
                                     T* __restrict__ stdv, T* __restrict__ var) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= B * half) return;
    const long long b = i / half, j = i - b * half;
    const float lv = fminf(fmaxf(static_cast<float>(params[b * 2 * half + half + j]), -30.0f), 20.0f);
    logvar[i] = static_cast<T>(lv);
    if (deterministic) {
        stdv[i] = static_cast<T>(0.0f);
        var[i] = static_cast<T>(0.0f);
    } else {
        const float hl = static_cast<float>(static_cast<T>(0.5f * lv));
        stdv[i] = static_cast<T>(expf(hl));
        var[i] = static_cast<T>(expf(lv));
    }
}

int launch_vae_posterior(const void* params, int dtype, long long B, long long half, int deterministic, void* logvar, void* stdv, void* var,
                         cudaStream_t st) {
    if (B * half == 0) return TPX_OK;
    ProfScope prof(PROF_VAE_MISC, st);
    const unsigned grid = static_cast<unsigned>((B * half + 255) / 256);
    if (dtype == TPX_DTYPE_F32)
        vae_posterior_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float*>(params), B, half, deterministic, static_cast<float*>(logvar),
                                                          static_cast<float*>(stdv), static_cast<float*>(var));
    else if (dtype == TPX_DTYPE_F16)
        vae_posterior_kernel<__half><<<grid, 256, 0, st>>>(static_cast<const __half*>(params), B, half, deterministic, static_cast<__half*>(logvar),
                                                           static_cast<__half*>(stdv), static_cast<__half*>(var));
    else { set_error("vae_posterior: unsupported dtype %d", dtype); return TPX_ERR_ARG; }
    TPX_LAUNCH_CHECK();
    return TPX_OK;
}

// ---------------------------------------------------------------------------------------------------------
// weight repacks (run once at load time)
// ---------------------------------------------------------------------------------------------------------
// Conv3d weight [Cout,Cin,3,3,3] -> [CoutPad, 27*CinP] with k = tap*CinP + ci, tap = (kz*3+ky)*3+kx; columns ci >= Cin are zero
// (CinP > Cin: the encoder's conv_in, whose input is zero-padded to CinP channels).
// transposed != 0: source is a ConvTranspose3d(k3,s1,p1) weight [Cin,Cout,3,3,3]; the equivalent correlation
// kernel is w'[co,ci,kz,ky,kx] = w[ci,co,2-kz,2-ky,2-kx]  (vae3d_dib.py:367).
template <typename T>
__global__ void pack_conv3_kernel(const T* __restrict__ src, __half* __restrict__ dst, int Cout, int Cin, int CinP, int transposed) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    const long long n = static_cast<long long>(Cout) * 27 * CinP;
    if (i >= n) return;
    const int co = static_cast<int>(i / (27 * CinP));
    const int r = static_cast<int>(i - static_cast<long long>(co) * 27 * CinP);
    const int tap = r / CinP, ci = r - tap * CinP;
    if (ci >= Cin) { dst[i] = __float2half_rn(0.f); return; }
    size_t s;
    if (!transposed) s = (static_cast<size_t>(co) * Cin + ci) * 27 + tap;
    else s = (static_cast<size_t>(ci) * Cout + co) * 27 + (26 - tap);
    dst[i] = __float2half_rn(static_cast<float>(src[s]));
}
// ConvTranspose3d(k2,s2) weight [Cin,Cout,2,2,2] -> [8*Cout, Cin]: row (abc*Cout + co), abc = (a*2+b)*2+c.
template <typename T>
__global__ void pack_convt2_kernel(const T* __restrict__ src, __half* __restrict__ dst, int Cin, int Cout) {
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    const long long n = 8LL * Cout * Cin;
    if (i >= n) return;
    const int row = static_cast<int>(i / Cin), ci = static_cast<int>(i - static_cast<long long>(row) * Cin);
    const int abc = row / Cout, co = row - abc * Cout;
    dst[i] = __float2half_rn(static_cast<float>(src[(static_cast<size_t>(ci) * Cout + co) * 8 + abc]));
}

int launch_pack_conv3(const void* src, int dtype, __half* dst, int Cout, int Cin, int transposed, cudaStream_t st, int CinP) {
    if (CinP < Cin) CinP = Cin;
    const long long n = static_cast<long long>(Cout) * 27 * CinP;
    const unsigned grid = static_cast<unsigned>((n + 255) / 256);
    if (dtype == TPX_DTYPE_F32) pack_conv3_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float*>(src), dst, Cout, Cin, CinP, transposed);
    else if (dtype == TPX_DTYPE_F16) pack_conv3_kernel<__half><<<grid, 256, 0, st>>>(static_cast<const __half*>(src), dst, Cout, Cin, CinP, transposed);
    else { set_error("pack_conv3: unsupported dtype %d", dtype); return TPX_ERR_ARG; }
    TPX_LAUNCH_CHECK();
    return TPX_OK;
}
int launch_pack_convt2(const void* src, int dtype, __half* dst, int Cin, int Cout, cudaStream_t st) {
    const long long n = 8LL * Cout * Cin;
    const unsigned grid = static_cast<unsigned>((n + 255) / 256);
    if (dtype == TPX_DTYPE_F32) pack_convt2_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float*>(src), dst, Cin, Cout);
    else if (dtype == TPX_DTYPE_F16) pack_convt2_kernel<__half><<<grid, 256, 0, st>>>(static_cast<const __half*>(src), dst, Cin, Cout);
    else { set_error("pack_convt2: unsupported dtype %d", dtype); return TPX_ERR_ARG; }
    TPX_LAUNCH_CHECK();
    return TPX_OK;
}

}  // namespace tpx
