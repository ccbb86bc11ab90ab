// Internal launcher declarations shared by the translation units of libtpx_b200.
#pragma once
#include "gemm_tc.cuh"

namespace tpx {

struct SamplerCoefs {
    float sqrt_ab, sqrt_1mab, sqrt_recip_ab, sqrt_recipm1_ab;  // _extract_into_tensor(...)[t] as fp32
    float c_x0, c_eps, sigma, nonzero;                           // DDIM: sqrt(ab_prev), sqrt(1-ab_prev-sigma^2), sigma, (t != 0)
    float coef1, coef2, min_log, max_log;                        // DDPM: posterior mean coefs, log-variance range
    int clip;
};

const char* last_error();
long long launch_count();
void prof_begin();
int prof_end(float* ms_by_class, long long* n_by_class);

// elementwise.cu
int launch_ln_modulate(float* x, int rows, int D, float eps, const __half* shift, const __half* scale, int mod_bstride, int rows_per_batch,
                       int mod_batches, __half* out, const __half* pre_gate, const __half* pre_const, int pre_row0, cudaStream_t st);
enum { GEMV_IN_TIMESTEP = 0, GEMV_IN_F32 = 1, GEMV_IN_F16 = 2 };
enum { GEMV_OUT_F32 = 0, GEMV_OUT_F32_SILU = 1, GEMV_OUT_F16 = 2, GEMV_OUT_F32_AND_SILU16 = 3 };
int launch_gemv(int in_mode, int out_mode, const __half* W, const __half* bias, const void* in, const long long* t, int B, int J, int K, void* out,
                __half* out2, int out_ld, cudaStream_t st);
int launch_x_embed(const float* x, const __half* W, const __half* bias, int rows, int Cin, int D, float* out, long long dup_offset, cudaStream_t st);
int launch_cfg_combine(const __half* both, long long n_half, float s, __half* out, cudaStream_t st);
int launch_sampler_step(int ddim, const float* x, const void* mo, int mo_is_half, const float* noise, long long n, int C, const SamplerCoefs& k,
                        float* x_prev, float* x0_out, cudaStream_t st);
int launch_to_half(const void* src, int src_dtype, __half* dst, long long n, cudaStream_t st);
int launch_from_half(const __half* src, void* dst, int dst_dtype, long long n, cudaStream_t st);
int launch_latent_split(const float* x, const float* mean, const float* stdv, float inv_nf, long long T, int C, float* srt, float* z, cudaStream_t st);
int launch_primvolume_pack(const float* srt, const void* dec, int dec_is_half, long long T, int F, int vox, int srt_fix, float* out, cudaStream_t st);
int launch_fill_rows_half(const __half* vec, __half* dst, long long rows, int K, cudaStream_t st);

// attention.cu :  q [B,H,Nq,DhP], k/v [B,H,Nk,DhP] fp16 (zero padded beyond Dh) -> out [B,Nq,H*Dh] fp16
int launch_attention(const __half* q, const __half* k, const __half* v, __half* out, int B, int H, int Nq, int Nk, int Dh, int DhP, float scale,
                     cudaStream_t st);

// attention_tc.cu : tcgen05 version for 64 < Dh <= 80; vT is V transposed [B,H,80,NkPad]
int launch_attention_tc(const __half* q, const __half* k, const __half* vT, __half* out, int B, int H, int Nq, int Nk, int NkPad, int Dh, float scale,
                        cudaStream_t st, long long* dbg = nullptr);
// gemm_tc.cu : cached 2-D TMA descriptor over a row-major fp16 matrix (swizzle = box_cols * 2 bytes: 128/64/32)
int make_tensor_map_2d(const void* ptr, long long rows, long long cols, long long ld, int box_rows, int box_cols, CUtensorMap* out);

int make_tensor_map_nd(const void* ptr, int rank, const long long* dims, const long long* strides_bytes, const int* box, int swizzle_bytes, CUtensorMap* out,
                       int l2_promotion_bytes = 256);
void set_gemm_timeline(long long* dev_buf);

// conv_halo.cu : 3x3x3 / pad 1 convolution on [P,8,8,8,C] volumes with the input block (+halo) staged ONCE per output tile
int launch_conv3_halo(const __half* x, const __half* W, const __half* bias, const __half* resid, float alpha, __half* out, float* out32, int n_valid, int P,
                      int C, int Cout, int epi, cudaStream_t st);
bool conv3_halo_supported(int S, int C, int Cout, int epi);

// vae_kernels.cu
int launch_vae_conv_in(const void* z, int z_dtype, const __half* w_pq, const __half* b_pq, const __half* W, const __half* bias, int P, int C,
                       __half* out, cudaStream_t st);
int launch_groupnorm_silu(const __half* x, const __half* gamma, const __half* beta, int P, int S3, int C, int groups, float eps, int apply_silu,
                          __half* out, cudaStream_t st);
int launch_vae_pack_input(const void* x, int dtype, int P, int Cin, int CP, __half* out, cudaStream_t st);
int launch_vae_posterior(const void* params, int dtype, long long B, long long half, int deterministic, void* logvar, void* stdv, void* var,
                         cudaStream_t st);

// primsdf.cu : PrimSDF point query; out [n,6] = (sdf, rgb clipped, rough/metal clipped)
int launch_primsdf_query(const float* x, const float* srt, const float* feat, long long n, int K, int S, int dim_feat, int inference, float* out,
                         cudaStream_t st);

// raymarch.cu : ray-march preview (compute_raydirs + mvpraymarch "fixedorder"), rgba [N,H,W,4]
int launch_raymarch_preview(const float* tpl, const float* primpos, const float* primrot, const float* primscale, const float* campos, const float* camrot,
                            const float* focal, const float* princpt, int N, int K, int S, int H, int W, float volradius, float stepsize, float fadescale,
                            float fadeexp, float* out, cudaStream_t st);
size_t primsdf_grid_bytes(long long cap_entries);
int launch_primsdf_grid_build(const float* srt, int K, void* ws, size_t ws_bytes, cudaStream_t st);
int launch_primsdf_query_grid(const float* x, const float* srt, const float* feat, const void* ws, size_t ws_bytes, long long n, int K, int S, int dim_feat,
                              int inference, float* out, cudaStream_t st);

}  // namespace tpx
