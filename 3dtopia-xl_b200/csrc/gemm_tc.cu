// Host launcher for the tcgen05 GEMM: tensor-map construction (cached), tile-shape dispatch.
#include "gemm_tc.cuh"

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <tuple>
#include <vector>

namespace tpx {

// ---- error plumbing -------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
const char* last_error() { return g_err; }
int cuda_fail(cudaError_t e, const char* what) {
    set_error("CUDA error %d (%s) at %s", static_cast<int>(e), cudaGetErrorString(e), what);
    return TPX_ERR_CUDA;
}

// ---- launch counter + optional event profiling ------------------------------------------------------------------
static std::atomic<long long> g_launches{0};
void note_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
long long launch_count() { return g_launches.load(); }

struct ProfRec { int cls; cudaEvent_t a, b; };
static bool g_prof_on = false;
static std::vector<ProfRec> g_prof_recs;
static std::vector<cudaEvent_t> g_prof_pool;
static cudaEvent_t prof_event() {
    if (!g_prof_pool.empty()) { cudaEvent_t e = g_prof_pool.back(); g_prof_pool.pop_back(); return e; }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}
ProfScope::ProfScope(int cls, cudaStream_t s) : idx(-1), st(s) {
    if (!g_prof_on) return;
    ProfRec r{cls, prof_event(), prof_event()};
    cudaEventRecord(r.a, st);
    idx = static_cast<int>(g_prof_recs.size());
    g_prof_recs.push_back(r);
}
ProfScope::~ProfScope() {
    if (idx >= 0) cudaEventRecord(g_prof_recs[idx].b, st);
}
void prof_begin() {
    for (auto& r : g_prof_recs) { g_prof_pool.push_back(r.a); g_prof_pool.push_back(r.b); }
    g_prof_recs.clear();
    g_prof_on = true;
}
int prof_end(float* ms_by_class, long long* n_by_class) {
    g_prof_on = false;
    TPX_CUDA(cudaDeviceSynchronize());
    for (int i = 0; i < PROF_NCLASS; ++i) { ms_by_class[i] = 0.f; n_by_class[i] = 0; }
    for (auto& r : g_prof_recs) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) { ms_by_class[r.cls] += ms; n_by_class[r.cls] += 1; }
        g_prof_pool.push_back(r.a);
        g_prof_pool.push_back(r.b);
    }
    g_prof_recs.clear();
    return TPX_OK;
}

// timeline probe target of the next GEMM launches (tools/gemm_timeline.py); nullptr = off
static long long* g_gemm_dbg = nullptr;
void set_gemm_timeline(long long* dev_buf) { g_gemm_dbg = dev_buf; }

int gemm_num_sms() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

// ---- tensor maps ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (fn == nullptr) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

static CUtensorMapSwizzle swizzle_for(int bk) {
    return bk == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : (bk == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
}

using MapKey = std::tuple<const void*, long long, long long, long long, int, int, int>;   // last: rank (2 / 5) * 16 + element bytes
static std::map<MapKey, CUtensorMap> g_maps;
static std::mutex g_maps_mu;

// 2-D: row-major [rows, K] matrix of fp16 (esz 2) or fp32 (esz 4) elements, box = [box_rows, bk], swizzle = box row bytes (128/64/32)
static int map_2d(const void* ptr, long long rows, long long K, long long ld, int box_rows, int bk, CUtensorMap* out, int esz = 2, bool swizzled = true) {
    MapKey key{ptr, rows, K, ld, box_rows, bk, 2 * 16 + esz + (swizzled ? 0 : 8)};
    std::lock_guard<std::mutex> lk(g_maps_mu);
    auto it = g_maps.find(key);
    if (it != g_maps.end()) { *out = it->second; return TPX_OK; }
    EncodeTiledFn enc = encode_fn();
    TPX_CHECK(enc != nullptr, TPX_ERR_CUDA, "cuTensorMapEncodeTiled unavailable (no driver?)");
    TPX_CHECK((reinterpret_cast<uintptr_t>(ptr) & 15) == 0 && (ld * esz) % 16 == 0, TPX_ERR_ARG,
              "TMA operand must be 16-B aligned (ptr %p, row stride %lld elements of %d bytes)", ptr, ld, esz);
    cuuint64_t gdim[2] = {static_cast<cuuint64_t>(K), static_cast<cuuint64_t>(rows)};
    cuuint64_t gstr[1] = {static_cast<cuuint64_t>(ld) * esz};
    cuuint32_t box[2] = {static_cast<cuuint32_t>(bk), static_cast<cuuint32_t>(box_rows)};
    cuuint32_t estr[2] = {1, 1};
    CUtensorMap m;
    CUresult r = enc(&m, esz == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(ptr), gdim, gstr, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, swizzled ? swizzle_for(bk * esz / 2) : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    TPX_CHECK(r == CUDA_SUCCESS, TPX_ERR_CUDA, "cuTensorMapEncodeTiled(2d) failed: %d (rows %lld K %lld ld %lld box %d x %d)", (int)r, rows, K, ld, box_rows, bk);
    if (g_maps.size() > 4096) g_maps.clear();
    g_maps[key] = m;
    *out = m;
    return TPX_OK;
}

// 5-D: channels-last volume [P, S, S, S, C] fp16; box = 128 voxel rows x bk channels.  stride2: S = 8 input traversed with element
// stride 2 in x / y / z, so the 8^3 x 2-primitive box lands as 4^3 x 2 = 128 rows (AMODE_CONV3_S2)
static int map_conv(const void* ptr, long long P, int S, int C, int bk, CUtensorMap* out, bool stride2 = false) {
    MapKey key{ptr, P, S, C, stride2 ? 2 : 0, bk, 5 * 16 + 2};
    std::lock_guard<std::mutex> lk(g_maps_mu);
    auto it = g_maps.find(key);
    if (it != g_maps.end()) { *out = it->second; return TPX_OK; }
    EncodeTiledFn enc = encode_fn();
    TPX_CHECK(enc != nullptr, TPX_ERR_CUDA, "cuTensorMapEncodeTiled unavailable (no driver?)");
    TPX_CHECK(S == 4 || S == 8, TPX_ERR_SHAPE, "conv volume edge must be 4 or 8, got %d", S);
    TPX_CHECK(!stride2 || S == 8, TPX_ERR_SHAPE, "stride-2 conv input edge must be 8, got %d", S);
    cuuint64_t gdim[5] = {(cuuint64_t)C, (cuuint64_t)S, (cuuint64_t)S, (cuuint64_t)S, (cuuint64_t)P};
    cuuint64_t gstr[4] = {(cuuint64_t)C * 2, (cuuint64_t)S * C * 2, (cuuint64_t)S * S * C * 2, (cuuint64_t)S * S * S * C * 2};
    cuuint32_t box[5] = {(cuuint32_t)bk, (cuuint32_t)S, (cuuint32_t)S, (cuuint32_t)(S == 4 ? 4 : 2), (cuuint32_t)(S == 4 ? 2 : 1)};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    if (stride2) {   // ceil(8 / 2) = 4 elements per spatial dimension land in shared memory
        box[1] = box[2] = box[3] = 8; box[4] = 2;
        estr[1] = estr[2] = estr[3] = 2;
    }
    CUtensorMap m;
    CUresult r = enc(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, const_cast<void*>(ptr), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     swizzle_for(bk), CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    TPX_CHECK(r == CUDA_SUCCESS, TPX_ERR_CUDA, "cuTensorMapEncodeTiled(5d) failed: %d (P %lld S %d C %d bk %d)", (int)r, P, S, C, bk);
    if (g_maps.size() > 4096) g_maps.clear();
    g_maps[key] = m;
    *out = m;
    return TPX_OK;
}

// General fp16 tensor map (rank <= 5, dims / strides innermost first, strides in bytes for dims 1..rank-1); not cached.
int make_tensor_map_nd(const void* ptr, int rank, const long long* dims, const long long* strides_bytes, const int* box, int swizzle_bytes,
                       CUtensorMap* out, int l2_promotion_bytes) {
    EncodeTiledFn enc = encode_fn();
    TPX_CHECK(enc != nullptr, TPX_ERR_CUDA, "cuTensorMapEncodeTiled unavailable (no driver?)");
    TPX_CHECK(rank >= 1 && rank <= 5 && (reinterpret_cast<uintptr_t>(ptr) & 15) == 0, TPX_ERR_ARG, "tensor map: rank %d / unaligned base", rank);
    cuuint64_t gdim[5];
    cuuint64_t gstr[4];
    cuuint32_t bx[5], estr[5];
    for (int i = 0; i < rank; ++i) {
        gdim[i] = static_cast<cuuint64_t>(dims[i]);
        bx[i] = static_cast<cuuint32_t>(box[i]);
        estr[i] = 1;
        if (i > 0) {
            TPX_CHECK(strides_bytes[i - 1] % 16 == 0, TPX_ERR_ARG, "tensor map: stride %lld of dim %d is not a multiple of 16 bytes", strides_bytes[i - 1], i);
            gstr[i - 1] = static_cast<cuuint64_t>(strides_bytes[i - 1]);
        }
    }
    const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                  : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                  : swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B
                                                        : CU_TENSOR_MAP_SWIZZLE_NONE;
    CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, rank, const_cast<void*>(ptr), gdim, gstr, bx, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                     l2_promotion_bytes >= 256  ? CU_TENSOR_MAP_L2_PROMOTION_L2_256B
                     : l2_promotion_bytes >= 128 ? CU_TENSOR_MAP_L2_PROMOTION_L2_128B
                     : l2_promotion_bytes >= 64  ? CU_TENSOR_MAP_L2_PROMOTION_L2_64B
                                                 : CU_TENSOR_MAP_L2_PROMOTION_NONE,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    TPX_CHECK(r == CUDA_SUCCESS, TPX_ERR_CUDA, "cuTensorMapEncodeTiled(rank %d) failed: %d", rank, static_cast<int>(r));
    return TPX_OK;
}

int make_tensor_map_2d(const void* ptr, long long rows, long long cols, long long ld, int box_rows, int box_cols, CUtensorMap* out) {
    return map_2d(ptr, rows, cols, ld, box_rows, box_cols, out);
}

// Output tensor maps of the bulk-store epilogues (tc / td / te default to copies of the A map when unused).  Validates the geometry the
// 24-column head-split stores need and clears a.heads_tma when it does not hold (the kernel then takes the per-thread path).
static int make_output_maps(const GemmProblem& p, GemmArgs& a, const CUtensorMap& ta, CUtensorMap& tc, CUtensorMap& td, CUtensorMap& te) {
    int rc = TPX_OK;
    tc = ta; td = ta; te = ta;
    if (p.epi == EPI_HEADS && a.heads_tma != 0) {
        const bool ok = p.a_mode == AMODE_LINEAR && p.BN % 24 == 0 && p.N % p.BN == 0 && a.Dh % 24 == 0 && a.split_cols % 24 == 0 && a.Nseq % 32 == 0 &&
                        a.Nseq > 0 && p.M % a.Nseq == 0 && a.DhP % 8 == 0 && (a.vt_which_plus1 == 0 || a.vt_ld % 8 == 0);
        a.heads_tma = ok ? 1 : 0;
        if (ok) {
            const long long rows = static_cast<long long>(p.M / a.Nseq) * a.H * a.Nseq, rows_t = static_cast<long long>(p.M / a.Nseq) * a.H * a.DhP;
            __half* outs[3] = {a.out0, a.out1, a.out2};
            CUtensorMap* maps[3] = {&tc, &td, &te};
            const int nwhich = p.N / a.split_cols;
            for (int w = 0; w < nwhich && w < 3; ++w) {
                TPX_CHECK(outs[w] != nullptr, TPX_ERR_ARG, "gemm: head-split output %d is null", w);
                if (w + 1 == a.vt_which_plus1) rc = map_2d(outs[w], rows_t, a.vt_ld, a.vt_ld, 24, 32, maps[w], 2, false);
                else rc = map_2d(outs[w], rows, a.DhP, a.DhP, 32, 24, maps[w], 2, false);
                if (rc != TPX_OK) return rc;
            }
        }
    } else {
        a.heads_tma = 0;
    }
    if (gemm_tma_epilogue(p.epi, p.BN)) {
        // fp16 [M, N] in 64-column x 32-row boxes, or the fp32 residual in 32 x 32 boxes
        if (p.epi == EPI_GATED) {
            TPX_CHECK(a.xres != nullptr && a.gate != nullptr, TPX_ERR_ARG, "gemm: gated epilogue without residual / gate");
            rc = map_2d(a.xres, p.M, p.N, a.ldx, 32, 32, &tc, 4);
        } else if (a.convt_store != 0) {
            // out0 already points at the (a,b,c) corner of the [P, 8, 8, 8, N] volume: the stride-2 sub-lattice as a 5-D tensor
            TPX_CHECK(a.out0 != nullptr && p.M % 64 == 0 && p.epi == EPI_STORE, TPX_ERR_ARG, "gemm: transposed-conv store needs EPI_STORE and M = P * 64");
            const long long C = p.N, dims[5] = {C, 4, 4, 4, p.M / 64};
            const long long strides[4] = {2 * C * 2, 16 * C * 2, 128 * C * 2, 512 * C * 2};
            const int box[5] = {64, 4, 4, 2, 1};
            rc = make_tensor_map_nd(a.out0, 5, dims, strides, box, 128, &tc, 256);
        } else {
            TPX_CHECK(a.out0 != nullptr && a.ldo >= p.N, TPX_ERR_ARG, "gemm: output pointer / row stride (%d < N %d)", a.ldo, p.N);
            rc = map_2d(a.out0, p.M, p.N, a.ldo, 32, 64, &tc, 2);
        }
    }
    return rc;
}

template <int BN, int BK, int AMODE, int EPI>
static int launch_one(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const CUtensorMap& td, const CUtensorMap& te, const GemmArgs& a,
                      cudaStream_t stream) {
    using Cfg = GemmCfg<BN, BK>;
    auto kern = gemm_tc_kernel<BN, BK, AMODE, EPI>;
    static bool attr_set = false;
    if (!attr_set) {
        TPX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
        attr_set = true;
    }
    const int tiles = ((a.M + 127) / 128) * ((a.N + BN - 1) / BN);
    const int grid = tiles < gemm_num_sms() ? tiles : gemm_num_sms();
    TPX_CUDA(launch_pdl(kern, dim3(grid), dim3(256), Cfg::SMEM_BYTES, stream, ta, tb, tc, td, te, a));
    TPX_LAUNCH_CHECK();
    return TPX_OK;
}

template <int BN, int EPI>
static int launch_one_2cta(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const CUtensorMap& td, const CUtensorMap& te, GemmArgs a,
                           cudaStream_t stream) {
    using Cfg = Gemm2Cfg<BN>;
    auto kern = gemm_tc2_kernel<BN, EPI>;
    static bool attr_set = false;
    if (!attr_set) {
        TPX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
        attr_set = true;
    }
    const int tiles = ((a.M + 255) / 256) * ((a.N + BN - 1) / BN);
    const int pairs = gemm_num_sms() / 2;
    const int clusters = tiles < pairs ? tiles : pairs;
    // TPX_2CTA_PDL: 0 = plain stream-serialised launch; 1 = programmatic dependent launch, trigger at exit; 2 = PDL with the early trigger
    static const int pdl_mode = getenv("TPX_2CTA_PDL") ? atoi(getenv("TPX_2CTA_PDL")) : 2;
    a.pdl_trigger = pdl_mode >= 2 ? 1 : 0;
    if (pdl_mode >= 1) {
        TPX_CUDA(launch_pdl(kern, dim3(2 * clusters), dim3(Cfg::THREADS), Cfg::SMEM_BYTES, stream, ta, tb, tc, td, te, a));
    } else {
        kern<<<2 * clusters, Cfg::THREADS, Cfg::SMEM_BYTES, stream>>>(ta, tb, tc, td, te, a);   // cluster dims are compiled in
    }
    TPX_LAUNCH_CHECK();
    return TPX_OK;
}

int launch_gemm_2cta(const GemmProblem& p, cudaStream_t stream) {
    TPX_CHECK(p.a_mode == AMODE_LINEAR && p.M > 0 && p.N > 0 && p.K > 0, TPX_ERR_SHAPE, "gemm_2cta: linear problems only");
    TPX_CHECK(p.N % 8 == 0 && p.K % 8 == 0, TPX_ERR_SHAPE, "gemm_2cta: N (%d) and K (%d) must be multiples of 8", p.N, p.K);
    ProfScope prof(PROF_GEMM, stream);
    GemmArgs a = p.args;
    a.M = p.M;
    a.N = p.N;
    a.num_kb = (p.K + 63) / 64;
    a.dbg = g_gemm_dbg;
    CUtensorMap ta, tb, tc, td, te;
    int rc = map_2d(p.A, p.M, p.K, p.lda, 128, 64, &ta);
    if (rc != TPX_OK) return rc;
    rc = map_2d(p.W, p.N, p.K, p.K, p.BN / 2, 64, &tb);
    if (rc != TPX_OK) return rc;
    rc = make_output_maps(p, a, ta, tc, td, te);
    if (rc != TPX_OK) return rc;
    TPX_CHECK(p.BN != 144 || a.heads_tma != 0, TPX_ERR_SHAPE, "gemm_2cta: the 144-wide tile exists for the bulk-store head split only");
#define TPX_CASE2(BN_, EP_) \
    if (p.BN == BN_ && p.epi == EP_) return launch_one_2cta<BN_, EP_>(ta, tb, tc, td, te, a, stream);
    TPX_CASE2(128, EPI_STORE) TPX_CASE2(128, EPI_GELU) TPX_CASE2(128, EPI_HEADS) TPX_CASE2(128, EPI_GATED)
    TPX_CASE2(144, EPI_HEADS)
    TPX_CASE2(192, EPI_STORE) TPX_CASE2(192, EPI_GELU) TPX_CASE2(192, EPI_HEADS) TPX_CASE2(192, EPI_GATED)
    TPX_CASE2(256, EPI_STORE) TPX_CASE2(256, EPI_GELU) TPX_CASE2(256, EPI_HEADS) TPX_CASE2(256, EPI_GATED)
#undef TPX_CASE2
    set_error("gemm_2cta: no kernel instantiated for BN=%d epi=%d", p.BN, p.epi);
    return TPX_ERR_SHAPE;
}

int launch_gemm(const GemmProblem& p, cudaStream_t stream) {
    TPX_CHECK(p.M > 0 && p.N > 0 && p.K > 0, TPX_ERR_SHAPE, "gemm: empty problem %d x %d x %d", p.M, p.N, p.K);
    TPX_CHECK(p.N % 8 == 0 && p.K % 8 == 0, TPX_ERR_SHAPE, "gemm: N (%d) and K (%d) must be multiples of 8", p.N, p.K);
    const bool conv = p.a_mode == AMODE_CONV3 || p.a_mode == AMODE_CONV3_S2;
    const int bk = (conv && p.conv_C == 32) ? 32 : 64;
    ProfScope prof(conv ? PROF_CONV_GEMM : PROF_GEMM, stream);
    GemmArgs a = p.args;
    a.M = p.M;
    a.N = p.N;
    a.num_kb = (p.K + bk - 1) / bk;
    a.dbg = g_gemm_dbg;
    a.conv_S = p.conv_S;
    a.chunks_per_tap = conv ? p.conv_C / bk : 1;
    CUtensorMap ta, tb;
    int rc;
    if (p.a_mode == AMODE_LINEAR) {
        rc = map_2d(p.A, p.M, p.K, p.lda, 128, bk, &ta);
    } else {
        TPX_CHECK(p.conv_C % bk == 0 && p.K == 27 * p.conv_C, TPX_ERR_SHAPE, "conv gemm: K (%d) must be 27*C (%d)", p.K, p.conv_C);
        const bool s2 = p.a_mode == AMODE_CONV3_S2;
        const int so = s2 ? p.conv_S / 2 : p.conv_S, s3 = so * so * so;   // output voxels per primitive
        TPX_CHECK(p.M % s3 == 0, TPX_ERR_SHAPE, "conv gemm: M (%d) must be P*S_out^3", p.M);
        rc = map_conv(p.A, p.M / s3, p.conv_S, p.conv_C, bk, &ta, s2);
    }
    TPX_CHECK(p.epi != EPI_NCDHW_MIX || (a.mix != nullptr && a.n_valid >= 1 && a.n_valid <= 4 && a.n_valid <= p.N), TPX_ERR_ARG,
              "gemm: channel-mix epilogue needs its weights and 1..4 valid channels (got %d)", a.n_valid);
    if (rc != TPX_OK) return rc;
    rc = map_2d(p.W, p.N, p.K, p.K, p.BN, bk, &tb);
    if (rc != TPX_OK) return rc;
    CUtensorMap tc, td, te;
    rc = make_output_maps(p, a, ta, tc, td, te);
    if (rc != TPX_OK) return rc;
    TPX_CHECK(p.BN != 144 || a.heads_tma != 0, TPX_ERR_SHAPE, "gemm: the 144-wide tile exists for the bulk-store head split only");

#define TPX_CASE(BN_, BK_, AM_, EP_) \
    if (p.BN == BN_ && bk == BK_ && p.a_mode == AM_ && p.epi == EP_) return launch_one<BN_, BK_, AM_, EP_>(ta, tb, tc, td, te, a, stream);
    // DiT (every tile width x every DiT epilogue, so any hidden size that is a multiple of 128 works)
    TPX_CASE(128, 64, AMODE_LINEAR, EPI_STORE)
    TPX_CASE(128, 64, AMODE_LINEAR, EPI_GELU)
    TPX_CASE(128, 64, AMODE_LINEAR, EPI_HEADS)
    TPX_CASE(128, 64, AMODE_LINEAR, EPI_GATED)
    TPX_CASE(144, 64, AMODE_LINEAR, EPI_HEADS)      // two 72-wide heads per tile: the N = 1152 head projections in one wave
    TPX_CASE(192, 64, AMODE_LINEAR, EPI_STORE)
    TPX_CASE(192, 64, AMODE_LINEAR, EPI_GELU)
    TPX_CASE(192, 64, AMODE_LINEAR, EPI_HEADS)
    TPX_CASE(192, 64, AMODE_LINEAR, EPI_GATED)
    TPX_CASE(256, 64, AMODE_LINEAR, EPI_STORE)
    TPX_CASE(256, 64, AMODE_LINEAR, EPI_GELU)
    TPX_CASE(256, 64, AMODE_LINEAR, EPI_HEADS)
    TPX_CASE(256, 64, AMODE_LINEAR, EPI_GATED)
    // VAE
    TPX_CASE(256, 64, AMODE_CONV3, EPI_STORE)
    TPX_CASE(256, 64, AMODE_CONV3, EPI_RESID_SCALE)
    TPX_CASE(256, 64, AMODE_LINEAR, EPI_RESID_SCALE)
    TPX_CASE(256, 64, AMODE_LINEAR, EPI_CONVT2)
    TPX_CASE(32, 64, AMODE_CONV3, EPI_STORE)
    TPX_CASE(32, 64, AMODE_LINEAR, EPI_STORE)
    TPX_CASE(32, 32, AMODE_CONV3, EPI_STORE)
    TPX_CASE(32, 32, AMODE_CONV3, EPI_RESID_SCALE)
    TPX_CASE(16, 32, AMODE_CONV3, EPI_NCDHW)
    // VAE encoder
    TPX_CASE(32, 32, AMODE_CONV3_S2, EPI_STORE)     // down_blocks.0.downsample 32 -> 32, 8^3 -> 4^3
    TPX_CASE(256, 32, AMODE_CONV3, EPI_STORE)       // down_blocks.1.nets.0.conv1 32 -> 256 at 4^3
    TPX_CASE(16, 64, AMODE_CONV3, EPI_NCDHW_MIX)    // conv_out 256 -> 2 (N padded to 16) with quant_conv folded in
#undef TPX_CASE
    set_error("gemm: no kernel instantiated for BN=%d BK=%d amode=%d epi=%d", p.BN, bk, p.a_mode, p.epi);
    return TPX_ERR_SHAPE;
}

}  // namespace tpx
