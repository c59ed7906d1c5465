// prcore.cu -- host side of libprcore.so: C ABI (include/prcore.h), workspaces, launches.
//
// Build (see passiveradar_b200/build.py):
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo \
//        -Xcompiler -fPIC -shared -Iinclude -o passiveradar_b200/libprcore.so prcore.cu
//
// Threading model: one workspace ("Ctx") per (device, caller stream), or per
// (device, calling thread) when the caller passes stream == NULL.  A Ctx owns grow-only
// device buffers; all work of one call is enqueued on the Ctx's stream, so buffer reuse
// is ordered by the stream.  Nothing here falls back to the CPU.
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "prcore.h"
#include "kernels.cuh"
#include "lagstream.cuh"
#include "toepcorr.cuh"
#include "firtc.cuh"
#include "frontend.cuh"
#include "detect.cuh"
#include "nlms.cuh"
#include "nlms_block.cuh"
#include "fftcorr.cuh"
#include "xcorr.cuh"

namespace {

using namespace prc;

// slide_mac tile shapes (DESIGN.md section 3.1): 10 x 10 complex MACs per step, lane stride
// 10 complex = 80 B (odd multiple of 16 B => conflict-free 128-bit shared loads).
constexpr int LC_TI = 10, LC_TD = 10;     // one-shot lagcorr kernel: samples x lags per step
constexpr int FIR_TK = 10, FIR_TO = 10;   // legacy fir variants: taps x outputs per step
// Register-tile variants of the pipelined kernels (PRC_TILE).  Shared-memory loads cost the FMA
// pipe ~9 cycles per 128-bit load (scripts/microbench/fma_peak2.cu), and a TI x TD tile needs
// 2*TI loads per TI*TD MACs, so a larger TD buys efficiency until registers run out.
//   0: 10 x 10   1: 6 x 18   2: 14 x 14      (TD*8 B must be an odd multiple of 16 B)
struct TileShape { int ti, td; };
constexpr TileShape kTiles[3] = {{10, 10}, {6, 18}, {14, 14}};
constexpr int FIR_THREADS = 128;
constexpr size_t SMEM_LIMIT = 200 * 1024;

thread_local std::string g_err;
std::atomic<uint64_t> g_launches{0};

// optional per-kernel timing (prc_profile_*): CUDA events on the launching stream around each launch
enum KernelId { K_LAGCORR_LS = 0, K_LEVINSON, K_FIR, K_LAGCORR_CAF, K_DOPPLER, K_NLMS, K_MISC, K_IIR, K_XCORR, K_COUNT };
const char* const kKernelNames[K_COUNT] = {"lagcorr_ls", "levinson", "fir_apply", "lagcorr_caf",
                                           "doppler_fft", "nlms", "misc", "iir_sos", "xcorr_fft"};
std::atomic<int> g_prof_on{0};
std::mutex g_prof_mu;
double g_prof_ms[K_COUNT] = {0};
uint64_t g_prof_n[K_COUNT] = {0};
struct ProfRec { int id; cudaEvent_t a, b; };

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CU(call)                                                                               \
    do {                                                                                       \
        cudaError_t e_ = (call);                                                               \
        if (e_ != cudaSuccess)                                                                 \
            return fail(PRC_E_CUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, \
                        __LINE__);                                                             \
    } while (0)

#define TRY(call)               \
    do {                        \
        int r_ = (call);        \
        if (r_ != PRC_OK) return r_; \
    } while (0)

struct DBuf {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return PRC_OK;
        if (p) {
            cudaError_t e = cudaFree(p);   // implicit device sync: nothing in flight still uses it
            p = nullptr;
            cap = 0;
            if (e != cudaSuccess) return fail(PRC_E_CUDA, "cudaFree: %s", cudaGetErrorString(e));
        }
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            p = nullptr;
            return fail(PRC_E_NOMEM, "cudaMalloc(%zu): %s", want, cudaGetErrorString(e));
        }
        cap = want;
        return PRC_OK;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <class T> T* as() const { return static_cast<T*>(p); }
};

struct Ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int nsm = 148;
    std::mutex mu;
    DBuf firb[3];             // Wm^T planes of the tensor-core FIR
    DBuf fe_in, fe_mid, fe_out, fe_hp, fe_ends;    // front end: raw IQ, mixed, resampled, polyphase taps, end points
    DBuf cf_in, cf_cr, cf_det, cf_part;            // CFAR_2D
    uint64_t fe_hp_key = 0;                        // which taps fe_hp holds
    // tensor maps of the last LS / CAF launch of this context: the planes live in DBufs, so the operand addresses
    // repeat from frame to frame and the nine cuTensorMapEncodeTiled calls per launch are paid once
    struct MapCache { bool valid = false; const void* ptr[9] = {nullptr}; int nk = 0, npass = 0; tc::ToepMaps maps; } map_cache[2];
    DBuf rs, clean2;          // LS_Filter_Toeplitz: rolled / frequency-shifted reference, ping-pong output
    DBuf cafplane[6];         // bf16 planes of the tensor-core CAF: x[3], s[3]
    DBuf tcplane[9];          // bf16 planes of the tensor-core path: x[3], s0[3], s1[3]
    DBuf refw, ref, srv, out, clean, partial, win32, win64, dtaps32, dtaps64, lstaps, tw, pbuf, status,
        nl_init, nl_taps;
    int tw_F = 0;
    int status_slot = 0;      // which int of `status` the direct-form Toeplitz solve reports to
    void* pin[2] = {nullptr, nullptr};      // page-locked bounce buffers for pageable host arrays (h2d / d2h below)
    cudaEvent_t pin_ev[2] = {nullptr, nullptr};
    bool pin_ready = false;
    DBuf fft_tw[3], wp_fir, wp_caf, fftP;     // FFT-domain path: twiddle tables (L = 1024 / 2048 / 4096), taps spectra, CAF block sums
    bool fft_tw_ready[3] = {false, false, false};
    // long-lag correlation / channel offset (xcorr.cuh): raw inputs, forward IIR pass, decimated channels,
    // transform planes, W_P tables (for xc_twP), argmax key + offset, |xc| / lag window staging
    DBuf xc_in1, xc_in2, xc_yf, xc_b1, xc_b2, xc_X, xc_Y, xc_S, xc_tw, xc_key, xc_out;
    long long xc_twP = 0;
    std::vector<ProfRec> recs;
    void release() {
        cudaSetDevice(device);
        for (DBuf& b : tcplane) b.release();
        for (DBuf& b : cafplane) b.release();
        for (DBuf& b : firb) b.release();
        rs.release();
        clean2.release();
        for (DBuf& b : fft_tw) b.release();
        for (bool& r : fft_tw_ready) r = false;
        for (DBuf* b : {&wp_fir, &wp_caf, &fftP}) b->release();
        for (DBuf* b : {&xc_in1, &xc_in2, &xc_yf, &xc_b1, &xc_b2, &xc_X, &xc_Y, &xc_S, &xc_tw, &xc_key, &xc_out}) b->release();
        xc_twP = 0;
        for (DBuf* b : {&fe_in, &fe_mid, &fe_out, &fe_hp, &fe_ends, &cf_in, &cf_cr, &cf_det, &cf_part}) b->release();
        for (DBuf* b : {&refw, &ref, &srv, &out, &clean, &partial, &win32, &win64, &dtaps32, &dtaps64, &lstaps,
                        &tw, &pbuf, &status, &nl_init, &nl_taps})
            b->release();
        if (pin_ready) {
            for (int k = 0; k < 2; ++k) { cudaFreeHost(pin[k]); cudaEventDestroy(pin_ev[k]); pin[k] = nullptr; pin_ev[k] = nullptr; }
            pin_ready = false;
        }
        if (own_stream && stream) cudaStreamDestroy(stream);
        stream = nullptr;
    }
};

std::mutex g_mu;
std::map<std::pair<int, void*>, Ctx*> g_stream_ctx;   // (device, caller stream)
std::vector<Ctx*> g_all_ctx;
std::atomic<bool> g_attrs_set[64];
std::atomic<uint64_t> g_epoch{1};                      // bumped by prc_shutdown
int g_tune_nchunk = -1, g_tune_g = -1;
int g_tile = 0;          // measured on B200: 10x10 beats 6x18 / 14x14 (109 vs 117 / 115 us, profiles/r01_tuning.md)
int g_nlms_block = 1;       // block-exact NLMS kernel for NLMS_filter (PRC_NLMS_BLOCK=0: sample-serial kernel)
int g_tma_l2 = 2;          // CUtensorMapL2promotion: 0 none, 1 64B, 2 128B, 3 256B (PRC_TMA_L2)
int g_tma = 1;             // TMA (cp.async.bulk.tensor) producers for the tcgen05 kernels (PRC_TMA=0: 16-byte cp.async loaders)
int g_tc_fir = 1;          // tensor-core path for the clutter FIR (PRC_TC_FIR=0: FP32 fir_apply_kernel)
int g_tc_caf = 1;          // tensor-core path for the CAF block sums as well (PRC_TC_CAF=0: FP32 lagstream)
int g_tc = 1;              // tcgen05 Toeplitz-GEMM for the LS correlations (PRC_TC=0: FP32 lagstream kernel)
int g_stream = 1;          // persistent pipelined lag-correlation kernel (PRC_STREAM=0: one-shot kernel)
int g_packed = 1;          // FFMA2 kernels (PRC_PACKED=0 selects the scalar-FFMA variant for A/B runs)
std::atomic<int> g_fft{1};            // FFT-domain correlation / overlap-save kernels (fftcorr.cuh); PRC_FFT=0: tcgen05 / FP32 direct form
std::atomic<int> g_fft_min_n{8192};   // ... for channels of at least this many samples (PRC_FFT_MIN_N)
std::atomic<int> g_caf_wave{0};       // 1: CAF kernel grid = one wave of CTAs walking several Doppler blocks (measured 4 % slower than one CTA per block)
std::once_flag g_env_once;

// Workspaces of a thread that called with stream == NULL.  They are released when the thread exits (dask's thread pool
// retires worker threads): otherwise every short-lived caller would strand ~60 MB of device memory until prc_shutdown.
struct TlsCtx {
    Ctx* ctx[64] = {nullptr};
    uint64_t epoch = 0;
    ~TlsCtx() {
        if (epoch != g_epoch.load()) return;              // prc_shutdown already freed them
        std::lock_guard<std::mutex> lk(g_mu);
        if (epoch != g_epoch.load()) return;
        for (Ctx*& c : ctx) {
            if (!c) continue;
            for (size_t i = 0; i < g_all_ctx.size(); ++i)
                if (g_all_ctx[i] == c) {
                    g_all_ctx.erase(g_all_ctx.begin() + i);
                    break;
                }
            if (c->stream) cudaStreamSynchronize(c->stream);
            for (ProfRec& r : c->recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
            c->release();
            delete c;
            c = nullptr;
        }
    }
};
thread_local TlsCtx g_tls;

void read_env() {
    if (const char* e = getenv("PRC_TUNE_NCHUNK")) g_tune_nchunk = atoi(e);
    if (const char* e = getenv("PRC_TUNE_G")) g_tune_g = atoi(e);
    if (const char* e = getenv("PRC_PACKED")) g_packed = atoi(e);
    if (const char* e = getenv("PRC_STREAM")) g_stream = atoi(e);
    if (const char* e = getenv("PRC_TC")) g_tc = atoi(e);
    if (const char* e = getenv("PRC_TC_CAF")) g_tc_caf = atoi(e);
    if (const char* e = getenv("PRC_TC_FIR")) g_tc_fir = atoi(e);
    if (const char* e = getenv("PRC_TMA")) g_tma = atoi(e);
    if (const char* e = getenv("PRC_NLMS_BLOCK")) g_nlms_block = atoi(e);
    if (const char* e = getenv("PRC_TMA_L2")) g_tma_l2 = atoi(e);
    if (const char* e = getenv("PRC_TILE")) g_tile = std::max(0, std::min(2, atoi(e)));
    if (const char* e = getenv("PRC_FFT")) g_fft.store(atoi(e));
    if (const char* e = getenv("PRC_FFT_MIN_N")) g_fft_min_n.store(atoi(e));
}

int set_kernel_attrs(int device) {
    if (g_attrs_set[device].load()) return PRC_OK;
    const int lim = (int)SMEM_LIMIT;
    CU(cudaFuncSetAttribute(lagcorr_kernel<LC_TI, LC_TD, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(lagcorr_kernel<LC_TI, LC_TD, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(tc::firtc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(tc::toepcorr_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(tc::toepcorr_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(tc::toepcorr_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(tc::toepcorr_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(lagstream_kernel<10, 10>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(lagstream_kernel<6, 18>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(lagstream_kernel<14, 14>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(fir_apply_kernel<FIR_TK, FIR_TO, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(fir_apply_kernel<FIR_TK, FIR_TO, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(fir_apply_kernel<10, 10, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(fir_apply_kernel<6, 18, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(fir_apply_kernel<14, 14, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(levinson_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(levinson_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(doppler_fft_pow2_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(doppler_fft_pow2_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(doppler_fft_pow2_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(nlms_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(nlms_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(nlms_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(nlms_block_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(nlms_block_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(nlms_block_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(nlms_block_kernel<1, 512>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(nlms_block_kernel<2, 512>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    CU(cudaFuncSetAttribute(nlms_block_kernel<4, 512>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
#define PRC_FFT_ATTRS(R3)                                                                                              \
    CU(cudaFuncSetAttribute(fftc::lscorr_fft_kernel<R3>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));           \
    CU(cudaFuncSetAttribute(fftc::taps_spectrum_kernel<R3>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));        \
    CU(cudaFuncSetAttribute(fftc::fir_fft_kernel<R3>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));              \
    CU(cudaFuncSetAttribute(fftc::caf_fft_kernel<R3, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));       \
    CU(cudaFuncSetAttribute(fftc::caf_fft_kernel<R3, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    PRC_FFT_ATTRS(4)
    PRC_FFT_ATTRS(8)
    PRC_FFT_ATTRS(16)
#undef PRC_FFT_ATTRS
#define PRC_XC_ATTRS(R1, R2)                                                                                           \
    CU(cudaFuncSetAttribute(xc::col_fwd_kernel<R1>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));                \
    CU(cudaFuncSetAttribute(xc::col_inv_kernel<R1>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));                \
    CU(cudaFuncSetAttribute(xc::row_fwd_kernel<R2>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));                \
    CU(cudaFuncSetAttribute(xc::row_prod_kernel<R1, R2>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
    PRC_XC_ATTRS(4, 4)
    PRC_XC_ATTRS(8, 4)
    PRC_XC_ATTRS(8, 8)
    PRC_XC_ATTRS(16, 8)
    PRC_XC_ATTRS(16, 16)
#undef PRC_XC_ATTRS
    g_attrs_set[device].store(true);
    return PRC_OK;
}

int get_ctx(int device, void* stream, Ctx** out) {
    std::call_once(g_env_once, read_env);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(PRC_E_CUDA, "no CUDA device available (%s); libprcore has no CPU fallback",
                    e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    if (device < 0 || device >= ndev || device >= 64) return fail(PRC_E_INVALID, "device %d out of range (0..%d)", device, ndev - 1);
    CU(cudaSetDevice(device));
    TRY(set_kernel_attrs(device));
    if (stream == nullptr) {
        if (g_tls.epoch != g_epoch.load()) {
            for (auto& c : g_tls.ctx) c = nullptr;
            g_tls.epoch = g_epoch.load();
        }
        Ctx*& c = g_tls.ctx[device];
        if (!c) {
            Ctx* n = new Ctx();
            n->device = device;
            n->own_stream = true;
            cudaError_t se = cudaStreamCreateWithFlags(&n->stream, cudaStreamNonBlocking);
            if (se != cudaSuccess) {
                delete n;
                return fail(PRC_E_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(se));
            }
            cudaDeviceGetAttribute(&n->nsm, cudaDevAttrMultiProcessorCount, device);
            std::lock_guard<std::mutex> lk(g_mu);
            g_all_ctx.push_back(n);
            c = n;
        }
        *out = c;
        return PRC_OK;
    }
    std::lock_guard<std::mutex> lk(g_mu);
    auto key = std::make_pair(device, stream);
    auto it = g_stream_ctx.find(key);
    if (it == g_stream_ctx.end()) {
        Ctx* n = new Ctx();
        n->device = device;
        n->stream = static_cast<cudaStream_t>(stream);
        n->own_stream = false;
        cudaDeviceGetAttribute(&n->nsm, cudaDevAttrMultiProcessorCount, device);
        g_all_ctx.push_back(n);
        it = g_stream_ctx.emplace(key, n).first;
    }
    *out = it->second;
    return PRC_OK;
}

int check_launch(const char* what) {
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(PRC_E_CUDA, "launch of %s failed: %s", what, cudaGetErrorString(e));
    return PRC_OK;
}

struct ProfScope {          // brackets one launch with events when profiling is enabled
    Ctx* c;
    int id;
    cudaEvent_t a = nullptr;
    ProfScope(Ctx* c_, int id_) : c(c_), id(id_) {
        if (g_prof_on.load(std::memory_order_relaxed)) {
            cudaEventCreate(&a);
            cudaEventRecord(a, c->stream);
        }
    }
    ~ProfScope() {
        if (a) {
            cudaEvent_t b;
            cudaEventCreate(&b);
            cudaEventRecord(b, c->stream);
            c->recs.push_back({id, a, b});
        }
    }
};

// --------------------------------------------------------------------------- geometry
struct Geo {
    int H, G, steps, nchunk, chunk_len, threads;
    size_t smem;
    int HT;
};

int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

int choose_geo(int blk_len, long long outer, int nlag, int nsm, Geo* g) {
    const int TI = LC_TI, TD = LC_TD;
    g->H = ceil_div(nlag, TD);
    g->HT = g->H * TD;
    if (g->H > 512) return fail(PRC_E_INVALID, "%d lags exceed the supported maximum of %d", nlag, 512 * TD);
    int gmax = std::max(1, std::min(32, 256 / g->H));
    if (g_tune_g > 0) gmax = std::max(1, std::min(g_tune_g, 512 / g->H));
    long long target = (long long)nsm * 8;
    long long nchunk = std::max<long long>(1, (target + outer - 1) / outer);
    const int min_chunk = TI * gmax * 2;
    nchunk = std::min<long long>(nchunk, std::max(1, blk_len / min_chunk));
    if (g_tune_nchunk > 0) nchunk = std::min<long long>(g_tune_nchunk, blk_len);
    for (;;) {
        g->chunk_len = ceil_div(blk_len, nchunk);
        g->nchunk = ceil_div(blk_len, g->chunk_len);
        g->G = std::max(1, std::min(gmax, ceil_div(g->chunk_len, TI * 4)));
        g->steps = ceil_div(ceil_div(g->chunk_len, g->G), TI);
        const size_t Lpad = (size_t)g->G * g->steps * TI;
        g->smem = std::max((g_packed ? 3 : 2) * Lpad + g->HT, (size_t)g->G * g->HT) * sizeof(float2);
        if (g->smem <= 100 * 1024 || g->chunk_len <= TI) break;
        nchunk = nchunk * 2;
    }
    if (g->smem > SMEM_LIMIT) return fail(PRC_E_INVALID, "lag-correlation tile needs %zu B of shared memory", g->smem);
    g->threads = ((g->H * g->G + 31) / 32) * 32;
    return PRC_OK;
}

struct StreamGeo {
    int H, HT, G, steps, threads, ncta, maxpieces;
    long long per_cta, total;
    size_t smem;
};

// CTAs per problem: fill every SM with two co-resident CTAs, but keep >= 2 full steps per CTA
int choose_stream(int blk_len, int nblk, int nprob, int nlag, int nsm, StreamGeo* g) {
    const int TI = kTiles[g_tile].ti, TD = kTiles[g_tile].td;
    g->H = ceil_div(nlag, TD);
    g->HT = g->H * TD;
    if (g->H > 512) return fail(PRC_E_INVALID, "%d lags exceed the supported maximum of %d", nlag, 512 * TD);
    const int max_threads = (TI * TD > 100) ? 256 : 512;     // the big tiles are compiled for <= 256 threads
    if (g->H > max_threads) return fail(PRC_E_INVALID, "%d lags exceed the supported maximum of %d", nlag, max_threads * TD);
    int G = std::max(1, std::min(32, 256 / g->H));
    if (g_tune_g > 0) G = std::max(1, std::min(g_tune_g, max_threads / g->H));
    g->total = (long long)nblk * blk_len;
    long long want = std::max(1, 2 * nsm / nprob);
    if (g_tune_nchunk > 0) want = g_tune_nchunk;
    const long long min_per_cta = (long long)G * TI * 2;
    want = std::min<long long>(want, std::max<long long>(1, g->total / min_per_cta));
    g->per_cta = (g->total + want - 1) / want;
    g->ncta = (int)((g->total + g->per_cta - 1) / g->per_cta);
    g->G = (int)std::max<long long>(1, std::min<long long>(G, (g->per_cta + TI - 1) / TI));
    g->steps = std::max(2, 100 / TI);
    while (g->steps > 1 && (long long)g->G * g->steps * TI > g->per_cta + g->G * TI) --g->steps;
    for (;;) {
        const size_t Lmax = (size_t)g->G * g->steps * TI;
        g->smem = (2 * (2 * Lmax + g->HT) + (size_t)g->G * g->HT) * sizeof(float2);
        if (g->smem <= 100 * 1024 || g->steps == 1) break;
        --g->steps;
    }
    if (g->smem > SMEM_LIMIT) return fail(PRC_E_INVALID, "lag-correlation tile needs %zu B of shared memory", g->smem);
    g->maxpieces = (int)std::min<long long>(g->ncta, (blk_len + g->per_cta - 2) / g->per_cta + 1);
    g->threads = ((g->H * g->G + 31) / 32) * 32;
    return PRC_OK;
}

void launch_lagstream(dim3 grid, int threads, size_t smem, cudaStream_t st, const LagStreamParams& sp) {
    switch (g_tile) {
        case 0: lagstream_kernel<10, 10><<<grid, threads, smem, st>>>(sp); break;
        case 1: lagstream_kernel<6, 18><<<grid, threads, smem, st>>>(sp); break;
        default: lagstream_kernel<14, 14><<<grid, threads, smem, st>>>(sp); break;
    }
}

// ---- tensor maps (TMA).  cuTensorMapEncodeTiled is a host-only driver call, resolved through the runtime
// (no link-time dependency on libcuda).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode_tiled = nullptr;
std::once_flag g_encode_once;

void resolve_encode() {
    std::call_once(g_encode_once, [] {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            g_encode_tiled = reinterpret_cast<EncodeTiledFn>(fn);
    });
}
// TMA producers need the driver's tensor-map encoder; without it the cp.async loaders (same layout family,
// same speed) are used
bool use_tma() {
    if (!g_tma) return false;
    resolve_encode();
    return g_encode_tiled != nullptr;
}

// BF16, 2-D: element (c0, c1) = base[c1 * stride_elems + c0]; rows may overlap (stride_elems < inner)
int make_map_bf16(CUtensorMap* tm, const void* base, uint64_t inner, uint64_t rows, uint64_t stride_elems,
                  uint32_t box_inner, uint32_t box_rows) {
    resolve_encode();
    if (!g_encode_tiled) return fail(PRC_E_CUDA, "cuTensorMapEncodeTiled is not available in this driver");
    const cuuint64_t dims[2] = {inner, rows};
    const cuuint64_t strides[1] = {stride_elems * 2};
    const cuuint32_t box[2] = {box_inner, box_rows};
    const cuuint32_t es[2] = {1, 1};
    const CUresult r = g_encode_tiled(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, es,
                                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                      (CUtensorMapL2promotion)g_tma_l2, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(PRC_E_CUDA, "cuTensorMapEncodeTiled failed (CUresult %d)", (int)r);
    return PRC_OK;
}

// maps of the Toeplitz-GEMM operands: x rows are 128 elements, s rows 256 * npass elements wide, both 128 apart
int make_toep_maps(const tc::ToepParams& tp, tc::ToepMaps* m) {
    const uint64_t rows = (uint64_t)tp.nk * tc::KSTEP;
    for (int k = 0; k < tc::NPLANE; ++k) {
        TRY(make_map_bf16(&m->x[k], tp.x[k], tc::ROW, rows, tc::ROW, 64, tc::KSTEP));
        for (int pr = 0; pr < 2; ++pr)
            TRY(make_map_bf16(&m->s[pr][k], tp.s[pr][k], (uint64_t)tp.npass * tc::NPASS, rows, tc::ROW, 64, tc::KSTEP));
    }
    return PRC_OK;
}

// cached variant: slot 0 = LS, slot 1 = CAF
int cached_toep_maps(Ctx* c, int slot, const tc::ToepParams& tp, const tc::ToepMaps** out) {
    Ctx::MapCache& mc = c->map_cache[slot];
    const void* ptr[9];
    for (int k = 0; k < 3; ++k) { ptr[k] = tp.x[k]; ptr[3 + k] = tp.s[0][k]; ptr[6 + k] = tp.s[1][k]; }
    bool same = mc.valid && mc.nk == tp.nk && mc.npass == tp.npass;
    for (int k = 0; same && k < 9; ++k) same = mc.ptr[k] == ptr[k];
    if (!same) {
        mc.valid = false;
        TRY(make_toep_maps(tp, &mc.maps));
        for (int k = 0; k < 9; ++k) mc.ptr[k] = ptr[k];
        mc.nk = tp.nk; mc.npass = tp.npass;
        mc.valid = true;
    }
    *out = &mc.maps;
    return PRC_OK;
}

// Tensor-core CAF eligibility and geometry (shared by the frame pipeline, which lets the LS stage's prep
// and FIR kernels write the CAF operands while the data is in registers, and by xambg_device)
struct CafTc {
    bool on = false;
    long long D = 0, nx = 0, slen = 0;
    int npass = 0, ht = 0;
    bool planes_ready = false;    // x and s planes already written by the LS stage
};

CafTc caf_tc_plan(const Ctx* c, long long n, int R, int F, bool has_taps) {
    CafTc t;
    if (!g_tc || !g_tc_caf || has_taps || F < 1) return t;
    const long long D = n / F;
    if (D < 1024 || D % 1024 != 0) return t;
    t.npass = ceil_div(2 * (64 + R + 1), tc::NPASS);
    t.ht = ceil_div(R + 1, 2) * 2;
    if ((long long)F * t.npass < c->nsm || tc::toep_smem_bytes(t.ht) > SMEM_LIMIT) return t;
    t.on = true;
    t.D = D;
    t.nx = (long long)F * D;
    t.slen = t.nx + (long long)t.npass * 128;
    return t;
}

// --------------------------------------------------------------------------- FFT-domain path (fftcorr.cuh)
// A batch of frames: nf channels pairs `stride` samples apart (inputs), results laid out frame after frame.
struct Batch {
    int nf = 1;
    long long stride = 0;
};

inline int r3_index(int r3) { return r3 == 4 ? 0 : (r3 == 8 ? 1 : 2); }
inline size_t fft_smem(int r3) { return (size_t)(2 * 16 * 17 * r3 + 256 * r3 + 16 * r3) * sizeof(float2); }   // fft::Geo<R3>::SMEM_FLOAT2: exchange buffers + twiddles, no staging
inline int ilog2(int v) { int l = 0; while ((1 << l) < v) ++l; return l; }

// R3 = 4 / 8 / 16  <->  L = 1024 / 2048 / 4096
#define PRC_R3_SWITCH(r3, STMT)                        \
    switch (r3) {                                      \
        case 4: { constexpr int R3 = 4; STMT; } break; \
        case 8: { constexpr int R3 = 8; STMT; } break; \
        default: { constexpr int R3 = 16; STMT; } break; \
    }

int fft_twiddles(Ctx* c, int r3, const float2** tw) {
    const int k = r3_index(r3);
    const int cnt = 256 * r3 + 16 * r3;
    if (!c->fft_tw_ready[k]) {
        TRY(c->fft_tw[k].ensure((size_t)cnt * sizeof(float2)));
        PRC_R3_SWITCH(r3, (fft::fft_twiddle_kernel<R3><<<ceil_div(cnt, 256), 256, 0, c->stream>>>(c->fft_tw[k].as<float2>())));
        TRY(check_launch("fft_twiddle_kernel"));
        c->fft_tw_ready[k] = true;
    }
    *tw = c->fft_tw[k].as<float2>();
    return PRC_OK;
}

// ---- LS correlations: segments of the channel
struct LsFftPlan {
    bool on = false;
    int r3 = 8, nseg = 0, Bs = 0, ncta = 0, HT = 0;
};

LsFftPlan ls_fft_plan(const Ctx* c, long long n, int M, int nf) {
    LsFftPlan pl;
    if (!g_fft.load() || n < g_fft_min_n.load() || M < 1 || M > 2048) return pl;
    pl.r3 = M <= 1024 ? 8 : 16;
    const int L = 256 * pl.r3;
    if (n < 2 * L) return pl;
    const int bmax = L - M + 1;                        // lags 0..M-1 of a segment stay inside its L-sample window
    pl.nseg = (int)((n + bmax - 1) / bmax);
    pl.Bs = (int)((n + pl.nseg - 1) / pl.nseg);
    pl.nseg = (int)((n + pl.Bs - 1) / pl.Bs);
    // CTAs of one transform group (16 R3 threads), 3 resident per SM: the whole batch is ONE wave of CTAs, every CTA
    // walks its share of a frame's segments (any split works: segments are independent)
    const long long slots = 3ll * c->nsm;
    pl.ncta = (int)std::max<long long>(1, std::min<long long>(pl.nseg, slots / nf));
    pl.HT = (M + 1) & ~1;
    pl.on = true;
    return pl;
}

int ls_fft_corr(Ctx* c, const LsFftPlan& pl, const float2* ref, const float2* srv, long long n, Batch bt, int M, int peek,
                bool linear) {
    const float2* tw;
    TRY(fft_twiddles(c, pl.r3, &tw));
    TRY(c->partial.ensure((size_t)bt.nf * 2 * pl.ncta * pl.HT * sizeof(float2)));
    fftc::LsCorrParams p{};
    p.ref = ref; p.srv = srv; p.frame_stride = bt.stride;
    p.n = (int)n; p.M = M; p.peek = peek; p.linear = linear ? 1 : 0;
    p.nseg = pl.nseg; p.Bs = pl.Bs;
    p.partial = c->partial.as<float2>(); p.HT = pl.HT; p.tw = tw;
    {
        ProfScope ps(c, K_LAGCORR_LS);
        PRC_R3_SWITCH(pl.r3, (fftc::lscorr_fft_kernel<R3><<<dim3(pl.ncta, bt.nf), 16 * R3, fftc::lscorr_smem_float2<R3>() * sizeof(float2), c->stream>>>(p)));
    }
    return check_launch("lscorr_fft_kernel");
}

// (T + reg I) w = rhs for nf frames: taps -> c->lstaps [nf][M], status -> c->status [nf]
int levinson_launch(Ctx* c, int nchunk, int HT, int M, double reg, int nf) {
    TRY(c->lstaps.ensure((size_t)nf * M * sizeof(float2)));
    TRY(c->status.ensure((size_t)nf * sizeof(int)));
    LevinsonParams lp{};
    lp.partial = c->partial.as<float2>();
    lp.nchunk = nchunk; lp.HT = HT; lp.M = M; lp.reg = reg;
    lp.taps = c->lstaps.as<float2>();
    lp.status = c->status.as<int>();
    {
        ProfScope ps(c, K_LEVINSON);
        // one thread per unknown (a CTA of 1024 threads would own a whole SM's registers and could not share it
        // with the other slots' transform CTAs; the recursion only ever uses ceil(M / 32) warps)
        const int thr = std::max(64, (M + 31) & ~31);
        if (M <= 1024) levinson_kernel<1><<<nf, thr, levinson_smem(M, thr), c->stream>>>(lp);
        else levinson_kernel<4><<<nf, 512, levinson_smem(M, 512), c->stream>>>(lp);
    }
    return check_launch("levinson_kernel");
}

// W' of c->lstaps for transform length 256 r3 -> wp [nf][L]
int taps_spectrum(Ctx* c, int r3, int M, int nf, DBuf* wp) {
    const float2* tw;
    TRY(fft_twiddles(c, r3, &tw));
    TRY(wp->ensure((size_t)nf * 256 * r3 * sizeof(float2)));
    fftc::TapSpecParams p{};
    p.taps = c->lstaps.as<float2>(); p.M = M; p.wp = wp->as<float2>(); p.tw = tw;
    {
        ProfScope ps(c, K_MISC);
        PRC_R3_SWITCH(r3, (fftc::taps_spectrum_kernel<R3><<<nf, 16 * R3, fft_smem(R3), c->stream>>>(p)));
    }
    return check_launch("taps_spectrum_kernel");
}

// out = srv - FIR(ref, c->lstaps) by overlap-save (circular, or zero-extended when linear)
int fir_fft(Ctx* c, int r3, const float2* ref, const float2* srv, float2* out, long long n, Batch bt, int M, int peek,
            bool linear) {
    const float2* tw;
    TRY(fft_twiddles(c, r3, &tw));
    TRY(taps_spectrum(c, r3, M, bt.nf, &c->wp_fir));
    const int L = 256 * r3;
    fftc::FirFftParams p{};
    p.ref = ref; p.srv = srv; p.out = out; p.frame_stride = bt.stride;
    p.wp = c->wp_fir.as<float2>();
    p.n = (int)n; p.M = M; p.peek = peek; p.linear = linear ? 1 : 0;
    p.nseg = ceil_div(n, L - M + 1);
    p.tw = tw;
    // one wave of CTAs for the whole batch (3 resident per SM: 68 KB of shared memory each)
    const int per_frame = (int)std::max<long long>(1, std::min<long long>(p.nseg, 3ll * c->nsm / bt.nf));
    {
        ProfScope ps(c, K_FIR);
        PRC_R3_SWITCH(r3, (fftc::fir_fft_kernel<R3><<<dim3(per_frame, bt.nf), 16 * R3, fftc::fir_smem_float2<R3>() * sizeof(float2), c->stream>>>(p)));
    }
    return check_launch("fir_fft_kernel");
}

// ---- CAF block sums
struct CafFftPlan {
    bool on = false;
    int r3 = 8, Bmax = 0, HT = 0;
};

// mfuse: taps of the clutter filter fused into the surveillance operand (0: none)
CafFftPlan caf_fft_plan(long long n, int R, int F, long long ntaps, long long D, bool boxcar, int mfuse) {
    CafFftPlan pl;
    if (!g_fft.load() || n < g_fft_min_n.load() || !boxcar || D < 32 || F < 1) return pl;
    double best = 0.0;
    for (int r3 : {4, 8, 16}) {
        const int L = 256 * r3;
        const long long bmax = (long long)L - R - std::max(mfuse - 1, 0);
        if (bmax < L / 4 || n < L) continue;
        const long long nseg = (ntaps + bmax - 1) / bmax;
        const double cost = (double)(nseg * (mfuse ? 3 : 2) + 1) * L * ilog2(L);
        if (!pl.on || cost < best) {
            pl.on = true; pl.r3 = r3; pl.Bmax = (int)bmax; best = cost;
        }
    }
    pl.HT = (R + 2) & ~1;
    return pl;
}

// P[frame][j][d] -> c->fftP; wp == nullptr: plain CAF of (ref, srv); else srv is cleaned on the fly with the taps
// spectrum wp ([nf][L], same r3)
int caf_fft(Ctx* c, const CafFftPlan& pl, const float2* ref, const float2* srv, long long n, Batch bt, int R, int F,
            const float* win32, long long D, int c0, long long ntaps, const float2* wp, int M, int peek) {
    const float2* tw;
    TRY(fft_twiddles(c, pl.r3, &tw));
    TRY(c->fftP.ensure((size_t)bt.nf * F * pl.HT * sizeof(float2)));
    fftc::CafFftParams p{};
    p.ref = ref; p.srv = srv; p.frame_stride = bt.stride; p.win = win32; p.wp = wp;
    p.n = (int)n; p.R = R; p.F = F; p.M = M; p.peek = peek;
    p.D = D; p.c0 = c0; p.ntaps = (int)ntaps; p.Bmax = pl.Bmax;
    p.P = c->fftP.as<float2>(); p.HT = pl.HT; p.tw = tw;
    // one wave of CTAs for the whole batch (3 resident per SM): a CTA walks several Doppler blocks of its frame, so the
    // twiddle tables are staged once per CTA and there is no partially filled last wave
    int gx = F;
    if (g_caf_wave.load()) gx = (int)std::max<long long>(1, std::min<long long>(F, 3ll * c->nsm / bt.nf));
    const dim3 grid(gx, bt.nf);
    {
        ProfScope ps(c, K_LAGCORR_CAF);
        if (wp) { PRC_R3_SWITCH(pl.r3, (fftc::caf_fft_kernel<R3, true><<<grid, 16 * R3, fftc::caf_smem_float2<R3>() * sizeof(float2), c->stream>>>(p))); }
        else { PRC_R3_SWITCH(pl.r3, (fftc::caf_fft_kernel<R3, false><<<grid, 16 * R3, fftc::caf_smem_float2<R3>() * sizeof(float2), c->stream>>>(p))); }
    }
    return check_launch("caf_fft_kernel");
}

// --------------------------------------------------------------------------- device pipelines
// All pointers are device pointers; everything is enqueued on c->stream.

int decimator_offset(long long ntaps, long long D) {   // resample_poly alignment, up = 1
    const long long half = (ntaps - 1) / 2;
    const long long pre_pad = D - half % D;
    const long long pre_remove = (half + pre_pad) / D;
    return (int)(pre_remove * D - pre_pad);
}

// bt.nf > 1 (a batch of frames) and fuse_wp != nullptr (clutter filter applied inside the CAF kernel, taps spectrum
// [nf][L] for the transform length of caf_fft_plan(..., fuse_M)) exist on the FFT-domain path only
int xambg_device(Ctx* c, const float2* ref, const float2* srv, long long n, int R, int F,
                 const float* win32, const float* dtaps32, long long ndtaps, float2* out,
                 bool refw_ready = false, bool caf_planes_ready = false, Batch bt = Batch{},
                 const float2* fuse_wp = nullptr, int fuse_M = 0, int fuse_peek = 0) {
    if (n <= 0 || n >= (1ll << 31) - 4096) return fail(PRC_E_INVALID, "n=%lld unsupported", n);
    if (F < 1 || R < 0) return fail(PRC_E_INVALID, "freq_bins=%d / range_bins=%d invalid", F, R);
    const long long D = n / F;
    if (D < 1) return fail(PRC_E_INVALID, "decimation factor int(n/freq_bins) is 0 (n=%lld, freq_bins=%d)", n, F);
    long long ntaps;
    int c0;
    const float* taps = nullptr;
    if (D == 1) {            // resample_poly(x, 1, 1) returns x (scipy _signaltools.py:4028)
        ntaps = 1;
        c0 = 0;
    } else if (dtaps32 == nullptr) {
        ntaps = D + 1;
        c0 = decimator_offset(ntaps, D);
    } else {
        ntaps = ndtaps;
        c0 = decimator_offset(ntaps, D);
        taps = dtaps32;
    }
    if (ntaps > (1ll << 30)) return fail(PRC_E_INVALID, "decimator too long");
    Geo g{};
    long long d_per_cta = 0;
    const float2* bnd_x = nullptr;                  // boundary-sample correction of the tensor-core path
    const float* bnd_w_all = nullptr;               // ... window to apply to bnd_x on the fly (bnd_x unweighted)
    const float2* dop_src = nullptr;                // Doppler-stage input when it is not c->partial
    const CafFftPlan fp = caf_fft_plan(n, R, F, ntaps, D, taps == nullptr && ntaps == D + 1, fuse_wp ? fuse_M : 0);
    if ((bt.nf > 1 || fuse_wp) && !fp.on)
        return fail(PRC_E_INVALID, "batched / fused CAF needs the FFT-domain path (n=%lld, F=%d, R=%d not eligible)", n, F, R);
    const CafTc ct = (!fp.on && ntaps == D + 1 && c0 == D / 2) ? caf_tc_plan(c, n, R, F, taps != nullptr) : CafTc{};
    if (fp.on) {
        // ---- FFT-domain block correlations (fftcorr.cuh): one CTA per Doppler block, P[j][d] straight from the channels
        TRY(caf_fft(c, fp, ref, srv, n, bt, R, F, win32, D, c0, ntaps, fuse_wp, fuse_M, fuse_peek));
        g.nchunk = 1;
        g.HT = fp.HT;
        dop_src = c->fftP.as<float2>();
    } else if (ct.on) {
        // ---- tensor-core CAF: one (Doppler block, pass) item per accumulation, persistent CTAs
        // ref * window as complex64 is needed to build the x planes here; when the LS stage already wrote them
        // (caf_planes_ready) only the F boundary samples use it, and those are weighted on the fly
        const float2* xw = ref;
        const float* bnd_w = nullptr;
        if (win32 && refw_ready) {
            xw = c->refw.as<float2>();
        } else if (win32 && caf_planes_ready) {
            bnd_w = win32;
        } else if (win32) {
            TRY(c->refw.ensure((size_t)n * sizeof(float2)));
            {
                ProfScope ps(c, K_MISC);
                weight_kernel<<<ceil_div(n, 256), 256, 0, c->stream>>>(ref, win32, c->refw.as<float2>(), (int)n);
            }
            TRY(check_launch("weight_kernel"));
            xw = c->refw.as<float2>();
        }
        for (int k = 0; k < 6; ++k) TRY(c->cafplane[k].ensure((size_t)(k < 3 ? ct.nx : ct.slen) * 2 * sizeof(uint16_t)));
        TRY(c->partial.ensure((size_t)F * ct.npass * ct.ht * sizeof(float2)));
        if (!caf_planes_ready) {
            tc::PrepParams px{};
            px.sig[0] = xw; px.sig[1] = xw;
            px.dmin[0] = px.dmin[1] = -(int)(D / 2);
            px.zero_outside[0] = px.zero_outside[1] = 1;
            for (int k = 0; k < 3; ++k) px.plane[0][k] = px.plane[1][k] = c->cafplane[k].as<uint16_t>();
            px.n = (int)n;
            px.len = ct.nx;
            tc::PrepParams py = px;
            py.sig[0] = py.sig[1] = srv;
            py.zero_outside[0] = py.zero_outside[1] = 0;
            for (int k = 0; k < 3; ++k) py.plane[0][k] = py.plane[1][k] = c->cafplane[3 + k].as<uint16_t>();
            py.len = ct.slen;
            {
                ProfScope ps(c, K_MISC);
                tc::tc_prep_kernel<<<dim3(ceil_div(ct.nx, 1024), 1), 256, 0, c->stream>>>(px);
                tc::tc_prep_kernel<<<dim3(ceil_div(ct.slen, 1024), 1), 256, 0, c->stream>>>(py);
            }
            TRY(check_launch("tc_prep_kernel(caf)"));
        }
        tc::ToepParams tp{};
        for (int k = 0; k < 3; ++k) {
            tp.x[k] = c->cafplane[k].as<uint16_t>();
            tp.s[0][k] = tp.s[1][k] = c->cafplane[3 + k].as<uint16_t>();
        }
        tp.nk = (int)(ct.nx / 1024); tp.nlag = R + 1; tp.npass = ct.npass; tp.ranges = 0;
        tp.kb = (int)(D / 1024); tp.nblk = F; tp.HT = ct.ht;
        tp.partial = c->partial.as<float2>();
        tp.debug_tile = nullptr; tp.debug_clk = nullptr;
        static const tc::ToepMaps no_maps{};
        const tc::ToepMaps* mp = &no_maps;
        const bool tma = use_tma();
        if (tma) TRY(cached_toep_maps(c, 1, tp, &mp));
        const tc::ToepMaps& maps = *mp;
        {
            ProfScope ps(c, K_LAGCORR_CAF);
            if (tma) tc::toepcorr_kernel<false, true><<<c->nsm, tc::THREADS, tc::toep_smem_bytes(ct.ht), c->stream>>>(tp, maps);
            else tc::toepcorr_kernel<false, false><<<c->nsm, tc::THREADS, tc::toep_smem_bytes(ct.ht), c->stream>>>(tp, maps);
        }
        TRY(check_launch("toepcorr_kernel(caf)"));
        g.nchunk = ct.npass;
        g.HT = ct.ht;
        bnd_x = xw;
        bnd_w_all = bnd_w;
    } else if (g_stream && taps == nullptr && ntaps >= 64) {   // tiny Doppler blocks: one flush per block would dominate
        StreamGeo sg;
        TRY(choose_stream((int)ntaps, F, 1, R + 1, c->nsm, &sg));
        TRY(c->partial.ensure((size_t)F * sg.maxpieces * sg.HT * sizeof(float2)));
        const float2* xw = ref;
        if (win32 && refw_ready) {
            xw = c->refw.as<float2>();           // ref * window already written by the LS stage's prep kernel
        } else if (win32) {
            TRY(c->refw.ensure((size_t)n * sizeof(float2)));
            {
                ProfScope ps(c, K_MISC);
                weight_kernel<<<ceil_div(n, 256), 256, 0, c->stream>>>(ref, win32, c->refw.as<float2>(), (int)n);
            }
            TRY(check_launch("weight_kernel"));
            xw = c->refw.as<float2>();
        }
        LagStreamParams sp{};
        sp.x = xw;
        sp.s[0] = srv; sp.s[1] = srv;
        sp.dmin[0] = 0; sp.dmin[1] = 0;
        sp.n = (int)n;
        sp.blk_first_lo = (long long)c0 - (ntaps - 1);
        sp.blk_stride = D;
        sp.blk_len = (int)ntaps;
        sp.nblk = F;
        sp.total = sg.total;
        sp.per_cta = sg.per_cta;
        sp.H = sg.H; sp.G = sg.G; sp.steps = sg.steps;
        sp.maxpieces = sg.maxpieces;
        sp.partial = c->partial.as<float2>();
        {
            ProfScope ps(c, K_LAGCORR_CAF);
            launch_lagstream(dim3(sg.ncta, 1), sg.threads, sg.smem, c->stream, sp);
        }
        TRY(check_launch("lagstream_kernel(caf)"));
        g.nchunk = sg.maxpieces;
        g.HT = sg.HT;
        d_per_cta = sg.per_cta;
    } else {
    TRY(choose_geo((int)ntaps, F, R + 1, c->nsm, &g));
    TRY(c->partial.ensure((size_t)F * g.nchunk * g.HT * sizeof(float2)));

    LagCorrParams p{};
    p.x = ref;
    p.s[0] = srv; p.s[1] = srv;
    p.dmin[0] = 0; p.dmin[1] = 0;
    p.win = win32;
    p.taps = taps;
    p.n = (int)n;
    p.blk_first_lo = (long long)c0 - (ntaps - 1);
    p.blk_stride = D;
    p.blk_len = (int)ntaps;
    p.nblk = F;
    p.nchunk = g.nchunk;
    p.chunk_len = g.chunk_len;
    p.H = g.H; p.G = g.G; p.steps = g.steps;
    p.partial = c->partial.as<float2>();
    {
        ProfScope ps(c, K_LAGCORR_CAF);
        const dim3 grid((unsigned)((long long)F * g.nchunk), 1);
        if (g_packed) lagcorr_kernel<LC_TI, LC_TD, true><<<grid, g.threads, g.smem, c->stream>>>(p);
        else lagcorr_kernel<LC_TI, LC_TD, false><<<grid, g.threads, g.smem, c->stream>>>(p);
    }
    TRY(check_launch("lagcorr_kernel(caf)"));
    }

    // Doppler stage
    if (c->tw_F != F) {
        TRY(c->tw.ensure((size_t)F * sizeof(float2)));
        twiddle_kernel<<<ceil_div(F, 256), 256, 0, c->stream>>>(c->tw.as<float2>(), F);
        TRY(check_launch("twiddle_kernel"));
        c->tw_F = F;
    }
    DopplerParams d{};
    d.partial = dop_src ? dop_src : c->partial.as<float2>();
    d.tw = c->tw.as<float2>();
    d.out = out;
    d.F = F; d.R = R; d.nchunk = g.nchunk; d.HT = g.HT;
    d.partial_fstride = (long long)F * g.nchunk * g.HT;
    d.out_fstride = (long long)F * (R + 1);
    d.blk_len = (int)ntaps; d.per_cta = d_per_cta;
    d.bx = bnd_x; d.bs = srv; d.bwin = bnd_x ? bnd_w_all : nullptr; d.bstride = D; d.boff = c0; d.n = (int)n;
    int logF = 0;
    while ((1 << logF) < F) ++logF;
    d.logF = logF;
    const bool pow2 = (1 << logF) == F && F >= 2;
    ProfScope ps_doppler(c, K_DOPPLER);
    if (pow2 && F <= 8192) {
        if (F <= 1024 && (long long)ceil_div(R + 1, 8) * bt.nf >= c->nsm) {
            const size_t sm = (size_t)2 * F * 8 * sizeof(float2);
            doppler_fft_pow2_kernel<8><<<dim3(ceil_div(R + 1, 8), bt.nf), 256, sm, c->stream>>>(d);
        } else if (F <= 4096) {     // also the small-grid case: 2 columns per CTA fill more SMs
            const size_t sm = (size_t)2 * F * 2 * sizeof(float2);
            doppler_fft_pow2_kernel<2><<<dim3(ceil_div(R + 1, 2), bt.nf), 256, sm, c->stream>>>(d);
        } else {
            const size_t sm = (size_t)2 * F * sizeof(float2);
            doppler_fft_pow2_kernel<1><<<dim3(R + 1, bt.nf), 256, sm, c->stream>>>(d);
        }
        TRY(check_launch("doppler_fft_pow2_kernel"));
    } else {
        TRY(c->pbuf.ensure((size_t)F * (R + 1) * sizeof(float2)));
        for (int fr = 0; fr < bt.nf; ++fr) {      // any F: chunk sum + direct DFT, frame by frame
            chunk_sum_kernel<<<ceil_div((long long)F * (R + 1), 256), 256, 0, c->stream>>>(
                d.partial + (size_t)fr * d.partial_fstride, c->pbuf.as<float2>(), F, R, g.nchunk, g.HT, (int)ntaps, d_per_cta, d);
            TRY(check_launch("chunk_sum_kernel"));
            doppler_dft_kernel<<<dim3(ceil_div(R + 1, 128), F), 128, 0, c->stream>>>(
                c->pbuf.as<float2>(), c->tw.as<float2>(), out + (size_t)fr * d.out_fstride, F, R);
            TRY(check_launch("doppler_dft_kernel"));
        }
    }
    return PRC_OK;
}

// bt.nf > 1 (a batch of frames; taps_out then receives [nf][M]) and need_out == false (only the taps are wanted: the
// caller applies them inside the CAF kernel) exist on the FFT-domain path only
int ls_device(Ctx* c, const float2* ref, const float2* srv, long long n, int filter_len, int peek,
              double reg, float2* out, float2* taps_out, const float* win32 = nullptr, bool* refw_ready = nullptr,
              CafTc* caf = nullptr, bool linear = false, Batch bt = Batch{}, bool need_out = true) {
    // linear: LS_Filter_Toeplitz semantics -- correlations and FIR treat ref/srv as zero outside [0, n)
    if (refw_ready) *refw_ready = false;
    bool caf_x_done = false;
    if (n <= 0 || n >= (1ll << 31) - 4096) return fail(PRC_E_INVALID, "n=%lld unsupported", n);
    if (filter_len < 0 || peek < 0 || filter_len + peek < 1)
        return fail(PRC_E_INVALID, "filter_len=%d peek=%d invalid", filter_len, peek);
    const int M = filter_len + peek;
    if (M > 2048) return fail(PRC_E_INVALID, "%d taps exceed the Toeplitz solver's maximum of 2048", M);
    const LsFftPlan lf = ls_fft_plan(c, n, M, bt.nf);
    if ((bt.nf > 1 || !need_out) && !lf.on)
        return fail(PRC_E_INVALID, "batched LS filter needs the FFT-domain path (n=%lld, %d taps not eligible)", n, M);
    if (lf.on) {
        // ---- FFT-domain path (fftcorr.cuh): block spectra -> lag sums -> float64 Toeplitz solve -> overlap-save FIR
        TRY(ls_fft_corr(c, lf, ref, srv, n, bt, M, peek, linear));
        TRY(levinson_launch(c, lf.ncta, lf.HT, M, reg, bt.nf));
        if (need_out) TRY(fir_fft(c, lf.r3, ref, srv, out, n, bt, M, peek, linear));
        if (taps_out)
            CU(cudaMemcpyAsync(taps_out, c->lstaps.p, (size_t)bt.nf * M * sizeof(float2), cudaMemcpyDeviceToDevice, c->stream));
        return PRC_OK;
    }
    Geo g{};
    bool use_fir_tc = false;
    int lead = 0, fir_shift = 0, fir_kv = 0, fir_nblk = 0;
    long long fir_zoff = 0;
    TRY(c->lstaps.ensure((size_t)M * sizeof(float2)));
    TRY(c->status.ensure(sizeof(int)));
    const int tc_npass = ceil_div(2 * (64 + M), tc::NPASS);
    const int tc_ranges = c->nsm / (2 * tc_npass);
    const int tc_nk = ceil_div(n, 1024);
    const int tc_ht = ceil_div(M, 2) * 2;
    if (g_tc && tc_ranges >= 1 && tc_nk >= 2 * tc_ranges && tc::toep_smem_bytes(tc_ht) <= SMEM_LIMIT) {
        // ---- tensor-core path: BF16x3 Toeplitz GEMM (toepcorr.cuh)
        const long long nx = (long long)tc_nk * 1024;
        long long slen = nx + (long long)tc_npass * 128;
        const bool alias_x = (nx == n) || linear;    // x (zero tail) and s0 (circular tail) only differ beyond n
        // tensor-core FIR geometry (firtc.cuh): the ref planes get a lead-in of `lead` samples so that the
        // window of output row a starts at plane sample 64 a + lead - pre
        const int fir_pre = std::max(0, ceil_div(M - 1 - peek, 4) * 4);
        const int fir_lead = ceil_div(fir_pre, 64) * 64;
        const int fir_kvp = ceil_div(2 * (64 + peek + fir_pre), 64) * 64;
        const long long fir_rows = ceil_div(n, 64);
        const int fir_grid = ceil_div(fir_rows, tc::FIR_ROWS);
        use_fir_tc = g_tc_fir && fir_grid >= 32 && fir_kvp <= 64 * tc::FIR_MAX_ATOMS && tc::firtc_smem_bytes() <= SMEM_LIMIT;
        lead = use_fir_tc ? fir_lead : 0;
        if (use_fir_tc) {
            fir_shift = peek + fir_pre;
            fir_kv = fir_kvp;
            fir_nblk = fir_grid;
            fir_zoff = 2ll * (fir_lead - fir_pre);
            slen = std::max(slen, ((long long)fir_grid * tc::FIR_ROWS + tc::FIR_MAX_ATOMS / 2 + 2) * 64);
        }
        for (int k = 0; k < 9; ++k) {
            if (k < 3 && alias_x) continue;
            TRY(c->tcplane[k].ensure((size_t)(k < 3 ? nx : slen + lead) * 2 * sizeof(uint16_t)));
        }
        TRY(c->partial.ensure((size_t)2 * tc_npass * tc_ranges * tc_ht * sizeof(float2)));
        const bool fold = win32 != nullptr && refw_ready != nullptr;
        if (fold) TRY(c->refw.ensure((size_t)n * sizeof(float2)));
        {
            ProfScope ps(c, K_MISC);
            if (!alias_x)
                tc::bf16_split_kernel<<<ceil_div(nx, 256), 256, 0, c->stream>>>(
                    ref, (int)n, 0, c->tcplane[0].as<uint16_t>(), c->tcplane[1].as<uint16_t>(), c->tcplane[2].as<uint16_t>(), nx, n);
            tc::PrepParams pp{};
            pp.sig[0] = ref; pp.sig[1] = srv;
            pp.dmin[0] = -lead; pp.dmin[1] = -peek;         // ref planes start `lead` samples early (FIR window)
            pp.zero_outside[0] = pp.zero_outside[1] = linear ? 1 : 0;
            for (int k = 0; k < 3; ++k) { pp.plane[0][k] = c->tcplane[3 + k].as<uint16_t>(); pp.plane[1][k] = c->tcplane[6 + k].as<uint16_t>(); }
            pp.win = fold ? win32 : nullptr;
            // the complex64 ref*window is only needed by the FP32 CAF; the tensor-core CAF takes its x planes (cafx)
            const bool need_refw = fold && !(caf && caf->on);
            pp.refw = need_refw ? c->refw.as<float2>() : nullptr;
            pp.n = (int)n;
            pp.len = slen + lead;
            if (fold && caf && caf->on) {          // also emit the CAF x operand (ref * window, shifted by D/2)
                for (int k = 0; k < 3; ++k) {
                    TRY(c->cafplane[k].ensure((size_t)caf->nx * 2 * sizeof(uint16_t)));
                    pp.cafx[k] = c->cafplane[k].as<uint16_t>();
                }
                pp.caf_off = caf->D / 2;
                pp.caf_nx = caf->nx;
                caf_x_done = true;
            }
            tc::tc_prep_kernel<<<dim3(ceil_div(slen + lead, 1024), 2), 256, 0, c->stream>>>(pp);
        }
        TRY(check_launch("tc_prep_kernel"));
        if (fold && !(caf && caf->on)) *refw_ready = true;
        tc::ToepParams tp{};
        for (int k = 0; k < 3; ++k) {
            tp.x[k] = alias_x ? c->tcplane[3 + k].as<uint16_t>() + 2 * lead : c->tcplane[k].as<uint16_t>();
            tp.s[0][k] = c->tcplane[3 + k].as<uint16_t>() + 2 * lead;
            tp.s[1][k] = c->tcplane[6 + k].as<uint16_t>();
        }
        tp.nk = tc_nk; tp.nlag = M; tp.npass = tc_npass; tp.ranges = tc_ranges; tp.HT = tc_ht;
        tp.partial = c->partial.as<float2>();
        tp.debug_tile = nullptr; tp.debug_clk = nullptr;
        static const tc::ToepMaps no_maps{};
        const tc::ToepMaps* mp = &no_maps;
        const bool tma = use_tma();
        if (tma) TRY(cached_toep_maps(c, 0, tp, &mp));
        const tc::ToepMaps& maps = *mp;
        {
            ProfScope ps(c, K_LAGCORR_LS);
            if (tma) tc::toepcorr_kernel<true, true><<<2 * tc_npass * tc_ranges, tc::THREADS, tc::toep_smem_bytes(tc_ht), c->stream>>>(tp, maps);
            else tc::toepcorr_kernel<true, false><<<2 * tc_npass * tc_ranges, tc::THREADS, tc::toep_smem_bytes(tc_ht), c->stream>>>(tp, maps);
        }
        TRY(check_launch("toepcorr_kernel"));
        g.nchunk = tc_npass * tc_ranges;
        g.HT = tc_ht;
    } else if (g_stream || linear) {
        StreamGeo sg;
        TRY(choose_stream((int)n, 1, 2, M, c->nsm, &sg));
        TRY(c->partial.ensure((size_t)2 * sg.maxpieces * sg.HT * sizeof(float2)));
        LagStreamParams sp{};
        sp.x = ref;
        sp.s[0] = ref; sp.s[1] = srv;
        sp.dmin[0] = 0; sp.dmin[1] = -peek;
        sp.n = (int)n;
        sp.blk_first_lo = 0;
        sp.blk_stride = 0;
        sp.blk_len = (int)n;
        sp.nblk = 1;
        sp.total = sg.total;
        sp.per_cta = sg.per_cta;
        sp.H = sg.H; sp.G = sg.G; sp.steps = sg.steps;
        sp.maxpieces = sg.maxpieces;
        sp.s_linear = linear ? 1 : 0;
        sp.partial = c->partial.as<float2>();
        {
            ProfScope ps(c, K_LAGCORR_LS);
            launch_lagstream(dim3(sg.ncta, 2), sg.threads, sg.smem, c->stream, sp);
        }
        TRY(check_launch("lagstream_kernel(ls)"));
        g.nchunk = sg.maxpieces;      // == pieces of the single block == ncta
        g.HT = sg.HT;
    } else {
    TRY(choose_geo((int)n, 2, M, c->nsm, &g));
    TRY(c->partial.ensure((size_t)2 * g.nchunk * g.HT * sizeof(float2)));

    LagCorrParams p{};
    p.x = ref;
    p.s[0] = ref; p.s[1] = srv;
    p.dmin[0] = 0; p.dmin[1] = -peek;
    p.win = nullptr; p.taps = nullptr;
    p.n = (int)n;
    p.blk_first_lo = 0;
    p.blk_stride = 0;
    p.blk_len = (int)n;
    p.nblk = 1;
    p.nchunk = g.nchunk;
    p.chunk_len = g.chunk_len;
    p.H = g.H; p.G = g.G; p.steps = g.steps;
    p.partial = c->partial.as<float2>();
    {
        ProfScope ps(c, K_LAGCORR_LS);
        if (g_packed) lagcorr_kernel<LC_TI, LC_TD, true><<<dim3(g.nchunk, 2), g.threads, g.smem, c->stream>>>(p);
        else lagcorr_kernel<LC_TI, LC_TD, false><<<dim3(g.nchunk, 2), g.threads, g.smem, c->stream>>>(p);
    }
    TRY(check_launch("lagcorr_kernel(ls)"));
    }

    LevinsonParams lp{};
    lp.partial = c->partial.as<float2>();
    lp.nchunk = g.nchunk;
    lp.HT = g.HT;
    lp.M = M;
    lp.reg = reg;
    lp.taps = c->lstaps.as<float2>();
    lp.status = c->status.as<int>() + c->status_slot;
    {
        ProfScope ps(c, K_LEVINSON);
        if (M <= 1024) levinson_kernel<1><<<1, 1024, levinson_smem(M, 1024), c->stream>>>(lp);
        else levinson_kernel<4><<<1, 512, levinson_smem(M, 512), c->stream>>>(lp);
    }
    TRY(check_launch("levinson_kernel"));

    if (use_fir_tc) {
        for (int k = 0; k < 3; ++k) TRY(c->firb[k].ensure((size_t)tc::FIR_N * fir_kv * sizeof(uint16_t)));
        {
            ProfScope ps(c, K_MISC);          // the taps-matrix builder is bookkeeping, not the FIR itself
            tc::fir_bmat_kernel<<<ceil_div(tc::FIR_N * fir_kv, 256), 256, 0, c->stream>>>(
                c->lstaps.as<float2>(), M, fir_shift, fir_kv, c->firb[0].as<uint16_t>(), c->firb[1].as<uint16_t>(), c->firb[2].as<uint16_t>());
        }
        {
            ProfScope ps(c, K_FIR);
            tc::FirTcParams ft{};
            for (int k = 0; k < 3; ++k) { ft.z[k] = c->tcplane[3 + k].as<uint16_t>(); ft.b[k] = c->firb[k].as<uint16_t>(); }
            ft.zoff = fir_zoff;
            ft.kvp = fir_kv;
            ft.srv = srv; ft.out = out; ft.n = (int)n;
            if (caf && caf->on && caf_x_done) {
                for (int k = 0; k < 3; ++k) {
                    TRY(c->cafplane[3 + k].ensure((size_t)caf->slen * 2 * sizeof(uint16_t)));
                    ft.cafs[k] = c->cafplane[3 + k].as<uint16_t>();
                }
                ft.caf_off = caf->D / 2;
                ft.caf_slen = caf->slen;
                caf->planes_ready = true;
            }
            static long long* dbg = nullptr;
            if (getenv("PRC_FIR_DEBUG")) {
                if (!dbg) cudaMalloc(&dbg, 256);
                cudaMemsetAsync(dbg, 0, 256, c->stream);
                ft.debug_clk = dbg;
            }
            tc::firtc_kernel<<<fir_nblk, tc::FIR_THREADS, tc::firtc_smem_bytes(), c->stream>>>(ft);
            if (ft.debug_clk) {
                long long h[32];
                cudaMemcpyAsync(h, dbg, 256, cudaMemcpyDeviceToHost, c->stream);
                cudaStreamSynchronize(c->stream);
                fprintf(stderr, "[firtc] grid=%d kvp=%d: last MMA commit %lld, tmem_full seen %lld, all done %lld cycles; full[kc] at",
                        fir_nblk, fir_kv, h[1] - h[0], h[2] - h[0], h[3] - h[0]);
                for (int k = 0; k < 12; ++k) fprintf(stderr, " %lld", h[4 + k] - h[0]);
                fprintf(stderr, "; slowest CTA %lld cycles, first start -> last end %lld ns\n", h[20], h[22] - (long long)~(unsigned long long)h[21]);
            }
        }
        TRY(check_launch("firtc_kernel"));
        if (taps_out)
            CU(cudaMemcpyAsync(taps_out, c->lstaps.p, (size_t)M * sizeof(float2), cudaMemcpyDeviceToDevice, c->stream));
        return PRC_OK;
    }
    FirParams fp{};
    fp.ref = ref; fp.srv = srv; fp.taps = c->lstaps.as<float2>(); fp.out = out;
    if (caf && caf->on && caf_x_done) {           // the FIR writes the CAF s operand (cleaned channel) as well
        for (int k = 0; k < 3; ++k) {
            TRY(c->cafplane[3 + k].ensure((size_t)caf->slen * 2 * sizeof(uint16_t)));
            fp.cafs[k] = c->cafplane[3 + k].as<uint16_t>();
        }
        fp.caf_off = caf->D / 2;
        fp.caf_slen = caf->slen;
        caf->planes_ready = true;
    }
    fp.n = (int)n; fp.M = M; fp.peek = peek;
    fp.linear = linear ? 1 : 0;
    const int mode = g_stream ? 2 : (g_packed ? 1 : 0);
    const int tk = mode == 2 ? kTiles[g_tile].ti : FIR_TK, to = mode == 2 ? kTiles[g_tile].td : FIR_TO;
    fp.Mpad = ceil_div(M, tk) * tk;
    if (fp.Mpad & 1) fp.Mpad += tk;          // keep the ref window 16-byte aligned behind the taps
    const int LO = FIR_THREADS * to;
    const size_t sm = (size_t)((mode == 1 ? 2 : 1) * fp.Mpad + LO + fp.Mpad) * sizeof(float2);
    if (sm > SMEM_LIMIT) return fail(PRC_E_INVALID, "%d taps exceed the FIR kernel's shared memory", M);
    {
        ProfScope ps(c, K_FIR);
        const int grid = ceil_div(n, LO);
        if (mode == 0) fir_apply_kernel<FIR_TK, FIR_TO, 0><<<grid, FIR_THREADS, sm, c->stream>>>(fp);
        else if (mode == 1) fir_apply_kernel<FIR_TK, FIR_TO, 1><<<grid, FIR_THREADS, sm, c->stream>>>(fp);
        else if (g_tile == 0) fir_apply_kernel<10, 10, 2><<<grid, FIR_THREADS, sm, c->stream>>>(fp);
        else if (g_tile == 1) fir_apply_kernel<6, 18, 2><<<grid, FIR_THREADS, sm, c->stream>>>(fp);
        else fir_apply_kernel<14, 14, 2><<<grid, FIR_THREADS, sm, c->stream>>>(fp);
    }
    TRY(check_launch("fir_apply_kernel"));
    if (taps_out)
        CU(cudaMemcpyAsync(taps_out, c->lstaps.p, (size_t)M * sizeof(float2), cudaMemcpyDeviceToDevice, c->stream));
    return PRC_OK;
}

// LS_Filter_Toeplitz (reference clutter_removal.py:109-160) on the device: roll (and optionally
// frequency-shift) the reference, then the LS pipeline in linear mode with reg = 0 and all
// filterLen + peek taps causal on the rolled reference.
// bt.nf > 1: a batch of frames, every buffer (ref, srv, out, the rolled reference) bt.stride samples apart (FFT-domain path)
int ls_toeplitz_device(Ctx* c, const float2* ref, const float2* srv, long long n, int filter_len, int peek,
                       bool shift, double fc, double fs, float2* out, float2* taps_out, Batch bt = Batch{}) {
    if (n <= 0 || n >= (1ll << 31) - 4096) return fail(PRC_E_INVALID, "n=%lld unsupported", n);
    if (filter_len < 0 || peek < 0 || filter_len + peek < 1)
        return fail(PRC_E_INVALID, "filter_len=%d peek=%d invalid", filter_len, peek);
    const long long stride = bt.nf > 1 ? bt.stride : n;
    TRY(c->rs.ensure(((size_t)(bt.nf - 1) * stride + n) * sizeof(float2)));
    // complex64(1j*2*pi*fc) * complex64(n) / Fs, evaluated like numpy does (see shift_roll_kernel)
    const float B = (float)(2.0 * 3.14159265358979323846 * fc);
    {
        ProfScope ps(c, K_MISC);
        shift_roll_kernel<<<dim3(ceil_div(n, 256), bt.nf), 256, 0, c->stream>>>(ref, c->rs.as<float2>(), (int)n, peek, shift ? 1 : 0, B,
                                                                                 1.0f / (float)fs, stride);
    }
    TRY(check_launch("shift_roll_kernel"));
    return ls_device(c, c->rs.as<float2>(), srv, n, filter_len + peek, 0, 0.0, out, taps_out, nullptr, nullptr, nullptr, true, bt);
}

// ---- front end (frontend.cuh) -------------------------------------------------------------------
size_t iq_bytes(int kind, long long n) {
    return (size_t)n * (kind == IQ_I8 ? 2 : kind == IQ_I16 ? 4 : 8);
}

MixParams make_mix(const void* in, int kind, long long n, int mode, double fc, double fs, double po) {
    MixParams m{};
    m.in = in; m.kind = kind; m.n = n; m.mode = mode;
    m.B = (float)(2.0 * 3.14159265358979323846 * fc);
    m.rFs = 1.0f / (float)fs;
    m.po = po;
    m.B64 = 2.0 * 3.14159265358979323846 * fc;
    m.rFs64 = 1.0 / fs;
    return m;
}

int mix_device(Ctx* c, const MixParams& m, float2* out) {
    ProfScope ps(c, K_MISC);
    iq_mix_kernel<<<ceil_div(m.n, 256), 256, 0, c->stream>>>(m, out);
    return check_launch("iq_mix_kernel");
}

// scipy.signal.resample_poly(x, up, down, padtype='line') geometry (scipy/signal/_signaltools.py, resample_poly)
struct ResampleGeo { int up, down, n_pre_pad, n_pre_remove, tpp; long long n_out; };

int resample_geo(long long n_in, int up, int down, int nh, ResampleGeo* g) {
    if (up < 1 || down < 1) return fail(PRC_E_INVALID, "up and down must be >= 1");
    if (nh < 1 || (nh & 1) == 0) return fail(PRC_E_INVALID, "nh=%d: the filter must have 2*half_len+1 taps", nh);
    long long a = up, b = down;
    while (b) { const long long t = a % b; a = b; b = t; }
    up /= (int)a; down /= (int)a;
    const int half_len = (nh - 1) / 2;
    g->up = up; g->down = down;
    g->n_pre_pad = down - half_len % down;
    g->n_pre_remove = (half_len + g->n_pre_pad) / down;
    g->n_out = (n_in * up + down - 1) / down;
    g->tpp = ceil_div(g->n_pre_pad + nh, up) | 1;     // odd row stride: the `up` phase rows of the table start in distinct shared-memory banks
    return PRC_OK;
}

// h: host doubles (already multiplied by `up`, as resample_poly does before upfirdn)
int resample_device(Ctx* c, const MixParams& mix, int up_in, int down_in, const double* h, int nh, float2* out,
                    long long* n_out) {
    ResampleGeo g;
    TRY(resample_geo(mix.n, up_in, down_in, nh, &g));
    if (mix.n < 1) return fail(PRC_E_INVALID, "n=%lld invalid", mix.n);
    if (n_out) *n_out = g.n_out;
    if (g.up == 1 && g.down == 1) {           // resample_poly returns a copy
        return mix_device(c, mix, out);
    }
    ResampleParams rp{};
    rp.mix = mix;
    rp.up = g.up; rp.down = g.down; rp.nh = nh;
    rp.n_pre_pad = g.n_pre_pad; rp.n_pre_remove = g.n_pre_remove; rp.tpp = g.tpp;
    rp.n_out = g.n_out;
    rp.span = (int)(((long long)(RS_THREADS - 1) * g.down) / g.up) + 2 + g.tpp;
    const size_t hp_bytes = (((size_t)g.up * g.tpp * 4 + 15) & ~(size_t)15);
    const size_t smem = hp_bytes + (size_t)rp.span * sizeof(float2);
    if (smem > SMEM_LIMIT)
        return fail(PRC_E_INVALID, "resample %d/%d with %d taps needs %zu bytes of shared memory per CTA", g.up, g.down, nh, smem);
    // polyphase table built on the host (nh ~ 2.4k taps) and cached per context: re-uploaded only when
    // the taps change (FNV-1a over the doubles), so steady-state calls enqueue kernels only
    uint64_t key = 1469598103934665603ull;
    auto mixin = [&key](const void* ptr, size_t bytes) {
        const unsigned char* b = static_cast<const unsigned char*>(ptr);
        for (size_t q = 0; q < bytes; ++q) { key ^= b[q]; key *= 1099511628211ull; }
    };
    mixin(h, (size_t)nh * sizeof(double));
    mixin(&g.up, sizeof(int));
    mixin(&g.down, sizeof(int));
    TRY(c->fe_ends.ensure(2 * sizeof(float2)));
    if (key != c->fe_hp_key || !c->fe_hp.p) {
        std::vector<float> hp((size_t)g.up * g.tpp, 0.f);
        for (int k = g.n_pre_pad; k < g.n_pre_pad + nh; ++k) hp[(size_t)(k % g.up) * g.tpp + k / g.up] = (float)h[k - g.n_pre_pad];
        TRY(c->fe_hp.ensure(hp.size() * sizeof(float)));
        CU(cudaMemcpyAsync(c->fe_hp.p, hp.data(), hp.size() * sizeof(float), cudaMemcpyHostToDevice, c->stream));
        CU(cudaStreamSynchronize(c->stream));     // hp is a stack-lifetime host buffer
        c->fe_hp_key = key;
    }
    rp.hp = c->fe_hp.as<float>();
    rp.ends = c->fe_ends.as<float2>();
    static std::atomic<bool> attr_set[64];
    if (!attr_set[c->device].exchange(true))
        CU(cudaFuncSetAttribute(resample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_LIMIT));
    {
        ProfScope ps(c, K_MISC);
        resample_ends_kernel<<<1, 32, 0, c->stream>>>(mix, c->fe_ends.as<float2>());
        resample_kernel<<<ceil_div(g.n_out, RS_THREADS), RS_THREADS, smem, c->stream>>>(rp, out);
    }
    return check_launch("resample_kernel");
}

// ---- CFAR_2D (detect.cuh) -----------------------------------------------------------------------
int cfar_device(Ctx* c, const void* x, bool is_complex, int rows, int cols, int fw, int gw, const float* thresh,
                float* cr, uint8_t* det) {
    if (rows < 1 || cols < 1) return fail(PRC_E_INVALID, "rows=%d cols=%d invalid", rows, cols);
    if (fw < 1 || fw > CFAR_MAX_FW) return fail(PRC_E_INVALID, "fw=%d outside [1, %d]", fw, CFAR_MAX_FW);
    if (gw < 0 || fw * fw - gw * gw == 0) return fail(PRC_E_INVALID, "fw=%d gw=%d: fw^2 - gw^2 must not be 0", fw, gw);
    TRY(c->cf_part.ensure(CFAR_MEAN_CTAS * sizeof(double)));
    CfarParams p{};
    p.x = x; p.is_complex = is_complex ? 1 : 0; p.rows = rows; p.cols = cols;
    p.fw = fw;
    // python: e1 = (fw - gw) // 2 (floor), e2 = fw - e1 + 1; slices clip to [0, fw]
    int e1 = (fw - gw) >= 0 ? (fw - gw) / 2 : -((gw - fw + 1) / 2);
    int e2 = fw - e1 + 1;
    if (e1 < 0) e1 = std::max(0, e1 + fw);     // negative slice start counts from the end
    p.e1 = std::min(e1, fw); p.e2 = std::min(std::max(e2, 0), fw);
    p.c = (fw - 1) / 2;
    p.scale = (float)(1.0 / ((double)fw * fw - (double)gw * gw));
    p.has_thresh = thresh ? 1 : 0;
    p.thresh = thresh ? *thresh : 0.f;
    p.partial = c->cf_part.as<double>();
    p.cr = cr; p.det = det;
    ProfScope ps(c, K_MISC);
    cfar_abssum_kernel<<<CFAR_MEAN_CTAS, 256, 0, c->stream>>>(p, c->cf_part.as<double>());
    const size_t smem = (size_t)(CFAR_TX + fw - 1) * (CFAR_TY + fw - 1) * sizeof(float);
    cfar2d_kernel<<<dim3(ceil_div(cols, CFAR_TX), ceil_div(rows, CFAR_TY)), dim3(CFAR_TX, CFAR_TY), smem, c->stream>>>(p);
    return check_launch("cfar2d_kernel");
}

// ---- direct_xambg (reference range_doppler_processing.py:93-124) ---------------------------------
// row f: xcorr(frequency_shift(ref, (f - F/2)/CPI, Fs), srv, R, 0): a LINEAR lag correlation of the
// frequency-shifted reference (float32 phase ramp, complex64 exp -- as the reference) with srv.
int direct_xambg_device(Ctx* c, const float2* ref, const float2* srv, long long n, int R, int F, double fs, float2* out) {
    if (n <= 0 || n >= (1ll << 31) - 4096) return fail(PRC_E_INVALID, "n=%lld unsupported", n);
    if (R < 0 || F < 1) return fail(PRC_E_INVALID, "range_bins=%d freq_bins=%d invalid", R, F);
    if (!(fs > 0)) return fail(PRC_E_INVALID, "sample_rate must be > 0");
    TRY(c->rs.ensure((size_t)n * sizeof(float2)));
    StreamGeo sg;
    TRY(choose_stream((int)n, 1, 1, R + 1, c->nsm, &sg));
    TRY(c->partial.ensure((size_t)sg.maxpieces * sg.HT * sizeof(float2)));
    const double cpi = (double)n / fs;
    for (int f = 0; f < F; ++f) {
        const double df = ((double)f - 0.5 * (double)F) / cpi;
        const MixParams m = make_mix(ref, IQ_C64, n, MIX_C64, df, fs, 0.0);
        TRY(mix_device(c, m, c->rs.as<float2>()));
        LagStreamParams sp{};
        sp.x = c->rs.as<float2>();
        sp.s[0] = srv; sp.s[1] = srv;
        sp.dmin[0] = 0; sp.dmin[1] = 0;
        sp.n = (int)n;
        sp.blk_first_lo = 0; sp.blk_stride = 0; sp.blk_len = (int)n; sp.nblk = 1;
        sp.total = sg.total; sp.per_cta = sg.per_cta;
        sp.H = sg.H; sp.G = sg.G; sp.steps = sg.steps;
        sp.maxpieces = sg.maxpieces;
        sp.s_linear = 1;
        sp.partial = c->partial.as<float2>();
        {
            ProfScope ps(c, K_LAGCORR_CAF);
            launch_lagstream(dim3(sg.ncta, 1), sg.threads, sg.smem, c->stream, sp);
            piece_sum_kernel<<<ceil_div(R + 1, 128), 128, 0, c->stream>>>(c->partial.as<float2>(), sg.maxpieces, sg.HT, R,
                                                                     out + (size_t)f * (R + 1));
        }
        TRY(check_launch("lagstream_kernel(direct_xambg)"));
    }
    return PRC_OK;
}

// bt.nf independent frames run as one CTA each (the recurrence of a frame is serial, the frames are not)
int nlms_device(Ctx* c, const float2* ref, const float2* srv, long long n, int filter_len, int peek, float mu,
                int block_len, const float2* init, float2* out, float2* taps_out, Batch bt = Batch{}, bool init_shared = true) {
    if (n <= 0 || n >= (1ll << 31) - 4096) return fail(PRC_E_INVALID, "n=%lld unsupported", n);
    if (filter_len < 0 || peek < 0 || filter_len + peek < 1)
        return fail(PRC_E_INVALID, "filter_len=%d peek=%d invalid", filter_len, peek);
    if (block_len < 1) return fail(PRC_E_INVALID, "block_len=%d invalid", block_len);
    const int M = filter_len + peek;
    if (M > 1024 * NLMS_MAXT) return fail(PRC_E_INVALID, "%d taps exceed the NLMS kernel's maximum of %d", M, 1024 * NLMS_MAXT);
    NlmsParams p{};
    p.ref = ref; p.srv = srv; p.init = init; p.out = out; p.taps_out = taps_out;
    p.n = (int)n; p.filter_len = filter_len; p.peek = peek; p.mu = mu; p.block_len = block_len;
    p.frame_stride = bt.nf > 1 ? bt.stride : 0; p.init_shared = init_shared ? 1 : 0;
    const int kt = M <= 1024 ? 1 : (M <= 2048 ? 2 : 4);
    const int threads = std::min(1024, ((ceil_div(M, kt) + 31) / 32) * 32);
    const size_t sm = (size_t)(NLMS_TILE + ((M + 1) & ~1) + NLMS_TILE) * sizeof(float2) + 64 * sizeof(float4);
    ProfScope ps(c, K_NLMS);
    if (g_nlms_block) {
        // exact evaluation 32 samples at a time (nlms_block.cuh), 4x the speed of the sample-serial kernel at
        // config 4; block_len > 1 (block_NLMS) freezes the taps inside a user block
        const size_t sb = nlms_block_smem(M);
        if (bt.nf > c->nsm && M <= 2048) {
            // more frames than SMs: 512-thread CTAs, two resident per SM (a 1024-thread CTA owns the SM's registers)
            if (M <= 512) nlms_block_kernel<1, 512><<<bt.nf, 512, sb, c->stream>>>(p);
            else if (M <= 1024) nlms_block_kernel<2, 512><<<bt.nf, 512, sb, c->stream>>>(p);
            else nlms_block_kernel<4, 512><<<bt.nf, 512, sb, c->stream>>>(p);
            return check_launch("nlms_block_kernel");
        }
        if (kt == 1) nlms_block_kernel<1><<<bt.nf, NB_THREADS, sb, c->stream>>>(p);
        else if (kt == 2) nlms_block_kernel<2><<<bt.nf, NB_THREADS, sb, c->stream>>>(p);
        else nlms_block_kernel<4><<<bt.nf, NB_THREADS, sb, c->stream>>>(p);
        return check_launch("nlms_block_kernel");
    }
    if (kt == 1) nlms_kernel<1><<<bt.nf, threads, sm, c->stream>>>(p);
    else if (kt == 2) nlms_kernel<2><<<bt.nf, threads, sm, c->stream>>>(p);
    else nlms_kernel<4><<<bt.nf, threads, sm, c->stream>>>(p);
    return check_launch("nlms_kernel");
}

// ---- host <-> device copies of caller arrays.  dask hands the operators ordinary (pageable) numpy arrays from several
// threads at once (main.py:169-194); cudaMemcpyAsync from pageable memory goes through the driver's own staging, one
// copy at a time for the whole process.  Each workspace therefore owns two page-locked bounce buffers: the calling
// thread copies a chunk into one while the DMA engine drains the other, so concurrent callers overlap their host-side
// copies and their transfers.  Page-locked arrays (FramePipeline, prc_host_alloc / prc_host_register) and asynchronous
// calls (PRC_FLAG_ASYNC: the caller owns the synchronisation) take the plain cudaMemcpyAsync path.
constexpr size_t PIN_CHUNK = 4u << 20;

bool host_is_pinned(const void* ptr) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

int ensure_pin(Ctx* c) {
    if (c->pin_ready) return PRC_OK;
    for (int k = 0; k < 2; ++k) {
        CU(cudaHostAlloc(&c->pin[k], PIN_CHUNK, cudaHostAllocPortable));
        CU(cudaEventCreateWithFlags(&c->pin_ev[k], cudaEventDisableTiming));
    }
    c->pin_ready = true;
    return PRC_OK;
}

int h2d(Ctx* c, void* dst, const void* src, size_t bytes, unsigned flags) {
    if ((flags & PRC_FLAG_ASYNC) || bytes < (256u << 10) || host_is_pinned(src)) {
        CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream));
        return PRC_OK;
    }
    TRY(ensure_pin(c));
    int k = 0;
    for (size_t off = 0; off < bytes; off += PIN_CHUNK, k ^= 1) {
        const size_t len = std::min(PIN_CHUNK, bytes - off);
        CU(cudaEventSynchronize(c->pin_ev[k]));           // the transfer that last used this buffer has finished
        memcpy(c->pin[k], static_cast<const char*>(src) + off, len);
        CU(cudaMemcpyAsync(static_cast<char*>(dst) + off, c->pin[k], len, cudaMemcpyHostToDevice, c->stream));
        CU(cudaEventRecord(c->pin_ev[k], c->stream));
    }
    return PRC_OK;
}

int d2h(Ctx* c, void* dst, const void* src, size_t bytes, unsigned flags) {
    if ((flags & PRC_FLAG_ASYNC) || bytes < (256u << 10) || host_is_pinned(dst)) {
        CU(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
        return PRC_OK;
    }
    TRY(ensure_pin(c));
    const size_t nchunk = (bytes + PIN_CHUNK - 1) / PIN_CHUNK;
    for (size_t i = 0; i <= nchunk; ++i) {                // transfer of chunk i overlaps the host copy of chunk i - 1
        if (i < nchunk) {
            const size_t off = i * PIN_CHUNK, len = std::min(PIN_CHUNK, bytes - off);
            CU(cudaMemcpyAsync(c->pin[i & 1], static_cast<const char*>(src) + off, len, cudaMemcpyDeviceToHost, c->stream));
            CU(cudaEventRecord(c->pin_ev[i & 1], c->stream));
        }
        if (i >= 1) {
            const size_t j = i - 1, off = j * PIN_CHUNK, len = std::min(PIN_CHUNK, bytes - off);
            CU(cudaEventSynchronize(c->pin_ev[j & 1]));
            memcpy(static_cast<char*>(dst) + off, c->pin[j & 1], len);
        }
    }
    return PRC_OK;
}

// window (host or device, double or float) -> device float
int stage_window(Ctx* c, const void* window, long long n, int mem_kind, unsigned flags, const float** win32) {
    *win32 = nullptr;
    if (!window) return PRC_OK;
    if (flags & PRC_FLAG_WINDOW_F32) {
        if (mem_kind == PRC_MEM_DEVICE) {
            *win32 = static_cast<const float*>(window);
            return PRC_OK;
        }
        TRY(c->win32.ensure((size_t)n * sizeof(float)));
        TRY(h2d(c, c->win32.p, window, (size_t)n * sizeof(float), flags));
        *win32 = c->win32.as<float>();
        return PRC_OK;
    }
    const double* w64 = static_cast<const double*>(window);
    TRY(c->win32.ensure((size_t)n * sizeof(float)));
    if (mem_kind == PRC_MEM_HOST) {
        TRY(c->win64.ensure((size_t)n * sizeof(double)));
        TRY(h2d(c, c->win64.p, window, (size_t)n * sizeof(double), flags));
        w64 = c->win64.as<double>();
    }
    f64_to_f32_kernel<<<ceil_div(n, 256), 256, 0, c->stream>>>(w64, c->win32.as<float>(), n);
    TRY(check_launch("f64_to_f32_kernel"));
    *win32 = c->win32.as<float>();
    return PRC_OK;
}

int finish(Ctx* c, unsigned flags) {
    if (flags & PRC_FLAG_ASYNC) return PRC_OK;
    CU(cudaStreamSynchronize(c->stream));
    return PRC_OK;
}

int check_ls_status(Ctx* c, unsigned flags, int nf = 1) {
    if (flags & PRC_FLAG_ASYNC) return PRC_OK;   // caller owns the synchronisation; status stays on the device (prc_ls_status)
    std::vector<int> st((size_t)nf, 0);
    CU(cudaMemcpyAsync(st.data(), c->status.p, (size_t)nf * sizeof(int), cudaMemcpyDeviceToHost, /*status*/ c->stream));
    CU(cudaStreamSynchronize(c->stream));
    for (int i = 0; i < nf; ++i)
        if (st[i] != 0)
            return fail(PRC_E_SINGULAR, "LS normal equations are not positive definite (singular Gram matrix, frame %d)", i);
    return PRC_OK;
}

// one frame (or, on the FFT-domain path, a batch of frames) of  LS_Filter -> fast_xambg  on device pointers
int frame_device(Ctx* c, const float2* ref, const float2* srv, long long n, Batch bt, int filter_len, int peek, double reg,
                 int R, int F, const float* win32, float2* maps, float2* taps_out, float2* cleaned_out) {
    const int M = filter_len + peek;
    const long long D = n / F;
    const LsFftPlan lf = (M >= 1 && M <= 2048) ? ls_fft_plan(c, n, M, bt.nf) : LsFftPlan{};
    const CafFftPlan cf = (D >= 2) ? caf_fft_plan(n, R, F, D + 1, D, true, M) : CafFftPlan{};
    if (lf.on && cf.on) {
        // FFT-domain frame: lag sums -> Toeplitz solve -> taps spectrum -> CAF with the clutter filter applied to the
        // surveillance spectrum inside the kernel (the cleaned channel exists only if the caller asks for it)
        TRY(ls_device(c, ref, srv, n, filter_len, peek, reg, cleaned_out, taps_out, nullptr, nullptr, nullptr, false, bt,
                      cleaned_out != nullptr));
        TRY(taps_spectrum(c, cf.r3, M, bt.nf, &c->wp_caf));
        return xambg_device(c, ref, srv, n, R, F, win32, nullptr, 0, maps, false, false, bt, c->wp_caf.as<float2>(), M, peek);
    }
    // direct-form kernels (tcgen05 / FP32), frame by frame
    TRY(c->clean.ensure((size_t)n * sizeof(float2)));
    TRY(c->status.ensure((size_t)bt.nf * sizeof(int)));
    for (int fr = 0; fr < bt.nf; ++fr) {
        const float2* r = ref + (size_t)fr * bt.stride;
        const float2* sv = srv + (size_t)fr * bt.stride;
        float2* dclean = cleaned_out ? cleaned_out + (size_t)fr * bt.stride : c->clean.as<float2>();
        bool refw_ready = false;
        CafTc caf = (n / F) % 2 == 0 ? caf_tc_plan(c, n, R, F, false) : CafTc{};
        c->status_slot = fr;            // frame fr reports its Toeplitz-solve status in status[fr]
        const int rc = ls_device(c, r, sv, n, filter_len, peek, reg, dclean, taps_out ? taps_out + (size_t)fr * M : nullptr, win32,
                                 &refw_ready, &caf);
        c->status_slot = 0;
        TRY(rc);
        TRY(xambg_device(c, r, dclean, n, R, F, win32, nullptr, 0, maps + (size_t)fr * F * (R + 1), refw_ready, caf.planes_ready));
    }
    return PRC_OK;
}

bool bad_mem_kind(int k) { return k != PRC_MEM_HOST && k != PRC_MEM_DEVICE; }

// --------------------------------------------------------------------------- long-lag correlation (xcorr.cuh)
// Tile plan: one circular transform of P = 2^20 .. 2^24 points holds Lseg x samples and nt lags without wrap-around
// when Lseg + nt - 1 <= P.  Lag windows longer than that are cut into tiles, x into segments whose spectra are
// accumulated before the transform back.
struct XcPlan {
    int r1 = 4, r2 = 4;
    long long P = 0, seg = 0, tile = 0;
    long long nseg = 0, ntile = 0;
};

constexpr long long XC_PMIN = 1ll << 20, XC_PMAX = 1ll << 24;

XcPlan xc_plan(long long nx, long long nlags) {
    XcPlan pl;
    const long long need = nx + nlags - 1;
    if (need <= XC_PMAX) {
        pl.P = XC_PMIN;
        while (pl.P < need) pl.P <<= 1;
        pl.seg = nx;
        pl.tile = nlags;
    } else {
        pl.P = XC_PMAX;
        pl.tile = std::min(nlags, XC_PMAX / 2);
        pl.seg = XC_PMAX - pl.tile + 1;
        if (nx < pl.seg) {
            pl.seg = nx;
            pl.tile = XC_PMAX - nx + 1;
        }
    }
    pl.nseg = (nx + pl.seg - 1) / pl.seg;
    pl.ntile = (nlags + pl.tile - 1) / pl.tile;
    // L1 x L2 = P, L1 >= L2
    const int lg = ilog2((int)(pl.P >> 20));      // P = 2^20 .. 2^24
    static const int r1s[5] = {4, 8, 8, 16, 16}, r2s[5] = {4, 4, 8, 8, 16};
    pl.r1 = r1s[lg];
    pl.r2 = r2s[lg];
    return pl;
}

int xc_p_twiddles(Ctx* c, long long P, const float2** lo, const float2** hi) {
    TRY(c->xc_tw.ensure(8192 * sizeof(float2)));
    if (c->xc_twP != P) {
        xc::p_twiddle_kernel<<<ceil_div(4096 + P / 4096, 256), 256, 0, c->stream>>>(c->xc_tw.as<float2>(),
                                                                                   c->xc_tw.as<float2>() + 4096, P);
        TRY(check_launch("p_twiddle_kernel"));
        c->xc_twP = P;
    }
    *lo = c->xc_tw.as<float2>();
    *hi = c->xc_tw.as<float2>() + 4096;
    return PRC_OK;
}

// out[j] = sum_i x[i] conj(y[i + lag0 - j]), j < nlags (device pointers).  out: complex lags, absout: |xc| (|Re xc| when
// real), best: argmax key (bits(|xc|) << 32 | ~j, max-reduced; caller zeroes it).  Any of the three may be NULL.
int xcorr_device(Ctx* c, const float2* x, long long nx, const float2* y, long long ny, long long lag0, long long nlags,
                 float2* out, float* absout, unsigned long long* best, bool real) {
    const XcPlan pl = xc_plan(nx, nlags);
    const int L1 = 256 * pl.r1, L2 = 256 * pl.r2;
    const float2 *tw1, *tw2, *plo, *phi;
    TRY(fft_twiddles(c, pl.r1, &tw1));
    TRY(fft_twiddles(c, pl.r2, &tw2));
    TRY(xc_p_twiddles(c, pl.P, &plo, &phi));
    TRY(c->xc_X.ensure((size_t)pl.P * sizeof(float2)));
    TRY(c->xc_Y.ensure((size_t)pl.P * sizeof(float2)));
    if (pl.nseg > 1) TRY(c->xc_S.ensure((size_t)pl.P * sizeof(float2)));
    float2* X = c->xc_X.as<float2>();
    float2* Y = c->xc_Y.as<float2>();
    const size_t sm1 = fft_smem(pl.r1), sm2 = fft_smem(pl.r2);
    ProfScope ps(c, K_XCORR);
    for (long long ti = 0; ti < pl.ntile; ++ti) {
        const long long j0 = ti * pl.tile, nt = std::min(pl.tile, nlags - j0);
        const long long m_lo = lag0 - j0 - nt + 1;
        for (long long si = 0; si < pl.nseg; ++si) {
            const long long s = si * pl.seg, ls = std::min(pl.seg, nx - s);
            xc::ColFwdParams cp{};
            cp.L2 = L2; cp.tw = tw1; cp.plo = plo; cp.phi = phi;
            xc::RowParams rp{};
            rp.L2 = L2; rp.tw = tw2; rp.plo = plo; rp.phi = phi;
            // x segment -> X spectrum
            cp.src = x; cp.off = s; cp.nsrc = nx; cp.lim = ls; cp.Z = X;
            rp.Z = X;
            PRC_R3_SWITCH(pl.r1, (xc::col_fwd_kernel<R3><<<L2 / xc::NCOL, 16 * R3, sm1, c->stream>>>(cp)));
            TRY(check_launch("col_fwd_kernel"));
            PRC_R3_SWITCH(pl.r2, (xc::row_fwd_kernel<R3><<<L1, 16 * R3, sm2, c->stream>>>(rp)));
            TRY(check_launch("row_fwd_kernel"));
            // the P samples of y that lags m_lo .. m_lo + nt - 1 of the segment reach -> product spectrum
            cp.src = y; cp.off = s + m_lo; cp.nsrc = ny; cp.lim = pl.P; cp.Z = Y;
            rp.Z = Y; rp.Xh = X; rp.S = c->xc_S.as<float2>();
            rp.acc_in = si > 0; rp.last = si + 1 == pl.nseg;
            PRC_R3_SWITCH(pl.r1, (xc::col_fwd_kernel<R3><<<L2 / xc::NCOL, 16 * R3, sm1, c->stream>>>(cp)));
            TRY(check_launch("col_fwd_kernel"));
            switch (pl.r1 * 100 + pl.r2) {
                case 404: xc::row_prod_kernel<4, 4><<<L1, 64, sm2, c->stream>>>(rp); break;
                case 804: xc::row_prod_kernel<8, 4><<<L1, 64, sm2, c->stream>>>(rp); break;
                case 808: xc::row_prod_kernel<8, 8><<<L1, 128, sm2, c->stream>>>(rp); break;
                case 1608: xc::row_prod_kernel<16, 8><<<L1, 128, sm2, c->stream>>>(rp); break;
                default: xc::row_prod_kernel<16, 16><<<L1, 256, sm2, c->stream>>>(rp); break;
            }
            TRY(check_launch("row_prod_kernel"));
        }
        xc::ColInvParams ip{};
        ip.Z = Y; ip.L2 = L2; ip.nt = nt; ip.j_hi = j0 + nt - 1;
        ip.scale = 1.0f / (float)pl.P;
        ip.out = out; ip.absout = absout; ip.best = best; ip.real = real ? 1 : 0;
        ip.tw = tw1;
        PRC_R3_SWITCH(pl.r1, (xc::col_inv_kernel<R3><<<L2 / xc::NCOL, 16 * R3, sm1, c->stream>>>(ip)));
        TRY(check_launch("col_inv_kernel"));
    }
    return PRC_OK;
}

// scipy.signal.sosfiltfilt's filter as the device runs it: normalised sections, sosfilt_zi, padlen, warm-up length
struct SosDesign {
    int ns = 0, pad = 0, warm = 0;
    double c[xc::SOS_MAX][5], zi[xc::SOS_MAX][2];
};

int sos_design(const double* sos, int nsec, SosDesign* d) {
    if (!sos || nsec < 1 || nsec > xc::SOS_MAX) return fail(PRC_E_INVALID, "nsections=%d invalid (1..%d)", nsec, xc::SOS_MAX);
    d->ns = nsec;
    int zb = 0, za = 0;
    double rho = 0.0, scale = 1.0;
    for (int s = 0; s < nsec; ++s) {
        const double* q = sos + 6 * s;
        if (q[3] != 1.0) return fail(PRC_E_INVALID, "sos[%d, 3] must be 1", s);
        zb += q[2] == 0.0;
        za += q[5] == 0.0;
        const double b0 = q[0], b1 = q[1], b2 = q[2], a1 = q[4], a2 = q[5];
        d->c[s][0] = b0; d->c[s][1] = b1; d->c[s][2] = b2; d->c[s][3] = a1; d->c[s][4] = a2;
        // lfilter_zi of the section: (I - companion(a)^T) zi = b[1:] - a[1:] b0
        const double B0 = b1 - a1 * b0, B1 = b2 - a2 * b0;
        const double den = 1.0 + a1 + a2;
        if (den == 0.0) return fail(PRC_E_INVALID, "section %d has a pole at z = 1", s);
        const double z0 = (B0 + B1) / den;
        d->zi[s][0] = scale * z0;
        d->zi[s][1] = scale * (B1 - a2 * z0);
        scale *= (b0 + b1 + b2) / den;
        // pole radius of z^2 + a1 z + a2
        const double disc = a1 * a1 - 4.0 * a2;
        const double r = disc < 0.0 ? std::sqrt(a2) : std::max(std::fabs(-a1 + std::sqrt(disc)), std::fabs(-a1 - std::sqrt(disc))) / 2.0;
        rho = std::max(rho, r);
    }
    for (int s = nsec; s < xc::SOS_MAX; ++s)
        for (int k = 0; k < 5; ++k) d->c[s][k] = 0.0, d->zi[s][k % 2] = 0.0;
    if (!(rho < 1.0)) return fail(PRC_E_INVALID, "unstable filter (pole radius %.6f)", rho);
    d->pad = 3 * (2 * nsec + 1 - std::min(zb, za));
    // free response below 1e-20 of the state it forgets
    d->warm = rho > 0.0 ? (int)std::min(1e7, std::ceil(std::log(1e-20) / std::log(rho))) : 0;
    d->warm = std::max(d->warm, 32);
    return PRC_OK;
}

size_t sig_elem(int kind) {
    switch (kind) {
        case xc::SIG_I8: return 1;
        case xc::SIG_I16: return 2;
        case xc::SIG_F64: return 8;
        case xc::SIG_C64: return 8;
        default: return 16;
    }
}
bool sig_complex(int kind) { return kind == xc::SIG_C64 || kind == xc::SIG_C128; }

// sosfiltfilt(sos, in)[::nd] -> out (complex64, ceil(n / nd) samples)
int decimate_device(Ctx* c, const void* in, int kind, long long n, const SosDesign& d, int nd, float2* out) {
    xc::IirParams p{};
    p.in = in; p.kind = kind; p.n = n; p.ns = d.ns; p.pad = d.pad;
    p.ne = n + 2ll * d.pad;
    p.chunk = 1024; p.warm = d.warm;
    memcpy(p.c, d.c, sizeof p.c);
    memcpy(p.zi, d.zi, sizeof p.zi);
    const bool cplx = sig_complex(kind);
    TRY(c->xc_yf.ensure((size_t)p.ne * (cplx ? sizeof(double2) : sizeof(double))));
    p.yf = c->xc_yf.p;
    p.out = out; p.nd = nd; p.nout = (n + nd - 1) / nd;
    const int nthr = ceil_div(p.ne, p.chunk);
    ProfScope ps(c, K_IIR);
    if (cplx) {
        xc::iir_fwd_kernel<double2><<<ceil_div(nthr, 32), 32, 0, c->stream>>>(p);
        TRY(check_launch("iir_fwd_kernel"));
        xc::iir_bwd_kernel<double2><<<ceil_div(nthr, 32), 32, 0, c->stream>>>(p);
    } else {
        xc::iir_fwd_kernel<double><<<ceil_div(nthr, 32), 32, 0, c->stream>>>(p);
        TRY(check_launch("iir_fwd_kernel"));
        xc::iir_bwd_kernel<double><<<ceil_div(nthr, 32), 32, 0, c->stream>>>(p);
    }
    return check_launch("iir_bwd_kernel");
}

// lag window of scipy.signal.correlate(s1, np.pad(s2, (nlag, nlead)), 'valid') (reference signal_utils.py:29-32):
// out[k] = c[lag0 - k], k < nlags
void xcorr_window(long long n1, long long n2, long long nlead, long long nlag, long long* lag0, long long* nlags) {
    const long long L2 = n2 + nlag + nlead;
    if (L2 >= n1) {
        *lag0 = n2 - n1 + nlead;
        *nlags = L2 - n1 + 1;
    } else {
        *lag0 = -nlag;
        *nlags = n1 - L2 + 1;
    }
}

constexpr long long XC_MAX_LAGS = 0x7FFFFFFFll;    // lag indices fit the 32 low bits of the argmax key

}  // namespace

// =========================================================================== C ABI
extern "C" {

int prc_version(void) { return PRC_VERSION; }

const char* prc_last_error(void) { return g_err.c_str(); }

int prc_device_count(int* count) {
    if (!count) return fail(PRC_E_INVALID, "count is NULL");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        *count = 0;
        return fail(PRC_E_CUDA, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    }
    *count = n;
    return PRC_OK;
}

int prc_init(int device) {
    Ctx* c;
    return get_ctx(device, nullptr, &c);
}

void prc_shutdown(void) {
    std::lock_guard<std::mutex> lk(g_mu);
    for (Ctx* c : g_all_ctx) {
        c->release();
        delete c;
    }
    g_all_ctx.clear();
    g_stream_ctx.clear();
    g_epoch.fetch_add(1);
}

int prc_sync(int device, void* stream) {
    Ctx* c;
    TRY(get_ctx(device, stream, &c));
    CU(cudaStreamSynchronize(c->stream));
    return PRC_OK;
}

uint64_t prc_launch_count(void) { return g_launches.load(); }

int prc_profile_enable(int on) {
    g_prof_on.store(on ? 1 : 0);
    return PRC_OK;
}

// Drains every workspace's pending event pairs (synchronising their streams) into the totals.
int prc_profile_collect(void) {
    std::lock_guard<std::mutex> lk(g_mu);
    std::lock_guard<std::mutex> lp(g_prof_mu);
    for (Ctx* c : g_all_ctx) {
        std::lock_guard<std::mutex> lc(c->mu);
        if (c->recs.empty()) continue;
        cudaSetDevice(c->device);
        for (ProfRec& r : c->recs) {
            cudaEventSynchronize(r.b);
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) {
                g_prof_ms[r.id] += ms;
                g_prof_n[r.id] += 1;
            }
            cudaEventDestroy(r.a);
            cudaEventDestroy(r.b);
        }
        c->recs.clear();
    }
    return PRC_OK;
}

int prc_profile_kernels(void) { return K_COUNT; }

int prc_profile_read(int idx, const char** name, double* total_ms, uint64_t* launches) {
    if (idx < 0 || idx >= K_COUNT) return fail(PRC_E_INVALID, "kernel index %d out of range", idx);
    std::lock_guard<std::mutex> lp(g_prof_mu);
    if (name) *name = kKernelNames[idx];
    if (total_ms) *total_ms = g_prof_ms[idx];
    if (launches) *launches = g_prof_n[idx];
    return PRC_OK;
}

int prc_profile_reset(void) {
    std::lock_guard<std::mutex> lp(g_prof_mu);
    for (int i = 0; i < K_COUNT; ++i) { g_prof_ms[i] = 0; g_prof_n[i] = 0; }
    return PRC_OK;
}

int prc_host_alloc(void** ptr, uint64_t bytes) {
    if (!ptr) return fail(PRC_E_INVALID, "ptr is NULL");
    CU(cudaHostAlloc(ptr, bytes ? bytes : 1, cudaHostAllocPortable));
    return PRC_OK;
}
int prc_host_free(void* ptr) {
    CU(cudaFreeHost(ptr));
    return PRC_OK;
}
int prc_host_register(void* ptr, uint64_t bytes) {
    CU(cudaHostRegister(ptr, bytes, cudaHostRegisterPortable));
    return PRC_OK;
}
int prc_host_unregister(void* ptr) {
    CU(cudaHostUnregister(ptr));
    return PRC_OK;
}

int prc_xambg_c64(const prc_c64* ref, const prc_c64* srv, int64_t n, int range_bins, int freq_bins,
                  const void* window, const double* dtaps, int64_t ndtaps, prc_c64* out, int mem_kind,
                  int device, void* stream, unsigned flags) {
    if (!ref || !srv || !out) return fail(PRC_E_INVALID, "ref/srv/out must not be NULL");
    if (bad_mem_kind(mem_kind)) return fail(PRC_E_INVALID, "mem_kind=%d invalid", mem_kind);
    if (n <= 0) return fail(PRC_E_INVALID, "n=%lld invalid", (long long)n);
    if (dtaps && ndtaps < 1) return fail(PRC_E_INVALID, "ndtaps=%lld invalid", (long long)ndtaps);
    Ctx* c;
    TRY(get_ctx(device, stream, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    const size_t nb = (size_t)n * sizeof(float2);
    const size_t ob = (size_t)freq_bins * (range_bins + 1) * sizeof(float2);
    const float2* dref = reinterpret_cast<const float2*>(ref);
    const float2* dsrv = reinterpret_cast<const float2*>(srv);
    float2* dout = reinterpret_cast<float2*>(out);
    if (mem_kind == PRC_MEM_HOST) {
        if (freq_bins < 1 || range_bins < 0) return fail(PRC_E_INVALID, "freq_bins=%d / range_bins=%d invalid", freq_bins, range_bins);
        TRY(c->ref.ensure(nb));
        TRY(c->srv.ensure(nb));
        TRY(c->out.ensure(ob));
        TRY(h2d(c, c->ref.p, ref, nb, flags));
        TRY(h2d(c, c->srv.p, srv, nb, flags));
        dref = c->ref.as<float2>();
        dsrv = c->srv.as<float2>();
        dout = c->out.as<float2>();
    }
    const float* win32;
    TRY(stage_window(c, window, n, mem_kind, flags, &win32));
    const float* taps32 = nullptr;
    if (dtaps) {
        TRY(c->dtaps32.ensure((size_t)ndtaps * sizeof(float)));
        const double* t64 = dtaps;
        if (mem_kind == PRC_MEM_HOST) {
            TRY(c->dtaps64.ensure((size_t)ndtaps * sizeof(double)));
            TRY(h2d(c, c->dtaps64.p, dtaps, (size_t)ndtaps * sizeof(double), flags));
            t64 = c->dtaps64.as<double>();
        }
        f64_to_f32_kernel<<<ceil_div(ndtaps, 256), 256, 0, c->stream>>>(t64, c->dtaps32.as<float>(), ndtaps);
        TRY(check_launch("f64_to_f32_kernel"));
        taps32 = c->dtaps32.as<float>();
    }
    TRY(xambg_device(c, dref, dsrv, n, range_bins, freq_bins, win32, taps32, ndtaps, dout));
    if (mem_kind == PRC_MEM_HOST) TRY(d2h(c, out, c->out.p, ob, flags));
    return finish(c, flags);
}

int prc_ls_filter_c64(const prc_c64* ref, const prc_c64* srv, int64_t n, int filter_len, int peek, float reg,
                      prc_c64* out, prc_c64* taps, int mem_kind, int device, void* stream, unsigned flags) {
    if (!ref || !srv || !out) return fail(PRC_E_INVALID, "ref/srv/out must not be NULL");
    if (bad_mem_kind(mem_kind)) return fail(PRC_E_INVALID, "mem_kind=%d invalid", mem_kind);
    if (n <= 0) return fail(PRC_E_INVALID, "n=%lld invalid", (long long)n);
    Ctx* c;
    TRY(get_ctx(device, stream, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    const size_t nb = (size_t)n * sizeof(float2);
    const float2* dref = reinterpret_cast<const float2*>(ref);
    const float2* dsrv = reinterpret_cast<const float2*>(srv);
    float2* dout = reinterpret_cast<float2*>(out);
    float2* dtaps = reinterpret_cast<float2*>(taps);
    if (mem_kind == PRC_MEM_HOST) {
        TRY(c->ref.ensure(nb));
        TRY(c->srv.ensure(nb));
        TRY(c->clean.ensure(nb));
        TRY(h2d(c, c->ref.p, ref, nb, flags));
        TRY(h2d(c, c->srv.p, srv, nb, flags));
        dref = c->ref.as<float2>();
        dsrv = c->srv.as<float2>();
        dout = c->clean.as<float2>();
        dtaps = nullptr;
    }
    TRY(ls_device(c, dref, dsrv, n, filter_len, peek, (double)reg, dout, dtaps));
    if (mem_kind == PRC_MEM_HOST) {
        TRY(d2h(c, out, c->clean.p, nb, flags));
        if (taps)
            TRY(d2h(c, taps, c->lstaps.p, (size_t)(filter_len + peek) * sizeof(float2), flags));
    }
    TRY(check_ls_status(c, flags));
    return finish(c, flags);
}

int prc_nlms_c64(const prc_c64* ref, const prc_c64* srv, int64_t n, int filter_len, int peek, float mu,
                 int block_len, const prc_c64* init_taps, prc_c64* out, prc_c64* taps_out, int mem_kind,
                 int device, void* stream, unsigned flags) {
    if (!ref || !srv || !out) return fail(PRC_E_INVALID, "ref/srv/out must not be NULL");
    if (bad_mem_kind(mem_kind)) return fail(PRC_E_INVALID, "mem_kind=%d invalid", mem_kind);
    if (n <= 0) return fail(PRC_E_INVALID, "n=%lld invalid", (long long)n);
    Ctx* c;
    TRY(get_ctx(device, stream, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    const size_t nb = (size_t)n * sizeof(float2);
    const int M = filter_len + peek;
    const size_t mb = (size_t)(M > 0 ? M : 1) * sizeof(float2);
    const float2* dref = reinterpret_cast<const float2*>(ref);
    const float2* dsrv = reinterpret_cast<const float2*>(srv);
    const float2* dinit = reinterpret_cast<const float2*>(init_taps);
    float2* dout = reinterpret_cast<float2*>(out);
    float2* dtaps = reinterpret_cast<float2*>(taps_out);
    if (mem_kind == PRC_MEM_HOST) {
        TRY(c->ref.ensure(nb));
        TRY(c->srv.ensure(nb));
        TRY(c->clean.ensure(nb));
        TRY(c->nl_taps.ensure(mb));
        TRY(h2d(c, c->ref.p, ref, nb, flags));
        TRY(h2d(c, c->srv.p, srv, nb, flags));
        if (init_taps) {
            TRY(c->nl_init.ensure(mb));
            TRY(h2d(c, c->nl_init.p, init_taps, mb, flags));
            dinit = c->nl_init.as<float2>();
        }
        dref = c->ref.as<float2>();
        dsrv = c->srv.as<float2>();
        dout = c->clean.as<float2>();
        dtaps = c->nl_taps.as<float2>();
    }
    TRY(nlms_device(c, dref, dsrv, n, filter_len, peek, mu, block_len, dinit, dout, dtaps));
    if (mem_kind == PRC_MEM_HOST) {
        TRY(d2h(c, out, c->clean.p, nb, flags));
        if (taps_out) TRY(d2h(c, taps_out, c->nl_taps.p, mb, flags));
    }
    return finish(c, flags);
}

int prc_nlms_frames_c64(const prc_c64* ref, const prc_c64* srv, int64_t n, int nframes, int64_t frame_stride,
                        int filter_len, int peek, float mu, int block_len, const prc_c64* init_taps, prc_c64* out,
                        prc_c64* taps_out, int mem_kind, int device, void* stream, unsigned flags) {
    if (!ref || !srv || !out) return fail(PRC_E_INVALID, "ref/srv/out must not be NULL");
    if (bad_mem_kind(mem_kind)) return fail(PRC_E_INVALID, "mem_kind=%d invalid", mem_kind);
    if (n <= 0) return fail(PRC_E_INVALID, "n=%lld invalid", (long long)n);
    if (nframes < 1) return fail(PRC_E_INVALID, "nframes=%d invalid", nframes);
    if (nframes > 1 && frame_stride < n) return fail(PRC_E_INVALID, "frame_stride=%lld smaller than n=%lld", (long long)frame_stride, (long long)n);
    Ctx* c;
    TRY(get_ctx(device, stream, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    const size_t nb = (size_t)n * sizeof(float2);
    const int M = filter_len + peek;
    const size_t mb = (size_t)(M > 0 ? M : 1) * sizeof(float2);
    Batch bt;
    bt.nf = nframes;
    bt.stride = nframes > 1 ? frame_stride : n;
    const float2* dref = reinterpret_cast<const float2*>(ref);
    const float2* dsrv = reinterpret_cast<const float2*>(srv);
    const float2* dinit = reinterpret_cast<const float2*>(init_taps);
    float2* dout = reinterpret_cast<float2*>(out);
    float2* dtaps = reinterpret_cast<float2*>(taps_out);
    if (mem_kind == PRC_MEM_HOST) {
        TRY(c->ref.ensure(nb * nframes));
        TRY(c->srv.ensure(nb * nframes));
        TRY(c->clean.ensure(nb * nframes));
        TRY(c->nl_taps.ensure(mb * nframes));
        for (int fr = 0; fr < nframes; ++fr) {
            TRY(h2d(c, c->ref.as<float2>() + (size_t)fr * n, ref + (size_t)fr * bt.stride, nb, flags));
            TRY(h2d(c, c->srv.as<float2>() + (size_t)fr * n, srv + (size_t)fr * bt.stride, nb, flags));
        }
        if (init_taps) {
            TRY(c->nl_init.ensure(mb));
            TRY(h2d(c, c->nl_init.p, init_taps, mb, flags));
            dinit = c->nl_init.as<float2>();
        }
        dref = c->ref.as<float2>();
        dsrv = c->srv.as<float2>();
        dout = c->clean.as<float2>();
        dtaps = c->nl_taps.as<float2>();
        bt.stride = n;
    }
    TRY(nlms_device(c, dref, dsrv, n, filter_len, peek, mu, block_len, dinit, dout, dtaps, bt, true));
    if (mem_kind == PRC_MEM_HOST) {
        const size_t fs = (size_t)(nframes > 1 ? frame_stride : n);
        for (int fr = 0; fr < nframes; ++fr)
            TRY(d2h(c, out + fr * fs, c->clean.as<float2>() + (size_t)fr * n, nb, flags));
        if (taps_out) TRY(d2h(c, taps_out, c->nl_taps.p, mb * nframes, flags));
    }
    return finish(c, flags);
}

int prc_xambg_frames_c64(const prc_c64* ref, const prc_c64* srv, int64_t n, int nframes, int64_t frame_stride,
                         int range_bins, int freq_bins, const void* window, prc_c64* out, int mem_kind, int device,
                         void* stream, unsigned flags) {
    if (!ref || !srv || !out) return fail(PRC_E_INVALID, "ref/srv/out must not be NULL");
    if (bad_mem_kind(mem_kind)) return fail(PRC_E_INVALID, "mem_kind=%d invalid", mem_kind);
    if (n <= 0) return fail(PRC_E_INVALID, "n=%lld invalid", (long long)n);
    if (nframes < 1) return fail(PRC_E_INVALID, "nframes=%d invalid", nframes);
    if (nframes > 1 && frame_stride < n) return fail(PRC_E_INVALID, "frame_stride=%lld smaller than n=%lld", (long long)frame_stride, (long long)n);
    if (freq_bins < 1 || range_bins < 0) return fail(PRC_E_INVALID, "freq_bins=%d / range_bins=%d invalid", freq_bins, range_bins);
    Ctx* c;
    TRY(get_ctx(device, stream, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    const size_t nb = (size_t)n * sizeof(float2);
    const size_t ob = (size_t)freq_bins * (range_bins + 1) * sizeof(float2);
    Batch bt;
    bt.nf = nframes;
    bt.stride = nframes > 1 ? frame_stride : n;
    const float2* dref = reinterpret_cast<const float2*>(ref);
    const float2* dsrv = reinterpret_cast<const float2*>(srv);
    float2* dout = reinterpret_cast<float2*>(out);
    if (mem_kind == PRC_MEM_HOST) {
        TRY(c->ref.ensure(nb * nframes));
        TRY(c->srv.ensure(nb * nframes));
        TRY(c->out.ensure(ob * nframes));
        for (int fr = 0; fr < nframes; ++fr) {
            TRY(h2d(c, c->ref.as<float2>() + (size_t)fr * n, ref + (size_t)fr * bt.stride, nb, flags));
            TRY(h2d(c, c->srv.as<float2>() + (size_t)fr * n, srv + (size_t)fr * bt.stride, nb, flags));
        }
        dref = c->ref.as<float2>();
        dsrv = c->srv.as<float2>();
        dout = c->out.as<float2>();
        bt.stride = n;
    }
    const float* win32;
    TRY(stage_window(c, window, n, mem_kind, flags, &win32));
    const long long D = n / freq_bins;
    const bool batched = D >= 2 && caf_fft_plan(n, range_bins, freq_bins, D + 1, D, true, 0).on;
    if (batched || nframes == 1) {
        TRY(xambg_device(c, dref, dsrv, n, range_bins, freq_bins, win32, nullptr, 0, dout, false, false, bt));
    } else {
        for (int fr = 0; fr < nframes; ++fr)       // direct-form kernels, frame by frame
            TRY(xambg_device(c, dref + (size_t)fr * bt.stride, dsrv + (size_t)fr * bt.stride, n, range_bins, freq_bins, win32,
                             nullptr, 0, dout + (size_t)fr * freq_bins * (range_bins + 1)));
    }
    if (mem_kind == PRC_MEM_HOST) TRY(d2h(c, out, c->out.p, ob * nframes, flags));
    return finish(c, flags);
}

int prc_frames_c64(const prc_c64* ref, const prc_c64* srv, int64_t n, int nframes, int64_t frame_stride,
                   int filter_len, int peek, float reg, int range_bins, int freq_bins, const void* window,
                   prc_c64* out_maps, prc_c64* taps_out, prc_c64* cleaned_out, int mem_kind, int device, void* stream,
                   unsigned flags) {
    if (!ref || !srv || !out_maps) return fail(PRC_E_INVALID, "ref/srv/out_maps must not be NULL");
    if (bad_mem_kind(mem_kind)) return fail(PRC_E_INVALID, "mem_kind=%d invalid", mem_kind);
    if (n <= 0) return fail(PRC_E_INVALID, "n=%lld invalid", (long long)n);
    if (nframes < 1) return fail(PRC_E_INVALID, "nframes=%d invalid", nframes);
    if (nframes > 1 && frame_stride < n) return fail(PRC_E_INVALID, "frame_stride=%lld smaller than n=%lld", (long long)frame_stride, (long long)n);
    if (freq_bins < 1 || range_bins < 0) return fail(PRC_E_INVALID, "freq_bins=%d / range_bins=%d invalid", freq_bins, range_bins);
    if (filter_len < 0 || peek < 0 || filter_len + peek < 1)
        return fail(PRC_E_INVALID, "filter_len=%d peek=%d invalid", filter_len, peek);
    Ctx* c;
    TRY(get_ctx(device, stream, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    const int M = filter_len + peek;
    const size_t nb = (size_t)n * sizeof(float2);
    const size_t ob = (size_t)freq_bins * (range_bins + 1) * sizeof(float2);
    Batch bt;
    bt.nf = nframes;
    bt.stride = nframes > 1 ? frame_stride : n;
    const float2* dref = reinterpret_cast<const float2*>(ref);
    const float2* dsrv = reinterpret_cast<const float2*>(srv);
    float2* dmap = reinterpret_cast<float2*>(out_maps);
    float2* dtaps = reinterpret_cast<float2*>(taps_out);
    float2* dclean = reinterpret_cast<float2*>(cleaned_out);
    if (mem_kind == PRC_MEM_HOST) {
        TRY(c->ref.ensure(nb * nframes));
        TRY(c->srv.ensure(nb * nframes));
        TRY(c->out.ensure(ob * nframes));
        if (cleaned_out) TRY(c->clean.ensure(nb * nframes));
        for (int fr = 0; fr < nframes; ++fr) {
            TRY(h2d(c, c->ref.as<float2>() + (size_t)fr * n, ref + (size_t)fr * bt.stride, nb, flags));
            TRY(h2d(c, c->srv.as<float2>() + (size_t)fr * n, srv + (size_t)fr * bt.stride, nb, flags));
        }
        dref = c->ref.as<float2>();
        dsrv = c->srv.as<float2>();
        dmap = c->out.as<float2>();
        dtaps = nullptr;
        dclean = cleaned_out ? c->clean.as<float2>() : nullptr;
        bt.stride = n;
    }
    const float* win32;
    TRY(stage_window(c, window, n, mem_kind, flags, &win32));
    TRY(frame_device(c, dref, dsrv, n, bt, filter_len, peek, (double)reg, range_bins, freq_bins, win32, dmap, dtaps, dclean));
    if (mem_kind == PRC_MEM_HOST) {
        TRY(d2h(c, out_maps, c->out.p, ob * nframes, flags));
        if (taps_out) {
            if (nframes > 1 && !(ls_fft_plan(c, n, M, nframes).on && caf_fft_plan(n, range_bins, freq_bins, n / freq_bins + 1, n / freq_bins, true, M).on))
                return fail(PRC_E_INVALID, "taps_out with host pointers and nframes > 1 needs the FFT-domain path");
            TRY(d2h(c, taps_out, c->lstaps.p, (size_t)nframes * M * sizeof(float2), flags));
        }
        if (cleaned_out) {
            const size_t fs = (size_t)(nframes > 1 ? frame_stride : n);
            for (int fr = 0; fr < nframes; ++fr)
                TRY(d2h(c, cleaned_out + fr * fs, c->clean.as<float2>() + (size_t)fr * n, nb, flags));
        }
    }
    TRY(check_ls_status(c, flags, nframes));
    return finish(c, flags);
}

int prc_frame_c64(const prc_c64* ref, const prc_c64* srv, int64_t n, int filter_len, int peek, float reg,
                  int range_bins, int freq_bins, const void* window, prc_c64* out_map, prc_c64* taps_out,
                  prc_c64* cleaned_out, int mem_kind, int device, void* stream, unsigned flags) {
    return prc_frames_c64(ref, srv, n, 1, n, filter_len, peek, reg, range_bins, freq_bins, window, out_map, taps_out,
                          cleaned_out, mem_kind, device, stream, flags);
}

int prc_ls_status(int device, void* stream, int* status, int nframes) {
    if (!status || nframes < 1) return fail(PRC_E_INVALID, "status must not be NULL, nframes >= 1");
    Ctx* c;
    TRY(get_ctx(device, stream, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    if (c->status.cap < (size_t)nframes * sizeof(int)) return fail(PRC_E_INVALID, "no LS solve of %d frames has run on this stream", nframes);
    CU(cudaMemcpyAsync(status, c->status.p, (size_t)nframes * sizeof(int), cudaMemcpyDeviceToHost, /*status*/ c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return PRC_OK;
}

int prc_set_option(const char* name, int value) {
    if (!name) return fail(PRC_E_INVALID, "name is NULL");
    std::call_once(g_env_once, read_env);
    const std::string k(name);
    if (k == "fft") g_fft.store(value);
    else if (k == "fft_min_n") g_fft_min_n.store(value);
    else if (k == "caf_wave") g_caf_wave.store(value);
    else return fail(PRC_E_INVALID, "unknown option '%s'", name);
    return PRC_OK;
}

int prc_get_option(const char* name, int* value) {
    if (!name || !value) return fail(PRC_E_INVALID, "name/value is NULL");
    std::call_once(g_env_once, read_env);
    const std::string k(name);
    if (k == "fft") *value = g_fft.load();
    else if (k == "fft_min_n") *value = g_fft_min_n.load();
    else if (k == "caf_wave") *value = g_caf_wave.load();
    else return fail(PRC_E_INVALID, "unknown option '%s'", name);
    return PRC_OK;
}

int prc_ls_toeplitz_c64(const prc_c64* ref, const prc_c64* srv, int64_t n, int filter_len, int peek,
                        prc_c64* out, prc_c64* taps, int mem_kind, int device, void* stream, unsigned flags) {
    const double bin0 = 0.0;
    (void)bin0;
    return prc_ls_multiple_c64(ref, srv, n, filter_len, peek, 1.0, nullptr, 1, out, taps, mem_kind, device, stream, flags);
}

int prc_ls_multiple_c64(const prc_c64* ref, const prc_c64* srv, int64_t n, int filter_len, int peek,
                        double sample_rate, const double* doppler_bins, int nbins, prc_c64* out, prc_c64* taps_last,
                        int mem_kind, int device, void* stream, unsigned flags) {
    if (!ref || !srv || !out) return fail(PRC_E_INVALID, "ref/srv/out must not be NULL");
    if (bad_mem_kind(mem_kind)) return fail(PRC_E_INVALID, "mem_kind=%d invalid", mem_kind);
    if (n <= 0) return fail(PRC_E_INVALID, "n=%lld invalid", (long long)n);
    if (nbins < 1) return fail(PRC_E_INVALID, "nbins=%d invalid", nbins);
    Ctx* c;
    TRY(get_ctx(device, stream, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    const size_t nb = (size_t)n * sizeof(float2);
    const int M = filter_len + peek;
    const float2* dref = reinterpret_cast<const float2*>(ref);
    const float2* dsrv = reinterpret_cast<const float2*>(srv);
    float2* dout = reinterpret_cast<float2*>(out);
    float2* dtaps = reinterpret_cast<float2*>(taps_last);
    TRY(c->clean.ensure(nb));
    TRY(c->clean2.ensure(nb));
    if (mem_kind == PRC_MEM_HOST) {
        TRY(c->ref.ensure(nb));
        TRY(c->srv.ensure(nb));
        TRY(h2d(c, c->ref.p, ref, nb, flags));
        TRY(h2d(c, c->srv.p, srv, nb, flags));
        dref = c->ref.as<float2>();
        dsrv = c->srv.as<float2>();
        dtaps = nullptr;
    }
    // bins are applied one after the other on the running residual (clutter_removal.py:178-187)
    const float2* cur = dsrv;
    float2* ping[2] = {c->clean.as<float2>(), c->clean2.as<float2>()};
    for (int b = 0; b < nbins; ++b) {
        const double fc = doppler_bins ? doppler_bins[b] : 0.0;
        const bool last = (b == nbins - 1);
        float2* dst = (last && mem_kind == PRC_MEM_DEVICE) ? dout : ping[b & 1];
        TRY(ls_toeplitz_device(c, dref, cur, n, filter_len, peek, fc != 0.0, fc, sample_rate, dst, last ? dtaps : nullptr));
        if (!(flags & PRC_FLAG_ASYNC)) TRY(check_ls_status(c, 0));      // singular systems are reported per bin
        cur = dst;
    }
    if (mem_kind == PRC_MEM_HOST) {
        TRY(d2h(c, out, cur, nb, flags));
        if (taps_last) TRY(d2h(c, taps_last, c->lstaps.p, (size_t)M * sizeof(float2), flags));
    }
    return finish(c, flags);
}

int prc_ls_multiple_frames_c64(const prc_c64* ref, const prc_c64* srv, int64_t n, int nframes, int64_t frame_stride,
                               int filter_len, int peek, double sample_rate, const double* doppler_bins, int nbins,
                               prc_c64* out, int mem_kind, int device, void* stream, unsigned flags) {
    if (!ref || !srv || !out) return fail(PRC_E_INVALID, "ref/srv/out must not be NULL");
    if (mem_kind != PRC_MEM_DEVICE) return fail(PRC_E_INVALID, "prc_ls_multiple_frames_c64 takes device pointers (mem_kind=%d)", mem_kind);
    if (n <= 0) return fail(PRC_E_INVALID, "n=%lld invalid", (long long)n);
    if (nframes < 1 || nbins < 1) return fail(PRC_E_INVALID, "nframes=%d nbins=%d invalid", nframes, nbins);
    if (nframes > 1 && frame_stride < n) return fail(PRC_E_INVALID, "frame_stride=%lld smaller than n=%lld", (long long)frame_stride, (long long)n);
    Ctx* c;
    TRY(get_ctx(device, stream, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    Batch bt;
    bt.nf = nframes;
    bt.stride = nframes > 1 ? frame_stride : n;
    const size_t span = ((size_t)(nframes - 1) * bt.stride + n) * sizeof(float2);
    const float2* dref = reinterpret_cast<const float2*>(ref);
    const float2* cur = reinterpret_cast<const float2*>(srv);
    float2* dout = reinterpret_cast<float2*>(out);
    if (nbins > 1) TRY(c->clean.ensure(span));
    if (nbins > 2) TRY(c->clean2.ensure(span));
    // bins are applied one after the other on the running residual (clutter_removal.py:178-187); the last one
    // writes the caller's buffer
    for (int b = 0; b < nbins; ++b) {
        const double fc = doppler_bins ? doppler_bins[b] : 0.0;
        const bool last = (b == nbins - 1);
        float2* dst = last ? dout : (((nbins - 1 - b) & 1) ? c->clean.as<float2>() : c->clean2.as<float2>());
        TRY(ls_toeplitz_device(c, dref, cur, n, filter_len, peek, fc != 0.0, fc, sample_rate, dst, nullptr, bt));
        if (!(flags & PRC_FLAG_ASYNC)) TRY(check_ls_status(c, 0, nframes));
        cur = dst;
    }
    return finish(c, flags);
}

int prc_iq_mix_c64(const void* in, int in_kind, int64_t n, int mode, double fc, double fs, double phase_offset,
                   prc_c64* out, int mem_kind, int device, void* stream, unsigned flags) {
    if (!in || !out) return fail(PRC_E_INVALID, "in/out must not be NULL");
    if (bad_mem_kind(mem_kind)) return fail(PRC_E_INVALID, "mem_kind=%d invalid", mem_kind);
    if (n <= 0) return fail(PRC_E_INVALID, "n=%lld invalid", (long long)n);
    if (in_kind < IQ_C64 || in_kind > IQ_I16) return fail(PRC_E_INVALID, "in_kind=%d invalid", in_kind);
    if (mode < MIX_NONE || mode > MIX_FS64) return fail(PRC_E_INVALID, "mode=%d invalid", mode);
    if (mode != MIX_NONE && !(fs != 0.0)) return fail(PRC_E_INVALID, "fs must not be 0");
    Ctx* c;
    TRY(get_ctx(device, stream, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    const void* din = in;
    float2* dout = reinterpret_cast<float2*>(out);
    if (mem_kind == PRC_MEM_HOST) {
        TRY(c->fe_in.ensure(iq_bytes(in_kind, n)));
        TRY(c->fe_out.ensure((size_t)n * sizeof(float2)));
        TRY(h2d(c, c->fe_in.p, in, iq_bytes(in_kind, n), flags));
        din = c->fe_in.p;
        dout = c->fe_out.as<float2>();
    }
    TRY(mix_device(c, make_mix(din, in_kind, n, mode, fc, fs, phase_offset), dout));
    if (mem_kind == PRC_MEM_HOST) TRY(d2h(c, out, dout, (size_t)n * sizeof(float2), flags));
    return finish(c, flags);
}

int prc_resample_out_len(int64_t n_in, int up, int down, int nh, int64_t* n_out) {
    if (!n_out) return fail(PRC_E_INVALID, "n_out must not be NULL");
    ResampleGeo g;
    TRY(resample_geo(n_in, up, down, nh, &g));
    *n_out = g.n_out;
    return PRC_OK;
}

int prc_frontend_c64(const void* in, int in_kind, int64_t n, int mode, double fc, double fs, double phase_offset,
                     int up, int down, const double* h, int nh, prc_c64* out, int64_t out_capacity,
                     int mem_kind, int device, void* stream, unsigned flags) {
    if (!in || !out || !h) return fail(PRC_E_INVALID, "in/out/h must not be NULL");
    if (bad_mem_kind(mem_kind)) return fail(PRC_E_INVALID, "mem_kind=%d invalid", mem_kind);
    if (n <= 0) return fail(PRC_E_INVALID, "n=%lld invalid", (long long)n);
    if (in_kind < IQ_C64 || in_kind > IQ_I16) return fail(PRC_E_INVALID, "in_kind=%d invalid", in_kind);
    if (mode < MIX_NONE || mode > MIX_FS64) return fail(PRC_E_INVALID, "mode=%d invalid", mode);
    if (mode != MIX_NONE && !(fs != 0.0)) return fail(PRC_E_INVALID, "fs must not be 0");
    ResampleGeo g;
    TRY(resample_geo(n, up, down, nh, &g));
    if (out_capacity < g.n_out) return fail(PRC_E_INVALID, "out holds %lld samples, %lld needed", (long long)out_capacity, g.n_out);
    Ctx* c;
    TRY(get_ctx(device, stream, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    const void* din = in;
    float2* dout = reinterpret_cast<float2*>(out);
    if (mem_kind == PRC_MEM_HOST) {
        TRY(c->fe_in.ensure(iq_bytes(in_kind, n)));
        TRY(c->fe_out.ensure((size_t)g.n_out * sizeof(float2)));
        TRY(h2d(c, c->fe_in.p, in, iq_bytes(in_kind, n), flags));
        din = c->fe_in.p;
        dout = c->fe_out.as<float2>();
    }
    long long n_out = 0;
    TRY(resample_device(c, make_mix(din, in_kind, n, mode, fc, fs, phase_offset), up, down, h, nh, dout, &n_out));
    if (mem_kind == PRC_MEM_HOST) TRY(d2h(c, out, dout, (size_t)n_out * sizeof(float2), flags));
    return finish(c, flags);
}

int prc_cfar2d_f32(const void* x, int rows, int cols, int fw, int gw, const float* thresh, float* cr_out,
                   uint8_t* det_out, int mem_kind, int device, void* stream, unsigned flags) {
    if (!x || (!cr_out && !det_out)) return fail(PRC_E_INVALID, "x and one of cr_out/det_out must not be NULL");
    if (det_out && !thresh) return fail(PRC_E_INVALID, "det_out needs a threshold");
    if (bad_mem_kind(mem_kind)) return fail(PRC_E_INVALID, "mem_kind=%d invalid", mem_kind);
    if (rows < 1 || cols < 1) return fail(PRC_E_INVALID, "rows=%d cols=%d invalid", rows, cols);
    const bool cplx = (flags & PRC_FLAG_ABS_C64) != 0;
    Ctx* c;
    TRY(get_ctx(device, stream, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    const size_t cells = (size_t)rows * cols;
    const void* dx = x;
    float* dcr = cr_out;
    uint8_t* ddet = det_out;
    if (mem_kind == PRC_MEM_HOST) {
        const size_t inb = cells * (cplx ? sizeof(float2) : sizeof(float));
        TRY(c->cf_in.ensure(inb));
        TRY(h2d(c, c->cf_in.p, x, inb, flags));
        dx = c->cf_in.p;
        if (cr_out) { TRY(c->cf_cr.ensure(cells * sizeof(float))); dcr = c->cf_cr.as<float>(); }
        if (det_out) { TRY(c->cf_det.ensure(cells)); ddet = c->cf_det.as<uint8_t>(); }
    }
    TRY(cfar_device(c, dx, cplx, rows, cols, fw, gw, thresh, dcr, ddet));
    if (mem_kind == PRC_MEM_HOST) {
        if (cr_out) TRY(d2h(c, cr_out, dcr, cells * sizeof(float), flags));
        if (det_out) TRY(d2h(c, det_out, ddet, cells, flags));
    }
    return finish(c, flags);
}

int prc_direct_xambg_c64(const prc_c64* ref, const prc_c64* srv, int64_t n, int range_bins, int freq_bins,
                         double sample_rate, prc_c64* out, int mem_kind, int device, void* stream, unsigned flags) {
    if (!ref || !srv || !out) return fail(PRC_E_INVALID, "ref/srv/out must not be NULL");
    if (bad_mem_kind(mem_kind)) return fail(PRC_E_INVALID, "mem_kind=%d invalid", mem_kind);
    if (n <= 0) return fail(PRC_E_INVALID, "n=%lld invalid", (long long)n);
    if (range_bins < 0 || freq_bins < 1) return fail(PRC_E_INVALID, "range_bins=%d freq_bins=%d invalid", range_bins, freq_bins);
    Ctx* c;
    TRY(get_ctx(device, stream, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    const size_t nb = (size_t)n * sizeof(float2);
    const size_t ob = (size_t)freq_bins * (range_bins + 1) * sizeof(float2);
    const float2* dref = reinterpret_cast<const float2*>(ref);
    const float2* dsrv = reinterpret_cast<const float2*>(srv);
    float2* dout = reinterpret_cast<float2*>(out);
    if (mem_kind == PRC_MEM_HOST) {
        TRY(c->ref.ensure(nb));
        TRY(c->srv.ensure(nb));
        TRY(c->out.ensure(ob));
        TRY(h2d(c, c->ref.p, ref, nb, flags));
        TRY(h2d(c, c->srv.p, srv, nb, flags));
        dref = c->ref.as<float2>();
        dsrv = c->srv.as<float2>();
        dout = c->out.as<float2>();
    }
    TRY(direct_xambg_device(c, dref, dsrv, n, range_bins, freq_bins, sample_rate, dout));
    if (mem_kind == PRC_MEM_HOST) TRY(d2h(c, out, dout, ob, flags));
    return finish(c, flags);
}

}  // extern "C"

extern "C" {

int prc_xcorr_c64(const prc_c64* x, int64_t nx, const prc_c64* y, int64_t ny, int64_t lag0, int64_t nlags,
                  prc_c64* out, int mem_kind, int device, void* stream, unsigned flags) {
    if (!x || !y || !out) return fail(PRC_E_INVALID, "x/y/out must not be NULL");
    if (bad_mem_kind(mem_kind)) return fail(PRC_E_INVALID, "mem_kind=%d invalid", mem_kind);
    if (nx <= 0 || ny <= 0) return fail(PRC_E_INVALID, "nx=%lld / ny=%lld invalid", (long long)nx, (long long)ny);
    if (nlags <= 0 || nlags > XC_MAX_LAGS) return fail(PRC_E_INVALID, "nlags=%lld invalid (1..%lld)", (long long)nlags, XC_MAX_LAGS);
    Ctx* c;
    TRY(get_ctx(device, stream, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    const float2* dx = reinterpret_cast<const float2*>(x);
    const float2* dy = reinterpret_cast<const float2*>(y);
    float2* dout = reinterpret_cast<float2*>(out);
    const size_t ob = (size_t)nlags * sizeof(float2);
    if (mem_kind == PRC_MEM_HOST) {
        TRY(c->xc_b1.ensure((size_t)nx * sizeof(float2)));
        TRY(c->xc_b2.ensure((size_t)ny * sizeof(float2)));
        TRY(c->xc_out.ensure(ob));
        TRY(h2d(c, c->xc_b1.p, x, (size_t)nx * sizeof(float2), flags));
        TRY(h2d(c, c->xc_b2.p, y, (size_t)ny * sizeof(float2), flags));
        dx = c->xc_b1.as<float2>();
        dy = c->xc_b2.as<float2>();
        dout = c->xc_out.as<float2>();
    }
    TRY(xcorr_device(c, dx, nx, dy, ny, lag0, nlags, dout, nullptr, nullptr, false));
    if (mem_kind == PRC_MEM_HOST) TRY(d2h(c, out, dout, ob, flags));
    return finish(c, flags);
}

int prc_channel_offset(const void* s1, int64_t n1, const void* s2, int64_t n2, int in_kind, int nd, int64_t nl,
                       const double* sos, int nsections, int64_t* offset, float* xc_abs,
                       int mem_kind, int device, void* stream, unsigned flags) {
    if (!s1 || !s2 || !offset) return fail(PRC_E_INVALID, "s1/s2/offset must not be NULL");
    if (bad_mem_kind(mem_kind)) return fail(PRC_E_INVALID, "mem_kind=%d invalid", mem_kind);
    if (in_kind < PRC_SIG_C64 || in_kind > PRC_SIG_C128) return fail(PRC_E_INVALID, "in_kind=%d invalid", in_kind);
    if (nd < 1) return fail(PRC_E_INVALID, "nd=%d invalid", nd);
    if (nl < 0) return fail(PRC_E_INVALID, "nl=%lld invalid", (long long)nl);
    SosDesign d;
    TRY(sos_design(sos, nsections, &d));
    if (n1 <= d.pad || n2 <= d.pad)
        return fail(PRC_E_INVALID, "n1=%lld / n2=%lld: the inputs must be longer than padlen=%d", (long long)n1, (long long)n2, d.pad);
    const long long n1d = (n1 + nd - 1) / nd, n2d = (n2 + nd - 1) / nd;
    long long lag0, nlags;
    xcorr_window(n1d, n2d, nl, nl, &lag0, &nlags);
    if (nlags > XC_MAX_LAGS) return fail(PRC_E_INVALID, "%lld lags exceed %lld", nlags, XC_MAX_LAGS);
    Ctx* c;
    TRY(get_ctx(device, stream, &c));
    std::lock_guard<std::mutex> lk(c->mu);
    const void* d1 = s1;
    const void* d2 = s2;
    if (mem_kind == PRC_MEM_HOST) {
        const size_t b1 = (size_t)n1 * sig_elem(in_kind), b2 = (size_t)n2 * sig_elem(in_kind);
        TRY(c->xc_in1.ensure(b1));
        TRY(c->xc_in2.ensure(b2));
        TRY(h2d(c, c->xc_in1.p, s1, b1, flags));
        TRY(h2d(c, c->xc_in2.p, s2, b2, flags));
        d1 = c->xc_in1.p;
        d2 = c->xc_in2.p;
    }
    TRY(c->xc_b1.ensure((size_t)n1d * sizeof(float2)));
    TRY(c->xc_b2.ensure((size_t)n2d * sizeof(float2)));
    TRY(decimate_device(c, d1, in_kind, n1, d, nd, c->xc_b1.as<float2>()));
    TRY(decimate_device(c, d2, in_kind, n2, d, nd, c->xc_b2.as<float2>()));
    TRY(c->xc_key.ensure(2 * sizeof(unsigned long long)));
    unsigned long long* key = c->xc_key.as<unsigned long long>();
    CU(cudaMemsetAsync(key, 0, sizeof(unsigned long long), c->stream));
    float* dabs = xc_abs;
    if (xc_abs && mem_kind == PRC_MEM_HOST) {
        TRY(c->xc_out.ensure((size_t)nlags * sizeof(float)));
        dabs = c->xc_out.as<float>();
    }
    TRY(xcorr_device(c, c->xc_b1.as<float2>(), n1d, c->xc_b2.as<float2>(), n2d, lag0, nlags, nullptr, dabs, key,
                     !sig_complex(in_kind)));
    long long* doff = mem_kind == PRC_MEM_HOST ? reinterpret_cast<long long*>(key + 1) : reinterpret_cast<long long*>(offset);
    xc::offset_kernel<<<1, 1, 0, c->stream>>>(key, nl, nd, doff);
    TRY(check_launch("offset_kernel"));
    if (mem_kind == PRC_MEM_HOST) {
        if (xc_abs) TRY(d2h(c, xc_abs, dabs, (size_t)nlags * sizeof(float), flags));
        CU(cudaMemcpyAsync(offset, doff, sizeof(long long), cudaMemcpyDeviceToHost, c->stream));
    }
    return finish(c, flags);
}

}  // extern "C"
