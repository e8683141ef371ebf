// jade_gpu.cu -- the C ABI of include/jade_gpu.h on top of the sm_100a kernels in jade_kernels.cuh.
//
// There is NO CPU fallback: every compute entry point launches CUDA kernels or fails with JADE_ERR_NOGPU /
// JADE_ERR_CUDA.  The only host arithmetic is one-off table generation (window, palette, twiddles, row maps),
// which the reference also does on the host at reconfiguration time.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/jade_gpu.h"
#include "jade_host_tables.h"
#define JADE_HELPER_KERNELS 1
#include "jade_kernels.cuh"
#include "jade_pk.cuh"
#include "jade_pk_cta.cuh"
#include "jade_pk_small.cuh"
#include "jade_pkz.cuh"
#include "jade_pk3.cuh"
#include "jade_pk_cluster3.cuh"
#include "jade_pk_cluster.cuh"

using jade::KParams;

namespace {

thread_local std::string t_last_error;

typedef void (*kernel_fn)(const KParams);

struct KernelChoice {
    kernel_fn fn = nullptr;
    kernel_fn fn_db = nullptr; // variant that also stores the float dB column (only where the two differ)
    kernel_fn fn_u8 = nullptr, fn_run_u8 = nullptr;  // pixel-only variants for palettes with KParams::pal_u8 (identical colours, no clamp instruction)
    kernel_fn fn_run = nullptr, fn_run_db = nullptr; // variant for long runs of evenly spaced columns run_hop samples apart (tensor-memory sample ring)
    int run_hop = 0;
    int threads = 0;
    int smem = 0;
    int blocks_per_sm = 1;
    int units_per_block = 1; // frames a block processes per loop iteration
    char name[32] = {0};
    int family = 0; // 0 warp, 1 cta, 2 cta2, 3 packed warp kernels, 4 cluster of two CTAs per frame
    int max_clusters = 0; // family 4: clusters that can be resident at once (cudaOccupancyMaxActiveClusters)
};

// Kernel instantiations live in their own translation units (jade_k_*.cu) so that they compile in parallel; each
// unit hands out function pointers.  (mix kind, general epilogue) -> instantiation; Max/Min only exist with the general
// epilogue.
} // namespace
namespace jade_k {
typedef void (*kernel_fn)(const jade::KParams);
kernel_fn warp_kernel(int T, int mixk, bool general);             // jade_k_warp_a.cu / jade_k_warp_b.cu
kernel_fn cta_kernel(int R1, int mixk, bool general);             // jade_k_cta.cu
kernel_fn pkcta_kernel(int R1, int mixk, bool want_db);           // jade_k_pkcta.cu
kernel_fn pkcta2_kernel(int mixk);                                // jade_k_pkcta.cu (N = 65536 on one CTA; experiments)
kernel_fn pkcl3_kernel();                                         // jade_k_pkcl.cu (N = 65536, one contributing channel)
kernel_fn pkcl65536_kernel(int mixk);                             // jade_k_pkcl.cu (N = 65536 on a cluster of two CTAs)
kernel_fn pk2048_kernel(int mixk, bool want_db, int load);        // jade_k_pk.cu (load = jade::PK_LD_*)
kernel_fn pk2048x2_kernel(bool want_db);                           // jade_k_pk2.cu (stereo: two real transforms per warp; experiments)
kernel_fn pkz2048_kernel(bool want_db, bool guard);                // jade_k_pkz.cu (stereo: one complex transform per frame)
kernel_fn pkz2048_run_kernel(bool want_db);
kernel_fn pkz2048_u8_kernel(bool run);
kernel_fn pk2048_run_kernel(bool want_db, int hop);                // jade_k_pk2.cu (one channel, hop 256 / 512: tensor-memory sample ring)
kernel_fn pk3_u8_kernel();
kernel_fn pk3_kernel(bool want_db, bool guard);                    // jade_k_pk3.cu (N = 16384, one contributing channel: three register passes)
kernel_fn pksmall_kernel(int T, int mixk, bool want_db, bool guard); // jade_k_pksmall_a.cu / _b.cu
} // namespace jade_k
namespace {

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    int ensure(size_t n)
    {
        if (n <= bytes) return 0;
        if (p) cudaFree(p);
        p = nullptr;
        bytes = 0;
        if (cudaMalloc(&p, n) != cudaSuccess) return -1;
        bytes = n;
        return 0;
    }
    void release()
    {
        if (p) cudaFree(p);
        p = nullptr;
        bytes = 0;
    }
};
struct PinBuf {
    void* p = nullptr;
    size_t bytes = 0;
    int ensure(size_t n)
    {
        if (n <= bytes) return 0;
        if (p) cudaFreeHost(p);
        p = nullptr;
        bytes = 0;
        if (cudaHostAlloc(&p, n, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) return -1;
        bytes = n;
        return 0;
    }
    void release()
    {
        if (p) cudaFreeHost(p);
        p = nullptr;
        bytes = 0;
    }
};

constexpr int kStageSlots = 8;
constexpr int kPipe = 6; // batch pipeline slots allocated; jade_render_batch uses pipe_depth() of them
// pipeline depth in use: 3 (H2D, kernel and D2H of consecutive chunks overlap); JADE_PIPE_DEPTH = 2..6 for experiments
inline int pipe_depth()
{
    static const int d = [] {
        const char* v = getenv("JADE_PIPE_DEPTH");
        const int n = v ? atoi(v) : 3;
        return n < 2 ? 2 : (n > kPipe ? kPipe : n);
    }();
    return d;
}

} // namespace

struct jade_engine {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    cudaStream_t pipe_stream[kPipe] = {};
    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr;
    bool timed = false;
    std::string err;
    // Locking (INTEGRATION.md section 2).  `mu` guards the plain engine state and is only ever held for short host-side
    // sections and asynchronous launches: no call holds it across a cudaStreamSynchronize / cudaEventSynchronize on GPU work
    // it has just submitted, a blocking cudaMemcpy or a ring-sized host copy, so the audio thread (jade_push_samples)
    // never waits behind the GUI thread's GPU work.  `ctl_mu` serialises the control operations (configure, reset,
    // set_window, set_palette, recolor) among themselves; lock order is ctl_mu, then mu.
    std::mutex mu, ctl_mu;
    std::atomic<long long> launches{0};
    int smem_optin = 227 * 1024; // largest dynamic shared-memory size a kernel may opt in to
    // pinned staging for table uploads that must not synchronise (palette, window): two slots, in-stream copies
    PinBuf h_tab[2];
    cudaEvent_t tab_ev[2] = {nullptr, nullptr};
    int tab_slot = 0;
    cudaEvent_t ctl_ev = nullptr;

    bool configured = false;
    jade_config cfg{};
    int N = 0, M = 0, B = 0, R = 0, W = 0;
    int k_lo = 0, k_hi = 0;
    KernelChoice kc;
    KernelChoice kc_edge;  // family 3 only: guarded-load instantiation for boundary columns / unaligned geometries
    KernelChoice kc_mid;   // N = 2048 only: LDG-to-register instantiation for 8- but not 16-byte aligned frames
    bool has_mid = false;
    KernelChoice kc_pair;  // N = 2048, AbsMean over exactly two channels: both channels of a frame per warp
    bool has_pair = false;
    int mixk = 0;          // jade::MIX_NONE / MIX_SUM / MIX_SEL
    bool general = false;  // general (rolled) epilogue: pooled / cropped rows, precise dB, non-2^n channel mean, Max/Min
    bool pooled = false;

    // tables
    std::vector<float> h_window;       // unit-RMS reference window
    std::vector<int32_t> h_palette;    // 0x00RRGGBB
    jade_host::ValueRange range;
    DevBuf d_window, d_twI, d_twP, d_twA, d_twH, d_palette, d_rowbins, d_scratch_e, d_scratch_p;
    int npal = 0;

    // streaming
    DevBuf d_hist, d_dbring;
    PinBuf h_pixring, h_stage;
    long long hist_cap = 0, hist_fill = 0, hist_base_abs = 0;
    long long pushed = 0;       // samples pushed per channel
    long long frames_done = 0;  // frames analysed (or skipped while paused): next frame index
    long long emitted = 0;      // columns published to the ring (the reference's running m_memCounter)
    long long fetched = 0;      // columns handed to fetch
    long long poll_from = 0;    // ring columns >= poll_from were zeroed before their launch: fetch may poll them (see fetch)
    int stage_slot = 0;
    size_t stage_slot_bytes = 0;
    cudaEvent_t stage_ev[kStageSlots] = {};
    cudaEvent_t last_push_ev = nullptr;
    bool paused = false;

    // batch pipeline
    DevBuf pipe_in[kPipe], pipe_pix[kPipe], pipe_db[kPipe];
    PinBuf pipe_hin[kPipe], pipe_hpix[kPipe], pipe_hdb[kPipe];
    cudaEvent_t pipe_done[kPipe] = {};
};

namespace {

int fail(jade_engine* e, int code, const char* fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    t_last_error = buf;
    if (e) e->err = buf;
    return code;
}
#define CU(e, call)                                                                                          \
    do {                                                                                                     \
        cudaError_t _r = (call);                                                                             \
        if (_r != cudaSuccess)                                                                               \
            return fail((e), JADE_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_r), __FILE__, __LINE__); \
    } while (0)

bool is_pow2(int n) { return n > 0 && (n & (n - 1)) == 0; }

int upload(jade_engine* e, DevBuf& b, const void* src, size_t bytes)
{
    if (b.ensure(bytes ? bytes : 16)) return fail(e, JADE_ERR_CUDA, "cudaMalloc(%zu) failed", bytes);
    if (bytes) CU(e, cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, e->stream));
    CU(e, cudaStreamSynchronize(e->stream));
    return 0;
}

// Table upload that never synchronises with the GPU work in flight: the bytes go through one of two pinned staging slots
// and are copied in stream order on the engine's stream (kernels launched earlier still see the old table, later ones the
// new one); the batch pipeline streams are made to wait for the copy.  `b` must already be large enough (no reallocation:
// cudaFree would synchronise the device).  Caller holds e->mu.
int upload_async(jade_engine* e, DevBuf& b, const void* src, size_t bytes)
{
    if (bytes > b.bytes) return fail(e, JADE_ERR_STATE, "internal: table buffer too small (%zu > %zu)", bytes, b.bytes);
    if (!bytes) return 0;
    const int slot = e->tab_slot;
    e->tab_slot ^= 1;
    if (e->h_tab[slot].ensure(std::max<size_t>(bytes, 256 * 1024))) return fail(e, JADE_ERR_CUDA, "pinned table staging allocation failed");
    CU(e, cudaEventSynchronize(e->tab_ev[slot])); // the copy that used this slot two uploads ago: long complete
    memcpy(e->h_tab[slot].p, src, bytes);
    CU(e, cudaMemcpyAsync(b.p, e->h_tab[slot].p, bytes, cudaMemcpyHostToDevice, e->stream));
    CU(e, cudaEventRecord(e->tab_ev[slot], e->stream));
    for (int i = 0; i < kPipe; ++i) CU(e, cudaStreamWaitEvent(e->pipe_stream[i], e->tab_ev[slot], 0));
    return 0;
}

int choose_kernel(jade_engine* e)
{
    KernelChoice kc;
    e->has_mid = e->has_pair = false;
    const int N = e->N;
    const int mu = e->mixk;
    const bool po = e->general;
    // Every kernel keeps the palette in shared memory, so a long table can push an instantiation over the opt-in limit.
    // Degrade instead of failing: two-channel complex kernel -> per-channel packed kernels -> general kernels; only when
    // nothing fits does configuration / jade_set_palette fail (and jade_set_palette then restores the previous table).
    const bool mono = mu == jade::MIX_NONE;
    auto pk_smem = [&](int T) {
        switch (T) {
        case 2: return mono ? jade::PkSmallCfg<2, true>::smem_bytes(e->npal) : jade::PkSmallCfg<2>::smem_bytes(e->npal);
        case 4: return mono ? jade::PkSmallCfg<4, true>::smem_bytes(e->npal) : jade::PkSmallCfg<4>::smem_bytes(e->npal);
        case 8: return mono ? jade::PkSmallCfg<8, true>::smem_bytes(e->npal) : jade::PkSmallCfg<8>::smem_bytes(e->npal);
        case 16: return mono ? jade::PkSmallCfg<16, true>::smem_bytes(e->npal) : jade::PkSmallCfg<16>::smem_bytes(e->npal);
        default: return mu == jade::MIX_NONE ? jade::PkCfgFor<jade::MIX_NONE>::smem_bytes(e->npal) : jade::PkCfg::smem_bytes(e->npal);
        }
    };
    if (N >= 128 && N <= 2048 && !po && mu != jade::MIX_SEL && pk_smem(N / 64) <= e->smem_optin) {
        // fast path: packed-FP32x2 kernels (jade_pk.cuh for N = 2048, jade_pk_small.cuh below)
        const int T = N / 64;
        kc.family = 3;
        int warps = mu == jade::MIX_NONE ? jade::PkCfgFor<jade::MIX_NONE>::WARPS : jade::PkCfg::WARPS;
        switch (T) {
        case 2: warps = mono ? jade::PkSmallCfg<2, true>::WARPS : jade::PkSmallCfg<2>::WARPS; break;
        case 4: warps = mono ? jade::PkSmallCfg<4, true>::WARPS : jade::PkSmallCfg<4>::WARPS; break;
        case 8: warps = mono ? jade::PkSmallCfg<8, true>::WARPS : jade::PkSmallCfg<8>::WARPS; break;
        case 16: warps = mono ? jade::PkSmallCfg<16, true>::WARPS : jade::PkSmallCfg<16>::WARPS; break;
        default: break;
        }
        kc.threads = warps * 32;
        kc.units_per_block = warps * (32 / T);
        switch (T) {
        case 2: kc.smem = pk_smem(2); break;
        case 4: kc.smem = pk_smem(4); break;
        case 8: kc.smem = pk_smem(8); break;
        case 16: kc.smem = pk_smem(16); break;
        default: kc.smem = pk_smem(32); break;
        }
        if (T == 32) snprintf(kc.name, sizeof kc.name, "pk2048");
        else snprintf(kc.name, sizeof kc.name, "pksmall<%d>", T);
        KernelChoice ke = kc; // boundary columns / unaligned geometries: same arithmetic, guarded loads
        snprintf(ke.name, sizeof ke.name, "%s-guard", kc.name);
        kc.fn = T == 32 ? jade_k::pk2048_kernel(mu, false, jade::PK_LD_ASYNC) : jade_k::pksmall_kernel(T, mu, false, false);
        kc.fn_db = T == 32 ? jade_k::pk2048_kernel(mu, true, jade::PK_LD_ASYNC) : jade_k::pksmall_kernel(T, mu, true, false);
        if (T == 32 && mu == jade::MIX_NONE && jade::PkCfg::TM && jade_k::pk2048_run_kernel(false, e->cfg.hop)) {
            kc.fn_run = jade_k::pk2048_run_kernel(false, e->cfg.hop);
            kc.fn_run_db = jade_k::pk2048_run_kernel(true, e->cfg.hop);
            kc.run_hop = e->cfg.hop;
            CU(e, cudaFuncSetAttribute((const void*)kc.fn_run, cudaFuncAttributeMaxDynamicSharedMemorySize, kc.smem));
            CU(e, cudaFuncSetAttribute((const void*)kc.fn_run_db, cudaFuncAttributeMaxDynamicSharedMemorySize, kc.smem));
        }
        ke.fn = T == 32 ? jade_k::pk2048_kernel(mu, true, jade::PK_LD_GUARD) : jade_k::pksmall_kernel(T, mu, true, true);
        if (!kc.fn || !kc.fn_db || !ke.fn) return fail(e, JADE_ERR_ARG, "unsupported fft_size %d", N);
        if (T == 32) {
            KernelChoice km = kc;
            snprintf(km.name, sizeof km.name, "pk2048-ldg");
            km.fn = jade_k::pk2048_kernel(mu, false, jade::PK_LD_DIRECT);
            km.fn_db = jade_k::pk2048_kernel(mu, true, jade::PK_LD_DIRECT);
            CU(e, cudaFuncSetAttribute((const void*)km.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, km.smem));
            CU(e, cudaFuncSetAttribute((const void*)km.fn_db, cudaFuncAttributeMaxDynamicSharedMemorySize, km.smem));
            int occ_m = 0;
            CU(e, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_m, (const void*)km.fn, km.threads, km.smem));
            if (occ_m < 1) return fail(e, JADE_ERR_CUDA, "kernel %s does not fit on an SM (smem %d)", km.name, km.smem);
            km.blocks_per_sm = occ_m;
            e->kc_mid = km;
            e->has_mid = true;
            // AbsMean over exactly two channels: both channels of a frame as ONE complex transform (jade_pkz.cuh).  Its
            // rounding differs from the per-channel kernels, so EVERY column of such a configuration goes through it:
            // interior aligned frames through the TMA-staged instantiation, everything else through its guarded one.
            const int contributing = (e->cfg.mix_mode == JADE_MIX_LEFT || e->cfg.mix_mode == JADE_MIX_RIGHT) ? 1 : e->cfg.channels;
            static const bool old_pair = [] { const char* v = getenv("JADE_PK_LOAD"); return v && !strcmp(v, "pair2"); }(); // experiments
            const int pair_smem = old_pair ? jade::PkPairCfg::smem_bytes(e->npal) : jade::PkzCfg::smem_bytes(e->npal);
            if (mu == jade::MIX_SUM && contributing == 2 && pair_smem <= e->smem_optin) {
                KernelChoice kp = kc;
                if (old_pair) {
                    snprintf(kp.name, sizeof kp.name, "pk2048x2");
                    kp.threads = jade::PkPairCfg::WARPS * 32;
                    kp.units_per_block = jade::PkPairCfg::WARPS;
                    kp.smem = jade::PkPairCfg::smem_bytes(e->npal);
                    kp.fn = jade_k::pk2048x2_kernel(false);
                    kp.fn_db = jade_k::pk2048x2_kernel(true);
                } else {
                    snprintf(kp.name, sizeof kp.name, "pkz2048");
                    kp.threads = jade::PkzCfg::WARPS * 32;
                    kp.units_per_block = jade::PkzCfg::WARPS;
                    kp.smem = jade::PkzCfg::smem_bytes(e->npal);
                    kp.fn = jade_k::pkz2048_kernel(false, false);
                    kp.fn_db = jade_k::pkz2048_kernel(true, false);
                    ke = kp;
                    kp.fn_run = jade_k::pkz2048_run_kernel(false);
                    kp.fn_run_db = jade_k::pkz2048_run_kernel(true);
                    kp.fn_u8 = jade_k::pkz2048_u8_kernel(false);
                    kp.fn_run_u8 = jade_k::pkz2048_u8_kernel(true);
                    kp.run_hop = 512;
                    snprintf(ke.name, sizeof ke.name, "pkz2048-guard");
                    ke.fn = jade_k::pkz2048_kernel(true, true);
                    e->has_mid = false; // 8- but not 16-byte aligned frames: the guarded instantiation
                }
                CU(e, cudaFuncSetAttribute((const void*)kp.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, kp.smem));
                CU(e, cudaFuncSetAttribute((const void*)kp.fn_db, cudaFuncAttributeMaxDynamicSharedMemorySize, kp.smem));
                for (kernel_fn f : {kp.fn_u8, kp.fn_run_u8})
                    if (f) CU(e, cudaFuncSetAttribute((const void*)f, cudaFuncAttributeMaxDynamicSharedMemorySize, kp.smem));
                if (kp.fn_run) {
                    CU(e, cudaFuncSetAttribute((const void*)kp.fn_run, cudaFuncAttributeMaxDynamicSharedMemorySize, kp.smem));
                    CU(e, cudaFuncSetAttribute((const void*)kp.fn_run_db, cudaFuncAttributeMaxDynamicSharedMemorySize, kp.smem));
                }
                int occ_p = 0;
                CU(e, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_p, (const void*)kp.fn, kp.threads, kp.smem));
                if (occ_p < 1) return fail(e, JADE_ERR_CUDA, "kernel %s does not fit on an SM (smem %d)", kp.name, kp.smem);
                kp.blocks_per_sm = occ_p;
                e->kc_pair = kp;
                e->has_pair = true;
            }
        }
        ke.fn_db = nullptr;
        CU(e, cudaFuncSetAttribute((const void*)kc.fn_db, cudaFuncAttributeMaxDynamicSharedMemorySize, kc.smem));
        CU(e, cudaFuncSetAttribute((const void*)ke.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, ke.smem));
        int occ_e = 0;
        CU(e, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_e, (const void*)ke.fn, ke.threads, ke.smem));
        if (occ_e < 1) return fail(e, JADE_ERR_CUDA, "kernel %s does not fit on an SM (smem %d)", ke.name, ke.smem);
        ke.blocks_per_sm = occ_e;
        e->kc_edge = ke;
    } else if (N <= 2048) {
        const int T = N / 64;
        // N >= 128 without the general epilogue only lands here when the palette does not fit the packed kernel: the warp
        // kernel of these sizes exists with the general epilogue only (jade_k_warp_*.cu)
        const bool gen = po || T > 1;
        kc.family = 0;
        kc.threads = jade::WARP_KERNEL_WARPS * 32;
        kc.units_per_block = jade::WARP_KERNEL_WARPS * (32 / T);
        snprintf(kc.name, sizeof kc.name, "warp<%d>", T);
        kc.fn = jade_k::warp_kernel(T, mu, gen);
        switch (T) {
        case 1: kc.smem = jade::WarpCfg<1>::smem_bytes(e->npal, gen); break;
        case 2: kc.smem = jade::WarpCfg<2>::smem_bytes(e->npal, gen); break;
        case 4: kc.smem = jade::WarpCfg<4>::smem_bytes(e->npal, gen); break;
        case 8: kc.smem = jade::WarpCfg<8>::smem_bytes(e->npal, gen); break;
        case 16: kc.smem = jade::WarpCfg<16>::smem_bytes(e->npal, gen); break;
        case 32: kc.smem = jade::WarpCfg<32>::smem_bytes(e->npal, gen); break;
        default: return fail(e, JADE_ERR_ARG, "unsupported fft_size %d", N);
        }
        if (!kc.fn) return fail(e, JADE_ERR_ARG, "unsupported fft_size %d", N);
    } else if (N == 16384 && !po && mu == jade::MIX_NONE && jade::Pk3Cfg::smem_bytes(e->npal) <= e->smem_optin / 2 &&
               !(getenv("JADE_N16384") && !strcmp(getenv("JADE_N16384"), "cta"))) { // (the environment switch: experiments)
        // one contributing channel: the three-pass kernel (jade_pk3.cuh); launch_stft routes interior, 16-byte aligned frames
        // to the TMA-staged instantiation and the rest to the guarded one, like the packed N <= 2048 kernels
        kc.family = 3;
        kc.threads = jade::Pk3Cfg::THREADS;
        kc.units_per_block = 1;
        kc.smem = jade::Pk3Cfg::smem_bytes(e->npal);
        snprintf(kc.name, sizeof kc.name, "pk3<16384>");
        KernelChoice ke = kc;
        snprintf(ke.name, sizeof ke.name, "pk3<16384>-guard");
        kc.fn = jade_k::pk3_kernel(false, false);
        kc.fn_db = jade_k::pk3_kernel(true, false);
        kc.fn_u8 = jade_k::pk3_u8_kernel();
        CU(e, cudaFuncSetAttribute((const void*)kc.fn_u8, cudaFuncAttributeMaxDynamicSharedMemorySize, kc.smem));
        ke.fn = jade_k::pk3_kernel(true, true);
        ke.fn_db = nullptr;
        CU(e, cudaFuncSetAttribute((const void*)kc.fn_db, cudaFuncAttributeMaxDynamicSharedMemorySize, kc.smem));
        CU(e, cudaFuncSetAttribute((const void*)ke.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, ke.smem));
        ke.blocks_per_sm = 2; // (see the note on the occupancy query below)
        e->kc_edge = ke;
        if (getenv("JADE_N16384") && !strcmp(getenv("JADE_N16384"), "mixed")) { // experiment: one launch, staged / guarded decided per frame
            kc.family = 1;
            kc.fn_u8 = nullptr;
            kc.fn = jade_k::pk3_kernel(false, true);
            kc.fn_db = jade_k::pk3_kernel(true, true);
            CU(e, cudaFuncSetAttribute((const void*)kc.fn_db, cudaFuncAttributeMaxDynamicSharedMemorySize, kc.smem));
        }
    } else if (N <= 32768) {
        const int R1 = N / 2048;
        kc.family = 1;
        kc.threads = 32 * R1;
        snprintf(kc.name, sizeof kc.name, "cta<%d>", R1);
        const bool packed = !po && mu != jade::MIX_SEL; // fast path: packed FP32x2 kernels (jade_pk_cta.cuh)
        if (packed) {
            snprintf(kc.name, sizeof kc.name, "pkcta<%d>", R1);
            kc.fn = jade_k::pkcta_kernel(R1, mu, false);
            kc.fn_db = jade_k::pkcta_kernel(R1, mu, true);
        } else {
            kc.fn = jade_k::cta_kernel(R1, mu, po);
        }
        switch (R1) {
        case 2: kc.smem = packed ? jade::PkCtaCfg<2>::smem_bytes(e->npal, false) : jade::CtaCfg<2>::smem_bytes(e->npal, po); break;
        case 4: kc.smem = packed ? jade::PkCtaCfg<4>::smem_bytes(e->npal, false) : jade::CtaCfg<4>::smem_bytes(e->npal, po); break;
        case 8: kc.smem = packed ? jade::PkCtaCfg<8>::smem_bytes(e->npal, false) : jade::CtaCfg<8>::smem_bytes(e->npal, po); break;
        case 16: kc.smem = packed ? jade::PkCtaCfg<16>::smem_bytes(e->npal, false) : jade::CtaCfg<16>::smem_bytes(e->npal, po); break;
        default: return fail(e, JADE_ERR_ARG, "unsupported fft_size %d", N);
        }
        if (!kc.fn) return fail(e, JADE_ERR_ARG, "unsupported fft_size %d", N);
    } else if (N == 65536) {
        static const bool one_cta = [] { const char* v = getenv("JADE_N65536"); return v && !strcmp(v, "cta2"); }(); // experiments
        kc.threads = 32 * 16;
        if (one_cta) {
            kc.family = 2;
            snprintf(kc.name, sizeof kc.name, "pkcta2<16>");
            kc.fn = jade_k::pkcta2_kernel(mu);
            kc.smem = jade::PkCtaCfg<16>::smem_bytes2(e->npal, e->pooled ? e->R : 0);
        } else {
            // one frame per cluster of two CTAs: the two half-size transforms run on two SMs and meet through DSMEM
            kc.family = 4;
            static const bool old_cl = [] { const char* v = getenv("JADE_N65536"); return v && !strcmp(v, "cl"); }(); // experiments
            const int smem3 = jade::PkCl3Cfg::smem_bytes(e->npal, e->pooled ? e->R : 0);
            if (mu == jade::MIX_NONE && !old_cl && smem3 <= e->smem_optin) {
                snprintf(kc.name, sizeof kc.name, "pkcl3<65536>");
                kc.fn = jade_k::pkcl3_kernel();
                kc.smem = smem3;
            } else {
                snprintf(kc.name, sizeof kc.name, "pkcl65536");
                kc.fn = jade_k::pkcl65536_kernel(mu);
                kc.smem = jade::PkClCfg::smem_bytes(e->npal, e->pooled ? e->R : 0);
            }
        }
    } else {
        return fail(e, JADE_ERR_ARG, "unsupported fft_size %d (power of two in [64,65536])", N);
    }
    if (kc.smem > e->smem_optin)
        return fail(e, JADE_ERR_ARG, "kernel %s needs %d bytes of shared memory with a %d-colour palette (limit %d)", kc.name, kc.smem,
                    e->npal, e->smem_optin);
    CU(e, cudaFuncSetAttribute((const void*)kc.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, kc.smem));
    if (kc.fn_db) CU(e, cudaFuncSetAttribute((const void*)kc.fn_db, cudaFuncAttributeMaxDynamicSharedMemorySize, kc.smem));
    int occ = 0;
    CU(e, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, (const void*)kc.fn, kc.threads, kc.smem));
    if (occ < 1) return fail(e, JADE_ERR_CUDA, "kernel %s does not fit on an SM (smem %d)", kc.name, kc.smem);
    kc.blocks_per_sm = occ;
    // (the occupancy query answers 1 for any kernel that contains tcgen05.alloc, whatever it allocates; the three-pass kernel
    // takes 256 of the 512 tensor-memory columns and two of its CTAs do share an SM -- launch__waves_per_multiprocessor in
    // profiles/r02c_pk3_16384.txt)
    if ((kc.family == 3 || kc.family == 1) && N == 16384 && kc.threads == jade::Pk3Cfg::THREADS && kc.smem == jade::Pk3Cfg::smem_bytes(e->npal)) kc.blocks_per_sm = 2;
    if (const char* v = getenv("JADE_BLOCKS_PER_SM")) { // experiments (kernels with tcgen05.alloc: the query above answers 1)
        if (atoi(v) > 0) kc.blocks_per_sm = e->kc_edge.blocks_per_sm = atoi(v);
    }
    if (kc.family == 4) {
        // how many clusters fit at once (GPCs with an odd number of SMs leave one unpaired): the persistent grid is exactly that
        cudaLaunchConfig_t lc = {};
        lc.gridDim = dim3(2 * e->sm_count);
        lc.blockDim = dim3(kc.threads);
        lc.dynamicSmemBytes = (size_t)kc.smem;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = 2;
        at[0].val.clusterDim.y = 1;
        at[0].val.clusterDim.z = 1;
        lc.attrs = at;
        lc.numAttrs = 1;
        int ncl = 0;
        CU(e, cudaOccupancyMaxActiveClusters(&ncl, (const void*)kc.fn, &lc));
        if (ncl < 1) return fail(e, JADE_ERR_CUDA, "kernel %s: no cluster of two CTAs fits (smem %d)", kc.name, kc.smem);
        kc.max_clusters = ncl;
    }
    e->kc = kc;
    return 0;
}

long long frame_start_abs(const jade_config& c, long long j)
{
    return (j / c.frames_per_block) * (long long)c.block_stride + (j % c.frames_per_block) * (long long)c.hop - c.preroll;
}
// number of columns available once `pushed` samples per channel exist
long long columns_available(const jade_config& c, long long pushed)
{
    const long long N = c.fft_size, fb = c.frames_per_block, S = c.block_stride;
    if (c.emit_mode == JADE_EMIT_BLOCK) {
        // block b complete when its last frame's samples are in: b*S + (fb-1)*hop - preroll + N <= pushed, and -- like
        // the reference, which consumes whole N-sample blocks -- when the block itself has been pushed entirely
        const long long last_off = (fb - 1) * (long long)c.hop - c.preroll + N;
        const long long need0 = std::max<long long>(last_off, S - c.preroll + N);
        if (pushed < need0) return 0;
        return ((pushed - need0) / S + 1) * fb;
    }
    // HOP mode: largest j with start(j)+N <= pushed
    long long lo = 0, hi = (pushed / std::max(1, c.hop) + 2) * 1 + fb + 2;
    // start() is monotone in j
    while (frame_start_abs(c, hi) + N <= pushed) hi *= 2;
    while (lo < hi) {
        const long long mid = (lo + hi) / 2;
        if (frame_start_abs(c, mid) + N <= pushed) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

void fill_params(jade_engine* e, KParams& P)
{
    memset(&P, 0, sizeof P);
    const jade_config& c = e->cfg;
    P.N = e->N;
    P.M = e->M;
    P.B = e->B;
    P.hop = c.hop;
    P.fb = c.frames_per_block;
    P.bstride = c.block_stride;
    if (c.frames_per_block > 1 && (long long)c.block_stride == (long long)c.frames_per_block * c.hop) {
        // evenly spaced columns (every reference geometry but perc10): one column per "block" of hop samples, so that
        // frame_start() in the kernels is a multiply-add instead of a 64-bit division and modulo per frame
        P.fb = 1;
        P.bstride = c.hop;
    }
    P.preroll = c.preroll;
    P.channels = c.channels;
    P.mix_mode = c.mix_mode;
    P.window = (const float*)e->d_window.p;
    P.twI = (const jade::cpx*)e->d_twI.p;
    P.twP = (const jade::cpx*)e->d_twP.p;
    P.twA = (const jade::cpx*)e->d_twA.p;
    P.twH = (const jade::cpx*)e->d_twH.p;
    P.palette = (const uint32_t*)e->d_palette.p;
    P.npal = e->npal;
    P.pmin = e->range.mn;
    P.pmax = e->range.mx;
    P.pmaxc = e->range.maxclamp();
    P.pmult = e->range.mult;
    jade::colour_fold(P);
    // 256 colours and the `>= m_Max` colour equal to the last one: the kernels' conversion to u8 saturates for them (colour_of_lg1)
    P.pal_u8 = (e->npal == 256 && (int)e->h_palette.size() == 256 && e->h_palette[P.ci_hi] == e->h_palette[255]) ? 1 : 0;
    P.db_precise = c.db_precise;
    P.pooled = e->pooled ? 1 : 0;
    P.R = e->R;
    P.k_lo = e->k_lo;
    P.k_hi = e->k_hi;
    P.flip = c.flip_y;
    P.row_bins = (const jade::i2*)e->d_rowbins.p;
    P.scratch_e = (jade::cpx*)e->d_scratch_e.p;
    P.scratch_p = (float*)e->d_scratch_p.p;
}

// grid size: persistent, a multiple of the SM count when there is enough work
int grid_for(jade_engine* e, const KernelChoice& kc, long long frames)
{
    if (kc.family == 4) return (int)(2 * std::max<long long>(1, std::min<long long>(frames, kc.max_clusters)));
    const long long blocks_needed = (frames + kc.units_per_block - 1) / kc.units_per_block;
    static const long long max_grid = [] { const char* v = getenv("JADE_MAX_GRID"); return v ? atoll(v) : 0ll; }(); // experiments / sanitizer runs
    const long long cap = max_grid > 0 ? max_grid : (long long)e->sm_count * kc.blocks_per_sm;
    return (int)std::max<long long>(1, std::min(blocks_needed, cap));
}

int launch_one(jade_engine* e, const KernelChoice& kc, KParams& P, cudaStream_t st)
{
    const long long frames = (long long)P.ncols * P.nstreams;
    if (frames <= 0) return 0;
    const int grid = grid_for(e, kc, frames);
    if (kc.family == 2) {
        const size_t need_e = (size_t)grid * (e->N / 4 + 1) * sizeof(jade::cpx);
        const size_t need_p = (size_t)grid * (e->N / 2 + 1) * sizeof(float);
        if (e->d_scratch_e.bytes < need_e || e->d_scratch_p.bytes < need_p)
            return fail(e, JADE_ERR_STATE, "scratch not sized for grid %d", grid);
    }
    void* args[] = {(void*)&P};
    static const bool trace = getenv("JADE_TRACE_LAUNCH") != nullptr; // one line per launch on stderr (tests/test_gpu_routes64.py)
    kernel_fn fn = (P.db && kc.fn_db) ? kc.fn_db : kc.fn;
    // long runs of evenly spaced columns, a quarter frame apart: the instantiation that walks contiguous columns per warp
    static const bool no_run = [] { const char* v = getenv("JADE_PK_LOAD"); return v && !strcmp(v, "norun"); }(); // experiments
    static const long long run_min = [] { const char* v = getenv("JADE_RUN_MIN"); return v ? atoll(v) : 16ll; }(); // frames per warp that make a "long run"
    if (kc.fn_run && !no_run && P.hop == kc.run_hop && (P.fb == 1 ? P.bstride == P.hop : P.bstride == P.fb * P.hop) &&
        frames >= run_min * grid * kc.units_per_block)
        fn = P.db ? kc.fn_run_db : ((P.pal_u8 && kc.fn_run_u8) ? kc.fn_run_u8 : kc.fn_run);
    else if (!P.db && P.pal_u8 && kc.fn_u8 && fn == kc.fn)
        fn = kc.fn_u8;
    if (trace) {
        // the suffixes name the instantiation: +run (long-run ring), +db (dB-storing form), +u8 (saturating u8 palette form)
        const bool is_run = fn == kc.fn_run || fn == kc.fn_run_db || fn == kc.fn_run_u8;
        const bool is_db = fn == kc.fn_db || fn == kc.fn_run_db;
        const bool is_u8 = fn == kc.fn_u8 || fn == kc.fn_run_u8;
        fprintf(stderr, "[jade] %s%s%s%s grid %d x %d threads, smem %d, blocks/SM %d, frames %lld, units/block %d\n", kc.name,
                is_run ? "+run" : "", is_db ? "+db" : "", is_u8 ? "+u8" : "", grid, kc.threads, kc.smem, kc.blocks_per_sm, frames,
                kc.units_per_block);
    }
    if (P.ring_w > 0) {
        // streaming push: programmatic dependent launch behind ingest_kernel (every STFT kernel calls grid_dep_wait()
        // after its table prologue, jade_kernels.cuh)
        cudaLaunchConfig_t lc = {};
        lc.gridDim = dim3(grid);
        lc.blockDim = dim3(kc.threads);
        lc.dynamicSmemBytes = (size_t)kc.smem;
        lc.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        lc.attrs = at;
        lc.numAttrs = 1;
        CU(e, cudaLaunchKernelExC(&lc, (const void*)fn, args));
    } else {
        CU(e, cudaLaunchKernel((const void*)fn, dim3(grid), dim3(kc.threads), args, kc.smem, st));
    }
    e->launches++;
    return 0;
}

// columns [a, b) of the launch described by P (same output buffers)
KParams sub_range(jade_engine* e, const KParams& P, long long a, long long b)
{
    KParams Q = P;
    const long long off = a - P.first_col;
    Q.first_col = a;
    Q.ncols = (int)(b - a);
    if (P.ring_w > 0) {
        Q.ring_col0 = P.ring_col0 + off;
    } else {
        if (Q.pix) Q.pix += off * e->R;
        if (Q.db) Q.db += off * e->B;
    }
    return Q;
}

int launch_stft(jade_engine* e, KParams& P, cudaStream_t st)
{
    if ((long long)P.ncols * P.nstreams <= 0) return 0;
    if (e->kc.family != 3) return launch_one(e, e->kc, P, st);
    // packed kernels: interior, aligned frames (16 bytes: cp.async staging for N = 2048; 8 bytes: LDG.64); the rest goes
    // to the guarded-load instantiation
    static const bool force_guard = [] { const char* v = getenv("JADE_PK_LOAD"); return v && !strcmp(v, "guard"); }(); // experiments
    if (!P.aligned2 || force_guard) return launch_one(e, e->kc_edge, P, st);
    if (!e->has_mid && !P.aligned4) return launch_one(e, e->kc_edge, P, st); // N < 2048: the staged kernel or the guarded one
    static const bool force_ldg = [] { const char* v = getenv("JADE_PK_LOAD"); return v && !strcmp(v, "ldg"); }(); // experiments
    static const bool no_pair = [] { const char* v = getenv("JADE_PK_LOAD"); return v && !strcmp(v, "single"); }();
    const KernelChoice& main_kc = (e->has_mid && (!P.aligned4 || force_ldg)) ? e->kc_mid : ((e->has_pair && !no_pair) ? e->kc_pair : e->kc);
    const long long j0 = P.first_col, j1 = P.first_col + P.ncols;
    auto start = [&](long long j) { return frame_start_abs(e->cfg, j) - P.sample_base; };
    long long lo = j0, hi = j1;
    while (lo < j1 && start(lo) < 0) ++lo;                       // frame starts are monotone in j
    while (hi > lo && start(hi - 1) + e->N > P.nsamples) --hi;
    if (hi > lo) {
        KParams Q = sub_range(e, P, lo, hi);
        if (int r = launch_one(e, main_kc, Q, st)) return r;
    }
    if (lo > j0) {
        KParams Q = sub_range(e, P, j0, lo);
        if (int r = launch_one(e, e->kc_edge, Q, st)) return r;
    }
    if (j1 > hi) {
        KParams Q = sub_range(e, P, hi, j1);
        if (int r = launch_one(e, e->kc_edge, Q, st)) return r;
    }
    return 0;
}

uint32_t bake_pixel(int32_t rgb, int fmt)
{
    const uint32_t r = (rgb >> 16) & 255, g = (rgb >> 8) & 255, b = rgb & 255;
    if (fmt == JADE_PIX_RGBA8) return 0xFF000000u | (b << 16) | (g << 8) | r; // bytes R,G,B,A on little endian
    return 0xFF000000u | (r << 16) | (g << 8) | b;                           // Spectrogram.cpp:637
}

constexpr int kMaxPalette = 65536; // jade_set_palette's argument limit; the device table is allocated for it once

// async = true: in stream order through pinned staging, no synchronisation (set_palette / set_window while streaming)
int upload_palette(jade_engine* e, bool async = false)
{
    std::vector<uint32_t> baked(e->h_palette.size());
    for (size_t i = 0; i < baked.size(); ++i) baked[i] = bake_pixel(e->h_palette[i], e->cfg.pixel_format);
    e->npal = (int)baked.size();
    if (e->d_palette.ensure((size_t)kMaxPalette * 4)) return fail(e, JADE_ERR_CUDA, "palette allocation failed");
    return async ? upload_async(e, e->d_palette, baked.data(), baked.size() * 4) : upload(e, e->d_palette, baked.data(), baked.size() * 4);
}

// device copy of a unit-RMS window: x 0.5 (real-FFT split without the 1/2; the two-channel complex transform folds its
// 1/4 the same way) x sqrt(power_scale)
void device_window(const jade_engine* e, const std::vector<float>& unit, std::vector<float>& w)
{
    w = unit;
    const float ps = e->cfg.power_scale;
    const float g = (ps == 1.0f) ? 0.5f : 0.5f * std::sqrt(ps);
    for (auto& v : w) v *= g;
}
int upload_window(jade_engine* e)
{
    jade_host::make_window(e->cfg.window, e->N, e->h_window);
    std::vector<float> w;
    device_window(e, e->h_window, w);
    return upload(e, e->d_window, w.data(), w.size() * 4);
}

int reset_stream_state(jade_engine* e)
{
    const jade_config& c = e->cfg;
    // history: [preroll zeros | samples ...]
    CU(e, cudaMemsetAsync(e->d_hist.p, 0, e->d_hist.bytes, e->stream));
    e->hist_base_abs = -(long long)c.preroll;
    e->hist_fill = c.preroll;
    e->pushed = 0;
    e->emitted = 0;
    e->frames_done = 0;
    e->fetched = 0;
    e->poll_from = 0;
    // ring filled with -120 dB (Spectrogram.cpp:223); pixel ring with the colour of -120 dB
    std::vector<float> init((size_t)e->W * e->B, -120.0f);
    CU(e, cudaMemcpyAsync(e->d_dbring.p, init.data(), init.size() * 4, cudaMemcpyHostToDevice, e->stream));
    CU(e, cudaStreamSynchronize(e->stream));
    if (e->npal > 0) {
        const int idx = jade_host::palette_index(-120.0f, e->range, e->npal);
        const uint32_t px = bake_pixel(e->h_palette[idx], c.pixel_format);
        uint32_t* p = (uint32_t*)e->h_pixring.p;
        for (size_t i = 0; i < (size_t)e->W * e->R; ++i) p[i] = px;
    }
    return 0;
}

} // namespace

// =========================================================================================================
extern "C" {

int jade_abi_version(void) { return JADE_ABI_VERSION; }

int jade_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

const char* jade_last_error(jade_engine* e) { return e ? e->err.c_str() : t_last_error.c_str(); }

int jade_create(int device, jade_engine** out)
{
    if (!out) return fail(nullptr, JADE_ERR_ARG, "out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t r = cudaGetDeviceCount(&n);
    if (r != cudaSuccess || n <= 0)
        return fail(nullptr, JADE_ERR_NOGPU, "no CUDA device (%s); libjade_gpu has no CPU fallback",
                    r == cudaSuccess ? "count=0" : cudaGetErrorString(r));
    if (device < 0 || device >= n) return fail(nullptr, JADE_ERR_ARG, "device %d out of range [0,%d)", device, n);
    jade_engine* e = new jade_engine();
    e->device = device;
    CU(e, cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(e, cudaGetDeviceProperties(&prop, device));
    e->sm_count = prop.multiProcessorCount;
    e->smem_optin = (int)prop.sharedMemPerBlockOptin;
    CU(e, cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    for (int i = 0; i < kPipe; ++i) {
        CU(e, cudaStreamCreateWithFlags(&e->pipe_stream[i], cudaStreamNonBlocking));
        CU(e, cudaEventCreateWithFlags(&e->pipe_done[i], cudaEventDisableTiming));
    }
    CU(e, cudaEventCreate(&e->ev_t0));
    CU(e, cudaEventCreate(&e->ev_t1));
    for (int i = 0; i < kStageSlots; ++i) CU(e, cudaEventCreateWithFlags(&e->stage_ev[i], cudaEventDisableTiming));
    CU(e, cudaEventCreateWithFlags(&e->last_push_ev, cudaEventDisableTiming));
    CU(e, cudaEventCreateWithFlags(&e->ctl_ev, cudaEventDisableTiming));
    for (int i = 0; i < 2; ++i) CU(e, cudaEventCreateWithFlags(&e->tab_ev[i], cudaEventDisableTiming));
    // default palette: the component's (256 colours, kJade, -50..50 dB; Spectrogram.cpp:337,342)
    e->h_palette.assign(256, 0);
    jade_host::palette_build(JADE_PAL_JADE, 256, 0, e->h_palette.data());
    e->range.set(-50.f, 50.f, 256);
    *out = e;
    return JADE_OK;
}

int jade_destroy(jade_engine* e)
{
    if (!e) return JADE_OK;
    cudaSetDevice(e->device);
    cudaDeviceSynchronize();
    for (DevBuf* b : {&e->d_window, &e->d_twI, &e->d_twP, &e->d_twA, &e->d_twH, &e->d_palette, &e->d_rowbins,
                      &e->d_scratch_e, &e->d_scratch_p, &e->d_hist, &e->d_dbring})
        b->release();
    e->h_pixring.release();
    e->h_stage.release();
    for (int i = 0; i < kPipe; ++i) {
        e->pipe_in[i].release();
        e->pipe_pix[i].release();
        e->pipe_db[i].release();
        e->pipe_hin[i].release();
        e->pipe_hpix[i].release();
        e->pipe_hdb[i].release();
        if (e->pipe_stream[i]) cudaStreamDestroy(e->pipe_stream[i]);
        if (e->pipe_done[i]) cudaEventDestroy(e->pipe_done[i]);
    }
    for (int i = 0; i < kStageSlots; ++i)
        if (e->stage_ev[i]) cudaEventDestroy(e->stage_ev[i]);
    if (e->last_push_ev) cudaEventDestroy(e->last_push_ev);
    if (e->ctl_ev) cudaEventDestroy(e->ctl_ev);
    for (int i = 0; i < 2; ++i) {
        if (e->tab_ev[i]) cudaEventDestroy(e->tab_ev[i]);
        e->h_tab[i].release();
    }
    if (e->ev_t0) cudaEventDestroy(e->ev_t0);
    if (e->ev_t1) cudaEventDestroy(e->ev_t1);
    if (e->stream) cudaStreamDestroy(e->stream);
    delete e;
    return JADE_OK;
}

int jade_config_default(jade_config* c)
{
    if (!c) return JADE_ERR_ARG;
    memset(c, 0, sizeof *c);
    c->sample_rate = 48000.f;
    c->fft_size = 2048; // PluginProcessor.cpp:13
    c->window = JADE_WIN_HANN;
    c->channels = 2;
    c->mix_mode = JADE_MIX_ABSMEAN;
    c->row_map = JADE_ROWS_IDENTITY;
    c->flip_y = 1;
    c->pixel_format = JADE_PIX_ARGB32;
    c->power_scale = 1.f;
    c->memory_time_s = 10.f; // PluginProcessor.cpp:110
    c->preroll = -1;
    c->emit_mode = JADE_EMIT_BLOCK;
    c->fmin = 0.f;
    c->fmax = 20000.f;
    return jade_config_set_feed_percent(c, 50); // PluginProcessor.cpp:112
}

int jade_config_set_feed_percent(jade_config* c, int percent)
{
    if (!c) return JADE_ERR_ARG;
    float pct;
    switch (percent) { // Spectrogram.cpp:189-211
    case 100: pct = 100.0; c->frames_per_block = 1; break;
    case 50: pct = 50.0; c->frames_per_block = 2; break;
    case 25: pct = 25.0; c->frames_per_block = 4; break;
    case 10: pct = 10.0; c->frames_per_block = 10; break;
    default: return JADE_ERR_ARG;
    }
    c->hop = int(pct * 0.01 * size_t(c->fft_size) + 0.5); // Spectrogram.cpp:216
    c->block_stride = c->fft_size;
    return JADE_OK;
}

int jade_configure(jade_engine* e, const jade_config* cin)
{
    if (!e || !cin) return fail(e, JADE_ERR_ARG, "null argument");
    // buildmem(): a stop-the-world reconfiguration like the reference's (setFFTSize holds m_protect, Spectrogram.cpp:162-167);
    // a concurrent jade_push_samples waits for it
    std::lock_guard<std::mutex> ctl(e->ctl_mu);
    std::lock_guard<std::mutex> lk(e->mu);
    CU(e, cudaSetDevice(e->device));
    jade_config c = *cin;
    if (!is_pow2(c.fft_size) || c.fft_size < 64 || c.fft_size > 65536)
        return fail(e, JADE_ERR_ARG, "fft_size %d must be a power of two in [64,65536]", c.fft_size);
    if (c.hop <= 0) return fail(e, JADE_ERR_ARG, "hop %d must be positive", c.hop);
    if (c.channels < 1 || c.channels > 16) return fail(e, JADE_ERR_ARG, "channels %d out of [1,16]", c.channels);
    if (c.mix_mode < 0 || c.mix_mode > JADE_MIX_RIGHT) return fail(e, JADE_ERR_ARG, "bad mix_mode %d", c.mix_mode);
    if (c.window < 0 || c.window > JADE_WIN_HANNPOISSON) return fail(e, JADE_ERR_ARG, "bad window %d", c.window);
    if (c.frames_per_block < 1) c.frames_per_block = 1;
    if (c.block_stride <= 0) c.block_stride = c.hop * c.frames_per_block;
    if (c.preroll < 0) c.preroll = c.fft_size;
    if (c.power_scale <= 0.f) c.power_scale = 1.f;
    if (c.sample_rate <= 0.f) return fail(e, JADE_ERR_ARG, "sample_rate must be positive");
    if (c.max_push <= 0) c.max_push = c.fft_size;
    // frame starts must be monotone in the column index (columns_available, the interior / boundary split of launch_stft and
    // the chunking of jade_render_batch rely on it): the last sub-frame of a block may not start after the next block
    if ((long long)(c.frames_per_block - 1) * c.hop > c.block_stride)
        return fail(e, JADE_ERR_ARG, "(frames_per_block-1)*hop = %lld exceeds block_stride %d: frame starts would not be monotone",
                    (long long)(c.frames_per_block - 1) * c.hop, c.block_stride);

    e->configured = false;
    e->cfg = c;
    e->N = c.fft_size;
    e->M = e->N / 2;
    e->B = e->M + 1;
    // ring width: Spectrogram.cpp:217  int(mem_s*fs/hop + 0.5) with float products
    if (c.ring_columns > 0) e->W = c.ring_columns;
    else {
        const float mem = c.memory_time_s > 0.f ? c.memory_time_s : 1.0f;
        e->W = int(mem * c.sample_rate / c.hop + 0.5);
        if (e->W < 1) e->W = 1;
    }
    e->cfg.ring_columns = e->W;

    // rows
    e->pooled = false;
    e->k_lo = 0;
    e->k_hi = e->B;
    std::vector<jade::i2> rb;
    if (c.row_map == JADE_ROWS_LINEAR_CROP) {
        jade_host::linear_crop(c.sample_rate, e->B, c.fmin, c.fmax, e->k_lo, e->k_hi);
        e->R = e->k_hi - e->k_lo;
    } else if (c.row_map == JADE_ROWS_LOG_MAXPOOL) {
        if (c.rows < 1) return fail(e, JADE_ERR_ARG, "rows must be >= 1 for LOG_MAXPOOL");
        std::vector<int32_t> lo, hi;
        jade_host::log_rows(c.sample_rate, e->N, c.rows, c.fmin, c.fmax, lo, hi);
        rb.resize(c.rows);
        for (int r = 0; r < c.rows; ++r) rb[r] = {lo[r], hi[r]};
        e->R = c.rows;
        e->pooled = true;
    } else if (c.row_map == JADE_ROWS_IDENTITY) {
        e->R = e->B;
    } else {
        return fail(e, JADE_ERR_ARG, "bad row_map %d", c.row_map);
    }
    e->cfg.rows = e->R;
    {
        const int contributing = (c.mix_mode == JADE_MIX_LEFT || c.mix_mode == JADE_MIX_RIGHT) ? 1 : c.channels;
        if (c.mix_mode == JADE_MIX_MIN || (c.mix_mode == JADE_MIX_MAX && contributing > 1)) e->mixk = jade::MIX_SEL;
        else if (c.mix_mode == JADE_MIX_ABSMEAN && contributing > 1) e->mixk = jade::MIX_SUM;
        else e->mixk = jade::MIX_NONE;
        const bool pow2ch = (c.channels & (c.channels - 1)) == 0;
        e->general = e->pooled || c.row_map != JADE_ROWS_IDENTITY || c.db_precise != 0 || c.flip_y == 0 || e->mixk == jade::MIX_SEL ||
                     (e->mixk == jade::MIX_SUM && !pow2ch);
    }

    // tables
    if (int r = upload_window(e)) return r;
    if (int r = upload_palette(e)) return r;
    if (int r = upload(e, e->d_rowbins, rb.data(), rb.size() * sizeof(jade::i2))) return r;
    std::vector<jade_host::cpxf> tw;
    jade_host::twiddles(e->N, e->M + 1, 1, tw); // W_N^k, k = 0..M
    if (int r = upload(e, e->d_twP, tw.data(), tw.size() * 8)) return r;
    if (e->N <= 2048) {
        const int T = e->N / 64;
        jade_host::twiddle_matrix(32 * T, 32, T, tw);
        if (int r = upload(e, e->d_twI, tw.data(), tw.size() * 8)) return r;
    } else {
        jade_host::twiddle_matrix(1024, 32, 32, tw);
        if (int r = upload(e, e->d_twI, tw.data(), tw.size() * 8)) return r;
        const int Mfft = (e->N == 65536) ? e->N / 4 : e->M; // complex points of the CTA transform
        const int R1 = Mfft / 1024;
        jade_host::twiddle_matrix(Mfft, R1, 1024, tw);
        if (int r = upload(e, e->d_twA, tw.data(), tw.size() * 8)) return r;
        if (e->N == 65536) {
            jade_host::twiddles(e->N / 2, e->N / 4 + 1, 1, tw); // split twiddles of the half-size real FFTs
            if (int r = upload(e, e->d_twH, tw.data(), tw.size() * 8)) return r;
        }
    }
    if (int r = choose_kernel(e)) return r;
    if (e->kc.family == 2) {
        const size_t g = (size_t)e->sm_count * e->kc.blocks_per_sm;
        if (e->d_scratch_e.ensure(g * (e->N / 4 + 1) * sizeof(jade::cpx)) || e->d_scratch_p.ensure(g * (e->N / 2 + 1) * 4))
            return fail(e, JADE_ERR_CUDA, "scratch allocation failed");
    }

    // streaming buffers
    const long long span = (long long)e->N + c.block_stride + (long long)(c.frames_per_block) * c.hop;
    e->hist_cap = 2 * span + 2LL * c.max_push + 64 + c.preroll;
    e->hist_cap = (e->hist_cap + 3) & ~3LL;
    if (e->d_hist.ensure((size_t)e->hist_cap * c.channels * 4)) return fail(e, JADE_ERR_CUDA, "history allocation failed");
    if (e->d_dbring.ensure((size_t)e->W * e->B * 4)) return fail(e, JADE_ERR_CUDA, "ring allocation failed");
    if (e->h_pixring.ensure((size_t)e->W * e->R * 4)) return fail(e, JADE_ERR_CUDA, "pinned ring allocation failed");
    e->stage_slot_bytes = ((size_t)c.max_push * c.channels * 4 + 255) & ~(size_t)255;
    if (e->h_stage.ensure(e->stage_slot_bytes * kStageSlots)) return fail(e, JADE_ERR_CUDA, "pinned staging allocation failed");
    if (int r = reset_stream_state(e)) return r;
    e->configured = true;
    return JADE_OK;
}

int jade_get_config(jade_engine* e, jade_config* out)
{
    if (!e || !out) return JADE_ERR_ARG;
    if (!e->configured) return fail(e, JADE_ERR_STATE, "engine not configured");
    *out = e->cfg;
    return JADE_OK;
}

int jade_set_pause(jade_engine* e, int on)
{
    if (!e) return JADE_ERR_ARG;
    std::lock_guard<std::mutex> lk(e->mu);
    e->paused = on != 0;
    return JADE_OK;
}

int jade_set_window(jade_engine* e, int window)
{
    if (!e || window < 0 || window > JADE_WIN_HANNPOISSON) return fail(e, JADE_ERR_ARG, "bad window");
    if (!e->configured) return fail(e, JADE_ERR_STATE, "engine not configured");
    std::lock_guard<std::mutex> ctl(e->ctl_mu);
    CU(e, cudaSetDevice(e->device));
    std::vector<float> unit, w;
    jade_host::make_window(window, e->N, unit); // outside e->mu: up to N double cos calls
    device_window(e, unit, w);
    std::lock_guard<std::mutex> lk(e->mu);
    e->cfg.window = window;
    e->h_window.swap(unit);
    return upload_async(e, e->d_window, w.data(), w.size() * 4); // pushes already launched keep the old table
}

int jade_get_window(jade_engine* e, float* out, int n)
{
    if (!e || !out) return JADE_ERR_ARG;
    if (!e->configured) return fail(e, JADE_ERR_STATE, "engine not configured");
    if (n != e->N) return fail(e, JADE_ERR_ARG, "window length %d != fft_size %d", n, e->N);
    memcpy(out, e->h_window.data(), (size_t)n * 4);
    return JADE_OK;
}

int jade_window_build(int window, int n, float* out)
{
    if (!out || n < 1 || window < 0 || window > JADE_WIN_HANNPOISSON) return JADE_ERR_ARG;
    std::vector<float> w;
    jade_host::make_window(window, n, w);
    memcpy(out, w.data(), (size_t)n * 4);
    return JADE_OK;
}

int jade_reset(jade_engine* e)
{
    if (!e) return JADE_ERR_ARG;
    if (!e->configured) return fail(e, JADE_ERR_STATE, "engine not configured");
    std::lock_guard<std::mutex> ctl(e->ctl_mu);
    std::lock_guard<std::mutex> lk(e->mu); // buildmem(): stop-the-world, see jade_configure
    CU(e, cudaSetDevice(e->device));
    CU(e, cudaStreamSynchronize(e->stream));
    return reset_stream_state(e);
}

// ---- palette ------------------------------------------------------------------------------------------
int jade_palette_build(int scheme, int n, int invert, int32_t* table)
{
    if (!table || n < 1 || scheme < 0 || scheme > JADE_PAL_JADE) return JADE_ERR_ARG;
    jade_host::palette_build(scheme, n, invert, table);
    return JADE_OK;
}

int jade_set_palette(jade_engine* e, const int32_t* rgb, int n)
{
    if (!e || !rgb || n < 1 || n > kMaxPalette) return fail(e, JADE_ERR_ARG, "bad palette (1..%d colours)", kMaxPalette);
    std::lock_guard<std::mutex> ctl(e->ctl_mu);
    std::lock_guard<std::mutex> lk(e->mu);
    CU(e, cudaSetDevice(e->device));
    const bool resize = (int)e->h_palette.size() != n;
    // transaction: everything the new table changes is saved and put back if no kernel fits it
    std::vector<int32_t> old_pal(e->h_palette);
    const int old_npal = e->npal;
    const float old_mult = e->range.mult;
    struct Choice {
        KernelChoice kc, kc_edge, kc_mid, kc_pair;
        bool has_mid, has_pair;
    } old_choice{e->kc, e->kc_edge, e->kc_mid, e->kc_pair, e->has_mid, e->has_pair};
    e->h_palette.assign(rgb, rgb + n);
    e->range.mult = float(n) / (e->range.mx - e->range.mn); // CColorpalette.cpp:55-61 setNrOfColors
    if (!e->configured) {
        e->npal = n;
        return JADE_OK;
    }
    e->npal = n;
    int r = resize ? choose_kernel(e) : 0; // shared-memory size depends on the table length
    if (!r) r = upload_palette(e, true);  // in stream order: no wait for the kernels in flight
    if (r) {
        const std::string why = e->err;
        e->h_palette.swap(old_pal);
        e->npal = old_npal;
        e->range.mult = old_mult;
        e->kc = old_choice.kc;
        e->kc_edge = old_choice.kc_edge;
        e->kc_mid = old_choice.kc_mid;
        e->kc_pair = old_choice.kc_pair;
        e->has_mid = old_choice.has_mid;
        e->has_pair = old_choice.has_pair;
        upload_palette(e, true);
        return fail(e, r, "%s; previous palette kept", why.c_str());
    }
    return JADE_OK;
}

int jade_set_palette_scheme(jade_engine* e, int scheme, int n, int invert)
{
    if (!e || n < 1 || n > 65536 || scheme < 0 || scheme > JADE_PAL_JADE) return fail(e, JADE_ERR_ARG, "bad palette scheme");
    std::vector<int32_t> t(n, 0);
    jade_host::palette_build(scheme, n, invert, t.data());
    return jade_set_palette(e, t.data(), n);
}

int jade_set_value_range(jade_engine* e, float mn, float mx)
{
    if (!e) return JADE_ERR_ARG;
    std::lock_guard<std::mutex> lk(e->mu);
    e->range.set(mn, mx, (int)e->h_palette.size());
    return JADE_OK;
}

int jade_get_value_range(jade_engine* e, float* mn, float* mx, float* mult)
{
    if (!e) return JADE_ERR_ARG;
    if (mn) *mn = e->range.mn;
    if (mx) *mx = e->range.mx;
    if (mult) *mult = e->range.mult;
    return JADE_OK;
}

int jade_lookup_color(jade_engine* e, float v, int32_t* rgb)
{
    if (!e || !rgb || e->h_palette.empty()) return JADE_ERR_ARG;
    *rgb = e->h_palette[jade_host::palette_index(v, e->range, (int)e->h_palette.size())];
    return JADE_OK;
}

int jade_colorbar(jade_engine* e, int height, float ramp_min, float ramp_max, uint32_t* out)
{
    if (!e || !out || height < 1 || e->h_palette.empty()) return fail(e, JADE_ERR_ARG, "bad colourbar arguments");
    std::lock_guard<std::mutex> lk(e->mu);
    for (int kk = 0; kk < height; ++kk) { // Spectrogram.cpp:511-517
        const float val = float(kk) / height * (ramp_max - ramp_min) + ramp_min;
        const int32_t rgb = e->h_palette[jade_host::palette_index(val, e->range, (int)e->h_palette.size())];
        out[height - 1 - kk] = bake_pixel(rgb, e->cfg.pixel_format);
    }
    return JADE_OK;
}

int jade_linear_crop(float fs, int bins, float fmin, float fmax, int* k_lo, int* k_hi)
{
    if (!k_lo || !k_hi || bins < 1 || fs <= 0.f) return JADE_ERR_ARG;
    jade_host::linear_crop(fs, bins, fmin, fmax, *k_lo, *k_hi);
    return JADE_OK;
}

int jade_log_rows(float fs, int fft_size, int rows, float fmin, float fmax, int32_t* lo, int32_t* hi)
{
    if (!lo || !hi || rows < 1 || fft_size < 2 || fs <= 0.f) return JADE_ERR_ARG;
    std::vector<int32_t> a, b;
    jade_host::log_rows(fs, fft_size, rows, fmin, fmax, a, b);
    memcpy(lo, a.data(), (size_t)rows * 4);
    memcpy(hi, b.data(), (size_t)rows * 4);
    return JADE_OK;
}

// ---- streaming ----------------------------------------------------------------------------------------
int jade_push_samples(jade_engine* e, const float* const* planar, int nch, int nsamples)
{
    if (!e || !planar) return fail(e, JADE_ERR_ARG, "null argument");
    if (!e->configured) return fail(e, JADE_ERR_STATE, "engine not configured");
    const jade_config& c = e->cfg;
    if (nch != c.channels) return fail(e, JADE_ERR_ARG, "got %d channels, configured %d", nch, c.channels);
    if (nsamples < 0 || nsamples > c.max_push) return fail(e, JADE_ERR_ARG, "nsamples %d exceeds max_push %d", nsamples, c.max_push);
    if (nsamples == 0) return JADE_OK;
    std::lock_guard<std::mutex> lk(e->mu);
    CU(e, cudaSetDevice(e->device));

    // stage into a pinned, device-mapped slot (the kernel reads it over PCIe: no memcpy call on this path)
    const int slot = e->stage_slot;
    e->stage_slot = (slot + 1) % kStageSlots;
    CU(e, cudaEventSynchronize(e->stage_ev[slot])); // normally long complete
    float* hs = (float*)((char*)e->h_stage.p + (size_t)slot * e->stage_slot_bytes);
    for (int ch = 0; ch < nch; ++ch) memcpy(hs + (size_t)ch * nsamples, planar[ch], (size_t)nsamples * 4);

    // slide the linear history when it would overflow
    long long slide_from = 0;
    int keep = 0;
    if (e->hist_fill + nsamples > e->hist_cap) {
        const long long next_start = frame_start_abs(c, e->frames_done); // oldest sample still needed
        long long from = next_start - e->hist_base_abs;
        // hop > fft_size: the next frame may start beyond everything pushed so far -- nothing older is needed then
        from = std::min<long long>(std::max<long long>(from, 0), e->hist_fill);
        from &= ~3LL; // keep frame starts 16-byte aligned relative to the buffer (TMA-staged kernels)
        keep = (int)(e->hist_fill - from);
        slide_from = from;
        e->hist_base_abs += from;
        e->hist_fill = keep;
    }
    const long long write_pos = e->hist_fill;
    {
        float* hist = (float*)e->d_hist.p;
        long long cs = e->hist_cap;
        int chn = nch, n = nsamples;
        const float* stage = hs;
        void* args[] = {&hist, &cs, &chn, &stage, &n, (void*)&write_pos, &slide_from, &keep};
        const int blocks = std::max(1, std::min(32, (std::max(n, keep) + 255) / 256));
        CU(e, cudaLaunchKernel((const void*)jade::ingest_kernel, dim3(blocks), dim3(256), args, 0, e->stream));
        e->launches++;
        CU(e, cudaEventRecord(e->stage_ev[slot], e->stream));
    }
    e->hist_fill += nsamples;
    e->pushed += nsamples;

    // Frames that became computable.  The reference always computes them; while paused it only skips the ring
    // write and the counters (Spectrogram.cpp:111-118) -- nothing observable is left, so the launch is skipped.
    const long long avail = columns_available(c, e->pushed);
    if (avail > e->frames_done) {
        if (!e->paused) {
            long long j0 = e->frames_done, n = avail - e->frames_done, skip = 0;
            if (n > e->W) { // more than a ring in one push: only the newest W survive
                skip = n - e->W;
                j0 += skip;
                n = e->W;
            }
            KParams P;
            fill_params(e, P);
            P.samples = (const float*)e->d_hist.p;
            P.stream_stride = 0;
            P.channel_stride = e->hist_cap;
            P.nsamples = e->hist_fill;
            P.sample_base = e->hist_base_abs;
            P.aligned2 = ((e->hist_cap % 2) == 0 && (c.hop % 2) == 0 && (c.block_stride % 2) == 0 &&
                          (c.preroll % 2) == 0 && (e->hist_base_abs % 2) == 0) ? 1 : 0;
            P.aligned4 = ((e->hist_cap % 4) == 0 && (c.hop % 4) == 0 && (c.block_stride % 4) == 0 &&
                          (c.preroll % 4) == 0 && (e->hist_base_abs % 4) == 0 && ((uintptr_t)e->d_hist.p % 16) == 0) ? 1 : 0;
            P.first_col = j0;
            P.ncols = (int)n;
            P.nstreams = 1;
            P.pix = (uint32_t*)e->h_pixring.p; // device-mapped pinned ring: columns land in host memory directly
            P.db = (float*)e->d_dbring.p;
            P.ring_w = e->W;
            P.ring_col0 = e->emitted + skip;
            // Arm the columns for polling: every pixel carries alpha 0xFF (bake_pixel), so a zeroed slot that has become
            // non-zero everywhere has been written completely -- jade_fetch_columns can hand it out without waiting for
            // the kernel to retire and its event to signal.  Only for a handful of columns of a long ring: up to kStageSlots
            // earlier pushes of <= 8 columns each can still be in flight, so with W >= (kStageSlots + 1) * 8 the slots
            // zeroed here cannot be the target of a launch that is still running; otherwise fetch falls back to the event.
            // INVARIANT: every pixel format bakes a non-zero alpha byte (bake_pixel), so no complete pixel is ever 0.
            // A recolour kernel still in flight rewrites every slot (with the old columns), so nothing is armed behind one.
            if (n <= 8 && e->W >= (kStageSlots + 1) * 8 && cudaEventQuery(e->ctl_ev) == cudaSuccess) {
                uint32_t* ring = (uint32_t*)e->h_pixring.p;
                for (long long i = 0; i < n; ++i) memset(ring + (size_t)((P.ring_col0 + i) % e->W) * e->R, 0, (size_t)e->R * 4);
            } else {
                e->poll_from = e->emitted + skip + n;
            }
            if (int r = launch_stft(e, P, e->stream)) return r;
            e->emitted += skip + n;
        }
        e->frames_done = avail;
    }
    CU(e, cudaEventRecord(e->last_push_ev, e->stream));
    return JADE_OK;
}

int jade_fetch_columns(jade_engine* e, uint32_t* pixels, float* db, int max_cols, int* ncols, int64_t* first_col)
{
    if (!e || !ncols) return fail(e, JADE_ERR_ARG, "null argument");
    if (!e->configured) return fail(e, JADE_ERR_STATE, "engine not configured");
    *ncols = 0;
    long long from, to, poll_from;
    {
        std::lock_guard<std::mutex> lk(e->mu);
        from = e->fetched;
        to = e->emitted;
        if (to - from > e->W) from = to - e->W;
        if (max_cols >= 0 && to - from > max_cols) from = to - max_cols;
        e->fetched = to;
        poll_from = e->poll_from;
    }
    if (first_col) *first_col = from;
    if (to <= from) return JADE_OK;
    CU(e, cudaSetDevice(e->device));
    const int W = e->W, R = e->R, B = e->B;
    const uint32_t* ring = (const uint32_t*)e->h_pixring.p;
    // Columns armed by jade_push_samples are complete once no pixel of their (pinned, device-mapped) slot is zero: poll
    // instead of waiting for the stream event (saves the kernel-retire + event-signal latency of the real-time path).
    bool landed = !db && from >= poll_from;
    if (landed) {
        const auto t_end = std::chrono::steady_clock::now() + std::chrono::milliseconds(20);
        for (long long j = from; j < to && landed; ++j) {
            const volatile uint32_t* slot = ring + (size_t)(j % W) * R;
            for (;;) {
                int r = R - 1;
                while (r >= 0 && slot[r] != 0u) --r;
                if (r < 0) break;
                if (std::chrono::steady_clock::now() > t_end) { // not expected: let the event decide
                    landed = false;
                    break;
                }
            }
        }
        std::atomic_thread_fence(std::memory_order_acquire);
    }
    if (!landed) CU(e, cudaEventSynchronize(e->last_push_ev));
    for (long long j = from; j < to; ++j) {
        const long long slot = j % W;
        if (pixels) memcpy(pixels + (size_t)(j - from) * R, ring + (size_t)slot * R, (size_t)R * 4);
    }
    if (db) {
        // contiguous runs of ring slots
        long long j = from;
        while (j < to) {
            const long long slot = j % W;
            const long long run = std::min<long long>(to - j, W - slot);
            CU(e, cudaMemcpy(db + (size_t)(j - from) * B, (const float*)e->d_dbring.p + (size_t)slot * B,
                             (size_t)run * B * 4, cudaMemcpyDeviceToHost));
            j += run;
        }
    }
    *ncols = (int)(to - from);
    return JADE_OK;
}

int jade_ring_info(jade_engine* e, int* ring_columns, int* rows, int* bins, int64_t* total_columns)
{
    if (!e) return JADE_ERR_ARG;
    if (!e->configured) return fail(e, JADE_ERR_STATE, "engine not configured");
    if (ring_columns) *ring_columns = e->W;
    if (rows) *rows = e->R;
    if (bins) *bins = e->B;
    if (total_columns) *total_columns = e->emitted;
    return JADE_OK;
}

int jade_recolor_ring(jade_engine* e, uint32_t* pixels)
{
    if (!e || !pixels) return fail(e, JADE_ERR_ARG, "null argument");
    if (!e->configured) return fail(e, JADE_ERR_STATE, "engine not configured");
    std::lock_guard<std::mutex> ctl(e->ctl_mu);
    CU(e, cudaSetDevice(e->device));
    {
        // only the launch happens under e->mu: a concurrent jade_push_samples waits microseconds, not for the kernel
        std::lock_guard<std::mutex> lk(e->mu);
        KParams P;
        fill_params(e, P);
        P.pix = (uint32_t*)e->h_pixring.p;
        const float* dbc = (const float*)e->d_dbring.p;
        long long ncolumns = e->W;
        void* args[] = {&P, &dbc, &ncolumns};
        const int grid = (int)std::min<long long>(ncolumns, (long long)e->sm_count * 8);
        CU(e, cudaLaunchKernel((const void*)jade::recolor_kernel, dim3(grid), dim3(256), args, 0, e->stream));
        e->launches++;
        CU(e, cudaEventRecord(e->ctl_ev, e->stream));
        e->poll_from = e->emitted; // slots the kernel rewrites cannot be polled for "non-zero = complete" any more
    }
    CU(e, cudaEventSynchronize(e->ctl_ev));
    // Columns pushed while this copy runs are written by later kernels and may be caught half-way; they are complete in
    // the next jade_fetch_columns, which returns every column emitted since the previous fetch.
    memcpy(pixels, e->h_pixring.p, (size_t)e->W * e->R * 4);
    return JADE_OK;
}

int jade_read_ring_db(jade_engine* e, float* db)
{
    if (!e || !db) return fail(e, JADE_ERR_ARG, "null argument");
    if (!e->configured) return fail(e, JADE_ERR_STATE, "engine not configured");
    CU(e, cudaSetDevice(e->device));
    CU(e, cudaEventSynchronize(e->last_push_ev));
    CU(e, cudaMemcpy(db, e->d_dbring.p, (size_t)e->W * e->B * 4, cudaMemcpyDeviceToHost));
    return JADE_OK;
}

// ---- batch --------------------------------------------------------------------------------------------
int64_t jade_columns_for(jade_engine* e, int64_t nsamples)
{
    if (!e || !e->configured || nsamples < 0) return -1;
    return columns_available(e->cfg, nsamples);
}

int jade_render_device(jade_engine* e, const float* d_samples, int nstreams, int64_t nsamples, int64_t stream_stride,
                       int64_t channel_stride, int64_t first_col, int64_t ncols, uint32_t* d_pixels, float* d_db,
                       void* cuda_stream)
{
    if (!e || !d_samples) return fail(e, JADE_ERR_ARG, "null argument");
    if (!e->configured) return fail(e, JADE_ERR_STATE, "engine not configured");
    if (nstreams < 0 || ncols < 0 || first_col < 0 || nsamples < 0) return fail(e, JADE_ERR_ARG, "negative size");
    if (ncols > 0x7fffffffLL) return fail(e, JADE_ERR_ARG, "ncols too large for one launch");
    CU(e, cudaSetDevice(e->device));
    const jade_config& c = e->cfg;
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : e->stream;
    KParams P;
    fill_params(e, P);
    P.samples = d_samples;
    P.stream_stride = stream_stride;
    P.channel_stride = channel_stride;
    P.nsamples = nsamples;
    P.sample_base = 0;
    P.aligned2 = ((stream_stride % 2) == 0 && (channel_stride % 2) == 0 && (c.hop % 2) == 0 && (c.block_stride % 2) == 0 &&
                  (c.preroll % 2) == 0 && ((uintptr_t)d_samples % 8) == 0) ? 1 : 0;
    P.aligned4 = ((stream_stride % 4) == 0 && (channel_stride % 4) == 0 && (c.hop % 4) == 0 && (c.block_stride % 4) == 0 &&
                  (c.preroll % 4) == 0 && ((uintptr_t)d_samples % 16) == 0) ? 1 : 0;
    P.first_col = first_col;
    P.ncols = (int)ncols;
    P.nstreams = nstreams;
    P.pix = d_pixels;
    P.db = d_db;
    P.pix_stream_stride = (long long)ncols * e->R;
    P.db_stream_stride = (long long)ncols * e->B;
    P.ring_w = 0;
    CU(e, cudaEventRecord(e->ev_t0, st));
    if (int r = launch_stft(e, P, st)) return r;
    CU(e, cudaEventRecord(e->ev_t1, st));
    e->timed = true;
    return JADE_OK;
}

int jade_sync(jade_engine* e)
{
    if (!e) return JADE_ERR_ARG;
    CU(e, cudaSetDevice(e->device));
    CU(e, cudaStreamSynchronize(e->stream));
    for (int i = 0; i < kPipe; ++i) CU(e, cudaStreamSynchronize(e->pipe_stream[i]));
    return JADE_OK;
}

double jade_last_kernel_seconds(jade_engine* e)
{
    if (!e || !e->timed) return -1.0;
    cudaSetDevice(e->device);
    if (cudaEventSynchronize(e->ev_t1) != cudaSuccess) return -1.0;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, e->ev_t0, e->ev_t1) != cudaSuccess) return -1.0;
    return ms * 1e-3;
}

// One pipelined pass: chunks of (stream group x column range); H2D, kernel and D2H of consecutive chunks overlap
// on kPipe streams.  Pageable caller buffers are staged through pinned memory; pinned ones are DMA'd directly.
int jade_render_batch(jade_engine* e, const float* samples, int nstreams, int64_t nsamples, int64_t first_col,
                      int64_t ncols, uint32_t* pixels, float* db)
{
    if (!e || !samples || (!pixels && !db)) return fail(e, JADE_ERR_ARG, "null argument");
    if (!e->configured) return fail(e, JADE_ERR_STATE, "engine not configured");
    if (nstreams <= 0 || ncols <= 0) return JADE_OK;
    CU(e, cudaSetDevice(e->device));
    const jade_config& c = e->cfg;
    const int C = c.channels, R = e->R, B = e->B, N = e->N;
    auto pinned = [](const void* p) {
        cudaPointerAttributes a;
        if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
            cudaGetLastError();
            return false;
        }
        return a.type == cudaMemoryTypeHost;
    };
    const bool in_pinned = pinned(samples);
    const bool pix_pinned = pixels && pinned(pixels);
    const bool db_pinned = db && pinned(db);

    // chunk shape
    // bytes of output per chunk: small enough that the pipeline's fill and drain (one chunk of H2D without a
    // concurrent D2H and vice versa) stay a small share of a call, large enough to keep DMA and launch overheads negligible
    static const size_t budget = []() {
        const char* v = getenv("JADE_CHUNK_MB"); // tuning knob
        const long mb = v ? atol(v) : 0;
        return (size_t)(mb > 0 ? mb : 32) << 20;
    }();
    const size_t col_bytes = (size_t)(pixels ? R * 4 : 0) + (size_t)(db ? B * 4 : 0);
    long long cols_per_chunk = ncols, streams_per_chunk = 1;
    if ((size_t)ncols * col_bytes > budget) {
        cols_per_chunk = std::max<long long>(1, (long long)(budget / col_bytes));
    } else {
        streams_per_chunk = std::max<long long>(1, std::min<long long>(nstreams, (long long)(budget / ((size_t)ncols * col_bytes))));
    }
    int slot = 0;
    bool used[kPipe] = {};
    const int depth = pipe_depth();
    struct Pending {
        bool active = false;
        uint32_t* dst_pix = nullptr;
        float* dst_db = nullptr;
        size_t pix_bytes = 0, db_bytes = 0;
    } pend[kPipe];
    auto drain = [&](int s) -> int {
        if (!used[s]) return 0;
        CU(e, cudaEventSynchronize(e->pipe_done[s]));
        if (pend[s].active) {
            if (pend[s].dst_pix) memcpy(pend[s].dst_pix, e->pipe_hpix[s].p, pend[s].pix_bytes);
            if (pend[s].dst_db) memcpy(pend[s].dst_db, e->pipe_hdb[s].p, pend[s].db_bytes);
            pend[s].active = false;
        }
        return 0;
    };

    for (long long s0 = 0; s0 < nstreams; s0 += streams_per_chunk) {
        const int ns = (int)std::min<long long>(streams_per_chunk, nstreams - s0);
        for (long long c0 = 0; c0 < ncols; c0 += cols_per_chunk) {
            const long long nc = std::min<long long>(cols_per_chunk, ncols - c0);
            if (int r = drain(slot)) return r;
            cudaStream_t st = e->pipe_stream[slot];
            // sample range needed by columns [first_col+c0, first_col+c0+nc)
            long long a = frame_start_abs(c, first_col + c0), b = frame_start_abs(c, first_col + c0 + nc - 1) + N;
            a = std::max<long long>(0, a) & ~3LL; // 16-byte aligned chunk origin (cp.async staging in the N = 2048 kernel)
            b = std::min<long long>(nsamples, b);
            long long len = std::max<long long>(0, b - a);
            const long long len_pad = (len + 3) & ~3LL;
            const size_t in_bytes = (size_t)ns * C * len_pad * 4;
            if (e->pipe_in[slot].ensure(std::max<size_t>(in_bytes, 16))) return fail(e, JADE_ERR_CUDA, "device input allocation failed");
            if (len > 0) {
                const float* src = samples + ((size_t)s0 * C) * nsamples + a;
                if (in_pinned) {
                    CU(e, cudaMemcpy2DAsync(e->pipe_in[slot].p, (size_t)len_pad * 4, src, (size_t)nsamples * 4, (size_t)len * 4,
                                            (size_t)ns * C, cudaMemcpyHostToDevice, st));
                } else {
                    if (e->pipe_hin[slot].ensure(in_bytes)) return fail(e, JADE_ERR_CUDA, "pinned input allocation failed");
                    float* h = (float*)e->pipe_hin[slot].p;
                    for (long long r = 0; r < (long long)ns * C; ++r)
                        memcpy(h + r * len_pad, src + r * nsamples, (size_t)len * 4);
                    CU(e, cudaMemcpyAsync(e->pipe_in[slot].p, h, in_bytes, cudaMemcpyHostToDevice, st));
                }
            }
            const size_t pix_bytes = pixels ? (size_t)ns * nc * R * 4 : 0, db_bytes = db ? (size_t)ns * nc * B * 4 : 0;
            if (pixels && e->pipe_pix[slot].ensure(pix_bytes)) return fail(e, JADE_ERR_CUDA, "device pixel allocation failed");
            if (db && e->pipe_db[slot].ensure(db_bytes)) return fail(e, JADE_ERR_CUDA, "device dB allocation failed");
            KParams P;
            fill_params(e, P);
            P.samples = (const float*)e->pipe_in[slot].p;
            P.stream_stride = (long long)C * len_pad;
            P.channel_stride = len_pad;
            P.nsamples = len;
            P.sample_base = a;
            P.aligned2 = ((c.hop % 2) == 0 && (c.block_stride % 2) == 0 && (c.preroll % 2) == 0) ? 1 : 0;
            P.aligned4 = ((c.hop % 4) == 0 && (c.block_stride % 4) == 0 && (c.preroll % 4) == 0) ? 1 : 0;
            P.first_col = first_col + c0;
            P.ncols = (int)nc;
            P.nstreams = ns;
            P.pix = pixels ? (uint32_t*)e->pipe_pix[slot].p : nullptr;
            P.db = db ? (float*)e->pipe_db[slot].p : nullptr;
            P.pix_stream_stride = nc * R;
            P.db_stream_stride = nc * B;
            if (int r = launch_stft(e, P, st)) return r;
            // outputs: the chunk is [ns][nc][R]; destination is [nstreams][ncols][R]
            const bool contiguous = (nc == ncols);
            if (pixels) {
                uint32_t* dst = pixels + ((size_t)s0 * ncols + c0) * R;
                if (pix_pinned) {
                    if (contiguous) CU(e, cudaMemcpyAsync(dst, e->pipe_pix[slot].p, pix_bytes, cudaMemcpyDeviceToHost, st));
                    else CU(e, cudaMemcpy2DAsync(dst, (size_t)ncols * R * 4, e->pipe_pix[slot].p, (size_t)nc * R * 4,
                                                 (size_t)nc * R * 4, ns, cudaMemcpyDeviceToHost, st));
                } else {
                    if (e->pipe_hpix[slot].ensure(pix_bytes)) return fail(e, JADE_ERR_CUDA, "pinned pixel allocation failed");
                    CU(e, cudaMemcpyAsync(e->pipe_hpix[slot].p, e->pipe_pix[slot].p, pix_bytes, cudaMemcpyDeviceToHost, st));
                }
            }
            if (db) {
                float* dst = db + ((size_t)s0 * ncols + c0) * B;
                if (db_pinned) {
                    if (contiguous) CU(e, cudaMemcpyAsync(dst, e->pipe_db[slot].p, db_bytes, cudaMemcpyDeviceToHost, st));
                    else CU(e, cudaMemcpy2DAsync(dst, (size_t)ncols * B * 4, e->pipe_db[slot].p, (size_t)nc * B * 4,
                                                 (size_t)nc * B * 4, ns, cudaMemcpyDeviceToHost, st));
                } else {
                    if (e->pipe_hdb[slot].ensure(db_bytes)) return fail(e, JADE_ERR_CUDA, "pinned dB allocation failed");
                    CU(e, cudaMemcpyAsync(e->pipe_hdb[slot].p, e->pipe_db[slot].p, db_bytes, cudaMemcpyDeviceToHost, st));
                }
            }
            CU(e, cudaEventRecord(e->pipe_done[slot], st));
            used[slot] = true;
            // pageable destinations need a host-side scatter after the chunk completes (only contiguous chunks or ns == 1)
            if ((pixels && !pix_pinned) || (db && !db_pinned)) {
                if (!contiguous && ns > 1) return fail(e, JADE_ERR_STATE, "internal: strided pageable chunk");
                pend[slot].active = true;
                pend[slot].dst_pix = (pixels && !pix_pinned) ? pixels + ((size_t)s0 * ncols + c0) * R : nullptr;
                pend[slot].dst_db = (db && !db_pinned) ? db + ((size_t)s0 * ncols + c0) * B : nullptr;
                pend[slot].pix_bytes = pix_bytes;
                pend[slot].db_bytes = db_bytes;
            }
            slot = (slot + 1) % depth;
        }
    }
    for (int s = 0; s < kPipe; ++s)
        if (int r = drain(s)) return r;
    return JADE_OK;
}

int jade_render_batch_multi(jade_engine* const* engines, int nengines, const float* samples, int nstreams,
                            int64_t nsamples, int64_t first_col, int64_t ncols, uint32_t* pixels, float* db)
{
    if (!engines || nengines < 1) return fail(nullptr, JADE_ERR_ARG, "no engines");
    if (nengines == 1) return jade_render_batch(engines[0], samples, nstreams, nsamples, first_col, ncols, pixels, db);
    std::vector<std::thread> th;
    std::vector<int> rc(nengines, 0);
    for (int g = 0; g < nengines; ++g) {
        th.emplace_back([&, g]() {
            jade_engine* e = engines[g];
            if (!e || !e->configured) {
                rc[g] = JADE_ERR_STATE;
                return;
            }
            const int C = e->cfg.channels, R = e->R, B = e->B;
            if (nstreams >= nengines) { // range-partition the streams
                const long long s0 = (long long)nstreams * g / nengines, s1 = (long long)nstreams * (g + 1) / nengines;
                if (s1 > s0)
                    rc[g] = jade_render_batch(e, samples + (size_t)s0 * C * nsamples, (int)(s1 - s0), nsamples, first_col, ncols,
                                              pixels ? pixels + (size_t)s0 * ncols * R : nullptr,
                                              db ? db + (size_t)s0 * ncols * B : nullptr);
            } else if (nstreams == 1) { // range-partition the columns; the N-hop input halo is re-read, not exchanged
                const long long c0 = ncols * g / nengines, c1 = ncols * (g + 1) / nengines;
                if (c1 > c0)
                    rc[g] = jade_render_batch(e, samples, 1, nsamples, first_col + c0, c1 - c0,
                                              pixels ? pixels + (size_t)c0 * R : nullptr, db ? db + (size_t)c0 * B : nullptr);
            } else {
                if (g < nstreams)
                    rc[g] = jade_render_batch(e, samples + (size_t)g * C * nsamples, 1, nsamples, first_col, ncols,
                                              pixels ? pixels + (size_t)g * ncols * R : nullptr,
                                              db ? db + (size_t)g * ncols * B : nullptr);
            }
        });
    }
    for (auto& t : th) t.join();
    for (int g = 0; g < nengines; ++g)
        if (rc[g]) return rc[g];
    return JADE_OK;
}

int jade_synth_device(jade_engine* e, float* d_out, int nstreams, int channels, int64_t nsamples, int64_t stream_stride,
                      int64_t channel_stride, int kind, uint64_t seed, void* cuda_stream)
{
    if (!e || !d_out) return fail(e, JADE_ERR_ARG, "null argument");
    CU(e, cudaSetDevice(e->device));
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : e->stream;
    long long ss = stream_stride, cs = channel_stride, n = nsamples;
    unsigned long long sd = seed;
    float fs = e->configured ? e->cfg.sample_rate : 48000.f;
    void* args[] = {&d_out, &ss, &cs, &nstreams, &channels, &n, &kind, &sd, &fs};
    CU(e, cudaLaunchKernel((const void*)jade::synth_kernel, dim3(e->sm_count * 8), dim3(256), args, 0, st));
    e->launches++;
    return JADE_OK;
}

void* jade_host_alloc(size_t bytes)
{
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
        fail(nullptr, JADE_ERR_CUDA, "cudaHostAlloc(%zu) failed", bytes);
        return nullptr;
    }
    return p;
}
int jade_host_free(void* p)
{
    if (p && cudaFreeHost(p) != cudaSuccess) return fail(nullptr, JADE_ERR_CUDA, "cudaFreeHost failed");
    return JADE_OK;
}

int64_t jade_kernel_launches(jade_engine* e) { return e ? (int64_t)e->launches.load() : 0; }
const char* jade_kernel_name(jade_engine* e)
{
    if (!e || !e->configured) return "";
    return e->has_pair ? e->kc_pair.name : e->kc.name; // the kernel interior, aligned frames go to
}

} // extern "C"
