// extern "C" boundary of libb200comms.so -- see include/b200comms.h for the contract and the
// reference interfaces (file:line) each entry point replaces.
#include <cuda.h>

#include <algorithm>
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "chan.hpp"
#include "common.hpp"
#include "fir_imma.hpp"
#include "fft.hpp"
#include "fir.hpp"
#include "rchan.hpp"
#include "rsynth.hpp"
#include "synth.hpp"

namespace b200c {

static thread_local std::string g_err;

void set_error(const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
}

struct DevInfo { int sm_count = 0; size_t smem_optin = 0; };

static int dev_info(int device, DevInfo &di)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
        (void)cudaGetLastError();
        set_error("no CUDA device available: the B200 path has no CPU fallback");
        return B200C_ERR_CUDA;
    }
    if (device < 0 || device >= n) { set_error("device ordinal %d out of range (have %d)", device, n); return B200C_ERR_INVALID; }
    int v = 0;
    B200C_CUDA_TRY(cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device));
    di.sm_count = v;
    B200C_CUDA_TRY(cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    di.smem_optin = (size_t)v;
    return B200C_OK;
}

constexpr int kHostSlotsMax = 8;
// Host-buffer entry points: chunk size and pipeline depth (streams / staging slots).  Defaults from the sweep in
// profiles/ (tools/sweep_host_path.py); B200C_HOST_CHUNK_MIB / B200C_HOST_SLOTS override for A/B runs.
static size_t host_chunk_bytes()
{
    static const size_t v = [] { const char *e = std::getenv("B200C_HOST_CHUNK_MIB"); const long m = e ? std::atol(e) : 0; return (size_t)(m > 0 ? m : 32) << 20; }();
    return v;
}
static int host_slots()
{
    static const int v = [] { const char *e = std::getenv("B200C_HOST_SLOTS"); const int n = e ? std::atoi(e) : 0; return n >= 2 && n <= kHostSlotsMax ? n : 3; }();
    return v;
}

struct HostPipe {   // staging for the *_run_host entry points
    cudaStream_t streams[kHostSlotsMax] = {};
    void *d_in[kHostSlotsMax] = {};
    void *d_out[kHostSlotsMax] = {};
    size_t in_bytes = 0, out_bytes = 0;
    bool streams_ok = false;
    int n = 3;             // slots in use

    int ensure(size_t need_in, size_t need_out)
    {
        if (!streams_ok) {
            n = host_slots();
            for (int i = 0; i < n; i++) B200C_CUDA_TRY(cudaStreamCreateWithFlags(&streams[i], cudaStreamNonBlocking));
            streams_ok = true;
        }
        if (need_in > in_bytes) {
            for (auto &p : d_in) { if (p) cudaFree(p); p = nullptr; }
            in_bytes = 0;
            for (int i = 0; i < n; i++) B200C_CUDA_TRY(cudaMalloc(&d_in[i], need_in));
            in_bytes = need_in;
        }
        if (need_out > out_bytes) {
            for (auto &p : d_out) { if (p) cudaFree(p); p = nullptr; }
            out_bytes = 0;
            for (int i = 0; i < n; i++) B200C_CUDA_TRY(cudaMalloc(&d_out[i], need_out));
            out_bytes = need_out;
        }
        return B200C_OK;
    }
    int sync_all()
    {
        for (int i = 0; i < n; i++) B200C_CUDA_TRY(cudaStreamSynchronize(streams[i]));
        return B200C_OK;
    }
    void release()
    {
        for (auto &p : d_in) { if (p) cudaFree(p); p = nullptr; }
        for (auto &p : d_out) { if (p) cudaFree(p); p = nullptr; }
        if (streams_ok) for (int i = 0; i < n; i++) cudaStreamDestroy(streams[i]);
        streams_ok = false; in_bytes = out_bytes = 0;
    }
};

} // namespace b200c

using namespace b200c;

struct b200c_fir {
    int device = 0;
    int dtype = B200C_CF32, taps_kind = B200C_TAPS_REAL;
    size_t M = 1, L = 1;
    std::vector<double> taps;   // as given to setTaps (interleaved if COMPLEX)
    size_t ntaps = 0;
    DevInfo di;
    FirTable table;
    FirDeviceState ds;
    HostPipe pipe;
    FirOsPlan os;               // fused overlap-save path (cf32, L = M = 1, long taps)
    bool use_os = false;
    FirImmaPlan imma;           // int8 tensor-core path (int16 / complex int16, L = M = 1)
    bool use_imma = false;
    FirUmmaPlan umma;           // tcgen05 / TMEM variant of the same path
    bool use_umma = false;
    FirUmma32Plan u32;          // tcgen05, 32 outputs per row (swizzled planes)
    bool use_u32 = false;
    FirUmmaPPlan up;            // tcgen05 polyphase resampler (int16, L, M <= 4)
    bool use_up = false;
};

struct b200c_fir_bank {
    int device = 0;
    int dtype = B200C_CF32, taps_kind = B200C_TAPS_REAL;
    DevInfo di;
    std::vector<b200c_fir *> ch;   // one /comms/fir_filter state per channel
    void *d_hf_all = nullptr;      // [nchan][N] tap spectra gathered for the one-launch path
    size_t hf_capacity = 0;
    bool dirty = true;
};

struct b200c_chan {
    int device = 0;
    DevInfo di;
    ChanPlan plan;
};

struct b200c_rchan {
    int device = 0;
    int dtype = B200C_F32;
    DevInfo di;
    ChanPlan plan;
};

struct b200c_synth {
    int device = 0;
    DevInfo di;
    SynthPlan plan;
};

struct b200c_rsynth {
    int device = 0;
    int dtype = B200C_F32;
    DevInfo di;
    SynthPlan plan;
};

struct b200c_fft {
    int device = 0;
    DevInfo di;
    FftPlan plan;
    HostPipe pipe;
};

struct b200c_ring {
    int device = 0;
    size_t bytes = 0;
    CUdeviceptr base = 0;
    CUmemGenericAllocationHandle handle = 0;
    bool mapped[2] = {false, false};
    bool have_handle = false, have_va = false;
};

static int fir_refresh(b200c_fir *h)
{
    DeviceGuard g(h->device);
    if (!g.ok) { set_error("cudaSetDevice(%d) failed", h->device); return B200C_ERR_CUDA; }
    FirTable t;
    // <= 100 KB per CTA keeps at least two CTAs resident per SM
    const size_t budget = std::min<size_t>(h->di.smem_optin, 100 * 1024);
    int rc = fir_build_table(t, h->dtype, h->taps_kind, h->taps.data(), h->ntaps, h->M, h->L, budget);
    if (rc) return rc;
    const size_t tb = t.taps.size(), ob = t.off.size() * sizeof(int);
    if (tb > h->ds.taps_capacity) {
        if (h->ds.d_taps) cudaFree(h->ds.d_taps);
        h->ds.d_taps = nullptr; h->ds.taps_capacity = 0;
        B200C_CUDA_TRY(cudaMalloc(&h->ds.d_taps, tb));
        h->ds.taps_capacity = tb;
    }
    if (ob > h->ds.off_capacity) {
        if (h->ds.d_off) cudaFree(h->ds.d_off);
        h->ds.d_off = nullptr; h->ds.off_capacity = 0;
        B200C_CUDA_TRY(cudaMalloc((void **)&h->ds.d_off, ob));
        h->ds.off_capacity = ob;
    }
    // setters are control-path calls serialised with work() by the actor model: a blocking
    // copy (which also orders against in-flight kernels on the legacy stream) is adequate
    B200C_CUDA_TRY(cudaDeviceSynchronize());
    B200C_CUDA_TRY(cudaMemcpy(h->ds.d_taps, t.taps.data(), tb, cudaMemcpyHostToDevice));
    B200C_CUDA_TRY(cudaMemcpy(h->ds.d_off, t.off.data(), ob, cudaMemcpyHostToDevice));
    h->table = std::move(t);
    // Long-tap complex float32 streams (no resampling) take the fused overlap-save kernel: one
    // pass over HBM whatever K is.  B200C_FIR_ALGO=direct|fft overrides the automatic choice
    // (fft: whenever applicable; direct: never).
    h->use_os = false;
    {
        const char *algo = std::getenv("B200C_FIR_ALGO");
        const bool force_direct = algo && std::strcmp(algo, "direct") == 0, force_fft = algo && std::strcmp(algo, "fft") == 0;
        if (!force_direct) {
            rc = fir_os_configure(h->os, h->dtype, h->taps.data(), h->ntaps, h->taps_kind == B200C_TAPS_COMPLEX, h->M, h->L,
                                  force_fft);
            if (rc) return rc;
            h->use_os = h->os.ready;
        }
        // int16 streams: byte-limb Toeplitz GEMMs on the int8 tensor cores, bit-exact
        // (B200C_FIR_ALGO=imma forces it below the automatic tap threshold, direct disables it)
        h->use_imma = false;
        if (!force_direct) {
            rc = fir_imma_configure(h->imma, h->dtype, h->taps.data(), h->ntaps, h->taps_kind == B200C_TAPS_COMPLEX, h->M, h->L,
                                    algo && std::strcmp(algo, "imma") == 0);
            if (rc) return rc;
            h->use_imma = h->imma.ready;
        }
        // tcgen05.mma (accumulators in tensor memory) where it applies; B200C_FIR_ALGO=imma keeps mma.sync
        h->use_umma = false;
        if (h->use_imma && !(algo && std::strcmp(algo, "imma") == 0)) {
            rc = fir_umma_configure(h->umma, h->imma, h->taps.data(), algo && std::strcmp(algo, "umma") == 0);
            if (rc) return rc;
            h->use_umma = h->umma.ready;
        }
        h->use_up = false;
        if (!force_direct) {
            rc = fir_ummap_configure(h->up, h->dtype, h->taps.data(), h->ntaps, h->taps_kind == B200C_TAPS_COMPLEX, h->M, h->L,
                                     algo && std::strcmp(algo, "ummap") == 0);
            if (rc) return rc;
            h->use_up = h->up.ready;
        }
        h->use_u32 = false;
        if (h->use_imma && !(algo && (std::strcmp(algo, "imma") == 0 || std::strcmp(algo, "umma") == 0))) {
            // umma32t: the operand-swapped variant (complex int16 data); umma32 pins the original formulation
            const bool t = algo && std::strcmp(algo, "umma32t") == 0, o = algo && std::strcmp(algo, "umma32") == 0;
            rc = fir_umma32_configure(h->u32, h->imma, h->taps.data(), t || o, t ? 1 : o ? 0 : -1);
            if (rc) return rc;
            h->use_u32 = h->u32.ready;
        }
    }
    return B200C_OK;
}

// one convolution pass over `nblocks` = N/M blocks with whichever kernel the setters selected
static int fir_dispatch(const b200c_fir *h, const void *d_in, size_t in_elems, void *d_out, size_t nblocks, cudaStream_t s)
{
    if (h->use_os) return fir_os_launch(h->os, d_in, in_elems, d_out, nblocks, h->di.sm_count, s);
    if (h->use_up) return fir_ummap_launch(h->up, d_in, in_elems, d_out, nblocks, h->di.sm_count, s);
    if (h->use_u32) return fir_umma32_launch(h->u32, d_in, in_elems, d_out, nblocks, h->di.sm_count, s);
    if (h->use_umma) return fir_umma_launch(h->umma, d_in, in_elems, d_out, nblocks, h->di.sm_count, s);
    if (h->use_imma) return fir_imma_launch(h->imma, d_in, in_elems, d_out, nblocks, h->di.sm_count, s);
    return fir_launch(h->table, h->ds, d_in, in_elems, d_out, nblocks, h->di.sm_count, s);
}

static void fir_plan_counts(const b200c_fir *h, size_t in_elems, size_t out_capacity, int zero_tail, size_t *consume,
                            size_t *produce)
{
    const size_t K = h->table.K, M = h->M, L = h->L;
    const size_t elems = in_elems + (zero_tail ? K - 1 : 0);
    size_t nb = 0;
    if (elems >= K - 1 + M) nb = std::min((elems - (K - 1)) / M, out_capacity / L);
    *consume = nb * M;
    *produce = nb * L;
}

extern "C" {

const char *b200c_last_error(void) { return g_err.c_str(); }
int b200c_abi_version(void) { return B200C_ABI_VERSION; }

int b200c_device_count(int *count)
{
    if (!count) return B200C_ERR_INVALID;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { (void)cudaGetLastError(); n = 0; }
    *count = n;
    return B200C_OK;
}

size_t b200c_dtype_size(int dtype) { return dtype_valid(dtype) ? dtype_bytes(dtype) : 0; }

/* ----------------------------------------------------------------------------- FIR --- */
int b200c_fir_create(b200c_fir **out, int dtype, int taps_kind, int device)
{
    if (!out) return B200C_ERR_INVALID;
    *out = nullptr;
    if (!dtype_valid(dtype) || (taps_kind != B200C_TAPS_REAL && taps_kind != B200C_TAPS_COMPLEX) ||
        (taps_kind == B200C_TAPS_COMPLEX && !dtype_is_complex(dtype))) {
        // FIRFilterFactory falls through its table and throws (filter/FIRFilter.cpp:383)
        set_error("FIRFilterFactory(dtype=%d, tapsType=%s): unsupported types", dtype,
                  taps_kind == B200C_TAPS_COMPLEX ? "COMPLEX" : taps_kind == B200C_TAPS_REAL ? "REAL" : "?");
        return B200C_ERR_UNSUPPORTED;
    }
    DevInfo di;
    int rc = dev_info(device, di);
    if (rc) return rc;
    b200c_fir *h = new (std::nothrow) b200c_fir();
    if (!h) { set_error("out of host memory"); return B200C_ERR_NOMEM; }
    h->device = device; h->dtype = dtype; h->taps_kind = taps_kind; h->di = di;
    // ctor: setTaps({1}) (filter/FIRFilter.cpp:125)
    h->taps.assign(taps_kind == B200C_TAPS_COMPLEX ? 2 : 1, 0.0);
    h->taps[0] = 1.0;
    h->ntaps = 1;
    rc = fir_refresh(h);
    if (rc) { b200c_fir_destroy(h); return rc; }
    *out = h;
    return B200C_OK;
}

int b200c_fir_destroy(b200c_fir *h)
{
    if (!h) return B200C_OK;
    {
        DeviceGuard g(h->device);
        if (h->ds.d_taps) cudaFree(h->ds.d_taps);
        if (h->ds.d_off) cudaFree(h->ds.d_off);
        fir_os_destroy(h->os);
        fir_imma_destroy(h->imma);
        fir_umma_destroy(h->umma);
        fir_umma32_destroy(h->u32);
        fir_ummap_destroy(h->up);
        h->pipe.release();
    }
    delete h;
    return B200C_OK;
}

int b200c_fir_set_taps(b200c_fir *h, const double *taps, size_t ntaps)
{
    if (!h) return B200C_ERR_INVALID;
    if (ntaps == 0 || !taps) { set_error("FIRFilter::setTaps(): taps cannot be empty"); return B200C_ERR_INVALID; }
    const size_t tc = h->taps_kind == B200C_TAPS_COMPLEX ? 2 : 1;
    std::vector<double> old = h->taps;
    const size_t old_n = h->ntaps;
    h->taps.assign(taps, taps + ntaps * tc);
    h->ntaps = ntaps;
    const int rc = fir_refresh(h);
    if (rc) {
        // a configure step failed half way (tables are committed before the kernel plans): put the old taps back and
        // rebuild EVERYTHING for them, so that info/plan/dispatch never see mixed state; the error text is the first one's
        const std::string first = g_err;
        h->taps = old; h->ntaps = old_n;
        (void)fir_refresh(h);
        g_err = first;
    }
    return rc;
}

int b200c_fir_set_rates(b200c_fir *h, size_t decim, size_t interp)
{
    if (!h) return B200C_ERR_INVALID;
    if (decim == 0) { set_error("FIRFilter::setDecimation(): decimation cannot be 0"); return B200C_ERR_INVALID; }
    if (interp == 0) { set_error("FIRFilter::setInterpolation(): interpolation cannot be 0"); return B200C_ERR_INVALID; }
    const size_t oM = h->M, oL = h->L;
    h->M = decim; h->L = interp;
    const int rc = fir_refresh(h);
    if (rc) {
        const std::string first = g_err;
        h->M = oM; h->L = oL;
        (void)fir_refresh(h);      // rebuild tables and kernel plans for the restored rates
        g_err = first;
    }
    return rc;
}

int b200c_fir_info(const b200c_fir *h, size_t *K, size_t *input_require, size_t *decim, size_t *interp)
{
    if (!h) return B200C_ERR_INVALID;
    if (K) *K = h->table.K;
    if (input_require) *input_require = h->M + h->table.K - 1;   // filter/FIRFilter.cpp:353
    if (decim) *decim = h->M;
    if (interp) *interp = h->L;
    return B200C_OK;
}

const char *b200c_fir_kernel(const b200c_fir *h)
{
    if (!h) return "";
    if (h->use_os) return fir_os_kernel_name(h->os);
    if (h->use_up) return "fir_ummap_kernel";
    if (h->use_u32) return h->u32.swapped ? "fir_umma32t_kernel" : "fir_umma32_kernel";
    if (h->use_umma) return "fir_umma_kernel";
    if (h->use_imma) return "fir_imma_kernel";
    return h->table.smem_path ? "fir_tile_kernel" : "fir_generic_kernel";
}

int b200c_fir_plan(const b200c_fir *h, size_t in_elems, size_t out_capacity, int zero_tail, size_t *consume,
                   size_t *produce)
{
    if (!h || !consume || !produce) return B200C_ERR_INVALID;
    fir_plan_counts(h, in_elems, out_capacity, zero_tail, consume, produce);
    return B200C_OK;
}

int b200c_fir_run(b200c_fir *h, const void *d_in, size_t in_elems, void *d_out, size_t out_capacity, int zero_tail,
                  size_t *consumed, size_t *produced, void *stream)
{
    if (!h) return B200C_ERR_INVALID;
    size_t c = 0, p = 0;
    fir_plan_counts(h, in_elems, out_capacity, zero_tail, &c, &p);
    if (consumed) *consumed = c;
    if (produced) *produced = p;
    if (c == 0) return B200C_OK;
    if (!d_in || !d_out) { set_error("b200c_fir_run: null device buffer"); return B200C_ERR_INVALID; }
    DeviceGuard g(h->device);
    if (!g.ok) { set_error("cudaSetDevice(%d) failed", h->device); return B200C_ERR_CUDA; }
    return fir_dispatch(h, d_in, in_elems, d_out, c / h->M, (cudaStream_t)stream);
}

int b200c_fir_run_host(b200c_fir *h, const void *h_in, size_t in_elems, void *h_out, size_t out_capacity, int zero_tail,
                       size_t *consumed, size_t *produced)
{
    if (!h) return B200C_ERR_INVALID;
    size_t c = 0, p = 0;
    fir_plan_counts(h, in_elems, out_capacity, zero_tail, &c, &p);
    if (consumed) *consumed = c;
    if (produced) *produced = p;
    if (c == 0) return B200C_OK;
    if (!h_in || !h_out) { set_error("b200c_fir_run_host: null host buffer"); return B200C_ERR_INVALID; }
    DeviceGuard g(h->device);
    if (!g.ok) { set_error("cudaSetDevice(%d) failed", h->device); return B200C_ERR_CUDA; }

    const size_t esz = dtype_bytes(h->dtype), M = h->M, L = h->L, K = h->table.K;
    const size_t nblocks = c / M;
    // chunks of ~32 MiB of input (host_chunk_bytes), a whole number of blocks each
    size_t cb = std::max<size_t>(1, host_chunk_bytes() / (esz * M));
    // overlap-save: chunk on a whole number of FFT hops so chunked and one-shot runs use the very
    // same block partition (bit-identical outputs)
    // ... and on a multiple of 4 KiB of input AND output where the chunk is large enough: a DMA that starts in the middle of
    // a host page runs ~8 % slower (the FFT path, whose chunks are 32 KiB multiples, measured 47 GB/s each way where this
    // path with hop-aligned chunks measured 43.4)
    {
        const size_t unit = h->use_os ? (size_t)h->os.hop() : 1;          // blocks per indivisible group
        size_t gran = unit;
        for (size_t k : {(size_t)512, (size_t)64, (size_t)8})
            if (cb >= unit * k * 2) { gran = unit * k; break; }               // 512 blocks x >= 8 B x M: whole pages for every type
        cb = std::max<size_t>(1, cb / gran) * gran;
    }
    cb = std::min(cb, nblocks);
    const size_t in_chunk_elems = cb * M + K - 1, out_chunk_elems = cb * L;
    int rc = h->pipe.ensure(in_chunk_elems * esz, out_chunk_elems * esz);
    if (rc) return rc;
    const char *src = static_cast<const char *>(h_in);
    char *dst = static_cast<char *>(h_out);
    size_t slot = 0;
    for (size_t b0 = 0; b0 < nblocks; b0 += cb, slot = (slot + 1) % (size_t)h->pipe.n) {
        const size_t nb = std::min(cb, nblocks - b0);
        const size_t first = b0 * M;                                  // element index of the chunk's history start
        const size_t want = nb * M + K - 1;
        const size_t have = in_elems > first ? std::min(want, in_elems - first) : 0;   // beyond: zero tail
        cudaStream_t s = h->pipe.streams[slot];
        if (have) B200C_CUDA_TRY(cudaMemcpyAsync(h->pipe.d_in[slot], src + first * esz, have * esz, cudaMemcpyHostToDevice, s));
        rc = fir_dispatch(h, h->pipe.d_in[slot], have, h->pipe.d_out[slot], nb, s);
        if (rc) return rc;
        B200C_CUDA_TRY(cudaMemcpyAsync(dst + b0 * L * esz, h->pipe.d_out[slot], nb * L * esz, cudaMemcpyDeviceToHost, s));
    }
    return h->pipe.sync_all();
}

/* ----------------------------------------------------------------------- filter bank --- */
int b200c_fir_bank_destroy(b200c_fir_bank *b)
{
    if (!b) return B200C_OK;
    for (auto *c : b->ch) b200c_fir_destroy(c);
    {
        DeviceGuard g(b->device);
        if (b->d_hf_all) cudaFree(b->d_hf_all);
    }
    delete b;
    return B200C_OK;
}

int b200c_fir_bank_create(b200c_fir_bank **out, int dtype, int taps_kind, size_t nchan, int device)
{
    if (!out) return B200C_ERR_INVALID;
    *out = nullptr;
    if (nchan == 0 || nchan > (1u << 20)) { set_error("filter bank: channel count %zu out of range", nchan); return B200C_ERR_INVALID; }
    b200c_fir_bank *b = new (std::nothrow) b200c_fir_bank();
    if (!b) { set_error("out of host memory"); return B200C_ERR_NOMEM; }
    b->device = device; b->dtype = dtype; b->taps_kind = taps_kind;
    b->ch.reserve(nchan);
    for (size_t i = 0; i < nchan; i++) {
        b200c_fir *c = nullptr;
        const int rc = b200c_fir_create(&c, dtype, taps_kind, device);
        if (rc) { b200c_fir_bank_destroy(b); return rc; }
        b->ch.push_back(c);
    }
    b->di = b->ch[0]->di;
    *out = b;
    return B200C_OK;
}

int b200c_fir_bank_set_taps(b200c_fir_bank *b, size_t chan, const double *taps, size_t ntaps)
{
    if (!b) return B200C_ERR_INVALID;
    if (chan >= b->ch.size()) { set_error("filter bank: channel %zu out of range (have %zu)", chan, b->ch.size()); return B200C_ERR_INVALID; }
    b->dirty = true;
    return b200c_fir_set_taps(b->ch[chan], taps, ntaps);
}

int b200c_fir_bank_set_rates(b200c_fir_bank *b, size_t decim, size_t interp)
{
    if (!b) return B200C_ERR_INVALID;
    b->dirty = true;
    const size_t oM = b->ch[0]->M, oL = b->ch[0]->L;
    for (size_t i = 0; i < b->ch.size(); i++) {
        const int rc = b200c_fir_set_rates(b->ch[i], decim, interp);
        if (rc) {
            // no channel may keep the new rates when one of them failed: undo the ones already switched
            const std::string first = g_err;
            for (size_t j = 0; j < i; j++) (void)b200c_fir_set_rates(b->ch[j], oM, oL);
            g_err = first;
            return rc;
        }
    }
    return B200C_OK;
}

int b200c_fir_bank_info(const b200c_fir_bank *b, size_t *nchan, size_t *K, size_t *input_require)
{
    if (!b) return B200C_ERR_INVALID;
    if (nchan) *nchan = b->ch.size();
    return b200c_fir_info(b->ch[0], K, input_require, nullptr, nullptr);
}

int b200c_fir_bank_run(b200c_fir_bank *b, const void *d_in, size_t in_stride, size_t in_elems, void *d_out, size_t out_stride,
                       size_t out_capacity, int zero_tail, size_t *consumed, size_t *produced, void *stream)
{
    if (!b) return B200C_ERR_INVALID;
    b200c_fir *h0 = b->ch[0];
    for (auto *c : b->ch)
        if (c->table.K != h0->table.K || c->ntaps != h0->ntaps) {
            set_error("filter bank: all channels must have the same number of taps (%zu vs %zu)", c->ntaps, h0->ntaps);
            return B200C_ERR_INVALID;
        }
    size_t c = 0, p = 0;
    fir_plan_counts(h0, in_elems, out_capacity, zero_tail, &c, &p);
    if (consumed) *consumed = c;
    if (produced) *produced = p;
    if (c == 0) return B200C_OK;
    if (!d_in || !d_out) { set_error("b200c_fir_bank_run: null device buffer"); return B200C_ERR_INVALID; }
    const size_t nch = b->ch.size(), esz = dtype_bytes(b->dtype);
    if (nch > 1 && (in_stride < in_elems || out_stride < p)) { set_error("filter bank: channel stride shorter than the channel"); return B200C_ERR_INVALID; }
    DeviceGuard g(b->device);
    if (!g.ok) { set_error("cudaSetDevice(%d) failed", b->device); return B200C_ERR_CUDA; }
    // one launch over (channel, block) where every channel's plan allows it (fir_os_batchable: complex float32, L = M = 1)
    bool fast = true;
    for (auto *ch : b->ch) fast = fast && ch->use_os && fir_os_batchable(ch->os) && ch->os.N == h0->os.N;
    if (fast) {
        // one launch over (channel, block): gather the channels' tap spectra once per setTaps()
        const size_t N = (size_t)h0->os.N, row = N * 2 * sizeof(float);
        if (b->dirty) {
            if (b->hf_capacity < nch * row) {
                if (b->d_hf_all) cudaFree(b->d_hf_all);
                b->d_hf_all = nullptr; b->hf_capacity = 0;
                B200C_CUDA_TRY(cudaMalloc(&b->d_hf_all, nch * row));
                b->hf_capacity = nch * row;
            }
            for (size_t i = 0; i < nch; i++) {
                const void *src = N == 1024 ? b->ch[i]->os.d_hf1k : b->ch[i]->os.d_hf;
                B200C_CUDA_TRY(cudaMemcpyAsync(static_cast<char *>(b->d_hf_all) + i * row, src, row, cudaMemcpyDeviceToDevice,
                                               (cudaStream_t)stream));
            }
            b->dirty = false;
        }
        FirOsBatch batch;
        batch.nchan = (int)nch; batch.in_stride = (long long)in_stride; batch.out_stride = (long long)out_stride;
        batch.d_hf = b->d_hf_all;
        return fir_os_launch(h0->os, d_in, in_elems, d_out, c / h0->M, b->di.sm_count, (cudaStream_t)stream, &batch);
    }
    // every other type / rate: the channels' own kernels back to back on the stream
    for (size_t i = 0; i < nch; i++) {
        b200c_fir *h = b->ch[i];
        const char *src = static_cast<const char *>(d_in) + i * in_stride * esz;
        char *dst = static_cast<char *>(d_out) + i * out_stride * esz;
        const int rc = fir_dispatch(h, src, in_elems, dst, c / h->M, (cudaStream_t)stream);
        if (rc) return rc;
    }
    return B200C_OK;
}

/* ------------------------------------------------------------------- channelizer --- */
int b200c_chan_create(b200c_chan **out, int dtype, size_t nchan, size_t decim, int device)
{
    if (!out) return B200C_ERR_INVALID;
    *out = nullptr;
    if (dtype != B200C_CF32) { set_error("channelizer: dtype %d unsupported (complex float32 only)", dtype); return B200C_ERR_UNSUPPORTED; }
    if (nchan < 2 || nchan > kChanMaxChannels || (nchan & (nchan - 1))) {
        set_error("channelizer: %zu channels unsupported (a power of two from 2 to %zu)", nchan, kChanMaxChannels);
        return B200C_ERR_UNSUPPORTED;
    }
    if (decim == 0 || nchan % decim) { set_error("channelizer: decimation %zu must divide the channel count %zu", decim, nchan); return B200C_ERR_INVALID; }
    DevInfo di;
    int rc = dev_info(device, di);
    if (rc) return rc;
    b200c_chan *h = new (std::nothrow) b200c_chan();
    if (!h) { set_error("out of host memory"); return B200C_ERR_NOMEM; }
    h->device = device; h->di = di;
    DeviceGuard g(device);
    if (!g.ok) { delete h; set_error("cudaSetDevice(%d) failed", device); return B200C_ERR_CUDA; }
    rc = chan_plan_create(h->plan, nchan, decim, di.smem_optin);
    const double one = 1.0;   // taps {1}, as FIRFilter() (filter/FIRFilter.cpp:125)
    if (!rc) rc = chan_set_taps(h->plan, &one, 1);
    if (rc) { b200c_chan_destroy(h); return rc; }
    *out = h;
    return B200C_OK;
}

int b200c_chan_destroy(b200c_chan *h)
{
    if (!h) return B200C_OK;
    {
        DeviceGuard g(h->device);
        chan_plan_destroy(h->plan);
    }
    delete h;
    return B200C_OK;
}

int b200c_chan_set_taps(b200c_chan *h, const double *taps, size_t ntaps)
{
    if (!h) return B200C_ERR_INVALID;
    if (ntaps == 0 || !taps) { set_error("channelizer: taps cannot be empty"); return B200C_ERR_INVALID; }
    if (ntaps > kChanMaxTapsPerBranch * (size_t)h->plan.M) {
        set_error("channelizer: %zu taps exceed 16 per branch (%zu for %d channels)", ntaps, kChanMaxTapsPerBranch * (size_t)h->plan.M, h->plan.M);
        return B200C_ERR_INVALID;
    }
    DeviceGuard g(h->device);
    if (!g.ok) { set_error("cudaSetDevice(%d) failed", h->device); return B200C_ERR_CUDA; }
    return chan_set_taps(h->plan, taps, ntaps);
}

int b200c_chan_info(const b200c_chan *h, size_t *nchan, size_t *decim, size_t *ntaps, size_t *input_require)
{
    if (!h) return B200C_ERR_INVALID;
    if (nchan) *nchan = (size_t)h->plan.M;
    if (decim) *decim = (size_t)h->plan.D;
    if (ntaps) *ntaps = h->plan.ntaps;
    if (input_require) *input_require = h->plan.ntaps - 1 + (size_t)h->plan.D;
    return B200C_OK;
}

int b200c_chan_run(b200c_chan *h, const void *d_in, size_t in_elems, uint64_t stream_index, void *d_out, size_t out_stride,
                   size_t out_capacity, size_t *consumed, size_t *produced, void *stream)
{
    if (!h) return B200C_ERR_INVALID;
    const size_t Km1 = h->plan.ntaps - 1, D = (size_t)h->plan.D;
    const size_t F = in_elems >= Km1 + D ? std::min((in_elems - Km1) / D, out_capacity) : 0;
    if (consumed) *consumed = F * D;
    if (produced) *produced = F;
    if (F == 0) return B200C_OK;
    if (!d_in || !d_out) { set_error("b200c_chan_run: null device buffer"); return B200C_ERR_INVALID; }
    if (out_stride < F) { set_error("channelizer: output stride %zu shorter than the %zu frames produced", out_stride, F); return B200C_ERR_INVALID; }
    DeviceGuard g(h->device);
    if (!g.ok) { set_error("cudaSetDevice(%d) failed", h->device); return B200C_ERR_CUDA; }
    return chan_launch(h->plan, d_in, F, stream_index, d_out, out_stride, (cudaStream_t)stream);
}

/* -------------------------------------------------------- real-input channelizer --- */
int b200c_rchan_create(b200c_rchan **out, int dtype, size_t m, size_t decim, int device)
{
    if (!out) return B200C_ERR_INVALID;
    *out = nullptr;
    if (dtype != B200C_F32 && dtype != B200C_I16) {
        set_error("real channelizer: dtype %d unsupported (float32 or int16 only)", dtype);
        return B200C_ERR_UNSUPPORTED;
    }
    if (m < 2 || m > kRChanMaxBranches || (m & (m - 1))) {
        set_error("real channelizer: %zu branches unsupported (a power of two from 2 to %zu)", m, kRChanMaxBranches);
        return B200C_ERR_UNSUPPORTED;
    }
    if (decim == 0 || m % decim) { set_error("real channelizer: decimation %zu must divide the branch count %zu", decim, m); return B200C_ERR_INVALID; }
    DevInfo di;
    int rc = dev_info(device, di);
    if (rc) return rc;
    b200c_rchan *h = new (std::nothrow) b200c_rchan();
    if (!h) { set_error("out of host memory"); return B200C_ERR_NOMEM; }
    h->device = device; h->dtype = dtype; h->di = di;
    DeviceGuard g(device);
    if (!g.ok) { delete h; set_error("cudaSetDevice(%d) failed", device); return B200C_ERR_CUDA; }
    rc = rchan_plan_create(h->plan, m, decim, di.smem_optin);
    const double one = 1.0;   // taps {1}, as FIRFilter() (filter/FIRFilter.cpp:125)
    if (!rc) rc = chan_set_taps(h->plan, &one, 1);
    if (rc) { b200c_rchan_destroy(h); return rc; }
    *out = h;
    return B200C_OK;
}

int b200c_rchan_destroy(b200c_rchan *h)
{
    if (!h) return B200C_OK;
    {
        DeviceGuard g(h->device);
        chan_plan_destroy(h->plan);
    }
    delete h;
    return B200C_OK;
}

int b200c_rchan_set_taps(b200c_rchan *h, const double *taps, size_t ntaps)
{
    if (!h) return B200C_ERR_INVALID;
    if (ntaps == 0 || !taps) { set_error("real channelizer: taps cannot be empty"); return B200C_ERR_INVALID; }
    if (ntaps > kChanMaxTapsPerBranch * (size_t)h->plan.M) {
        set_error("real channelizer: %zu taps exceed 16 per branch (%zu for %d branches)", ntaps, kChanMaxTapsPerBranch * (size_t)h->plan.M, h->plan.M);
        return B200C_ERR_INVALID;
    }
    DeviceGuard g(h->device);
    if (!g.ok) { set_error("cudaSetDevice(%d) failed", h->device); return B200C_ERR_CUDA; }
    return chan_set_taps(h->plan, taps, ntaps);
}

int b200c_rchan_info(const b200c_rchan *h, size_t *m, size_t *nchan, size_t *decim, size_t *ntaps, size_t *input_require)
{
    if (!h) return B200C_ERR_INVALID;
    if (m) *m = (size_t)h->plan.M;
    if (nchan) *nchan = (size_t)h->plan.M / 2 + 1;
    if (decim) *decim = (size_t)h->plan.D;
    if (ntaps) *ntaps = h->plan.ntaps;
    if (input_require) *input_require = h->plan.ntaps - 1 + (size_t)h->plan.D;
    return B200C_OK;
}

int b200c_rchan_run(b200c_rchan *h, const void *d_in, size_t in_elems, uint64_t stream_index, void *d_out,
                    size_t out_stride, size_t out_capacity, size_t *consumed, size_t *produced, void *stream)
{
    if (!h) return B200C_ERR_INVALID;
    const size_t Km1 = h->plan.ntaps - 1, D = (size_t)h->plan.D;
    const size_t F = in_elems >= Km1 + D ? std::min((in_elems - Km1) / D, out_capacity) : 0;
    if (consumed) *consumed = F * D;
    if (produced) *produced = F;
    if (F == 0) return B200C_OK;
    if (!d_in || !d_out) { set_error("b200c_rchan_run: null device buffer"); return B200C_ERR_INVALID; }
    if (out_stride < F) { set_error("real channelizer: output stride %zu shorter than the %zu frames produced", out_stride, F); return B200C_ERR_INVALID; }
    DeviceGuard g(h->device);
    if (!g.ok) { set_error("cudaSetDevice(%d) failed", h->device); return B200C_ERR_CUDA; }
    return rchan_launch(h->plan, h->dtype, d_in, F, stream_index, d_out, out_stride, (cudaStream_t)stream);
}

/* ------------------------------------------------------------------- synthesizer --- */
int b200c_synth_create(b200c_synth **out, int dtype, size_t nchan, size_t interp, int device)
{
    if (!out) return B200C_ERR_INVALID;
    *out = nullptr;
    if (dtype != B200C_CF32) { set_error("synthesizer: dtype %d unsupported (complex float32 only)", dtype); return B200C_ERR_UNSUPPORTED; }
    if (nchan < 2 || nchan > kSynthMaxChannels || (nchan & (nchan - 1))) {
        set_error("synthesizer: %zu channels unsupported (a power of two from 2 to %zu)", nchan, kSynthMaxChannels);
        return B200C_ERR_UNSUPPORTED;
    }
    if (interp == 0 || nchan % interp) { set_error("synthesizer: interpolation %zu must divide the channel count %zu", interp, nchan); return B200C_ERR_INVALID; }
    DevInfo di;
    int rc = dev_info(device, di);
    if (rc) return rc;
    b200c_synth *h = new (std::nothrow) b200c_synth();
    if (!h) { set_error("out of host memory"); return B200C_ERR_NOMEM; }
    h->device = device; h->di = di;
    DeviceGuard g(device);
    if (!g.ok) { delete h; set_error("cudaSetDevice(%d) failed", device); return B200C_ERR_CUDA; }
    rc = synth_plan_create(h->plan, nchan, interp, di.smem_optin);
    const double one = 1.0;   // taps {1}, as FIRFilter() (filter/FIRFilter.cpp:125)
    if (!rc) rc = synth_set_taps(h->plan, &one, 1);
    if (rc) { b200c_synth_destroy(h); return rc; }
    *out = h;
    return B200C_OK;
}

int b200c_synth_destroy(b200c_synth *h)
{
    if (!h) return B200C_OK;
    {
        DeviceGuard g(h->device);
        synth_plan_destroy(h->plan);
    }
    delete h;
    return B200C_OK;
}

int b200c_synth_set_taps(b200c_synth *h, const double *taps, size_t ntaps)
{
    if (!h) return B200C_ERR_INVALID;
    if (ntaps == 0 || !taps) { set_error("synthesizer: taps cannot be empty"); return B200C_ERR_INVALID; }
    const size_t M = (size_t)h->plan.M, D = (size_t)h->plan.D;
    const size_t limit = std::min(kSynthMaxTapsPerChannel * M, kSynthMaxTapsPerPhase * D);
    if (ntaps > limit) {
        set_error("synthesizer: %zu taps exceed min(16 M, 32 D) = %zu for %zu channels, interpolation %zu", ntaps, limit, M, D);
        return B200C_ERR_INVALID;
    }
    DeviceGuard g(h->device);
    if (!g.ok) { set_error("cudaSetDevice(%d) failed", h->device); return B200C_ERR_CUDA; }
    return synth_set_taps(h->plan, taps, ntaps);
}

int b200c_synth_info(const b200c_synth *h, size_t *nchan, size_t *interp, size_t *ntaps, size_t *input_require)
{
    if (!h) return B200C_ERR_INVALID;
    if (nchan) *nchan = (size_t)h->plan.M;
    if (interp) *interp = (size_t)h->plan.D;
    if (ntaps) *ntaps = h->plan.ntaps;
    if (input_require) *input_require = (size_t)h->plan.K;
    return B200C_OK;
}

int b200c_synth_run(b200c_synth *h, const void *d_in, size_t in_stride, size_t in_frames, uint64_t stream_index, void *d_out,
                    size_t out_capacity, size_t *consumed, size_t *produced, void *stream)
{
    if (!h) return B200C_ERR_INVALID;
    if (consumed) *consumed = 0;
    if (produced) *produced = 0;
    if (in_stride < in_frames) { set_error("synthesizer: input stride %zu shorter than the %zu frames given", in_stride, in_frames); return B200C_ERR_INVALID; }
    const size_t Km1 = (size_t)h->plan.K - 1, D = (size_t)h->plan.D;
    const size_t F = in_frames > Km1 ? std::min(in_frames - Km1, out_capacity / D) : 0;
    if (consumed) *consumed = F;
    if (produced) *produced = F * D;
    if (F == 0) return B200C_OK;
    if (!d_in || !d_out) { set_error("b200c_synth_run: null device buffer"); return B200C_ERR_INVALID; }
    DeviceGuard g(h->device);
    if (!g.ok) { set_error("cudaSetDevice(%d) failed", h->device); return B200C_ERR_CUDA; }
    return synth_launch(h->plan, d_in, in_stride, F, stream_index, d_out, (cudaStream_t)stream);
}

/* ------------------------------------------------------- real-output synthesizer --- */
int b200c_rsynth_create(b200c_rsynth **out, int dtype, size_t m, size_t interp, int device)
{
    if (!out) return B200C_ERR_INVALID;
    *out = nullptr;
    if (dtype != B200C_F32 && dtype != B200C_I16) {
        set_error("real synthesizer: dtype %d unsupported (float32 or int16 only)", dtype);
        return B200C_ERR_UNSUPPORTED;
    }
    if (m < 2 || m > kRSynthMaxBranches || (m & (m - 1))) {
        set_error("real synthesizer: %zu branches unsupported (a power of two from 2 to %zu)", m, kRSynthMaxBranches);
        return B200C_ERR_UNSUPPORTED;
    }
    if (interp == 0 || m % interp) { set_error("real synthesizer: interpolation %zu must divide the branch count %zu", interp, m); return B200C_ERR_INVALID; }
    DevInfo di;
    int rc = dev_info(device, di);
    if (rc) return rc;
    b200c_rsynth *h = new (std::nothrow) b200c_rsynth();
    if (!h) { set_error("out of host memory"); return B200C_ERR_NOMEM; }
    h->device = device; h->dtype = dtype; h->di = di;
    DeviceGuard g(device);
    if (!g.ok) { delete h; set_error("cudaSetDevice(%d) failed", device); return B200C_ERR_CUDA; }
    rc = rsynth_plan_create(h->plan, m, interp, di.smem_optin);
    const double one = 1.0;   // taps {1}, as FIRFilter() (filter/FIRFilter.cpp:125)
    if (!rc) rc = rsynth_set_taps(h->plan, &one, 1);
    if (rc) { b200c_rsynth_destroy(h); return rc; }
    *out = h;
    return B200C_OK;
}

int b200c_rsynth_destroy(b200c_rsynth *h)
{
    if (!h) return B200C_OK;
    {
        DeviceGuard g(h->device);
        synth_plan_destroy(h->plan);
    }
    delete h;
    return B200C_OK;
}

int b200c_rsynth_set_taps(b200c_rsynth *h, const double *taps, size_t ntaps)
{
    if (!h) return B200C_ERR_INVALID;
    if (ntaps == 0 || !taps) { set_error("real synthesizer: taps cannot be empty"); return B200C_ERR_INVALID; }
    const size_t M = (size_t)h->plan.M, D = (size_t)h->plan.D;
    const size_t limit = std::min(kSynthMaxTapsPerChannel * M, kSynthMaxTapsPerPhase * D);
    if (ntaps > limit) {
        set_error("real synthesizer: %zu taps exceed min(16 M, 32 D) = %zu for %zu branches, interpolation %zu", ntaps, limit, M, D);
        return B200C_ERR_INVALID;
    }
    DeviceGuard g(h->device);
    if (!g.ok) { set_error("cudaSetDevice(%d) failed", h->device); return B200C_ERR_CUDA; }
    return rsynth_set_taps(h->plan, taps, ntaps);
}

int b200c_rsynth_info(const b200c_rsynth *h, size_t *m, size_t *nchan, size_t *interp, size_t *ntaps, size_t *input_require)
{
    if (!h) return B200C_ERR_INVALID;
    if (m) *m = (size_t)h->plan.M;
    if (nchan) *nchan = (size_t)h->plan.M / 2 + 1;
    if (interp) *interp = (size_t)h->plan.D;
    if (ntaps) *ntaps = h->plan.ntaps;
    if (input_require) *input_require = (size_t)h->plan.K;
    return B200C_OK;
}

int b200c_rsynth_run(b200c_rsynth *h, const void *d_in, size_t in_stride, size_t in_frames, uint64_t stream_index,
                     void *d_out, size_t out_capacity, size_t *consumed, size_t *produced, void *stream)
{
    if (!h) return B200C_ERR_INVALID;
    if (consumed) *consumed = 0;
    if (produced) *produced = 0;
    if (in_stride < in_frames) { set_error("real synthesizer: input stride %zu shorter than the %zu frames given", in_stride, in_frames); return B200C_ERR_INVALID; }
    const size_t Km1 = (size_t)h->plan.K - 1, D = (size_t)h->plan.D;
    const size_t F = in_frames > Km1 ? std::min(in_frames - Km1, out_capacity / D) : 0;
    if (consumed) *consumed = F;
    if (produced) *produced = F * D;
    if (F == 0) return B200C_OK;
    if (!d_in || !d_out) { set_error("b200c_rsynth_run: null device buffer"); return B200C_ERR_INVALID; }
    DeviceGuard g(h->device);
    if (!g.ok) { set_error("cudaSetDevice(%d) failed", h->device); return B200C_ERR_CUDA; }
    return rsynth_launch(h->plan, h->dtype, d_in, in_stride, F, stream_index, d_out, (cudaStream_t)stream);
}

/* ----------------------------------------------------------------------------- FFT --- */
int b200c_fft_create(b200c_fft **out, int dtype, size_t nbins, int inverse, int device)
{
    if (!out) return B200C_ERR_INVALID;
    *out = nullptr;
    if (dtype != B200C_CF32 && dtype != B200C_CF64 && dtype != B200C_CI16) {
        set_error("FFTFactory(dtype=%d): unsupported type", dtype);   // fft/FFT.cpp:92
        return B200C_ERR_UNSUPPORTED;
    }
    DevInfo di;
    int rc = dev_info(device, di);
    if (rc) return rc;
    b200c_fft *h = new (std::nothrow) b200c_fft();
    if (!h) { set_error("out of host memory"); return B200C_ERR_NOMEM; }
    h->device = device; h->di = di;
    DeviceGuard g(device);
    if (!g.ok) { delete h; set_error("cudaSetDevice(%d) failed", device); return B200C_ERR_CUDA; }
    rc = fft_plan_create(h->plan, dtype, nbins, inverse, std::min<size_t>(di.smem_optin, 200 * 1024));
    if (rc) { fft_plan_destroy(h->plan); delete h; return rc; }
    *out = h;
    return B200C_OK;
}

int b200c_fft_destroy(b200c_fft *h)
{
    if (!h) return B200C_OK;
    {
        DeviceGuard g(h->device);
        fft_plan_destroy(h->plan);
        h->pipe.release();
    }
    delete h;
    return B200C_OK;
}

int b200c_fft_info(const b200c_fft *h, size_t *nbins, int *inverse)
{
    if (!h) return B200C_ERR_INVALID;
    if (nbins) *nbins = (size_t)h->plan.n;
    if (inverse) *inverse = h->plan.inverse;
    return B200C_OK;
}

int b200c_fft_run(b200c_fft *h, const void *d_in, void *d_out, size_t batch, void *stream)
{
    if (!h) return B200C_ERR_INVALID;
    if (batch == 0) return B200C_OK;
    if (!d_in || !d_out) { set_error("b200c_fft_run: null device buffer"); return B200C_ERR_INVALID; }
    DeviceGuard g(h->device);
    if (!g.ok) { set_error("cudaSetDevice(%d) failed", h->device); return B200C_ERR_CUDA; }
    return fft_launch(h->plan, d_in, d_out, batch, h->di.sm_count, (cudaStream_t)stream);
}

int b200c_fft_run_host(b200c_fft *h, const void *h_in, void *h_out, size_t batch)
{
    if (!h) return B200C_ERR_INVALID;
    if (batch == 0) return B200C_OK;
    if (!h_in || !h_out) { set_error("b200c_fft_run_host: null host buffer"); return B200C_ERR_INVALID; }
    DeviceGuard g(h->device);
    if (!g.ok) { set_error("cudaSetDevice(%d) failed", h->device); return B200C_ERR_CUDA; }
    const size_t tb = (size_t)h->plan.n * dtype_bytes(h->plan.dtype);
    size_t cb = std::max<size_t>(1, host_chunk_bytes() / tb);
    cb = std::min(cb, batch);
    int rc = h->pipe.ensure(cb * tb, cb * tb);
    if (rc) return rc;
    const char *src = static_cast<const char *>(h_in);
    char *dst = static_cast<char *>(h_out);
    size_t slot = 0;
    for (size_t b0 = 0; b0 < batch; b0 += cb, slot = (slot + 1) % (size_t)h->pipe.n) {
        const size_t nb = std::min(cb, batch - b0);
        cudaStream_t s = h->pipe.streams[slot];
        B200C_CUDA_TRY(cudaMemcpyAsync(h->pipe.d_in[slot], src + b0 * tb, nb * tb, cudaMemcpyHostToDevice, s));
        rc = fft_launch(h->plan, h->pipe.d_in[slot], h->pipe.d_out[slot], nb, h->di.sm_count, s);
        if (rc) return rc;
        B200C_CUDA_TRY(cudaMemcpyAsync(dst + b0 * tb, h->pipe.d_out[slot], nb * tb, cudaMemcpyDeviceToHost, s));
    }
    return h->pipe.sync_all();
}

/* ------------------------------------------------------- device-resident ring (CUDA VMM) --- */
// The driver entry points are fetched through the runtime so that libb200comms.so has no
// link-time dependency on libcuda.so.1 (it must load, and fail loudly, on GPU-less hosts).
#define DRV_FN(name, type)                                                                          \
    static type p_##name = nullptr;                                                                 \
    if (!p_##name) {                                                                                \
        cudaDriverEntryPointQueryResult qr;                                                         \
        void *fp = nullptr;                                                                         \
        if (cudaGetDriverEntryPoint(#name, &fp, cudaEnableDefault, &qr) != cudaSuccess || !fp) {    \
            (void)cudaGetLastError();                                                               \
            set_error("CUDA driver entry point %s unavailable", #name);                             \
            return B200C_ERR_CUDA;                                                                  \
        }                                                                                           \
        p_##name = (type)fp;                                                                        \
    }

#define DRV_TRY(expr)                                                                               \
    do {                                                                                            \
        CUresult r__ = (expr);                                                                      \
        if (r__ != CUDA_SUCCESS) { set_error("%s failed: CUresult %d", #expr, (int)r__); rc = B200C_ERR_CUDA; goto fail; } \
    } while (0)

typedef CUresult (*fn_cuMemGetAllocationGranularity)(size_t *, const CUmemAllocationProp *, CUmemAllocationGranularity_flags);
typedef CUresult (*fn_cuMemCreate)(CUmemGenericAllocationHandle *, size_t, const CUmemAllocationProp *, unsigned long long);
typedef CUresult (*fn_cuMemAddressReserve)(CUdeviceptr *, size_t, size_t, CUdeviceptr, unsigned long long);
typedef CUresult (*fn_cuMemMap)(CUdeviceptr, size_t, size_t, CUmemGenericAllocationHandle, unsigned long long);
typedef CUresult (*fn_cuMemSetAccess)(CUdeviceptr, size_t, const CUmemAccessDesc *, size_t);
typedef CUresult (*fn_cuMemUnmap)(CUdeviceptr, size_t);
typedef CUresult (*fn_cuMemAddressFree)(CUdeviceptr, size_t);
typedef CUresult (*fn_cuMemRelease)(CUmemGenericAllocationHandle);

int b200c_ring_destroy(b200c_ring *r)
{
    if (!r) return B200C_OK;
    DRV_FN(cuMemUnmap, fn_cuMemUnmap)
    DRV_FN(cuMemAddressFree, fn_cuMemAddressFree)
    DRV_FN(cuMemRelease, fn_cuMemRelease)
    DeviceGuard g(r->device);
    cudaDeviceSynchronize();
    for (int i = 0; i < 2; i++) if (r->mapped[i]) p_cuMemUnmap(r->base + (CUdeviceptr)i * r->bytes, r->bytes);
    if (r->have_va) p_cuMemAddressFree(r->base, 2 * r->bytes);
    if (r->have_handle) p_cuMemRelease(r->handle);
    delete r;
    return B200C_OK;
}

int b200c_ring_create(b200c_ring **out, size_t min_bytes, int device)
{
    if (!out || min_bytes == 0) return B200C_ERR_INVALID;
    *out = nullptr;
    DevInfo di;
    int rc = dev_info(device, di);
    if (rc) return rc;
    DRV_FN(cuMemGetAllocationGranularity, fn_cuMemGetAllocationGranularity)
    DRV_FN(cuMemCreate, fn_cuMemCreate)
    DRV_FN(cuMemAddressReserve, fn_cuMemAddressReserve)
    DRV_FN(cuMemMap, fn_cuMemMap)
    DRV_FN(cuMemSetAccess, fn_cuMemSetAccess)
    DeviceGuard g(device);
    if (!g.ok) { set_error("cudaSetDevice(%d) failed", device); return B200C_ERR_CUDA; }
    B200C_CUDA_TRY(cudaFree(0));   // make sure the primary context exists

    b200c_ring *r = new (std::nothrow) b200c_ring();
    if (!r) { set_error("out of host memory"); return B200C_ERR_NOMEM; }
    r->device = device;
    CUmemAllocationProp prop;
    std::memset(&prop, 0, sizeof(prop));
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = device;
    CUmemAccessDesc acc;
    std::memset(&acc, 0, sizeof(acc));
    acc.location = prop.location;
    acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    size_t gran = 0;
    DRV_TRY(p_cuMemGetAllocationGranularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_MINIMUM));
    r->bytes = (min_bytes + gran - 1) / gran * gran;
    DRV_TRY(p_cuMemCreate(&r->handle, r->bytes, &prop, 0));
    r->have_handle = true;
    DRV_TRY(p_cuMemAddressReserve(&r->base, 2 * r->bytes, gran, 0, 0));
    r->have_va = true;
    for (int i = 0; i < 2; i++) {
        DRV_TRY(p_cuMemMap(r->base + (CUdeviceptr)i * r->bytes, r->bytes, 0, r->handle, 0));
        r->mapped[i] = true;
    }
    DRV_TRY(p_cuMemSetAccess(r->base, 2 * r->bytes, &acc, 1));
    *out = r;
    return B200C_OK;
fail:
    b200c_ring_destroy(r);
    return rc;
}

void *b200c_ring_base(const b200c_ring *r) { return r ? (void *)r->base : nullptr; }
size_t b200c_ring_bytes(const b200c_ring *r) { return r ? r->bytes : 0; }

/* ------------------------------------------------------------- plain device buffers --- */
#define WITH_DEVICE(dev)                                                                            \
    DeviceGuard g(dev);                                                                             \
    if (!g.ok) { set_error("cudaSetDevice(%d) failed", dev); return B200C_ERR_CUDA; }

int b200c_dev_alloc(void **d_ptr, size_t bytes, int device)
{
    if (!d_ptr) return B200C_ERR_INVALID;
    *d_ptr = nullptr;
    DevInfo di;
    int rc = dev_info(device, di);
    if (rc) return rc;
    WITH_DEVICE(device)
    B200C_CUDA_TRY(cudaMalloc(d_ptr, bytes ? bytes : 1));
    return B200C_OK;
}
int b200c_dev_free(void *d_ptr, int device)
{
    if (!d_ptr) return B200C_OK;
    WITH_DEVICE(device)
    B200C_CUDA_TRY(cudaFree(d_ptr));
    return B200C_OK;
}
int b200c_host_alloc_pinned(void **h_ptr, size_t bytes)
{
    if (!h_ptr) return B200C_ERR_INVALID;
    *h_ptr = nullptr;
    B200C_CUDA_TRY(cudaMallocHost(h_ptr, bytes ? bytes : 1));
    return B200C_OK;
}
int b200c_host_free_pinned(void *h_ptr)
{
    if (!h_ptr) return B200C_OK;
    B200C_CUDA_TRY(cudaFreeHost(h_ptr));
    return B200C_OK;
}
int b200c_copy_h2d(void *d_dst, const void *h_src, size_t bytes, int device, void *stream)
{
    WITH_DEVICE(device)
    B200C_CUDA_TRY(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    return B200C_OK;
}
int b200c_copy_d2h(void *h_dst, const void *d_src, size_t bytes, int device, void *stream)
{
    WITH_DEVICE(device)
    B200C_CUDA_TRY(cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return B200C_OK;
}
int b200c_copy_d2d(void *d_dst, const void *d_src, size_t bytes, int device, void *stream)
{
    WITH_DEVICE(device)
    B200C_CUDA_TRY(cudaMemcpyAsync(d_dst, d_src, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return B200C_OK;
}
int b200c_memset(void *d_dst, int value, size_t bytes, int device, void *stream)
{
    WITH_DEVICE(device)
    B200C_CUDA_TRY(cudaMemsetAsync(d_dst, value, bytes, (cudaStream_t)stream));
    return B200C_OK;
}
int b200c_stream_sync(int device, void *stream)
{
    WITH_DEVICE(device)
    B200C_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    return B200C_OK;
}

} // extern "C"
