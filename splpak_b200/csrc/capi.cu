// capi.cu -- the C ABI of include/splpak_b200.h: argument validation in the reference's order,
// device-memory ownership, host<->device staging, and the launch sequences of the kernels in
// eval.cu / assemble.cu / solve.cu.  There is no CPU fallback anywhere in this file: without a
// usable CUDA device every compute entry point returns SPLPAK_ERR_CUDA.
#include <condition_variable>
#include <dlfcn.h>
#include <math.h>
#include <mutex>
#include <new>
#include <stdlib.h>
#include <string.h>
#include <thread>
#include <vector>

#include "common.cuh"

unsigned long long g_spl_launches = 0;

// ---- kernels' host launchers (other translation units) ----
int spl_assemble_scratch_init(const GridParams &gp, AssembleScratch &sc, cudaStream_t st);
int spl_assemble_scratch_reserve(const GridParams &gp, AssembleScratch &sc, long long n);
void spl_assemble_scratch_free(AssembleScratch &sc);
int spl_eval_launch(const GridParams &gp, const int *nderiv, int order, const real_t *d_x, int l1x, long long nq,
                    const double *d_coef, long long ncol_padded, real_t *d_out, cudaStream_t stream,
                    int nsm, size_t smem_optin, unsigned long long *d_counter, double *d_pad);
long long spl_eval_regroup_elems(const GridParams &gp, long long nq, int nsm, size_t smem_optin);
long long spl_eval_scratch_elems(const GridParams &gp, const int *nderiv, int order, long long nq, int nsm,
                                 size_t smem_optin);
#ifdef SPLPAK_REAL32
int spl_eval_f32_launch(const GridParams &gp, const real_t *d_x, int l1x, long long nq, const real_t *d_coef,
                        real_t *d_out, cudaStream_t stream, int nsm, size_t smem_optin, unsigned long long *d_counter);
int spl_eval_f32_mixed4_launch(const GridParams &gp, const real_t *d_x, int l1x, long long nq, const real_t *d_coef,
                               const double *d_coef64, double *d_pad, real_t *d_out, cudaStream_t stream, int nsm,
                               size_t smem_optin, unsigned long long *d_counter);
long long spl_eval_uni_f32_elems(const GridParams &gp, long long nq, int nsm, size_t smem_optin);
int spl_eval_uni_f32_launch(const GridParams &gp, const real_t *d_x, int l1x, long long nq, const real_t *d_coef,
                            real_t *d_ext, real_t *d_out, cudaStream_t stream, int nsm, size_t smem_optin);
#endif
long long spl_grid_tmp_elems(const GridParams &gp, const long long *naxis);
int spl_eval_grid_launch(const GridParams &gp, const int *nderiv, const real_t *const *d_axis, const long long *naxis,
                         const double *d_coef64, real_t *d_out, double *d_tmp, long long tmp_elems, int *d_iws,
                         double *d_w4, cudaStream_t st, int nsm);
int spl_assemble_chunk(const GridParams &gp, const real_t *d_x, int l1x, const real_t *d_y,
                       const real_t *d_w, int weighted, long long n, int do_hist, int rhs_only,
                       const AssembleScratch &sc, double *d_S, double *d_g, double *d_cnt,
                       double *d_totals, cudaStream_t st, int nsm, cudaEvent_t *ev);
int spl_constraints_launch(const GridParams &gp, double xtrap, const double *d_cnt,
                           const double *d_totals_in, double *d_S, double *d_totals_out,
                           cudaStream_t st, int nsm);
long long spl_band_lda(int bw);
int spl_half_bandwidth(const GridParams &gp);
long long spl_band_elems(const GridParams &gp);
long long spl_solve_workspace(const GridParams &gp);
int spl_solve_launch(const GridParams &gp, const double *d_S, double *d_AB, double *d_g, double *d_work,
                     double **d_coef_out, int *d_fail, cudaStream_t st, cudaStream_t st_aux, int nsm, cudaEvent_t *ev,
                     void **cache);
void spl_solve_cache_free(void *cache);
int spl_resolve_launch(const GridParams &gp, const double *d_AB, double *d_g, double *d_work, double **d_coef_out,
                       int *d_fail, cudaStream_t st, int nsm);
int spl_constraints_residual_launch(const GridParams &gp, double xtrap, const double *d_cnt,
                                    const double *d_totals_in, const double *d_coef, double *d_g,
                                    cudaStream_t st, int nsm);
long long spl_penalty_table_len(const GridParams &gp);
int spl_penalty_add_launch(const GridParams &gp, double lambda, int penalty, double *d_tab, double *d_S,
                           cudaStream_t st, int nsm);
int spl_penalty_residual_launch(const GridParams &gp, double lambda, int penalty, const double *d_tab,
                                const double *d_coef, double *d_g, cudaStream_t st, int nsm);
int spl_measure_peaks_impl(double *out, int n);
int spl_ortho_supported(const GridParams &gp);
void spl_ortho_free(OrthoScratch &os);
int spl_ortho_init(const GridParams &gp, OrthoScratch &os, cudaStream_t st, size_t smem_optin);
int spl_ortho_reset(const GridParams &gp, OrthoScratch &os, cudaStream_t st);
int spl_ortho_add_chunk(const GridParams &gp, const real_t *d_x, int l1x, const real_t *d_y, const real_t *d_w,
                        int weighted, long long n, int do_hist, OrthoScratch &os, double *d_cnt, double *d_totals,
                        cudaStream_t st, int nsm);
int spl_ortho_compute(const GridParams &gp, double xtrap, OrthoScratch &os, const double *d_cnt, double *d_totals,
                      int *d_fail, cudaStream_t st, int nsm);
int spl_pivot_range_launch(const GridParams &gp, const double *d_work, double *d_out2, cudaStream_t st);
int spl_penalty_diag_launch(const GridParams &gp, int penalty, double *d_tab, const double *d_S, double *d_out2,
                            cudaStream_t st);
long long spl_selinv_scratch(const GridParams &gp);
int spl_selinv_launch(const GridParams &gp, double *d_AB, const double *d_work, double *d_scr, cudaStream_t st,
                      void **cache);
void spl_selinv_cache_free(void *cache);
int spl_gcv_ywy_launch(const real_t *d_y, const real_t *d_w, int weighted, long long n, double *d_part, double *d_ywy,
                       cudaStream_t st);
long long spl_gcv_part_len();
int spl_reml_stencil_launch(const GridParams &gp, const double *d_M, const double *d_c, const double *d_g,
                            const double *d_linv, double *d_part, double *d_out3, cudaStream_t st);
int spl_gcv_stencil_launch(const GridParams &gp, const double *d_S, const double *d_AB, const double *d_c,
                           const double *d_g0, double *d_part, double *d_out3, cudaStream_t st);
long long spl_variance_table_len(const GridParams &gp);
int spl_variance_table_launch(const GridParams &gp, const double *d_AB, long long lda, double *d_W, cudaStream_t st,
                              int nsm);
int spl_variance_launch(const GridParams &gp, const int *nderiv, const real_t *d_x, int l1x, long long nq,
                        const double *d_W, real_t *d_out, cudaStream_t st, int nsm);

// ------------------------------------------------------------------------------------------
// small conversion kernels
// ------------------------------------------------------------------------------------------
__global__ void spl_to_double_kernel(const real_t *__restrict__ in, double *__restrict__ out,
                                     long long n, long long npad) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < npad; i += stride)
        out[i] = (i < n) ? (double)in[i] : 0.0;
}
// residual of a chunk, in place: r[i] = y[i] - r[i]   (r holds the spline values on entry)
__global__ void spl_residual_kernel(const real_t *__restrict__ y, real_t *__restrict__ r, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) r[i] = (real_t)((double)y[i] - (double)r[i]);
}
__global__ void spl_axpy_kernel(double *__restrict__ c, const double *__restrict__ d, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) c[i] += d[i];
}

__global__ void spl_from_double_kernel(const double *__restrict__ in, real_t *__restrict__ out,
                                       long long n) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        out[i] = (real_t)in[i];
}

// ------------------------------------------------------------------------------------------
// device context
// ------------------------------------------------------------------------------------------
struct DeviceInfo {
    int ok = 0, dev = 0, nsm = SPL_NSM_DEFAULT;
    size_t smem_optin = 0;
};
static int get_device(DeviceInfo &di) {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count < 1) {
        cudaGetLastError();
        return SPLPAK_ERR_CUDA;
    }
    SPL_CUDA_TRY(cudaGetDevice(&di.dev));
    // the two attributes are cached per device (cudaGetDeviceProperties costs milliseconds per call)
    static std::mutex mu;
    static int c_nsm[64] = {0};
    static size_t c_smem[64] = {0};
    std::lock_guard<std::mutex> lk(mu);
    const int slot = (di.dev >= 0 && di.dev < 64) ? di.dev : -1;
    if (slot < 0 || c_nsm[slot] == 0) {
        int nsm = 0, smem = 0;
        SPL_CUDA_TRY(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, di.dev));
        SPL_CUDA_TRY(cudaDeviceGetAttribute(&smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, di.dev));
        di.nsm = nsm;
        di.smem_optin = (size_t)smem;
        if (slot >= 0) {
            c_nsm[slot] = nsm;
            c_smem[slot] = (size_t)smem;
        }
    } else {
        di.nsm = c_nsm[slot];
        di.smem_optin = c_smem[slot];
    }
    di.ok = 1;
    return SPLPAK_OK;
}

// ------------------------------------------------------------------------------------------
// Pageable host memory.  The reference's caller arrays are ordinary Fortran arrays (src/splpak.F90:537-559), i.e.
// pageable: cudaMemcpyAsync from/to them is staged by the driver through one internal bounce buffer by ONE thread
// and serialises with everything else.  The host-array entry points therefore stage pageable ranges themselves:
// a small per-device ring of pinned slots, filled (or drained) by a pool of host threads, one cudaMemcpyAsync per
// slot, so the host-side memcpy of piece k+1 overlaps the DMA of piece k.  Ranges that are already pinned
// (cudaHostAlloc / cudaHostRegister / torch pin_memory) are copied directly.
// ------------------------------------------------------------------------------------------
class CopyPool {
  public:
    static CopyPool &get() {
        static CopyPool *pool = new CopyPool();      // leaked on purpose: its detached workers outlive static destructors
        return *pool;
    }
    void copy(void *dst, const void *src, size_t bytes) {
        if (nthr_ <= 1 || bytes < (1u << 20)) {
            memcpy(dst, src, bytes);
            return;
        }
        std::unique_lock<std::mutex> lk(mu_);
        dst_ = static_cast<char *>(dst);
        src_ = static_cast<const char *>(src);
        bytes_ = bytes;
        pending_ = nthr_;
        ++gen_;
        cv_work_.notify_all();
        cv_done_.wait(lk, [&] { return pending_ == 0; });
    }

  private:
    CopyPool() {
        int n = 0;
        if (const char *e = getenv("SPLPAK_B200_COPY_THREADS")) n = atoi(e);
        if (n <= 0) {
            int hw = (int)std::thread::hardware_concurrency();
            int ranks = 1;
            if (const char *e = getenv("LOCAL_WORLD_SIZE")) ranks = atoi(e) > 0 ? atoi(e) : 1;
            // measured on the 16-core GPU box, 1e8 pageable points / queries (scripts/pageable_ab.py): 4 / 8 / 12 / 16 / 24
            // threads -> fit 120 / 97 / 83 / 84 / 85 ms, evaluation 139 / 94 / 83 / 84 / 93 ms
            n = (hw * 3 / 4) / ranks;
            if (n > 12) n = 12;
        }
        if (n < 1) n = 1;
        nthr_ = n;
        for (int t = 0; t < nthr_; ++t) workers_.emplace_back([this, t] { run(t); });
        for (auto &w : workers_) w.detach();         // process-lifetime pool
    }
    void run(int t) {
        unsigned long long seen = 0;
        for (;;) {
            const char *src;
            char *dst;
            size_t bytes;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_work_.wait(lk, [&] { return gen_ != seen; });
                seen = gen_;
                src = src_;
                dst = dst_;
                bytes = bytes_;
            }
            const size_t per = ((bytes + nthr_ - 1) / nthr_ + 4095) & ~(size_t)4095;
            const size_t lo = per * t, hi = lo + per < bytes ? lo + per : bytes;
            if (lo < bytes) memcpy(dst + lo, src + lo, hi - lo);
            {
                std::lock_guard<std::mutex> lk(mu_);
                if (--pending_ == 0) cv_done_.notify_all();
            }
        }
    }
    std::mutex mu_;
    std::condition_variable cv_work_, cv_done_;
    std::vector<std::thread> workers_;
    int nthr_ = 1, pending_ = 0;
    unsigned long long gen_ = 0;
    char *dst_ = nullptr;
    const char *src_ = nullptr;
    size_t bytes_ = 0;
};

#define STAGE_SLOTS 4
#define STAGE_SLOT_BYTES ((size_t)16 << 20)
struct HostStager {
    std::mutex mu;
    char *up[STAGE_SLOTS] = {nullptr}, *down[STAGE_SLOTS] = {nullptr};
    cudaEvent_t up_ev[STAGE_SLOTS] = {nullptr}, down_ev[STAGE_SLOTS] = {nullptr};
    int up_next = 0, down_next = 0;
    // device -> pageable host copies whose DMA into the pinned slot has been issued but not yet drained
    struct Pending {
        void *dst = nullptr;
        size_t bytes = 0;
    } down_pending[STAGE_SLOTS];
    bool ok = false, tried = false;
};
static HostStager &host_stager(int device) {
    static HostStager st[64];
    return st[(device >= 0 && device < 64) ? device : 0];
}
static bool stager_init(HostStager &hs) {
    if (hs.tried) return hs.ok;
    hs.tried = true;
    bool ok = true;
    for (int k = 0; k < STAGE_SLOTS && ok; ++k) {
        ok = ok && cudaHostAlloc((void **)&hs.up[k], STAGE_SLOT_BYTES, cudaHostAllocDefault) == cudaSuccess;
        ok = ok && cudaHostAlloc((void **)&hs.down[k], STAGE_SLOT_BYTES, cudaHostAllocDefault) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&hs.up_ev[k], cudaEventDisableTiming) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&hs.down_ev[k], cudaEventDisableTiming) == cudaSuccess;
    }
    if (!ok) cudaGetLastError();
    hs.ok = ok;
    return ok;
}
// true when the driver can DMA straight from/to p (pinned or registered host memory, or managed/device memory)
static bool host_range_is_pinned(const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type != cudaMemoryTypeUnregistered;
}
static bool stage_disabled() {
    static int v = -1;
    if (v < 0) v = getenv("SPLPAK_B200_NO_STAGING") ? 1 : 0;
    return v == 1;
}

// host -> device, asynchronous on st for pinned sources; pageable sources go through the pinned ring (the call then
// returns once the LAST piece has been handed to the DMA engine; the source may be reused immediately)
static cudaError_t spl_h2d(void *d_dst, const void *h_src, size_t bytes, cudaStream_t st, int dev) {
    if (bytes == 0) return cudaSuccess;
    if (bytes < (256u << 10) || stage_disabled() || host_range_is_pinned(h_src))
        return cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, st);
    HostStager &hs = host_stager(dev);
    std::lock_guard<std::mutex> lk(hs.mu);
    if (!stager_init(hs)) return cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, st);
    cudaError_t e = cudaSuccess;
    for (size_t off = 0; off < bytes && e == cudaSuccess; off += STAGE_SLOT_BYTES) {
        const size_t nb = bytes - off < STAGE_SLOT_BYTES ? bytes - off : STAGE_SLOT_BYTES;
        const int k = hs.up_next;
        hs.up_next = (k + 1) % STAGE_SLOTS;
        if ((e = cudaEventSynchronize(hs.up_ev[k])) != cudaSuccess) break;        // the slot's previous DMA is done
        CopyPool::get().copy(hs.up[k], static_cast<const char *>(h_src) + off, nb);
        if ((e = cudaMemcpyAsync(static_cast<char *>(d_dst) + off, hs.up[k], nb, cudaMemcpyHostToDevice, st)) != cudaSuccess) break;
        e = cudaEventRecord(hs.up_ev[k], st);
    }
    return e;
}

static cudaError_t drain_slot(HostStager &hs, int k) {
    if (!hs.down_pending[k].dst) return cudaSuccess;
    cudaError_t e = cudaEventSynchronize(hs.down_ev[k]);
    if (e == cudaSuccess) CopyPool::get().copy(hs.down_pending[k].dst, hs.down[k], hs.down_pending[k].bytes);
    hs.down_pending[k].dst = nullptr;
    return e;
}
// device -> host on st.  Pageable destinations: the DMA lands in a pinned slot and the host-side copy is DEFERRED
// until the slot is needed again or spl_d2h_flush() is called -- callers must flush before they return.
static cudaError_t spl_d2h(void *h_dst, const void *d_src, size_t bytes, cudaStream_t st, int dev) {
    if (bytes == 0) return cudaSuccess;
    if (bytes < (256u << 10) || stage_disabled() || host_range_is_pinned(h_dst))
        return cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, st);
    HostStager &hs = host_stager(dev);
    std::lock_guard<std::mutex> lk(hs.mu);
    if (!stager_init(hs)) return cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, st);
    cudaError_t e = cudaSuccess;
    for (size_t off = 0; off < bytes && e == cudaSuccess; off += STAGE_SLOT_BYTES) {
        const size_t nb = bytes - off < STAGE_SLOT_BYTES ? bytes - off : STAGE_SLOT_BYTES;
        const int k = hs.down_next;
        hs.down_next = (k + 1) % STAGE_SLOTS;
        if ((e = drain_slot(hs, k)) != cudaSuccess) break;
        if ((e = cudaMemcpyAsync(hs.down[k], static_cast<const char *>(d_src) + off, nb, cudaMemcpyDeviceToHost, st)) != cudaSuccess) break;
        if ((e = cudaEventRecord(hs.down_ev[k], st)) != cudaSuccess) break;
        hs.down_pending[k].dst = static_cast<char *>(h_dst) + off;
        hs.down_pending[k].bytes = nb;
    }
    return e;
}
static cudaError_t spl_d2h_flush(int dev) {
    HostStager &hs = host_stager(dev);
    std::lock_guard<std::mutex> lk(hs.mu);
    cudaError_t e = cudaSuccess;
    for (int i = 0; i < STAGE_SLOTS; ++i) {
        const int k = (hs.down_next + i) % STAGE_SLOTS;       // oldest first
        const cudaError_t ek = drain_slot(hs, k);
        if (e == cudaSuccess) e = ek;
    }
    return e;
}

// Grid validation shared by fit and evaluation, in the reference's order
// (fit :718-750, evaluation :1168-1198).  nderiv != NULL adds the 104 check of :1190.
static int make_grid(int ndim, const real_t *xmin, const real_t *xmax, const int *nodes,
                     const int *nderiv, GridParams &gp, int *soft104) {
    memset(&gp, 0, sizeof(gp));
    if (soft104) *soft104 = 0;
    if (ndim < 1 || ndim > SPL_MAXDIM) return SPLPAK_ERR_NDIM;
    gp.ndim = ndim;
    gp.ncol = 1;
    gp.nwindows = 1;
    gp.nsten = 1;
    for (int d = 0; d < ndim; ++d) {
        const int nod = nodes[d];
        if (nod < 4) return SPLPAK_ERR_NODES;
        const real_t xrng = xmax[d] - xmin[d];
        if (xrng == (real_t)0) return SPLPAK_ERR_RANGE;
        if (nderiv && soft104 && (nderiv[d] < 0 || nderiv[d] > 2)) *soft104 = 1;   // no return, :1190-1194
        // working-precision arithmetic exactly as :747-748, then widened
        const real_t dx = xrng / (real_t)(nod - 1);
        const real_t dxin = (real_t)1.0 / dx;
        gp.nodes[d] = nod;
        gp.nwin[d] = nod - 3;
        gp.xmin[d] = (double)xmin[d];
        gp.dx[d] = (double)dx;
        gp.dxin[d] = (double)dxin;
        gp.ncol *= nod;
        gp.nwindows *= (nod - 3);
        gp.nsten *= 4;
    }
    for (int d = ndim; d < SPL_MAXDIM; ++d) {
        gp.nodes[d] = 4;
        gp.nwin[d] = 1;
        gp.dx[d] = 1.0;
        gp.dxin[d] = 1.0;
    }
    return SPLPAK_OK;
}

extern "C" int splpak_b200_sizeof_real(void) { return (int)sizeof(real_t); }

extern "C" const char *splpak_b200_strerror(int code, int evaluation) {
    if (evaluation) {
        switch (code) {   // src/splpak.F90:1170-1193
        case 0: return "";
        case 101: return " splfe or splde - NDIM is less than 1";
        case 102: return " splfe or splde - NODES(IDIM) is less than  4for some IDIM";
        case 103: return " splfe or splde - XMIN(IDIM) = XMAX(IDIM) for some IDIM";
        case 104: return " splde - NDERIV(IDIM) IS less than 0 or greater than 2 for some IDIM";
        }
    } else {
        switch (code) {   // src/splpak.F90:720-779, :852
        case 0: return "";
        case 101: return " splcc or splcw - NDIM is less than 1";
        case 102: return " splcc or splcw - NODES(IDIM) is less than 4 for some IDIM";
        case 103: return " splcc or splcw - XMIN(IDIM) equals XMAX(IDIM) for some IDIM";
        case 104: return " splcc or splcw - NCF (size of COEF) is too small";
        case 105: return " splcc or splcw - Ndata Is less than 1";
        case 106: return " splcc or splcw - NWRK (size of WORK) is too small";
        case 107: return " splcc or splcw - suprls failure (this usually indicates insufficient input data)";
        }
    }
    switch (code) {
    case SPLPAK_ERR_CUDA: return " splpak_b200 - CUDA failure (no usable device, or a runtime error)";
    case SPLPAK_ERR_NCCL: return " splpak_b200 - NCCL failure";
    case SPLPAK_ERR_HANDLE: return " splpak_b200 - invalid handle or argument";
    case SPLPAK_ERR_ALLOC: return " splpak_b200 - device allocation failed";
    }
    return " splpak_b200 - unknown error";
}

// ------------------------------------------------------------------------------------------
// evaluation
// ------------------------------------------------------------------------------------------
static cudaMemPool_t eval_scratch_pool(int device) {
    static std::mutex mu;
    static cudaMemPool_t pools[64] = {nullptr};
    static bool tried[64] = {false};
    if (device < 0 || device >= 64) return nullptr;
    std::lock_guard<std::mutex> lk(mu);
    if (!tried[device]) {
        tried[device] = true;
        cudaMemPoolProps props;
        memset(&props, 0, sizeof(props));
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = device;
        cudaMemPool_t p = nullptr;
        if (cudaMemPoolCreate(&p, &props) == cudaSuccess) {
            unsigned long long keep = ~0ULL;
            cudaMemPoolSetAttribute(p, cudaMemPoolAttrReleaseThreshold, &keep);
            pools[device] = p;
        } else {
            cudaGetLastError();
        }
    }
    return pools[device];
}

#define EVAL_COUNTERS 1024
static unsigned long long *eval_counter_slot(int device) {
    static std::mutex mu;
    static unsigned long long *pool[64] = {nullptr};
    static unsigned next[64] = {0};
    if (device < 0 || device >= 64) return nullptr;
    std::lock_guard<std::mutex> lk(mu);
    if (!pool[device]) {
        if (cudaMalloc((void **)&pool[device], sizeof(unsigned long long) * EVAL_COUNTERS) != cudaSuccess) {
            pool[device] = nullptr;
            return nullptr;
        }
    }
    return pool[device] + (next[device]++ % EVAL_COUNTERS);
}

// order 0: one output per query (nderiv, NULL = splfe); order 1 / 2: the derivative sets, ncomp outputs per query
static int eval_device_impl(const GridParams &gp, const DeviceInfo &di, const int *nderiv, int order,
                            const real_t *d_x, int l1x, long long nq, const real_t *d_coef,
                            real_t *d_out, cudaStream_t st) {
#ifdef SPLPAK_REAL32
    {
        // splfe of the REAL32 library runs in working precision (float), like the reference built with -DREAL32; the
        // derivative sets keep float I/O with float64 arithmetic, as splde does
        bool value = order == 0;
        for (int d = 0; d < gp.ndim; ++d)
            if (nderiv && nderiv[d] != 0) value = false;
        const char *mode = getenv("SPLPAK_B200_R32");
        if (value && !(mode && strcmp(mode, "f64") == 0)) {
            unsigned long long *counter = eval_counter_slot(di.dev);
            if (!counter) return SPLPAK_ERR_ALLOC;
            cudaMemPool_t pool = eval_scratch_pool(di.dev);
            // uniform (phantom-node) form in float: extended float table (padded when the 32-class regrouping kernel runs)
            const long long ext_floats = spl_eval_uni_f32_elems(gp, nq, di.nsm, di.smem_optin);
            if (ext_floats > 0) {
                real_t *ext = nullptr;
                cudaError_t e = pool ? cudaMallocFromPoolAsync((void **)&ext, sizeof(float) * (size_t)ext_floats, pool, st)
                                     : cudaMallocAsync((void **)&ext, sizeof(float) * (size_t)ext_floats, st);
                if (e == cudaSuccess) {
                    const int rcu = spl_eval_uni_f32_launch(gp, d_x, l1x, nq, d_coef, ext, d_out, st, di.nsm, di.smem_optin);
                    cudaFreeAsync(ext, st);
                    return rcu;
                }
                cudaGetLastError();
            }
            const long long pad_elems4 = (gp.ndim == 4) ? spl_eval_regroup_elems(gp, nq, di.nsm, di.smem_optin) : 0;
            if (pad_elems4 > 0) {
                // 4-D, large batch, exact form: scattered queries go to the float64 regrouping kernel (order probe decides)
                const long long npad4 = (gp.ncol + 1) & ~1LL;
                double *blk = nullptr;
                const size_t bytes = sizeof(double) * (size_t)(npad4 + pad_elems4 + 2);
                cudaError_t e = pool ? cudaMallocFromPoolAsync((void **)&blk, bytes, pool, st) : cudaMallocAsync((void **)&blk, bytes, st);
                if (e == cudaSuccess) {
                    spl_to_double_kernel<<<spl_div_up(npad4, 256), 256, 0, st>>>(d_coef, blk, gp.ncol, npad4);
                    ++g_spl_launches;
                    const int rc4 = spl_eval_f32_mixed4_launch(gp, d_x, l1x, nq, d_coef, blk, blk + npad4, d_out, st, di.nsm,
                                                               di.smem_optin, counter);
                    cudaFreeAsync(blk, st);
                    return rc4;
                }
                cudaGetLastError();
            }
            return spl_eval_f32_launch(gp, d_x, l1x, nq, d_coef, d_out, st, di.nsm, di.smem_optin, counter);
        }
    }
#endif
    const long long npad = (gp.ncol + 1) & ~1LL;
    const double *coef64 = nullptr;
    double *tmp = nullptr;
    const bool direct = sizeof(real_t) == sizeof(double) && (gp.ncol % 2 == 0) &&
                        ((uintptr_t)d_coef % 16 == 0);
    if (direct) {
        coef64 = reinterpret_cast<const double *>(d_coef);
    } else {
        // stream-ordered scratch from a private pool that keeps its memory across synchronisations (the
        // default pool hands everything back to the driver at every sync: ~1 ms per call to get it again)
        cudaMemPool_t pool = eval_scratch_pool(di.dev);
        if (pool) SPL_CUDA_TRY(cudaMallocFromPoolAsync((void **)&tmp, sizeof(double) * npad, pool, st));
        else SPL_CUDA_TRY(cudaMallocAsync((void **)&tmp, sizeof(double) * npad, st));
        spl_to_double_kernel<<<spl_div_up(npad, 256), 256, 0, st>>>(d_coef, tmp, gp.ncol, npad);
        ++g_spl_launches;
        coef64 = tmp;
    }
    // tile counter of the dynamic scheduler: one slot of a persistent per-device pool, handed out round
    // robin (a slot is reused only after EVAL_COUNTERS further launches; each launch zeroes its slot
    // on its own stream)
    unsigned long long *counter = eval_counter_slot(di.dev);
    if (!counter) return SPLPAK_ERR_ALLOC;
    // image of the table the kernels read: extended (uniform form) and/or padded (regrouping kernel) copy
    double *pad = nullptr;
    const long long pad_elems = spl_eval_scratch_elems(gp, nderiv, order, nq, di.nsm, di.smem_optin);
    if (pad_elems > 0) {
        cudaMemPool_t pool = eval_scratch_pool(di.dev);
        cudaError_t e = pool ? cudaMallocFromPoolAsync((void **)&pad, sizeof(double) * (size_t)(pad_elems + 2), pool, st)
                             : cudaMallocAsync((void **)&pad, sizeof(double) * (size_t)(pad_elems + 2), st);   // + the order flag
        if (e != cudaSuccess) {
            cudaGetLastError();
            pad = nullptr;                                     // the exact plain kernel needs no scratch
        }
    }
    int rc = spl_eval_launch(gp, nderiv, order, d_x, l1x, nq, coef64, npad, d_out, st, di.nsm, di.smem_optin, counter, pad);
    if (pad) cudaFreeAsync(pad, st);
    if (tmp) cudaFreeAsync(tmp, st);
    return rc;
}

extern "C" int splpak_b200_eval_device(int ndim, const real_t *d_x, int l1x, int64_t nq,
                                       const int *nderiv, const real_t *d_coef, const real_t *xmin,
                                       const real_t *xmax, const int *nodes, real_t *d_out,
                                       void *stream, int *ierror) {
    GridParams gp;
    int soft = 0;
    int rc = make_grid(ndim, xmin, xmax, nodes, nderiv, gp, &soft);
    if (rc == SPLPAK_OK) {
        DeviceInfo di;
        rc = get_device(di);
        if (rc == SPLPAK_OK)
            rc = eval_device_impl(gp, di, nderiv, 0, d_x, l1x, nq, d_coef, d_out, (cudaStream_t)stream);
    }
    if (rc == SPLPAK_OK && soft) rc = SPLPAK_ERR_NDERIV;
    if (ierror) *ierror = rc;
    return rc;
}

// ------------------------------------------------------------------------------------------
// evaluation on a regular output grid (grid.cu)
// ------------------------------------------------------------------------------------------
static int eval_grid_device_impl(const GridParams &gp, const DeviceInfo &di, const int *nderiv,
                                 const real_t *const *d_axis, const long long *naxis, const real_t *d_coef,
                                 real_t *d_out, cudaStream_t st) {
    long long nsum = 0;
    for (int d = 0; d < gp.ndim; ++d) {
        if (naxis[d] <= 0) return SPLPAK_OK;
        nsum += naxis[d];
    }
    const long long tmp_elems = spl_grid_tmp_elems(gp, naxis);
    const bool direct = sizeof(real_t) == sizeof(double);
    // one stream-ordered scratch block: [coef64 (if converted) | 2 x tmp | w4 | iws]
    const size_t coef_d = direct ? 0 : (size_t)gp.ncol;
    const size_t bytes = sizeof(double) * (coef_d + 2 * (size_t)tmp_elems + 4 * (size_t)nsum) + sizeof(int) * (size_t)nsum + 64;
    char *blk = nullptr;
    cudaMemPool_t pool = eval_scratch_pool(di.dev);
    if (pool) SPL_CUDA_TRY(cudaMallocFromPoolAsync((void **)&blk, bytes, pool, st));
    else SPL_CUDA_TRY(cudaMallocAsync((void **)&blk, bytes, st));
    double *c64 = reinterpret_cast<double *>(blk);
    double *tmp = c64 + coef_d;
    double *w4 = tmp + 2 * tmp_elems;
    int *iws = reinterpret_cast<int *>(w4 + 4 * nsum);
    const double *coef64 = reinterpret_cast<const double *>(d_coef);
    if (!direct) {
        spl_to_double_kernel<<<spl_div_up(gp.ncol, 256), 256, 0, st>>>(d_coef, c64, gp.ncol, gp.ncol);
        ++g_spl_launches;
        coef64 = c64;
    }
    const int rc = spl_eval_grid_launch(gp, nderiv, d_axis, naxis, coef64, d_out, tmp, tmp_elems, iws, w4, st, di.nsm);
    cudaFreeAsync(blk, st);
    return rc;
}

// axes: the ndim axes concatenated (axis d has naxis[d] points); out(naxis(1),...,naxis(ndim)), dimension 1 fastest
extern "C" int splpak_b200_eval_grid_device(int ndim, const real_t *d_axes, const int64_t *naxis, const int *nderiv,
                                            const real_t *d_coef, const real_t *xmin, const real_t *xmax,
                                            const int *nodes, real_t *d_out, void *stream, int *ierror) {
    GridParams gp;
    int soft = 0;
    int rc = make_grid(ndim, xmin, xmax, nodes, nderiv, gp, &soft);
    if (rc == SPLPAK_OK) {
        DeviceInfo di;
        rc = get_device(di);
        if (rc == SPLPAK_OK) {
            const real_t *ax[SPL_MAXDIM] = {nullptr, nullptr, nullptr, nullptr};
            long long na[SPL_MAXDIM] = {0, 0, 0, 0}, off = 0;
            for (int d = 0; d < gp.ndim; ++d) {
                ax[d] = d_axes + off;
                na[d] = (long long)naxis[d];
                off += na[d] > 0 ? na[d] : 0;
            }
            rc = eval_grid_device_impl(gp, di, nderiv, ax, na, d_coef, d_out, (cudaStream_t)stream);
        }
    }
    if (rc == SPLPAK_OK && soft) rc = SPLPAK_ERR_NDERIV;
    if (ierror) *ierror = rc;
    return rc;
}

// HOST arrays; the output is produced in slabs along the last axis so that device memory stays bounded
extern "C" int splpak_b200_eval_grid(int ndim, const real_t *axes, const int64_t *naxis, const int *nderiv,
                                     const real_t *coef, const real_t *xmin, const real_t *xmax, const int *nodes,
                                     real_t *out, int *ierror) {
    GridParams gp;
    int soft = 0;
    int rc = make_grid(ndim, xmin, xmax, nodes, nderiv, gp, &soft);
    DeviceInfo di;
    if (rc == SPLPAK_OK) rc = get_device(di);
    if (rc != SPLPAK_OK) {
        if (ierror) *ierror = rc;
        return rc;
    }
    long long na[SPL_MAXDIM] = {0, 0, 0, 0}, nsum = 0, plane = 1;
    for (int d = 0; d < gp.ndim; ++d) {
        na[d] = (long long)naxis[d];
        if (na[d] <= 0) {
            if (ierror) *ierror = soft ? SPLPAK_ERR_NDERIV : SPLPAK_OK;
            return soft ? SPLPAK_ERR_NDERIV : SPLPAK_OK;
        }
        nsum += na[d];
        if (d + 1 < gp.ndim) plane *= na[d];
    }
    long long slab = (1LL << 25) / plane;                      // ~32M outputs (256 MB) per slab
    if (slab < 1) slab = 1;
    if (slab > na[gp.ndim - 1]) slab = na[gp.ndim - 1];
    real_t *d_axes = nullptr, *d_coef = nullptr, *d_out = nullptr;
    cudaStream_t st = nullptr;
    auto cleanup = [&]() {
        if (d_axes) cudaFree(d_axes);
        if (d_coef) cudaFree(d_coef);
        if (d_out) cudaFree(d_out);
        if (st) cudaStreamDestroy(st);
    };
#define GR_TRY(expr)                                        \
    do {                                                    \
        if ((expr) != cudaSuccess) {                        \
            cudaGetLastError();                             \
            cleanup();                                      \
            if (ierror) *ierror = SPLPAK_ERR_CUDA;          \
            return SPLPAK_ERR_CUDA;                         \
        }                                                   \
    } while (0)
    GR_TRY(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    GR_TRY(cudaMalloc((void **)&d_axes, sizeof(real_t) * (size_t)nsum));
    GR_TRY(cudaMalloc((void **)&d_coef, sizeof(real_t) * (size_t)(gp.ncol + 2)));
    GR_TRY(cudaMalloc((void **)&d_out, sizeof(real_t) * (size_t)(plane * slab)));
    GR_TRY(cudaMemcpyAsync(d_axes, axes, sizeof(real_t) * (size_t)nsum, cudaMemcpyHostToDevice, st));
    GR_TRY(cudaMemcpyAsync(d_coef, coef, sizeof(real_t) * (size_t)gp.ncol, cudaMemcpyHostToDevice, st));
    const real_t *ax[SPL_MAXDIM] = {nullptr, nullptr, nullptr, nullptr};
    long long off = 0;
    for (int d = 0; d < gp.ndim; ++d) {
        ax[d] = d_axes + off;
        off += na[d];
    }
    const real_t *last0 = ax[gp.ndim - 1];
    const long long nlast = na[gp.ndim - 1];
    for (long long lo = 0; lo < nlast && rc == SPLPAK_OK; lo += slab) {
        const long long ns = (nlast - lo < slab) ? nlast - lo : slab;
        ax[gp.ndim - 1] = last0 + lo;
        na[gp.ndim - 1] = ns;
        rc = eval_grid_device_impl(gp, di, nderiv, ax, na, d_coef, d_out, st);
        if (rc != SPLPAK_OK) break;
        GR_TRY(cudaMemcpyAsync(out + lo * plane, d_out, sizeof(real_t) * (size_t)(plane * ns), cudaMemcpyDeviceToHost, st));
        GR_TRY(cudaStreamSynchronize(st));
    }
#undef GR_TRY
    cleanup();
    if (rc == SPLPAK_OK && soft) rc = SPLPAK_ERR_NDERIV;
    if (ierror) *ierror = rc;
    return rc;
}

// Grow-only device buffer: afterwards *p holds at least `need` elements (*cap of them).  The old buffer is released with
// the synchronising cudaFree: the kernels of an earlier call may still be reading it.
template <class T>
static cudaError_t grow(T **p, long long *cap, long long need) {
    if (need <= *cap) return cudaSuccess;
    if (*p) cudaFree(*p);
    *p = nullptr;
    *cap = 0;
    const cudaError_t e = cudaMalloc((void **)p, sizeof(T) * (size_t)need);
    if (e != cudaSuccess) {
        cudaGetLastError();
        *p = nullptr;
        return e;
    }
    *cap = need;
    return cudaSuccess;
}

struct EvalHostCtx {
    std::mutex mu;
    cudaStream_t st = nullptr, st2 = nullptr;
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr};
    real_t *d_coef = nullptr, *d_x[2] = {nullptr, nullptr}, *d_out[2] = {nullptr, nullptr};
    long long coef_cap = 0, x_cap[2] = {0, 0}, out_cap[2] = {0, 0};
    // host shadow of the table that d_coef holds: a call with the same coefficients (the reference's usage is
    // `evaluate` once per point in a loop, test/splpak_test.f90:72-80) skips the upload after one memcmp
    std::vector<char> coef_shadow;
    bool coef_valid = false;
};
static EvalHostCtx &eval_host_ctx(int device) {
    static EvalHostCtx ctx[64];
    return ctx[(device >= 0 && device < 64) ? device : 0];
}

// The host-array path of splpak_b200_eval / splpak_b200_eval_derivs / splpak_b200_fit_variance: ncomp outputs per query,
// launch(d_x, nc, d_coef, d_out, st) evaluates nc staged queries.  coef == NULL: the launch reads no coefficient table
// (the variance kernel reads the handle's tables), so none is uploaded and d_coef is NULL.  Returns the code of the
// call (ierror is the caller's business).
template <class Launch>
static int eval_host_staged(const GridParams &gp, const DeviceInfo &di, const real_t *x, int l1x, long long nq,
                            const real_t *coef, real_t *out, int ncomp, Launch launch) {
    // Streams, events and device staging buffers of the host path are cached per device (grow-only) and
    // the call holds the device's lock: creating and freeing ~270 MB of device memory per call made
    // identical calls take anywhere between 52 and 900 ms.
    EvalHostCtx &cx = eval_host_ctx(di.dev);
    std::lock_guard<std::mutex> lk(cx.mu);
    const long long chunk = nq < (1LL << 22) ? nq : (1LL << 22);
    const int nbuf = nq > chunk ? 2 : 1;
#define EV_TRY(expr)                                        \
    do {                                                    \
        if ((expr) != cudaSuccess) {                        \
            cudaGetLastError();                             \
            return SPLPAK_ERR_CUDA;                         \
        }                                                   \
    } while (0)
    if (!cx.st) {
        EV_TRY(cudaStreamCreateWithFlags(&cx.st, cudaStreamNonBlocking));
        EV_TRY(cudaStreamCreateWithFlags(&cx.st2, cudaStreamNonBlocking));
        for (int k = 0; k < 2; ++k) {
            EV_TRY(cudaEventCreateWithFlags(&cx.ev_in[k], cudaEventDisableTiming));
            EV_TRY(cudaEventCreateWithFlags(&cx.ev_done[k], cudaEventDisableTiming));
        }
    }
    if (coef && gp.ncol + 2 > cx.coef_cap) {
        cx.coef_valid = false;                                   // a new buffer holds no table
        EV_TRY(grow(&cx.d_coef, &cx.coef_cap, gp.ncol + 2));
    }
    for (int k = 0; k < nbuf; ++k) {
        EV_TRY(grow(&cx.d_x[k], &cx.x_cap[k], chunk * l1x));
        EV_TRY(grow(&cx.d_out[k], &cx.out_cap[k], chunk * ncomp));
    }
    cudaStream_t st = cx.st, st2 = cx.st2;
    real_t *d_coef = coef ? cx.d_coef : nullptr;
    if (coef) {
        const size_t cbytes = sizeof(real_t) * (size_t)gp.ncol;
        if (!(cx.coef_valid && cx.coef_shadow.size() == cbytes && memcmp(cx.coef_shadow.data(), coef, cbytes) == 0)) {
            cx.coef_valid = false;
            try {
                cx.coef_shadow.assign(reinterpret_cast<const char *>(coef), reinterpret_cast<const char *>(coef) + cbytes);
            } catch (...) {                                        // no C++ exception may cross the C ABI
                return SPLPAK_ERR_ALLOC;
            }
            // from the shadow, not from the caller's array: the copy may still be in flight when we return on an error path
            EV_TRY(cudaMemcpyAsync(d_coef, cx.coef_shadow.data(), cbytes, cudaMemcpyHostToDevice, st));
            EV_TRY(cudaStreamSynchronize(st));                   // pageable source: complete before the shadow can change
            cx.coef_valid = true;
        }
    }
    int rc = SPLPAK_OK;
    if (nq <= 4096) {
        // latency path (scalar splfe / splde and small batches): one stream, one synchronisation
        EV_TRY(cudaMemcpyAsync(cx.d_x[0], x, sizeof(real_t) * (size_t)nq * l1x, cudaMemcpyHostToDevice, st));
        rc = launch(cx.d_x[0], nq, d_coef, cx.d_out[0], st);
        if (rc == SPLPAK_OK) {
            EV_TRY(cudaMemcpyAsync(out, cx.d_out[0], sizeof(real_t) * (size_t)nq * ncomp, cudaMemcpyDeviceToHost, st));
            EV_TRY(cudaStreamSynchronize(st));
        }
        return rc;
    }
    // chunked, double-buffered: H2D of chunk k+1 (st2) overlaps the kernel + D2H of chunk k (st)
    int k = 0;
    for (long long q0 = 0; q0 < nq; q0 += chunk, k ^= 1) {
        const long long nc = (nq - q0 < chunk) ? nq - q0 : chunk;
        EV_TRY(cudaStreamWaitEvent(st2, cx.ev_done[k], 0));      // buffer k free again
        EV_TRY(spl_h2d(cx.d_x[k], x + q0 * (long long)l1x, sizeof(real_t) * (size_t)nc * l1x, st2, di.dev));
        EV_TRY(cudaEventRecord(cx.ev_in[k], st2));
        EV_TRY(cudaStreamWaitEvent(st, cx.ev_in[k], 0));
        rc = launch(cx.d_x[k], nc, d_coef, cx.d_out[k], st);
        if (rc != SPLPAK_OK) break;
        EV_TRY(spl_d2h(out + q0 * ncomp, cx.d_out[k], sizeof(real_t) * (size_t)nc * ncomp, st, di.dev));
        EV_TRY(cudaEventRecord(cx.ev_done[k], st));
    }
    EV_TRY(spl_d2h_flush(di.dev));
    EV_TRY(cudaStreamSynchronize(st));
    EV_TRY(cudaStreamSynchronize(st2));
#undef EV_TRY
    return rc;
}

extern "C" int splpak_b200_eval(int ndim, const real_t *x, int l1x, int64_t nq, const int *nderiv,
                                const real_t *coef, const real_t *xmin, const real_t *xmax,
                                const int *nodes, real_t *out, int *ierror) {
    GridParams gp;
    int soft = 0;
    int rc = make_grid(ndim, xmin, xmax, nodes, nderiv, gp, &soft);
    if (rc != SPLPAK_OK || nq <= 0) {
        if (ierror) *ierror = rc;
        return rc;
    }
    DeviceInfo di;
    rc = get_device(di);
    if (rc == SPLPAK_OK)
        rc = eval_host_staged(gp, di, x, l1x, nq, coef, out, 1,
                              [&](const real_t *d_x, long long n, const real_t *d_coef, real_t *d_out, cudaStream_t st) {
                                  return eval_device_impl(gp, di, nderiv, 0, d_x, l1x, n, d_coef, d_out, st);
                              });
    if (rc == SPLPAK_OK && soft) rc = SPLPAK_ERR_NDERIV;
    if (ierror) *ierror = rc;
    return rc;
}

// ------------------------------------------------------------------------------------------
// derivative sets: every partial derivative up to total order `order` of each query in one pass
// ------------------------------------------------------------------------------------------
static int derivs_ncomp(int ndim, int order) { return order == 1 ? ndim + 1 : (ndim + 1) * (ndim + 2) / 2; }

extern "C" int splpak_b200_eval_derivs_device(int ndim, const real_t *d_x, int l1x, int64_t nq, int order,
                                              const real_t *d_coef, const real_t *xmin, const real_t *xmax,
                                              const int *nodes, real_t *d_out, void *stream, int *ierror) {
    GridParams gp;
    int rc = make_grid(ndim, xmin, xmax, nodes, nullptr, gp, nullptr);
    if (rc == SPLPAK_OK && order != 1 && order != 2) rc = SPLPAK_ERR_NDERIV;
    if (rc == SPLPAK_OK && nq > 0) {
        DeviceInfo di;
        rc = get_device(di);
        if (rc == SPLPAK_OK)
            rc = eval_device_impl(gp, di, nullptr, order, d_x, l1x, nq, d_coef, d_out, (cudaStream_t)stream);
    }
    if (ierror) *ierror = rc;
    return rc;
}

extern "C" int splpak_b200_eval_derivs(int ndim, const real_t *x, int l1x, int64_t nq, int order, const real_t *coef,
                                       const real_t *xmin, const real_t *xmax, const int *nodes, real_t *out,
                                       int *ierror) {
    GridParams gp;
    int rc = make_grid(ndim, xmin, xmax, nodes, nullptr, gp, nullptr);
    if (rc == SPLPAK_OK && order != 1 && order != 2) rc = SPLPAK_ERR_NDERIV;
    if (rc == SPLPAK_OK && nq > 0) {
        DeviceInfo di;
        rc = get_device(di);
        if (rc == SPLPAK_OK)
            rc = eval_host_staged(gp, di, x, l1x, nq, coef, out, derivs_ncomp(ndim, order),
                                  [&](const real_t *d_x, long long n, const real_t *d_c, real_t *d_out, cudaStream_t st) {
                                      return eval_device_impl(gp, di, nullptr, order, d_x, l1x, n, d_c, d_out, st);
                                  });
    }
    if (ierror) *ierror = rc;
    return rc;
}

extern "C" real_t splpak_b200_splde(int ndim, const real_t *x, const int *nderiv, const real_t *coef,
                                    const real_t *xmin, const real_t *xmax, const int *nodes,
                                    int *ierror) {
    real_t out = (real_t)0;
    int nd0[SPL_MAXDIM] = {0, 0, 0, 0};
    splpak_b200_eval(ndim, x, ndim > 0 ? ndim : 1, 1, nderiv ? nderiv : nd0, coef, xmin, xmax, nodes,
                     &out, ierror);
    return out;
}

extern "C" real_t splpak_b200_splfe(int ndim, const real_t *x, const real_t *coef, const real_t *xmin,
                                    const real_t *xmax, const int *nodes, int *ierror) {
    real_t out = (real_t)0;
    splpak_b200_eval(ndim, x, ndim > 0 ? ndim : 1, 1, nullptr, coef, xmin, xmax, nodes, &out, ierror);
    return out;
}

// ------------------------------------------------------------------------------------------
// streaming fit handle
// ------------------------------------------------------------------------------------------
#define FIT_MAGIC 0x53504c42u
#define SPLPAK_REFINE_STEPS 2
#define NTIMER 7

struct splpak_b200_fit_s {
    GridParams gp_fx;             // gp with the fixed-point limb arrays: the constraint kernels ALWAYS accumulate through them
    unsigned magic;
    GridParams gp;
    DeviceInfo di;
    double xtrap;
    cudaStream_t st, st_copy, st_aux;   // st_aux: look-ahead stream of the solve
    // partial sums, one contiguous buffer (layout_partial): [S | g | cnt | totals(2) (| ywy)]
    double *d_part;
    long long n_part;
    double *d_S, *d_g, *d_cnt, *d_totals;
    // chunk scratch
    AssembleScratch sc;
    real_t *d_stage[2][3];        // host-path staging: x, y, w double-buffered
    long long stage_cap[2][3];    // reals each staging buffer holds
    cudaEvent_t ev_stage_in[2], ev_stage_free[2];
    // solve
    double *d_AB;
    long long ab_elems;
    int *d_fail;
    void *solve_cache;            // CUDA graphs of the factor / back-substitution loops (solve.cu)
    // refinement (corrected semi-normal equations): current solution, residual scratch
    double *d_coef64;             // ncol: solution of the last compute / refine step
    real_t *d_res;                // residuals y - s(x) of the chunk being re-assembled
    long long res_cap;
    double *d_dummy_tot;          // [0,1] classify's row/weight totals of refinement passes (discarded); [2] row count before the constraint rows
    int solved;                   // compute succeeded: d_coef64 is valid
    int solver;                   // SPLPAK_SOLVER_CHOLESKY (default) or SPLPAK_SOLVER_ORTHOGONAL (ortho.cuh)
    OrthoScratch *os;             // scratch of the orthogonal path (allocated on first use)
    double cond_est;              // (max L_jj / min L_jj)^2 of the last Cholesky factor: a LOWER bound of cond(G); 0: unknown
    int factor_valid;             // d_AB / the workspace behind it hold the Cholesky factor of the current G
    real_t *d_out_tmp;            // ncol reals: working-precision copy of the solution for the D2H of real32 builds
    int refining;
    int constraints_fired;        // derivative-constraint rows were added by compute
    // smoothing (penalty.cu): lambda * R is added to S by compute when lambda > 0; kept across fit_reset
    double lambda;
    int penalty;                  // SPLPAK_PENALTY_CURVATURE or SPLPAK_PENALTY_THIN_PLATE
    double *d_pen;                // 1-D penalty tables (spl_penalty_table_len doubles): ensure_penalty_tables
    // generalized cross-validation (selinv.cu): enable_gcv; kept across fit_reset
    int gcv;
    double *d_ywy;                // the last slot of the partial buffer: sum (w y)^2
    double *d_ywy_part;           // per-CTA partials of one chunk's sum
    double *d_gcv;                // score scratch: S1 = G0 + C, S2 = S1 + lambda R, g2, totals1, results, reductions,
                                  // selected-inverse scratch (allocated by the first score call)
    int s1_valid;                 // d_gcv holds S1 of the current assembly
    int sigma_valid;              // d_AB holds Sigma of the last score call
    double sigma_lambda;          // (lambda, penalty) of that score call and its {V, RSS, edf, N, ywy}
    int sigma_penalty;
    double sigma_out[5];
    // posterior variances (variance.cu): per-window tables of Sigma, built by prepare_variance, outside d_AB so that
    // they survive compute and the refinement steps
    double *d_var;                // spl_variance_table_len doubles, allocated by the first prepare_variance
    int var_valid;                // d_var holds the tables of the current assembly and (lambda, penalty)
    void *score_cache;            // solve graphs of the score calls (their own buffers: compute keeps its graphs)
    void *selinv_cache;           // graph of the selected inverse
    // timing: accumulated event pairs
    double ms[NTIMER];
    cudaEvent_t ev[12];           // 0-3 assembly, 4-5 constraints, 8-11 solve stages
    unsigned long long launches0;
    int finalized;
    int timers_pending;           // ev[0..3] hold an unharvested assembly measurement
    long long total_points;
};

static bool valid(splpak_b200_fit_t h) { return h && h->magic == FIT_MAGIC; }

static void free_handle(splpak_b200_fit_t h) {
    if (!h) return;
    if (h->d_part) cudaFree(h->d_part);
    spl_assemble_scratch_free(h->sc);
    for (int k = 0; k < 2; ++k) {
        for (int a = 0; a < 3; ++a)
            if (h->d_stage[k][a]) cudaFree(h->d_stage[k][a]);
        if (h->ev_stage_in[k]) cudaEventDestroy(h->ev_stage_in[k]);
        if (h->ev_stage_free[k]) cudaEventDestroy(h->ev_stage_free[k]);
    }
    if (h->d_AB) cudaFree(h->d_AB);
    if (h->d_fail) cudaFree(h->d_fail);
    for (int k = 0; k < 12; ++k)
        if (h->ev[k]) cudaEventDestroy(h->ev[k]);
    if (h->st) cudaStreamDestroy(h->st);
    if (h->solve_cache) spl_solve_cache_free(h->solve_cache);
    if (h->d_coef64) cudaFree(h->d_coef64);
    if (h->d_res) cudaFree(h->d_res);
    if (h->d_dummy_tot) cudaFree(h->d_dummy_tot);
    if (h->d_out_tmp) cudaFree(h->d_out_tmp);
    if (h->d_pen) cudaFree(h->d_pen);
    if (h->d_ywy_part) cudaFree(h->d_ywy_part);
    if (h->d_gcv) cudaFree(h->d_gcv);
    if (h->d_var) cudaFree(h->d_var);
    if (h->score_cache) spl_solve_cache_free(h->score_cache);
    if (h->selinv_cache) spl_selinv_cache_free(h->selinv_cache);
    if (h->os) {
        spl_ortho_free(*h->os);
        delete h->os;
        h->os = nullptr;
    }
    if (h->st_copy) cudaStreamDestroy(h->st_copy);
    if (h->st_aux) cudaStreamDestroy(h->st_aux);
    h->magic = 0;
    delete h;
}

// Pointers into the partial buffer [S | g | cnt | totals(2)], and with GCV one more slot: ywy = sum (w y)^2
static void layout_partial(splpak_b200_fit_t h, bool ywy) {
    const GridParams &gp = h->gp;
    h->d_S = h->d_part;
    h->d_g = h->d_S + gp.ncol * gp.nsten;
    h->d_cnt = h->d_g + gp.ncol;
    h->d_totals = h->d_cnt + gp.ncol;
    h->d_ywy = ywy ? h->d_totals + 2 : nullptr;
}

extern "C" int splpak_b200_fit_create(int ndim, const real_t *xmin, const real_t *xmax,
                                      const int *nodes, real_t xtrap, splpak_b200_fit_t *handle,
                                      int *ierror) {
    if (handle) *handle = nullptr;
    GridParams gp;
    int rc = make_grid(ndim, xmin, xmax, nodes, nullptr, gp, nullptr);
    if (rc != SPLPAK_OK || !handle) {
        if (rc == SPLPAK_OK) rc = SPLPAK_ERR_HANDLE;
        if (ierror) *ierror = rc;
        return rc;
    }
    DeviceInfo di;
    rc = get_device(di);
    if (rc != SPLPAK_OK) {
        if (ierror) *ierror = rc;
        return rc;
    }
    splpak_b200_fit_t h = new (std::nothrow) splpak_b200_fit_s();
    if (!h) {
        if (ierror) *ierror = SPLPAK_ERR_ALLOC;
        return SPLPAK_ERR_ALLOC;
    }
    memset(h, 0, sizeof(*h));
    h->magic = FIT_MAGIC;
    h->gp = gp;
    h->di = di;
    h->xtrap = (double)xtrap;
    h->launches0 = g_spl_launches;
    {
        const char *mode = getenv("SPLPAK_B200_FIT");
        if (mode && strcmp(mode, "orthogonal") == 0 && spl_ortho_supported(gp)) h->solver = SPLPAK_SOLVER_ORTHOGONAL;
    }
    bool ok = true;
    ok = ok && cudaStreamCreateWithFlags(&h->st, cudaStreamNonBlocking) == cudaSuccess;
    ok = ok && cudaStreamCreateWithFlags(&h->st_copy, cudaStreamNonBlocking) == cudaSuccess;
    ok = ok && cudaStreamCreateWithFlags(&h->st_aux, cudaStreamNonBlocking) == cudaSuccess;
    h->n_part = gp.ncol * gp.nsten + gp.ncol + gp.ncol + 2;
    ok = ok && cudaMalloc((void **)&h->d_part, sizeof(double) * (size_t)h->n_part) == cudaSuccess;
    ok = ok && cudaMalloc((void **)&h->d_fail, SPL_FAIL_WORDS * sizeof(int)) == cudaSuccess;   // [failure flag, grid-barrier counter of the persistent kernels, ..., flags of the data-flow factor kernel from word 32]
    ok = ok && cudaMalloc((void **)&h->d_coef64, sizeof(double) * (size_t)(gp.ncol + 2)) == cudaSuccess;
    ok = ok && cudaMalloc((void **)&h->d_dummy_tot, sizeof(double) * 4) == cudaSuccess;
    if (sizeof(real_t) != sizeof(double))
        ok = ok && cudaMalloc((void **)&h->d_out_tmp, sizeof(real_t) * (size_t)(gp.ncol + 2)) == cudaSuccess;
    for (int k = 0; k < 12 && ok; ++k) ok = cudaEventCreate(&h->ev[k]) == cudaSuccess;
    for (int k = 0; k < 2 && ok; ++k) {
        ok = ok && cudaEventCreateWithFlags(&h->ev_stage_in[k], cudaEventDisableTiming) == cudaSuccess;
        ok = ok && cudaEventCreateWithFlags(&h->ev_stage_free[k], cudaEventDisableTiming) == cudaSuccess;
    }
    if (ok) {
        layout_partial(h, false);
        ok = cudaMemsetAsync(h->d_part, 0, sizeof(double) * (size_t)h->n_part, h->st) == cudaSuccess;
    }
    if (!ok) {
        cudaGetLastError();
        free_handle(h);
        if (ierror) *ierror = SPLPAK_ERR_ALLOC;
        return SPLPAK_ERR_ALLOC;
    }
    *handle = h;
    if (ierror) *ierror = SPLPAK_OK;
    return SPLPAK_OK;
}

extern "C" int splpak_b200_fit_reset(splpak_b200_fit_t h) {
    if (!valid(h)) return SPLPAK_ERR_HANDLE;
    SPL_CUDA_TRY(cudaMemsetAsync(h->d_part, 0, sizeof(double) * (size_t)h->n_part, h->st));
    for (int k = 0; k < NTIMER; ++k) h->ms[k] = 0.0;
    h->launches0 = g_spl_launches;
    h->finalized = 0;
    h->timers_pending = 0;
    h->total_points = 0;
    h->solved = h->refining = h->constraints_fired = h->factor_valid = 0;
    h->s1_valid = h->sigma_valid = h->var_valid = 0;
    h->cond_est = 0.0;
    if (h->os) return spl_ortho_reset(h->gp, *h->os, h->st);
    return SPLPAK_OK;
}

// The assembly scratch for chunks of up to n points (assemble.cu), created by the first chunk.
static int ensure_scratch(splpak_b200_fit_t h, long long n) {
    AssembleScratch &sc = h->sc;
    if (!sc.wincount) {
        const int rc = spl_assemble_scratch_init(h->gp, sc, h->st);
        if (rc != SPLPAK_OK) return rc;
    }
    // The constraint rows always go through the fixed-point limbs (tiny work): after an all-reduce every rank holds the
    // same S, adds the same rows in an order-independent way and -- the solver being deterministic -- gets the SAME
    // coefficients, bit for bit.  With unordered FP64 atomics the replicas differed by ~eps cond(G), every rank formed the
    // residual of its shard with its own coefficients, and a multi-GPU refinement stalled at that difference.
    h->gp_fx = h->gp;
    h->gp_fx.fxS = sc.fxS;
    h->gp_fx.fxg = sc.fxg;
    h->gp_fx.fxmax = sc.fxmax;
    h->gp_fx.fxe = sc.fxe;
    h->gp_fx.fxpass = 0;
    // SPLPAK_B200_DETERMINISTIC=1: the assembly too (the assembly kernels find the limb arrays in gp)
    if (sc.deterministic) h->gp = h->gp_fx;
    return spl_assemble_scratch_reserve(h->gp, sc, n);
}

static void collect_assemble_timers(splpak_b200_fit_t h);
static void add_ms(splpak_b200_fit_t h, int slot, cudaEvent_t a, cudaEvent_t b) {
    float f = 0.f;
    if (cudaEventElapsedTime(&f, a, b) == cudaSuccess) h->ms[slot] += f;
    else cudaGetLastError();
}

#define DEVICE_CHUNK (1LL << 27)   // points per device-resident chunk (bounds the 4-byte/point permutation scratch)
#define HOST_CHUNK (1LL << 22)     // points per host->device staging chunk

static int add_device_chunk(splpak_b200_fit_t h, const real_t *d_x, int l1x, const real_t *d_y,
                            const real_t *d_w, int weighted, long long n) {
    collect_assemble_timers(h);   // the events are re-recorded below
    if (h->solver == SPLPAK_SOLVER_ORTHOGONAL) {
        if (!h->os) {
            h->os = new (std::nothrow) OrthoScratch();
            if (!h->os) return SPLPAK_ERR_ALLOC;
        }
        int ro = spl_ortho_init(h->gp, *h->os, h->st, h->di.smem_optin);
        if (ro != SPLPAK_OK) return ro;
        return spl_ortho_add_chunk(h->gp, d_x, l1x, d_y, d_w, weighted, n, h->xtrap != 0.0, *h->os, h->d_cnt, h->d_totals,
                                   h->st, h->di.nsm);
    }
    int rc = ensure_scratch(h, n);
    if (rc != SPLPAK_OK) return rc;
    h->timers_pending = 1;
    rc = spl_assemble_chunk(h->gp, d_x, l1x, d_y, d_w, weighted, n, h->xtrap != 0.0, 0, h->sc, h->d_S,
                            h->d_g, h->d_cnt, h->d_totals, h->st, h->di.nsm, h->ev);
    if (rc == SPLPAK_OK && h->gcv) {
        h->s1_valid = h->sigma_valid = h->var_valid = 0;
        rc = spl_gcv_ywy_launch(d_y, weighted ? d_w : nullptr, weighted, n, h->d_ywy_part, h->d_ywy, h->st);
    }
    return rc;
}

static void collect_assemble_timers(splpak_b200_fit_t h) {
    if (!h->timers_pending) return;
    h->timers_pending = 0;
    if (cudaEventSynchronize(h->ev[3]) != cudaSuccess) {
        cudaGetLastError();
        return;
    }
    add_ms(h, 0, h->ev[0], h->ev[1]);
    add_ms(h, 1, h->ev[1], h->ev[2]);
    add_ms(h, 2, h->ev[2], h->ev[3]);
}

// Device points in chunks of DEVICE_CHUNK; chunk(h, d_x, l1x, d_y, d_w, weighted, n) takes one chunk (add_device_chunk
// or refine_device_chunk).
template <class Chunk>
static int feed_device(splpak_b200_fit_t h, const real_t *d_x, int l1x, const real_t *d_y, const real_t *d_w,
                       int weighted, long long n, Chunk chunk) {
    for (long long i0 = 0; i0 < n; i0 += DEVICE_CHUNK) {
        const long long nc = (n - i0 < DEVICE_CHUNK) ? n - i0 : DEVICE_CHUNK;
        const int rc = chunk(h, d_x + i0 * (long long)l1x, l1x, d_y + i0, weighted ? d_w + i0 : nullptr, weighted, nc);
        if (rc != SPLPAK_OK) return rc;
    }
    return SPLPAK_OK;
}

// Host-path staging buffers, grow-only.  The x buffer is sized in REALS (chunk * l1x): a later call with
// a larger leading dimension must not reuse a buffer sized for a smaller one.
static int ensure_stage(splpak_b200_fit_t h, long long chunk, int l1x) {
    for (int k = 0; k < 2; ++k)
        for (int a = 0; a < 3; ++a)
            SPL_CUDA_TRY(grow(&h->d_stage[k][a], &h->stage_cap[k][a], a == 0 ? chunk * (long long)l1x : chunk));
    return SPLPAK_OK;
}

// Host points through the double-buffered staging buffers, HOST_CHUNK at a time: the copy stream uploads chunk k+1
// while the handle's stream works on chunk k.  chunk: as in feed_device.
template <class Chunk>
static int feed_host(splpak_b200_fit_t h, const real_t *x, int l1x, const real_t *y, const real_t *w, int weighted,
                     long long n, Chunk chunk) {
    const long long nch = n < HOST_CHUNK ? n : HOST_CHUNK;
    const int rcs = ensure_stage(h, nch, l1x);
    if (rcs != SPLPAK_OK) return rcs;
    int k = 0;
    for (long long i0 = 0; i0 < n; i0 += nch, k ^= 1) {
        const long long nc = (n - i0 < nch) ? n - i0 : nch;
        real_t *const *buf = h->d_stage[k];
        // copy stream: wait until the kernels that read staging buffer k have finished
        SPL_CUDA_TRY(cudaStreamWaitEvent(h->st_copy, h->ev_stage_free[k], 0));
        SPL_CUDA_TRY(spl_h2d(buf[0], x + i0 * (long long)l1x, sizeof(real_t) * (size_t)nc * l1x, h->st_copy, h->di.dev));
        SPL_CUDA_TRY(spl_h2d(buf[1], y + i0, sizeof(real_t) * (size_t)nc, h->st_copy, h->di.dev));
        if (weighted) SPL_CUDA_TRY(spl_h2d(buf[2], w + i0, sizeof(real_t) * (size_t)nc, h->st_copy, h->di.dev));
        SPL_CUDA_TRY(cudaEventRecord(h->ev_stage_in[k], h->st_copy));
        SPL_CUDA_TRY(cudaStreamWaitEvent(h->st, h->ev_stage_in[k], 0));
        const int rc = chunk(h, buf[0], l1x, buf[1], weighted ? buf[2] : nullptr, weighted, nc);
        if (rc != SPLPAK_OK) return rc;
        SPL_CUDA_TRY(cudaEventRecord(h->ev_stage_free[k], h->st));
    }
    return SPLPAK_OK;
}

extern "C" int splpak_b200_fit_add_points_device(splpak_b200_fit_t h, const real_t *d_x, int l1x,
                                                 const real_t *d_y, const real_t *d_w, int weighted,
                                                 int64_t n) {
    if (!valid(h) || h->finalized) return SPLPAK_ERR_HANDLE;
    if (n <= 0) return SPLPAK_OK;
    if (l1x < h->gp.ndim) return SPLPAK_ERR_HANDLE;
    if (!d_w) weighted = 0;
    const int rc = feed_device(h, d_x, l1x, d_y, d_w, weighted, n, add_device_chunk);
    if (rc != SPLPAK_OK) return rc;
    h->total_points += n;
    return SPLPAK_OK;   // asynchronous: timers are harvested by the next chunk / compute / fit_timings
}

extern "C" int splpak_b200_fit_add_points(splpak_b200_fit_t h, const real_t *x, int l1x,
                                          const real_t *y, const real_t *w, int weighted, int64_t n) {
    if (!valid(h) || h->finalized) return SPLPAK_ERR_HANDLE;
    if (n <= 0) return SPLPAK_OK;
    if (l1x < h->gp.ndim) return SPLPAK_ERR_HANDLE;
    if (!w) weighted = 0;
    const int rc = feed_host(h, x, l1x, y, w, weighted, n, add_device_chunk);
    if (rc != SPLPAK_OK) return rc;
    collect_assemble_timers(h);
    h->total_points += n;
    return SPLPAK_OK;
}

extern "C" int splpak_b200_fit_partial_buffer(splpak_b200_fit_t h, void **d_ptr, int64_t *count) {
    if (!valid(h)) return SPLPAK_ERR_HANDLE;
    h->s1_valid = h->var_valid = 0;   // the caller may write the sums through the pointer (all-reduce)
    if (d_ptr) *d_ptr = h->d_part;
    if (count) *count = h->n_part;
    return SPLPAK_OK;
}

// ---- lazily bound NCCL (libnccl.so.2), so the library has no link-time NCCL dependency ----
// A Fortran / C host has no torch.distributed to create communicators for it, so the few NCCL calls a
// one-process-per-GPU (or one-process-many-GPUs) fit needs are re-exported with plain C types.
struct Id128 {
    char b[128];
};
struct NcclApi {
    int (*AllReduce)(const void *, void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    int (*Bcast)(void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    int (*CommInitAll)(void **, int, const int *) = nullptr;
    int (*GetUniqueId)(void *) = nullptr;
    int (*CommInitRank)(void **, int, /* ncclUniqueId by value: 128 bytes */ Id128, int) = nullptr;
    int (*CommDestroy)(void *) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    bool ok = false;
};
static NcclApi &nccl_api() {
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        void *lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) return;
        api.AllReduce = (decltype(api.AllReduce))dlsym(lib, "ncclAllReduce");
        api.Bcast = (decltype(api.Bcast))dlsym(lib, "ncclBcast");
        api.CommInitAll = (decltype(api.CommInitAll))dlsym(lib, "ncclCommInitAll");
        api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(lib, "ncclGetUniqueId");
        api.CommInitRank = (decltype(api.CommInitRank))dlsym(lib, "ncclCommInitRank");
        api.CommDestroy = (decltype(api.CommDestroy))dlsym(lib, "ncclCommDestroy");
        api.GroupStart = (decltype(api.GroupStart))dlsym(lib, "ncclGroupStart");
        api.GroupEnd = (decltype(api.GroupEnd))dlsym(lib, "ncclGroupEnd");
        api.ok = api.AllReduce && api.Bcast && api.CommInitAll && api.GetUniqueId && api.CommInitRank && api.CommDestroy &&
                 api.GroupStart && api.GroupEnd;
    });
    return api;
}
extern "C" int splpak_b200_fit_allreduce(splpak_b200_fit_t h, void *nccl_comm) {
    if (!valid(h) || !nccl_comm) return SPLPAK_ERR_HANDLE;
    NcclApi &api = nccl_api();
    if (!api.ok) return SPLPAK_ERR_NCCL;
    // ncclFloat64 = 8, ncclSum = 0 (nccl.h)
    h->s1_valid = h->sigma_valid = h->var_valid = 0;
    const int rc = api.AllReduce(h->d_part, h->d_part, (size_t)h->n_part, 8, 0, nccl_comm, h->st);
    return rc == 0 ? SPLPAK_OK : SPLPAK_ERR_NCCL;
}
// refinement steps: the ncol-long right-hand side A^T r is what the ranks have to sum
extern "C" int splpak_b200_fit_allreduce_rhs(splpak_b200_fit_t h, void *nccl_comm) {
    if (!valid(h) || !nccl_comm) return SPLPAK_ERR_HANDLE;
    NcclApi &api = nccl_api();
    if (!api.ok) return SPLPAK_ERR_NCCL;
    const int rc = api.AllReduce(h->d_g, h->d_g, (size_t)h->gp.ncol, 8, 0, nccl_comm, h->st);
    return rc == 0 ? SPLPAK_OK : SPLPAK_ERR_NCCL;
}
// one process driving ndev GPUs: comms[i] belongs to device devs[i] (ncclCommInitAll)
extern "C" int splpak_b200_comm_init_all(int ndev, const int *devs, void **comms) {
    NcclApi &api = nccl_api();
    if (!api.ok || ndev < 1 || !comms) return SPLPAK_ERR_NCCL;
    return api.CommInitAll(comms, ndev, devs) == 0 ? SPLPAK_OK : SPLPAK_ERR_NCCL;
}
// one process per GPU: rank 0 calls comm_unique_id and hands the 128 bytes to the others (MPI, a file, a socket);
// then every rank calls comm_init_rank on its own device
extern "C" int splpak_b200_comm_unique_id(char id[128]) {
    NcclApi &api = nccl_api();
    if (!api.ok || !id) return SPLPAK_ERR_NCCL;
    return api.GetUniqueId(id) == 0 ? SPLPAK_OK : SPLPAK_ERR_NCCL;
}
extern "C" int splpak_b200_comm_init_rank(int nranks, int rank, const char id[128], void **comm) {
    NcclApi &api = nccl_api();
    if (!api.ok || !id || !comm) return SPLPAK_ERR_NCCL;
    Id128 v;
    memcpy(v.b, id, 128);
    return api.CommInitRank(comm, nranks, v, rank) == 0 ? SPLPAK_OK : SPLPAK_ERR_NCCL;
}
extern "C" int splpak_b200_comm_destroy(void *comm) {
    NcclApi &api = nccl_api();
    if (!api.ok || !comm) return SPLPAK_ERR_NCCL;
    return api.CommDestroy(comm) == 0 ? SPLPAK_OK : SPLPAK_ERR_NCCL;
}
// several handles of ONE process (one per device) must issue their all-reduces inside a group
extern "C" int splpak_b200_comm_group_start(void) {
    NcclApi &api = nccl_api();
    return api.ok && api.GroupStart() == 0 ? SPLPAK_OK : SPLPAK_ERR_NCCL;
}
extern "C" int splpak_b200_comm_group_end(void) {
    NcclApi &api = nccl_api();
    return api.ok && api.GroupEnd() == 0 ? SPLPAK_OK : SPLPAK_ERR_NCCL;
}

// the band matrix and the solve workspace behind it (grow-only): *band_elems doubles of band, *need in all
static int ensure_band(splpak_b200_fit_t h, long long *band_elems, long long *need) {
    *band_elems = spl_band_elems(h->gp);
    *need = *band_elems + spl_solve_workspace(h->gp);
    return grow(&h->d_AB, &h->ab_elems, *need) == cudaSuccess ? SPLPAK_OK : SPLPAK_ERR_ALLOC;
}

// The solution (ncol doubles at d_sol) to the caller's coef, on st: a device array, or a host array of real_t (REAL32:
// through d_out_tmp; d_AB keeps the factor for refinement steps).  The host copy is complete at the next synchronisation.
static int write_coef(splpak_b200_fit_t h, const double *d_sol, real_t *coef, int coef_on_device) {
    const long long n = h->gp.ncol;
    if (!coef_on_device && sizeof(real_t) == sizeof(double)) {
        SPL_CUDA_TRY(cudaMemcpyAsync(coef, d_sol, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, h->st));
        return SPLPAK_OK;
    }
    real_t *dst = coef_on_device ? coef : h->d_out_tmp;
    spl_from_double_kernel<<<spl_div_up(n, 256), 256, 0, h->st>>>(d_sol, dst, n);
    ++g_spl_launches;
    if (!coef_on_device)
        SPL_CUDA_TRY(cudaMemcpyAsync(coef, dst, sizeof(real_t) * (size_t)n, cudaMemcpyDeviceToHost, h->st));
    return SPLPAK_OK;
}

// The end of both compute paths: read back the failure flag and the row counts (one synchronisation), set solved and
// constraints_fired.  Not solved: a non-positive pivot, or fewer rows than columns (suprls error 33, :1650; not an error
// with smoothing, whose penalty makes such a fit well posed).
static int read_back_solve(splpak_b200_fit_t h) {
    cudaStream_t st = h->st;
    int fail = 0;
    double totals[2] = {0.0, 0.0}, rows_before = 0.0;
    SPL_CUDA_TRY(cudaMemcpyAsync(&fail, h->d_fail, sizeof(int), cudaMemcpyDeviceToHost, st));
    SPL_CUDA_TRY(cudaMemcpyAsync(totals, h->d_totals, sizeof(double) * 2, cudaMemcpyDeviceToHost, st));
    SPL_CUDA_TRY(cudaMemcpyAsync(&rows_before, h->d_dummy_tot + 2, sizeof(double), cudaMemcpyDeviceToHost, st));
    SPL_CUDA_TRY(cudaStreamSynchronize(st));
    h->solved = !fail && !(h->lambda == 0.0 && totals[1] < (double)h->gp.ncol);
    h->constraints_fired = (h->xtrap != 0.0) && (totals[1] > rows_before);
    return SPLPAK_OK;
}

// Householder path (ortho.cuh): constraint rows, band QR of the stacked window triangles, back-substitution
static int compute_orthogonal(splpak_b200_fit_t h, real_t *coef, int coef_on_device) {
    cudaStream_t st = h->st;
    // no point was ever added: fewer rows than columns (suprls error 33)
    if (!h->os || !h->os->ready) return SPLPAK_ERR_SOLVER;
    SPL_CUDA_TRY(cudaMemcpyAsync(h->d_dummy_tot + 2, h->d_totals + 1, sizeof(double), cudaMemcpyDeviceToDevice, st));
    SPL_CUDA_TRY(cudaMemsetAsync(h->d_fail, 0, sizeof(int), st));
    SPL_CUDA_TRY(cudaEventRecord(h->ev[8], st));
    int rc = spl_ortho_compute(h->gp, h->xtrap, *h->os, h->d_cnt, h->d_totals, h->d_fail, st, h->di.nsm);
    SPL_CUDA_TRY(cudaEventRecord(h->ev[9], st));
    if (rc != SPLPAK_OK) return rc;
    const double *d_sol = h->os->csol;
    SPL_CUDA_TRY(cudaMemcpyAsync(h->d_coef64, d_sol, sizeof(double) * (size_t)h->gp.ncol, cudaMemcpyDeviceToDevice, st));
    rc = write_coef(h, d_sol, coef, coef_on_device);
    if (rc == SPLPAK_OK) rc = read_back_solve(h);
    if (rc != SPLPAK_OK) return rc;
    add_ms(h, 5, h->ev[8], h->ev[9]);                      // reported in the "factor" slot
    return h->solved ? SPLPAK_OK : SPLPAK_ERR_SOLVER;
}

// Band Cholesky path: constraint rows and penalty into S, band expansion, factor and solve in d_AB (band_elems doubles
// of band, need in all)
static int compute_cholesky(splpak_b200_fit_t h, real_t *coef, int coef_on_device, long long band_elems,
                            long long need) {
    const GridParams &gp = h->gp;
    cudaStream_t st = h->st;
    // row count before the constraint rows, kept on the device until the one synchronisation after the solve
    SPL_CUDA_TRY(cudaMemcpyAsync(h->d_dummy_tot + 2, h->d_totals + 1, sizeof(double), cudaMemcpyDeviceToDevice, st));
    SPL_CUDA_TRY(cudaEventRecord(h->ev[4], st));
    int rc = SPLPAK_OK;
    if (h->xtrap != 0.0) {
        rc = spl_constraints_launch(h->gp_fx.fxS ? h->gp_fx : gp, h->xtrap, h->d_cnt, h->d_totals, h->d_S, h->d_totals, st, h->di.nsm);
        if (rc != SPLPAK_OK) return rc;
    }
    // smoothing: S += lambda R after the constraint rows (and the fixed-point finish of the deterministic mode); after the
    // all-reduce of a multi-GPU fit, so the penalty counts once.  Timed in the constraints slot.
    if (h->lambda > 0.0) {
        rc = spl_penalty_add_launch(gp, h->lambda, h->penalty, h->d_pen, h->d_S, st, h->di.nsm);
        if (rc != SPLPAK_OK) return rc;
    }
    SPL_CUDA_TRY(cudaEventRecord(h->ev[5], st));
    SPL_CUDA_TRY(cudaMemsetAsync(h->d_AB, 0, sizeof(double) * (size_t)need, st));
    SPL_CUDA_TRY(cudaMemsetAsync(h->d_fail, 0, sizeof(int), st));
    h->sigma_valid = 0;
    cudaEvent_t *sev = h->ev + 8;
    // the solve destroys g; the solution comes back in the workspace behind the band matrix
    double *d_sol = nullptr;
    rc = spl_solve_launch(gp, h->d_S, h->d_AB, h->d_g, h->d_AB + band_elems, &d_sol, h->d_fail, st, h->st_aux, h->di.nsm, sev,
                          &h->solve_cache);
    if (rc != SPLPAK_OK) return rc;
    SPL_CUDA_TRY(cudaMemcpyAsync(h->d_coef64, d_sol, sizeof(double) * (size_t)gp.ncol, cudaMemcpyDeviceToDevice, st));
    rc = write_coef(h, d_sol, coef, coef_on_device);
    if (rc != SPLPAK_OK) return rc;
    // smallest / largest diagonal entry of L (from the stored block inverses): a cheap LOWER bound of cond(G)
    double prange[2] = {0.0, 0.0};
    if (spl_pivot_range_launch(gp, h->d_AB + band_elems, h->d_dummy_tot, st) == SPLPAK_OK)
        SPL_CUDA_TRY(cudaMemcpyAsync(prange, h->d_dummy_tot, sizeof(double) * 2, cudaMemcpyDeviceToHost, st));
    rc = read_back_solve(h);
    if (rc != SPLPAK_OK) return rc;
    collect_assemble_timers(h);
    add_ms(h, 3, h->ev[4], h->ev[5]);
    add_ms(h, 4, sev[0], sev[1]);
    add_ms(h, 5, sev[1], sev[2]);
    add_ms(h, 6, sev[2], sev[3]);
    h->cond_est = (prange[0] > 0.0 && prange[1] > 0.0) ? (prange[1] / prange[0]) * (prange[1] / prange[0]) : 0.0;
    h->factor_valid = h->solved;
    return h->solved ? SPLPAK_OK : SPLPAK_ERR_SOLVER;
}

static int fit_compute_impl(splpak_b200_fit_t h, real_t *coef, int coef_on_device, int64_t ncf,
                            int64_t nwrk, int *ierror) {
    int rc = valid(h) ? SPLPAK_OK : SPLPAK_ERR_HANDLE;
    if (rc == SPLPAK_OK && h->gp.ncol > ncf) rc = SPLPAK_ERR_NCF;                // :751
    if (rc == SPLPAK_OK && nwrk >= 0) {
        // :757-781 and suprls :1443-1454
        const long long ncol = h->gp.ncol;
        const long long nwrk1 = (h->xtrap != 0.0) ? ncol + 1 : 1;
        const long long nwlft = (long long)nwrk - nwrk1 + 1;
        const long long nreq = ((ncol + 5) * ncol + 2) / 2;
        if (nwlft < 1) rc = SPLPAK_ERR_NWRK;
        else if (nwlft < nreq) rc = SPLPAK_ERR_SOLVER;
    }
    if (rc == SPLPAK_OK && h->finalized) rc = SPLPAK_ERR_HANDLE;
    // a failed band allocation (204) leaves the handle open; every later outcome finalizes it
    long long band_elems = 0, need = 0;
    const bool ortho = rc == SPLPAK_OK && h->solver == SPLPAK_SOLVER_ORTHOGONAL;
    if (rc == SPLPAK_OK && !ortho) rc = ensure_band(h, &band_elems, &need);
    if (rc == SPLPAK_OK) {
        h->finalized = 1;
        h->solved = 0;
        rc = ortho ? compute_orthogonal(h, coef, coef_on_device) : compute_cholesky(h, coef, coef_on_device, band_elems, need);
    }
    if (ierror) *ierror = rc;
    return rc;
}

extern "C" int splpak_b200_fit_compute(splpak_b200_fit_t h, real_t *coef, int64_t ncf, int64_t nwrk,
                                       int *ierror) {
    return fit_compute_impl(h, coef, 0, ncf, nwrk, ierror);
}
extern "C" int splpak_b200_fit_compute_device(splpak_b200_fit_t h, real_t *d_coef, int64_t ncf,
                                              int64_t nwrk, int *ierror) {
    return fit_compute_impl(h, d_coef, 1, ncf, nwrk, ierror);
}

// ------------------------------------------------------------------------------------------
// refinement: corrected semi-normal equations (Bjorck 1987).  The Cholesky solve of G c = g loses
// eps*cond(G) = eps*cond(A)^2, which is what separates it from the reference's QR (suprls) when
// derivative-constraint rows with weights ~dxin^2 sit next to O(1) data rows.  One step
//     r = b - A c  (row by row: data rows through a second pass over the points, constraint rows from the
//                   node histogram),   G dc = A^T r  (same factorisation),   c += dc
// recovers the accuracy of the orthogonal method as long as eps*cond(G) < 1.
// ------------------------------------------------------------------------------------------
extern "C" int splpak_b200_fit_refine_begin(splpak_b200_fit_t h) {
    if (!valid(h) || !h->finalized || !h->solved) return SPLPAK_ERR_HANDLE;
    if (h->solver == SPLPAK_SOLVER_ORTHOGONAL) return SPLPAK_ERR_HANDLE;   // already at cond(A): nothing to refine
    if (sizeof(real_t) != sizeof(double)) return SPLPAK_OK;            // fp32 I/O: nothing to gain
    SPL_CUDA_TRY(cudaMemsetAsync(h->d_g, 0, sizeof(double) * (size_t)h->gp.ncol, h->st));
    h->refining = 1;
    return SPLPAK_OK;
}

static int refine_device_chunk(splpak_b200_fit_t h, const real_t *d_x, int l1x, const real_t *d_y,
                               const real_t *d_w, int weighted, long long n) {
    int rc = ensure_scratch(h, n);
    if (rc != SPLPAK_OK) return rc;
    SPL_CUDA_TRY(grow(&h->d_res, &h->res_cap, n));
    // s(x_i) with the current coefficients, then r_i = y_i - s(x_i), then g += sum (w phi)(w r)
    rc = eval_device_impl(h->gp, h->di, nullptr, 0, d_x, l1x, n, reinterpret_cast<const real_t *>(h->d_coef64), h->d_res,
                          h->st);
    if (rc != SPLPAK_OK) return rc;
    spl_residual_kernel<<<spl_div_up(n, 256), 256, 0, h->st>>>(d_y, h->d_res, n);
    ++g_spl_launches;
    return spl_assemble_chunk(h->gp, d_x, l1x, h->d_res, d_w, weighted, n, 0, 1, h->sc, h->d_S, h->d_g, h->d_cnt,
                              h->d_dummy_tot, h->st, h->di.nsm, nullptr);
}

extern "C" int splpak_b200_fit_refine_add_points_device(splpak_b200_fit_t h, const real_t *d_x, int l1x,
                                                        const real_t *d_y, const real_t *d_w, int weighted,
                                                        int64_t n) {
    if (!valid(h) || !h->refining) return SPLPAK_ERR_HANDLE;
    if (sizeof(real_t) != sizeof(double) || n <= 0) return SPLPAK_OK;
    if (l1x < h->gp.ndim) return SPLPAK_ERR_HANDLE;
    if (!d_w) weighted = 0;
    return feed_device(h, d_x, l1x, d_y, d_w, weighted, n, refine_device_chunk);
}

// the staging buffers of add_points are reused (and grown if this call needs more)
extern "C" int splpak_b200_fit_refine_add_points(splpak_b200_fit_t h, const real_t *x, int l1x,
                                                 const real_t *y, const real_t *w, int weighted, int64_t n) {
    if (!valid(h) || !h->refining) return SPLPAK_ERR_HANDLE;
    if (sizeof(real_t) != sizeof(double) || n <= 0) return SPLPAK_OK;
    if (l1x < h->gp.ndim) return SPLPAK_ERR_HANDLE;
    if (!w) weighted = 0;
    return feed_host(h, x, l1x, y, w, weighted, n, refine_device_chunk);
}

// One refinement step's solve: the constraint rows' and the penalty's share of the residual, then G dc = A^T r with the
// factor compute left in d_AB, c += dc, and c to the caller.
static int refine_solve(splpak_b200_fit_t h, real_t *coef, int coef_on_device) {
    const GridParams &gp = h->gp;
    cudaStream_t st = h->st;
    if (sizeof(real_t) == sizeof(double)) {
        int rc = SPLPAK_OK;
        if (h->xtrap != 0.0) {
            rc = spl_constraints_residual_launch(h->gp_fx.fxS ? h->gp_fx : gp, h->xtrap, h->d_cnt, h->d_totals, h->d_coef64, h->d_g, st, h->di.nsm);
            if (rc != SPLPAK_OK) return rc;
        }
        if (h->lambda > 0.0) {
            // the penalty's share of the residual, -lambda R c: without it the steps would converge to the unsmoothed fit
            rc = spl_penalty_residual_launch(gp, h->lambda, h->penalty, h->d_pen, h->d_coef64, h->d_g, st, h->di.nsm);
            if (rc != SPLPAK_OK) return rc;
        }
        const long long band_elems = spl_band_elems(gp);
        const long long need = band_elems + spl_solve_workspace(gp);
        if (need > h->ab_elems) return SPLPAK_ERR_HANDLE;               // compute allocated it
        double *d_sol = nullptr;
        // G is unchanged: reuse its factor (forward + back substitution only); re-factor only where the persistent
        // substitution kernels are not available for this shape
        rc = h->factor_valid ? spl_resolve_launch(gp, h->d_AB, h->d_g, h->d_AB + band_elems, &d_sol, h->d_fail, st, h->di.nsm)
                             : SPLPAK_ERR_HANDLE;
        if (rc != SPLPAK_OK) {
            h->factor_valid = 0;
            SPL_CUDA_TRY(cudaMemsetAsync(h->d_AB, 0, sizeof(double) * (size_t)need, st));
            SPL_CUDA_TRY(cudaMemsetAsync(h->d_fail, 0, sizeof(int), st));
            rc = spl_solve_launch(gp, h->d_S, h->d_AB, h->d_g, h->d_AB + band_elems, &d_sol, h->d_fail, st, h->st_aux,
                                  h->di.nsm, nullptr, &h->solve_cache);
            if (rc != SPLPAK_OK) return rc;
            h->factor_valid = 1;
        }
        spl_axpy_kernel<<<spl_div_up(gp.ncol, 256), 256, 0, st>>>(h->d_coef64, d_sol, gp.ncol);
        ++g_spl_launches;
    }
    int fail = 0;
    SPL_CUDA_TRY(cudaMemcpyAsync(&fail, h->d_fail, sizeof(int), cudaMemcpyDeviceToHost, st));
    const int rc = write_coef(h, h->d_coef64, coef, coef_on_device);
    if (rc != SPLPAK_OK) return rc;
    SPL_CUDA_TRY(cudaStreamSynchronize(st));
    return fail ? SPLPAK_ERR_SOLVER : SPLPAK_OK;
}

static int fit_refine_compute_impl(splpak_b200_fit_t h, real_t *coef, int coef_on_device, int64_t ncf, int *ierror) {
    int rc = SPLPAK_OK;
    if (!valid(h) || !h->refining) rc = SPLPAK_ERR_HANDLE;
    else if (h->gp.ncol > ncf) rc = SPLPAK_ERR_NCF;
    if (rc == SPLPAK_OK) {
        h->refining = 0;
        rc = refine_solve(h, coef, coef_on_device);
        if (rc == SPLPAK_ERR_CUDA) h->factor_valid = 0;
    }
    if (ierror) *ierror = rc;
    return rc;
}

extern "C" int splpak_b200_fit_refine_compute(splpak_b200_fit_t h, real_t *coef, int64_t ncf, int *ierror) {
    return fit_refine_compute_impl(h, coef, 0, ncf, ierror);
}
extern "C" int splpak_b200_fit_refine_compute_device(splpak_b200_fit_t h, real_t *d_coef, int64_t ncf, int *ierror) {
    return fit_refine_compute_impl(h, d_coef, 1, ncf, ierror);
}
extern "C" int splpak_b200_fit_set_solver(splpak_b200_fit_t h, int solver) {
    if (!valid(h) || h->total_points != 0 || h->finalized) return SPLPAK_ERR_HANDLE;    // before the first point
    if (solver == SPLPAK_SOLVER_CHOLESKY) {
        h->solver = solver;
        return SPLPAK_OK;
    }
    // the penalty couples nodes across the windows of the orthogonal path: no smoothing there
    if (solver == SPLPAK_SOLVER_ORTHOGONAL && spl_ortho_supported(h->gp) && h->lambda == 0.0 && !h->gcv) {
        h->solver = solver;
        return SPLPAK_OK;
    }
    return SPLPAK_ERR_HANDLE;
}
extern "C" int splpak_b200_fit_get_solver(splpak_b200_fit_t h) { return valid(h) ? h->solver : -1; }
// The 1-D penalty tables (penalty.cu), allocated by the first call that needs them
static int ensure_penalty_tables(splpak_b200_fit_t h) {
    if (h->d_pen) return SPLPAK_OK;
    if (cudaMalloc((void **)&h->d_pen, sizeof(double) * (size_t)spl_penalty_table_len(h->gp)) != cudaSuccess) {
        cudaGetLastError();
        h->d_pen = nullptr;
        return SPLPAK_ERR_ALLOC;
    }
    return SPLPAK_OK;
}

extern "C" int splpak_b200_fit_set_smoothing(splpak_b200_fit_t h, double lambda, int penalty) {
    if (!valid(h) || h->finalized) return SPLPAK_ERR_HANDLE;
    if (!(lambda >= 0.0) || !isfinite(lambda)) return SPLPAK_ERR_HANDLE;                  // negative, NaN, inf
    if (penalty != SPLPAK_PENALTY_CURVATURE && penalty != SPLPAK_PENALTY_THIN_PLATE) return SPLPAK_ERR_HANDLE;
    if (lambda > 0.0 && h->solver == SPLPAK_SOLVER_ORTHOGONAL) return SPLPAK_ERR_HANDLE;
    if (lambda > 0.0 && ensure_penalty_tables(h) != SPLPAK_OK) return SPLPAK_ERR_ALLOC;
    if (lambda != h->lambda || (lambda > 0.0 && penalty != h->penalty)) h->var_valid = 0;   // another system
    h->lambda = lambda;
    h->penalty = penalty;
    return SPLPAK_OK;
}
// ---- generalized cross-validation (selinv.cu; DESIGN §4.12) ----
extern "C" int splpak_b200_fit_enable_gcv(splpak_b200_fit_t h) {
    if (!valid(h) || h->finalized || h->total_points != 0 || h->solver == SPLPAK_SOLVER_ORTHOGONAL)
        return SPLPAK_ERR_HANDLE;
    if (h->gcv) return SPLPAK_OK;
    // one more slot at the end of the partial buffer, so that the one all-reduce sums ywy too
    double *part = nullptr;
    if (cudaMalloc((void **)&part, sizeof(double) * (size_t)(h->n_part + 1)) != cudaSuccess ||
        (!h->d_ywy_part && cudaMalloc((void **)&h->d_ywy_part, sizeof(double) * 256) != cudaSuccess)) {
        cudaGetLastError();
        if (part) cudaFree(part);
        return SPLPAK_ERR_ALLOC;
    }
    SPL_CUDA_TRY(cudaStreamSynchronize(h->st));
    cudaFree(h->d_part);
    h->d_part = part;
    h->n_part += 1;
    layout_partial(h, true);
    SPL_CUDA_TRY(cudaMemsetAsync(h->d_part, 0, sizeof(double) * (size_t)h->n_part, h->st));
    h->gcv = 1;
    h->s1_valid = h->sigma_valid = h->var_valid = 0;
    return SPLPAK_OK;
}

// Score scratch layout: S1, S2 (ncol * nsten each), g2 (ncol), totals1 (2), results (8), reductions, selected-inverse
// scratch.  Every part starts at a multiple of 32 doubles (256 bytes): the selected inverse stages its X panel with
// 16-byte cp.async, and with ncol odd an unpadded layout would put it at an odd double offset.
struct GcvScratch {
    long long S1, S2, g2, tot1, res, red, sel, len;
};
static GcvScratch gcv_scratch_layout(const GridParams &gp) {
    auto up = [](long long v) { return (v + 31) & ~31LL; };
    const long long ns = gp.ncol * gp.nsten;
    GcvScratch L;
    L.S1 = 0;
    L.S2 = up(L.S1 + ns);
    L.g2 = up(L.S2 + ns);
    L.tot1 = up(L.g2 + gp.ncol);
    L.res = up(L.tot1 + 2);
    L.red = up(L.res + 8);
    L.sel = up(L.red + spl_gcv_part_len());
    L.len = L.sel + spl_selinv_scratch(gp);
    return L;
}

// The part both scores share: M = S1 + lambda R into S2 (S1 = G0 + C cached per assembly), then the factor and solve
// of M c = g in d_AB / the workspace behind it (band_elems doubles in), c at *d_sol.  Leaves S, g, cnt and totals as
// they are.  Clears sigma_valid: d_AB no longer holds Sigma.  SPLPAK_ERR_SOLVER for a non-positive pivot.
static int score_factor(splpak_b200_fit_t h, double lambda, int penalty, long long *band_elems_out, double **d_sol_out) {
    const GridParams &gp = h->gp;
    cudaStream_t st = h->st;
    long long band_elems = 0, need = 0;
    int rc = ensure_band(h, &band_elems, &need);
    if (rc != SPLPAK_OK) return rc;
    const GcvScratch L = gcv_scratch_layout(gp);
    if (!h->d_gcv) {
        if (cudaMalloc((void **)&h->d_gcv, sizeof(double) * (size_t)L.len) != cudaSuccess) {
            cudaGetLastError();
            h->d_gcv = nullptr;
            return SPLPAK_ERR_ALLOC;
        }
        h->s1_valid = 0;
    }
    if (lambda > 0.0 && ensure_penalty_tables(h) != SPLPAK_OK) return SPLPAK_ERR_ALLOC;
    const long long ns = gp.ncol * gp.nsten;
    double *d_S1 = h->d_gcv + L.S1, *d_S2 = h->d_gcv + L.S2, *d_g2 = h->d_gcv + L.g2, *d_tot1 = h->d_gcv + L.tot1;
    h->sigma_valid = 0;
    if (!h->s1_valid) {
        // S1 = G0 + C: the constraint rows through the fixed-point limbs, as in compute, on copies of S and the totals
        SPL_CUDA_TRY(cudaMemcpyAsync(d_S1, h->d_S, sizeof(double) * (size_t)ns, cudaMemcpyDeviceToDevice, st));
        SPL_CUDA_TRY(cudaMemcpyAsync(d_tot1, h->d_totals, sizeof(double) * 2, cudaMemcpyDeviceToDevice, st));
        if (h->xtrap != 0.0) {
            rc = spl_constraints_launch(h->gp_fx.fxS ? h->gp_fx : gp, h->xtrap, h->d_cnt, d_tot1, d_S1, d_tot1, st,
                                        h->di.nsm);
            if (rc != SPLPAK_OK) return rc;
        }
        h->s1_valid = 1;
    }
    SPL_CUDA_TRY(cudaMemcpyAsync(d_S2, d_S1, sizeof(double) * (size_t)ns, cudaMemcpyDeviceToDevice, st));
    SPL_CUDA_TRY(cudaMemcpyAsync(d_g2, h->d_g, sizeof(double) * (size_t)gp.ncol, cudaMemcpyDeviceToDevice, st));
    if (lambda > 0.0) {
        rc = spl_penalty_add_launch(gp, lambda, penalty, h->d_pen, d_S2, st, h->di.nsm);
        if (rc != SPLPAK_OK) return rc;
    }
    SPL_CUDA_TRY(cudaMemsetAsync(h->d_AB, 0, sizeof(double) * (size_t)need, st));
    SPL_CUDA_TRY(cudaMemsetAsync(h->d_fail, 0, sizeof(int), st));
    h->factor_valid = 0;
    double *d_sol = nullptr;
    rc = spl_solve_launch(gp, d_S2, h->d_AB, d_g2, h->d_AB + band_elems, &d_sol, h->d_fail, st, h->st_aux, h->di.nsm,
                          nullptr, &h->score_cache);
    if (rc != SPLPAK_OK) return rc;
    int fail = 0;
    SPL_CUDA_TRY(cudaMemcpyAsync(&fail, h->d_fail, sizeof(int), cudaMemcpyDeviceToHost, st));
    SPL_CUDA_TRY(cudaStreamSynchronize(st));
    if (fail) return SPLPAK_ERR_SOLVER;
    *band_elems_out = band_elems;
    *d_sol_out = d_sol;
    return SPLPAK_OK;
}

// {V, RSS, edf, N, ywy} of one lambda.  Leaves S, g, cnt and totals as they are; d_AB then holds Sigma.
static int gcv_score_impl(splpak_b200_fit_t h, double lambda, int penalty, double out5[5]) {
    const GridParams &gp = h->gp;
    cudaStream_t st = h->st;
    long long band_elems = 0;
    double *d_sol = nullptr;
    int rc = score_factor(h, lambda, penalty, &band_elems, &d_sol);
    if (rc != SPLPAK_OK) return rc;
    const GcvScratch L = gcv_scratch_layout(gp);
    double *d_res = h->d_gcv + L.res, *d_red = h->d_gcv + L.red, *d_sel = h->d_gcv + L.sel;
    rc = spl_selinv_launch(gp, h->d_AB, h->d_AB + band_elems, d_sel, st, &h->selinv_cache);
    if (rc != SPLPAK_OK) return rc;
    rc = spl_gcv_stencil_launch(gp, h->d_S, h->d_AB, d_sol, h->d_g, d_red, d_res, st);
    if (rc != SPLPAK_OK) return rc;
    double r[3], totals[2], ywy = 0.0;
    SPL_CUDA_TRY(cudaMemcpyAsync(r, d_res, sizeof(r), cudaMemcpyDeviceToHost, st));
    SPL_CUDA_TRY(cudaMemcpyAsync(totals, h->d_totals, sizeof(totals), cudaMemcpyDeviceToHost, st));
    SPL_CUDA_TRY(cudaMemcpyAsync(&ywy, h->d_ywy, sizeof(double), cudaMemcpyDeviceToHost, st));
    SPL_CUDA_TRY(cudaStreamSynchronize(st));
    const double edf = r[0], N = totals[1];
    // the cancellation of ywy - 2 c.g + c^T G0 c: relative error ~ eps ywy / RSS
    const double rss = ywy - 2.0 * r[2] + r[1];
    const double dof = N - edf;
    out5[0] = dof > 0.0 ? N * rss / (dof * dof) : INFINITY;
    out5[1] = rss;
    out5[2] = edf;
    out5[3] = N;
    out5[4] = ywy;
    h->sigma_valid = 1;
    h->sigma_lambda = lambda;
    h->sigma_penalty = penalty;
    memcpy(h->sigma_out, out5, sizeof(h->sigma_out));
    return SPLPAK_OK;
}

static int gcv_check(splpak_b200_fit_t h, int penalty) {
    if (!valid(h) || h->finalized || !h->gcv || h->solver == SPLPAK_SOLVER_ORTHOGONAL) return SPLPAK_ERR_HANDLE;
    if (penalty != SPLPAK_PENALTY_CURVATURE && penalty != SPLPAK_PENALTY_THIN_PLATE) return SPLPAK_ERR_HANDLE;
    return SPLPAK_OK;
}

extern "C" int splpak_b200_fit_smoothing_score(splpak_b200_fit_t h, double lambda, int penalty, double *out, int nout,
                                               int *ierror) {
    int rc = gcv_check(h, penalty);
    if (rc == SPLPAK_OK && (!(lambda >= 0.0) || !isfinite(lambda) || !out || nout < 5)) rc = SPLPAK_ERR_HANDLE;
    if (rc == SPLPAK_OK) rc = gcv_score_impl(h, lambda, penalty, out);
    if (ierror) *ierror = rc;
    return rc;
}

// ---- REML (selinv.cu: spl_reml_stencil_kernel; DESIGN §4.14) ----
// Dimension Mp of the penalty's null space: the multilinear functions (curvature), the affine ones (thin plate); 2 in 1-D.
static int penalty_null_dim(int ndim, int penalty) {
    return penalty == SPLPAK_PENALTY_CURVATURE ? 1 << ndim : ndim + 1;
}

// {V_R, D_p, log|M|, n, ywy, phi} of one lambda > 0.  Leaves S, g, cnt and totals as they are; d_AB then holds the
// factor of M, not Sigma (score_factor clears sigma_valid).
static int reml_score_impl(splpak_b200_fit_t h, double lambda, int penalty, double out6[6]) {
    const GridParams &gp = h->gp;
    cudaStream_t st = h->st;
    long long band_elems = 0;
    double *d_sol = nullptr;
    int rc = score_factor(h, lambda, penalty, &band_elems, &d_sol);
    if (rc != SPLPAK_OK) return rc;
    const GcvScratch L = gcv_scratch_layout(gp);
    double *d_res = h->d_gcv + L.res, *d_red = h->d_gcv + L.red;
    // M = S2: the band expansion and the solve only read it
    rc = spl_reml_stencil_launch(gp, h->d_gcv + L.S2, d_sol, h->d_g, h->d_AB + band_elems, d_red, d_res, st);
    if (rc != SPLPAK_OK) return rc;
    double r[3], tot1[2], ywy = 0.0;
    SPL_CUDA_TRY(cudaMemcpyAsync(r, d_res, sizeof(r), cudaMemcpyDeviceToHost, st));
    SPL_CUDA_TRY(cudaMemcpyAsync(tot1, h->d_gcv + L.tot1, sizeof(tot1), cudaMemcpyDeviceToHost, st));
    SPL_CUDA_TRY(cudaMemcpyAsync(&ywy, h->d_ywy, sizeof(double), cudaMemcpyDeviceToHost, st));
    SPL_CUDA_TRY(cudaStreamSynchronize(st));
    // n: the data rows and the constraint rows (their totals after the constraint kernel)
    const double n = tot1[1], mp = (double)penalty_null_dim(gp.ndim, penalty), p = (double)gp.ncol;
    // the quadratic form, not ywy - c.g: at the minimiser its error is second order in the solve's error
    const double dp = ywy - 2.0 * r[1] + r[0];
    const double logdet = 2.0 * r[2];
    const double dof = n - mp;
    out6[0] = dof > 0.0 ? dof * log(dp / dof) + logdet - (p - mp) * log(lambda) : INFINITY;
    out6[1] = dp;
    out6[2] = logdet;
    out6[3] = n;
    out6[4] = ywy;
    out6[5] = dof > 0.0 ? dp / dof : INFINITY;
    return SPLPAK_OK;
}

extern "C" int splpak_b200_fit_reml_score(splpak_b200_fit_t h, double lambda, int penalty, double *out, int nout,
                                          int *ierror) {
    int rc = gcv_check(h, penalty);
    if (rc == SPLPAK_OK && (!(lambda > 0.0) || !isfinite(lambda) || !out || nout < 6)) rc = SPLPAK_ERR_HANDLE;
    if (rc == SPLPAK_OK) rc = reml_score_impl(h, lambda, penalty, out);
    if (ierror) *ierror = rc;
    return rc;
}

// The search of select_smoothing and select_smoothing_reml: `score` writes nres outputs, the criterion first, and
// returns SPLPAK_ERR_SOLVER for a non-positive pivot.  rescore: when the best point was not the last one evaluated,
// score it again at the end (the GCV score leaves that point's Sigma behind).
typedef int (*ScoreFn)(splpak_b200_fit_t, double, int, double *);
static int select_smoothing_search(splpak_b200_fit_t h, int penalty, double lambda_lo, double lambda_hi, ScoreFn score,
                                   int nres, bool rescore, double *lambda, double *out, int nout, double *trace,
                                   int64_t trace_cap, int64_t *ntrace, int *ierror) {
    int rc = gcv_check(h, penalty);
    if (rc == SPLPAK_OK && (isnan(lambda_lo) || isnan(lambda_hi) || isinf(lambda_lo) || isinf(lambda_hi)))
        rc = SPLPAK_ERR_HANDLE;
    if (rc == SPLPAK_OK && lambda_lo > lambda_hi) rc = SPLPAK_ERR_HANDLE;
    if (rc == SPLPAK_OK && out && nout < nres) rc = SPLPAK_ERR_HANDLE;
    if (rc != SPLPAK_OK) {
        if (ierror) *ierror = rc;
        return rc;
    }
    if (ntrace) *ntrace = 0;
    if (!(lambda_lo > 0.0) || !(lambda_hi > 0.0)) {
        // default range rho * [1e-10, 1e4], rho = sum G0_ii / sum R_ii on the device
        double sums[2] = {0.0, 0.0};
        rc = ensure_penalty_tables(h);
        if (rc == SPLPAK_OK) rc = spl_penalty_diag_launch(h->gp, penalty, h->d_pen, h->d_S, h->d_dummy_tot, h->st);
        if (rc == SPLPAK_OK && (cudaMemcpyAsync(sums, h->d_dummy_tot, sizeof(sums), cudaMemcpyDeviceToHost, h->st) !=
                                    cudaSuccess ||
                                cudaStreamSynchronize(h->st) != cudaSuccess))
            rc = SPLPAK_ERR_CUDA;
        if (rc != SPLPAK_OK) {
            if (ierror) *ierror = rc;
            return rc;
        }
        const double rho = (sums[0] > 0.0 && sums[1] > 0.0) ? sums[0] / sums[1] : 1.0;
        lambda_lo = rho * 1e-10;
        lambda_hi = rho * 1e4;
    }
    // every evaluated point, in order; the best is the smallest V, ties to the larger lambda
    int64_t neval = 0;
    double best_t = 0.0, best_v = INFINITY, best_out[6] = {0, 0, 0, 0, 0, 0}, last_t = 0.0;
    bool any_ok = false, have_best = false;
    auto eval = [&](double t, double *v) -> int {
        const double lam = pow(10.0, t);
        last_t = t;
        double o[6];
        const int r = score(h, lam, penalty, o);
        if (r != SPLPAK_OK && r != SPLPAK_ERR_SOLVER) return r;
        if (r == SPLPAK_ERR_SOLVER) {
            o[0] = INFINITY;
            o[1] = o[2] = NAN;
        } else {
            any_ok = true;
        }
        if (trace && neval < trace_cap) {
            trace[4 * neval + 0] = lam;
            trace[4 * neval + 1] = o[0];
            trace[4 * neval + 2] = o[1];
            trace[4 * neval + 3] = o[2];
        }
        ++neval;
        if (r == SPLPAK_OK && (!have_best || o[0] < best_v || (o[0] == best_v && t > best_t))) {
            have_best = true;
            best_t = t;
            best_v = o[0];
            memcpy(best_out, o, sizeof(double) * (size_t)nres);
        }
        *v = o[0];
        return SPLPAK_OK;
    };
    const double t_lo = log10(lambda_lo), t_hi = log10(lambda_hi);
    int K = (int)ceil(2.0 * (t_hi - t_lo) - 1e-9);
    if (K < 0) K = 0;
    int kbest = 0;
    double vbest = INFINITY;
    for (int k = 0; k <= K && rc == SPLPAK_OK; ++k) {
        const double t = K > 0 ? t_lo + (t_hi - t_lo) * k / K : t_lo;
        double v = 0.0;
        rc = eval(t, &v);
        if (rc == SPLPAK_OK && (k == 0 || v <= vbest)) {
            vbest = v;
            kbest = k;
        }
    }
    if (rc == SPLPAK_OK && K > 0) {
        // golden section on the grid bracket of the best point
        auto grid_t = [&](int k) { return t_lo + (t_hi - t_lo) * k / K; };
        double a = grid_t(kbest > 0 ? kbest - 1 : 0), b = grid_t(kbest < K ? kbest + 1 : K);
        const double gr = 0.5 * (sqrt(5.0) - 1.0);
        double c = b - gr * (b - a), d = a + gr * (b - a), fc = 0.0, fd = 0.0;
        rc = eval(c, &fc);
        if (rc == SPLPAK_OK) rc = eval(d, &fd);
        while (rc == SPLPAK_OK && b - a > 0.02) {
            if (fc < fd) {
                b = d;
                d = c;
                fd = fc;
                c = b - gr * (b - a);
                rc = eval(c, &fc);
            } else {
                a = c;
                c = d;
                fc = fd;
                d = a + gr * (b - a);
                rc = eval(d, &fd);
            }
        }
    }
    if (ntrace) *ntrace = (trace && neval > trace_cap) ? trace_cap : neval;
    if (rc == SPLPAK_OK && !any_ok) rc = SPLPAK_ERR_SOLVER;
    if (rescore && rc == SPLPAK_OK && last_t != best_t) {
        // d_AB holds Sigma of the last point evaluated: score the selected lambda again, so that get_selected_inverse
        // returns the inverse of the system the handle now carries (the same inputs: the same scores, bit for bit)
        double o[5];
        rc = gcv_score_impl(h, pow(10.0, best_t), penalty, o);
    }
    if (rc == SPLPAK_OK) {
        const double lam = pow(10.0, best_t);
        rc = splpak_b200_fit_set_smoothing(h, lam, penalty);
        if (rc == SPLPAK_OK) {
            if (lambda) *lambda = lam;
            if (out) memcpy(out, best_out, sizeof(double) * (size_t)nres);
        }
    }
    if (ierror) *ierror = rc;
    return rc;
}

extern "C" int splpak_b200_fit_select_smoothing(splpak_b200_fit_t h, int penalty, double lambda_lo, double lambda_hi,
                                                double *lambda, double *out, int nout, double *trace, int64_t trace_cap,
                                                int64_t *ntrace, int *ierror) {
    return select_smoothing_search(h, penalty, lambda_lo, lambda_hi, gcv_score_impl, 5, true, lambda, out, nout, trace,
                                   trace_cap, ntrace, ierror);
}

extern "C" int splpak_b200_fit_select_smoothing_reml(splpak_b200_fit_t h, int penalty, double lambda_lo,
                                                     double lambda_hi, double *lambda, double *out, int nout,
                                                     double *trace, int64_t trace_cap, int64_t *ntrace, int *ierror) {
    return select_smoothing_search(h, penalty, lambda_lo, lambda_hi, reml_score_impl, 6, false, lambda, out, nout,
                                   trace, trace_cap, ntrace, ierror);
}

extern "C" int splpak_b200_fit_get_selected_inverse(splpak_b200_fit_t h, double *out, int64_t capacity, int64_t *count) {
    if (!valid(h) || !h->sigma_valid) return SPLPAK_ERR_HANDLE;
    const GridParams &gp = h->gp;
    const int bw = spl_half_bandwidth(gp);
    const long long lda = spl_band_lda(bw);
    const int64_t n = (int64_t)gp.ncol * (bw + 1);
    if (count) *count = n;
    if (!out) return SPLPAK_OK;
    if (capacity < n) return SPLPAK_ERR_HANDLE;
    // row i = Sigma(i..i+b, i): b + 1 consecutive doubles from AB + i (lda + 1); the entries past n are zero
    SPL_CUDA_TRY(cudaStreamSynchronize(h->st));
    SPL_CUDA_TRY(cudaMemcpy2D(out, sizeof(double) * (size_t)(bw + 1), h->d_AB, sizeof(double) * (size_t)(lda + 1),
                              sizeof(double) * (size_t)(bw + 1), (size_t)gp.ncol, cudaMemcpyDeviceToHost));
    return SPLPAK_OK;
}

// Parity-test hook of the Cholesky factor (layout: spl_solve_launch).  which = 0: columns first_col .. first_col+ncols-1
// of the band, each its lda doubles AB[j (lda+1) ..], rows j .. j+lda-1; which = 1: the block inverses L11^-1 of the
// panels those columns belong to, 64 x 64 row-major each.  *count returns the size.
extern "C" int splpak_b200_fit_get_cholesky_factor(splpak_b200_fit_t h, int which, int64_t first_col, int64_t ncols,
                                                   double *out, int64_t capacity, int64_t *count) {
    if (!valid(h) || !h->factor_valid) return SPLPAK_ERR_HANDLE;
    const GridParams &gp = h->gp;
    if (which < 0 || which > 1 || first_col < 0 || ncols < 1 || first_col + ncols > gp.ncol) return SPLPAK_ERR_HANDLE;
    const long long lda = spl_band_lda(spl_half_bandwidth(gp));
    const long long band_elems = spl_band_elems(gp);
    const long long kb0 = first_col / 64, kb1 = (first_col + ncols - 1) / 64;
    const int64_t n = which == 0 ? ncols * lda : (kb1 - kb0 + 1) * 4096;
    if (count) *count = n;
    if (!out) return SPLPAK_OK;
    if (capacity < n) return SPLPAK_ERR_HANDLE;
    SPL_CUDA_TRY(cudaStreamSynchronize(h->st));
    if (which == 0)
        SPL_CUDA_TRY(cudaMemcpy2D(out, sizeof(double) * (size_t)lda, h->d_AB + first_col * (lda + 1),
                                  sizeof(double) * (size_t)(lda + 1), sizeof(double) * (size_t)lda, (size_t)ncols,
                                  cudaMemcpyDeviceToHost));
    else
        SPL_CUDA_TRY(cudaMemcpy(out, h->d_AB + band_elems + kb0 * 4096, sizeof(double) * (size_t)n,
                                cudaMemcpyDeviceToHost));
    return SPLPAK_OK;
}

// ---- posterior variances (variance.cu; DESIGN §4.13) ----
extern "C" int splpak_b200_fit_prepare_variance(splpak_b200_fit_t h, double *out, int nout, int *ierror) {
    int rc = SPLPAK_OK;
    if (!valid(h) || h->finalized || !h->gcv || h->solver == SPLPAK_SOLVER_ORTHOGONAL || !out || nout < 6)
        rc = SPLPAK_ERR_HANDLE;
    double o[5];
    if (rc == SPLPAK_OK) {
        // Sigma of exactly the handle's current system is already in d_AB (after select_smoothing): no second score
        const bool same = h->sigma_valid && h->s1_valid && h->sigma_lambda == h->lambda &&
                          (h->lambda == 0.0 || h->sigma_penalty == h->penalty);
        h->var_valid = 0;
        if (same) memcpy(o, h->sigma_out, sizeof(o));
        else rc = gcv_score_impl(h, h->lambda, h->penalty, o);
    }
    if (rc == SPLPAK_OK && !h->d_var &&
        cudaMalloc((void **)&h->d_var, sizeof(double) * (size_t)spl_variance_table_len(h->gp)) != cudaSuccess) {
        cudaGetLastError();
        h->d_var = nullptr;
        rc = SPLPAK_ERR_ALLOC;
    }
    if (rc == SPLPAK_OK) {
        const long long lda = spl_band_lda(spl_half_bandwidth(h->gp));
        rc = spl_variance_table_launch(h->gp, h->d_AB, lda, h->d_var, h->st, h->di.nsm);
        // complete before returning: variance_device may run on any stream
        if (rc == SPLPAK_OK && cudaStreamSynchronize(h->st) != cudaSuccess) {
            cudaGetLastError();
            rc = SPLPAK_ERR_CUDA;
        }
    }
    if (rc == SPLPAK_OK) {
        h->var_valid = 1;
        const double dof = o[3] - o[2];
        memcpy(out, o, sizeof(o));
        out[5] = dof > 0.0 ? o[1] / dof : INFINITY;
    }
    if (ierror) *ierror = rc;
    return rc;
}

static int variance_check(splpak_b200_fit_t h, int l1x, const int *nderiv) {
    if (!valid(h) || !h->var_valid || l1x < h->gp.ndim) return SPLPAK_ERR_HANDLE;
    for (int d = 0; d < h->gp.ndim && nderiv; ++d)
        if (nderiv[d] < 0 || nderiv[d] > 2) return SPLPAK_ERR_NDERIV;
    return SPLPAK_OK;
}

extern "C" int splpak_b200_fit_variance_device(splpak_b200_fit_t h, const real_t *d_x, int l1x, int64_t nq,
                                               const int *nderiv, real_t *d_out, void *stream, int *ierror) {
    int rc = variance_check(h, l1x, nderiv);
    if (rc == SPLPAK_OK && nq > 0)
        rc = spl_variance_launch(h->gp, nderiv, d_x, l1x, nq, h->d_var, d_out,
                                 stream ? (cudaStream_t)stream : h->st, h->di.nsm);
    if (ierror) *ierror = rc;
    return rc;
}

extern "C" int splpak_b200_fit_variance(splpak_b200_fit_t h, const real_t *x, int l1x, int64_t nq, const int *nderiv,
                                        real_t *out, int *ierror) {
    int rc = variance_check(h, l1x, nderiv);
    if (rc == SPLPAK_OK && nq > 0)
        rc = eval_host_staged(h->gp, h->di, x, l1x, nq, nullptr, out, 1,
                              [&](const real_t *d_x, long long n, const real_t *, real_t *d_out, cudaStream_t st) {
                                  return spl_variance_launch(h->gp, nderiv, d_x, l1x, n, h->d_var, d_out, st,
                                                             h->di.nsm);
                              });
    if (ierror) *ierror = rc;
    return rc;
}

// Parity-test hook of the orthogonal path: which = 0 -> the per-window triangles [nwindows][ncw][ncw + 1] (R_w | z_w),
// which = 1 -> the band factor [ncol][bw + 2] (row i: R[i][i..i+bw], then (Q^T r)_i).  *count returns the size.
extern "C" int splpak_b200_fit_get_orthogonal_factor(splpak_b200_fit_t h, int which, double *out, int64_t capacity,
                                                     int64_t *count) {
    if (!valid(h) || !h->os || !h->os->ready) return SPLPAK_ERR_HANDLE;
    const OrthoScratch &os = *h->os;
    const int64_t n = which == 0 ? (int64_t)h->gp.nwindows * os.ncw * (os.ncw + 1) : (int64_t)h->gp.ncol * (os.bw + 2);
    if (count) *count = n;
    if (!out) return SPLPAK_OK;
    if (capacity < n) return SPLPAK_ERR_HANDLE;
    SPL_CUDA_TRY(cudaStreamSynchronize(h->st));
    SPL_CUDA_TRY(cudaMemcpy(out, which == 0 ? os.Rw : os.Rb, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost));
    return SPLPAK_OK;
}
extern "C" int splpak_b200_fit_condition_estimate(splpak_b200_fit_t h, double *cond_lower_bound) {
    if (!valid(h) || !cond_lower_bound) return SPLPAK_ERR_HANDLE;
    *cond_lower_bound = h->cond_est;
    return SPLPAK_OK;
}
extern "C" int splpak_b200_fit_constraints_fired(splpak_b200_fit_t h) {
    return valid(h) ? h->constraints_fired : 0;
}
extern "C" int splpak_b200_fit_rhs_buffer(splpak_b200_fit_t h, void **d_ptr, int64_t *count) {
    if (!valid(h)) return SPLPAK_ERR_HANDLE;
    if (d_ptr) *d_ptr = h->d_g;
    if (count) *count = h->gp.ncol;
    return SPLPAK_OK;
}

extern "C" void *splpak_b200_fit_stream(splpak_b200_fit_t h) { return valid(h) ? (void *)h->st : nullptr; }

extern "C" int splpak_b200_fit_timings(splpak_b200_fit_t h, double *ms, int n) {
    if (!valid(h)) return SPLPAK_ERR_HANDLE;
    SPL_CUDA_TRY(cudaStreamSynchronize(h->st));
    collect_assemble_timers(h);
    for (int k = 0; k < n && k < NTIMER; ++k) ms[k] = h->ms[k];
    return SPLPAK_OK;
}

extern "C" int64_t splpak_b200_fit_launch_count(splpak_b200_fit_t h) {
    return valid(h) ? (int64_t)(g_spl_launches - h->launches0) : -1;
}
extern "C" int64_t splpak_b200_total_launches(void) { return (int64_t)g_spl_launches; }

extern "C" int splpak_b200_fit_get_normal_equations(splpak_b200_fit_t h, double *S, double *g,
                                                    double *cnt, double *totals) {
    if (!valid(h)) return SPLPAK_ERR_HANDLE;
    const GridParams &gp = h->gp;
    SPL_CUDA_TRY(cudaStreamSynchronize(h->st));
    if (S) SPL_CUDA_TRY(cudaMemcpy(S, h->d_S, sizeof(double) * (size_t)(gp.ncol * gp.nsten), cudaMemcpyDeviceToHost));
    if (g) SPL_CUDA_TRY(cudaMemcpy(g, h->d_g, sizeof(double) * (size_t)gp.ncol, cudaMemcpyDeviceToHost));
    if (cnt) SPL_CUDA_TRY(cudaMemcpy(cnt, h->d_cnt, sizeof(double) * (size_t)gp.ncol, cudaMemcpyDeviceToHost));
    if (totals) SPL_CUDA_TRY(cudaMemcpy(totals, h->d_totals, sizeof(double) * 2, cudaMemcpyDeviceToHost));
    return SPLPAK_OK;
}

extern "C" int splpak_b200_fit_destroy(splpak_b200_fit_t h) {
    if (!valid(h)) return SPLPAK_ERR_HANDLE;
    cudaStreamSynchronize(h->st);
    cudaStreamSynchronize(h->st_copy);
    free_handle(h);
    return SPLPAK_OK;
}

// ------------------------------------------------------------------------------------------
// one-shot fit (splcw / splcc)
// ------------------------------------------------------------------------------------------
extern "C" int splpak_b200_splcw(int ndim, const real_t *xdata, int l1xdat, const real_t *ydata,
                                 const real_t *wdata, int64_t ndata, const real_t *xmin,
                                 const real_t *xmax, const int *nodes, real_t xtrap, real_t *coef,
                                 int64_t ncf, real_t *work, int64_t nwrk, int *ierror) {
    (void)work;
    int rc = SPLPAK_OK;
    // validation in the reference's order: 101, 102, 103 (:718-750), 104 (:751), 105 (:759), 106 (:776)
    GridParams gp;
    rc = make_grid(ndim, xmin, xmax, nodes, nullptr, gp, nullptr);
    if (rc == SPLPAK_OK && gp.ncol > ncf) rc = SPLPAK_ERR_NCF;
    if (rc == SPLPAK_OK && ndata < 1) rc = SPLPAK_ERR_NDATA;
    if (rc == SPLPAK_OK) {
        const long long nwrk1 = (xtrap != (real_t)0) ? gp.ncol + 1 : 1;
        if ((long long)nwrk - nwrk1 + 1 < 1) rc = SPLPAK_ERR_NWRK;
    }
    if (rc != SPLPAK_OK) {
        if (ierror) *ierror = rc;
        return rc;
    }
    splpak_b200_fit_t h = nullptr;
    rc = splpak_b200_fit_create(ndim, xmin, xmax, nodes, xtrap, &h, ierror);
    if (rc != SPLPAK_OK) return rc;
    const int weighted = (wdata != nullptr) && (wdata[0] >= (real_t)0);        // :796
    const int first_solver = splpak_b200_fit_get_solver(h);
    rc = splpak_b200_fit_add_points(h, xdata, l1xdat, ydata, wdata, weighted, ndata);
    if (rc == SPLPAK_OK) rc = splpak_b200_fit_compute(h, coef, ncf, nwrk, ierror);
    else if (ierror) *ierror = rc;
    // The reference reduces the rows with orthogonal transformations (suprls), i.e. at cond(A); the Cholesky path works
    // at cond(A)^2.  When the factor says that is too much -- a non-positive pivot (107 from the solver although there
    // are enough rows), or eps * (pivot-ratio bound of cond(G)) above 1e-3, where the refinement below no longer
    // contracts -- the fit is repeated with the Householder path (ortho.cuh) over the same, still valid, host arrays.
    // SPLPAK_B200_FIT=cholesky disables the fallback.
    if (first_solver == SPLPAK_SOLVER_CHOLESKY && sizeof(real_t) == sizeof(double)) {
        const char *mode = getenv("SPLPAK_B200_FIT");
        const bool allow = !(mode && strcmp(mode, "cholesky") == 0);
        double est = 0.0;
        splpak_b200_fit_condition_estimate(h, &est);
        const bool pivot_failed = (rc == SPLPAK_ERR_SOLVER) && h->total_points >= h->gp.ncol;
        const bool too_ill = (rc == SPLPAK_OK) && est * 2.220446049250313e-16 > 1e-3;
        if (allow && (pivot_failed || too_ill) && splpak_b200_fit_reset(h) == SPLPAK_OK &&
            splpak_b200_fit_set_solver(h, SPLPAK_SOLVER_ORTHOGONAL) == SPLPAK_OK) {
            rc = splpak_b200_fit_add_points(h, xdata, l1xdat, ydata, wdata, weighted, ndata);
            if (rc == SPLPAK_OK) rc = splpak_b200_fit_compute(h, coef, ncf, nwrk, ierror);
            else if (ierror) *ierror = rc;
        }
    }
    // Data-sparse constraint rows fired: their weights make cond(G) = cond(A)^2 explode, so two refinement
    // steps over the same (still valid) host arrays bring the coefficients back to the accuracy of the
    // reference's orthogonal solver (see the refinement section above).
    // Round 2 (ADVICE r1): the same when NO constraint row fired but the factor says the system is ill-conditioned
    // (clustered data, tiny weights, xtrap = 0).  Calibration on 29 1-D..3-D problems (scripts/cond_calib.py): the
    // pivot-ratio bound `est` is 0.01..0.5 x cond(G), and the unrefined coefficients differ from the reference's suprls solution by
    // <= 1e-16 x est -- so below est = 3e6 they are good to 3e-10 as they are (cfg3's dense data: est ~ 1e6).
    double est_now = 0.0;
    splpak_b200_fit_condition_estimate(h, &est_now);
    if (rc == SPLPAK_OK && sizeof(real_t) == sizeof(double) && splpak_b200_fit_get_solver(h) == SPLPAK_SOLVER_CHOLESKY &&
        (splpak_b200_fit_constraints_fired(h) || est_now > 3e6)) {
        for (int step = 0; step < SPLPAK_REFINE_STEPS && rc == SPLPAK_OK; ++step) {
            rc = splpak_b200_fit_refine_begin(h);
            if (rc == SPLPAK_OK) rc = splpak_b200_fit_refine_add_points(h, xdata, l1xdat, ydata, wdata, weighted, ndata);
            if (rc == SPLPAK_OK) rc = splpak_b200_fit_refine_compute(h, coef, ncf, ierror);
            else if (ierror) *ierror = rc;
        }
    }
    splpak_b200_fit_destroy(h);
    return rc;
}

extern "C" int splpak_b200_splcc(int ndim, const real_t *xdata, int l1xdat, const real_t *ydata,
                                 int64_t ndata, const real_t *xmin, const real_t *xmax,
                                 const int *nodes, real_t xtrap, real_t *coef, int64_t ncf,
                                 real_t *work, int64_t nwrk, int *ierror) {
    const real_t wdata[1] = {(real_t)-1.0};    // :440
    return splpak_b200_splcw(ndim, xdata, l1xdat, ydata, wdata, ndata, xmin, xmax, nodes, xtrap, coef,
                             ncf, work, nwrk, ierror);
}

extern "C" int splpak_b200_measure_peaks(double *out, int n) { return spl_measure_peaks_impl(out, n); }
