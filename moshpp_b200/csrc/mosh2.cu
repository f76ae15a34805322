// mosh2.cu -- libmosh2.so: kernels and the C-ABI declared in include/mosh2.h.
//
// One CUDA thread block per chunk of frames runs the whole Stage-II schedule of
// src/moshpp/chmosh.py:584-724 on device (mosh2_device.cuh).  Built for sm_100a only.
#include "../../include/mosh2.h"

#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "mesh_distance.cuh"
#include "mosh2_device.cuh"
#include "mosh2_host.h"

namespace {

thread_local std::string g_err;

int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CU(expr)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (expr);                                                                   \
        if (e_ != cudaSuccess) return fail(MOSH2_E_CUDA, "%s: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// ---------------------------------------------------------------------------------------------------------------------
// Caching allocator for job buffers.  A Stage-II call creates a job, runs it and destroys it; cudaMallocHost / cudaMalloc /
// cudaFree(Host) of its few tens of megabytes cost more wall clock than the solve itself and vary by 10x between calls.
// Freed blocks are therefore kept (per device, pinned host memory apart) and handed to the next job that fits; the cache
// is bounded and mosh2_release_cached_memory() empties it.
// ---------------------------------------------------------------------------------------------------------------------
class BlockCache {
  public:
    // dev >= 0: device memory of that device; dev == -1: pinned host memory
    cudaError_t get(int dev, size_t bytes, void **out) {
        const size_t need = round_up(bytes);
        {
            std::lock_guard<std::mutex> lock(mu_);
            auto &pool = pools_[dev];
            auto it = pool.lower_bound(need);
            if (it != pool.end() && it->first <= 2 * need + (1u << 20)) {
                *out = it->second;
                sizes_[*out] = it->first;
                cached_ -= it->first;
                pool.erase(it);
                return cudaSuccess;
            }
        }
        cudaError_t e = dev < 0 ? cudaMallocHost(out, need) : cudaMalloc(out, need);
        if (e != cudaSuccess) {             // make room and try once more
            release_all();
            cudaGetLastError();
            e = dev < 0 ? cudaMallocHost(out, need) : cudaMalloc(out, need);
        }
        if (e == cudaSuccess) { std::lock_guard<std::mutex> lock(mu_); sizes_[*out] = need; }
        return e;
    }
    void put(int dev, void *p) {
        if (!p) return;
        size_t bytes = 0;
        {
            std::lock_guard<std::mutex> lock(mu_);
            auto it = sizes_.find(p);
            if (it == sizes_.end()) { lock_free(dev, p); return; }
            bytes = it->second;
            sizes_.erase(it);
            if (cached_ + bytes <= kLimit) { pools_[dev].emplace(bytes, p); cached_ += bytes; return; }
        }
        lock_free(dev, p);
    }
    void release_all() {
        std::map<int, std::multimap<size_t, void *>> pools;
        { std::lock_guard<std::mutex> lock(mu_); pools.swap(pools_); cached_ = 0; }
        for (auto &dp : pools)
            for (auto &b : dp.second) lock_free(dp.first, b.second);
    }

  private:
    static constexpr size_t kLimit = size_t(1) << 30;      // cached bytes, all pools together
    static size_t round_up(size_t b) { const size_t g = b < (1u << 20) ? 4096 : (1u << 18); return (b + g - 1) / g * g; }
    static void lock_free(int dev, void *p) {
        if (dev < 0) cudaFreeHost(p);
        else { int cur = 0; cudaGetDevice(&cur); cudaSetDevice(dev); cudaFree(p); cudaSetDevice(cur); }
    }
    std::mutex mu_;
    std::map<int, std::multimap<size_t, void *>> pools_;
    std::map<void *, size_t> sizes_;
    size_t cached_ = 0;
};
BlockCache g_blocks;

constexpr size_t kMaxSmem = 227 * 1024;
#ifndef MOSH2_F32_THREADS
#define MOSH2_F32_THREADS 384      // 168 registers per thread: measured best of 256 / 320 / 384 / 512 (profiles/)
#endif
template <class real> constexpr int threads_for() { return sizeof(real) == 4 ? MOSH2_F32_THREADS : 256; }

template <class real, bool BIG>
__global__ void __launch_bounds__(threads_for<real>(), 1)
mosh2_stageii_kernel(const __grid_constant__ mosh2::Model<real> m, const __grid_constant__ mosh2::Job<real> job,
                     const __grid_constant__ mosh2::Work<real, BIG> w, const __grid_constant__ mosh2::Dims d) {
    // The workspace layout `w` was computed on the host (mosh2::carve) and arrives in the constant bank: every array
    // is shared-memory base + a parameter word.  BIG = true (f64 / oversized models): A, its factor and the Jacobian
    // tiles live in a per-CTA global workspace whose base is parked in the shared-memory header.
    if (BIG) {
        if (threadIdx.x == 0) *reinterpret_cast<char **>(mosh2::m2_smem()) = job.gws + size_t(blockIdx.x) * job.gws_stride;   // (per block, not per chunk)
        __syncthreads();
    }
    mosh2::Cta c{int(threadIdx.x), int(blockDim.x)};
    mosh2::Solver<real, BIG> s(m, job, w, d, c);
    // f32 with the workspace in shared memory: J^T J accumulates on the tensor cores (tcgen05, accumulator in
    // tensor memory); warp 0 owns the allocation
    if (w.tc) {
        if (threadIdx.x < 32) mosh2::tc::tmem_alloc(mosh2::tc::smem_u32(w.tmem_slot), mosh2::kTcCols);
        if (threadIdx.x == 32) mosh2::tc::mbar_init(mosh2::tc::smem_u32(w.mbar), 1);
        mosh2::tc::fence_before();
        __syncthreads();
        mosh2::tc::fence_after();
        s.tc_tmem = *w.tmem_slot;
        s.tc_kt = 4 * d.tmk;
    }
    s.run_chunk(job.chunk_ids ? job.chunk_ids[blockIdx.x] : int(blockIdx.x));
    if (w.tc) {
        mosh2::tc::fence_before();
        __syncthreads();
        if (threadIdx.x < 32) mosh2::tc::tmem_dealloc(s.tc_tmem, mosh2::kTcCols);
    }
}

// device copy of every model array in one precision
template <class real>
struct DevModel {
    mosh2::Model<real> m{};
    std::vector<void *> owned;
    int device = 0;
    ~DevModel() {
        for (void *p : owned) g_blocks.put(device, p);
    }
    template <class T, class U>
    int up(const U *src, size_t n, const T **dst) {
        *dst = nullptr;
        if (n == 0) {       // keep a valid pointer so kernels can form addresses
            void *p = nullptr;
            CU(g_blocks.get(device, 16, &p));
            owned.push_back(p);
            *dst = static_cast<const T *>(p);
            return 0;
        }
        std::vector<T> tmp(n);
        for (size_t i = 0; i < n; ++i) tmp[i] = static_cast<T>(src[i]);
        void *p = nullptr;
        CU(g_blocks.get(device, n * sizeof(T), &p));
        owned.push_back(p);
        CU(cudaMemcpy(p, tmp.data(), n * sizeof(T), cudaMemcpyHostToDevice));
        *dst = static_cast<const T *>(p);
        return 0;
    }
    int build(const mosh2_model_desc &d) {
        return mosh2_host::build_model(d, m, [this](const auto *src, size_t n, auto **dst) { return up(src, n, dst); });
    }
};

}  // namespace

template <class S, class D>
__global__ void convert_kernel(const S *__restrict__ src, D *__restrict__ dst, size_t n) {
    const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = D(src[i]);
}

// one packed float32 row per frame: [fullpose PF | trans 3 | dmpls nd | errs N_ERR | status | jacobian builds]
template <class real>
__global__ void pack_rows_kernel(const real *__restrict__ fullpose, const real *__restrict__ trans, const real *__restrict__ dmpls,
                                 const real *__restrict__ errs, const int *__restrict__ status, const int *__restrict__ counters,
                                 float *__restrict__ rows, int n_frames, int PF, int nd) {
    const int width = PF + 3 + nd + mosh2::N_ERR + 2;
    const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= size_t(n_frames) * width) return;
    const int f = int(i / width);
    int c = int(i - size_t(f) * width);
    float v;
    if (c < PF) v = float(fullpose[size_t(f) * PF + c]);
    else if ((c -= PF) < 3) v = float(trans[size_t(f) * 3 + c]);
    else if ((c -= 3) < nd) v = float(dmpls[size_t(f) * nd + c]);
    else if ((c -= nd) < mosh2::N_ERR) v = float(errs[size_t(f) * mosh2::N_ERR + c]);
    else if ((c -= mosh2::N_ERR) == 0) v = float(status[f]);
    else v = float(counters[4 * f + 2]);
    rows[i] = v;
}

// boundary check on the device: per chunk max |state on the last warm-up frame - emitted row of that frame| over
// (root+body pose, other pose coefficients, translation, linear coefficients); one warp per chunk
template <class real>
__global__ void boundary_delta_kernel(const real *__restrict__ warm_x, const int *__restrict__ warm_f, const real *__restrict__ pose,
                                      const real *__restrict__ trans, const real *__restrict__ dmpls, float *__restrict__ out,
                                      int n_chunks, int PR, int nd, int body) {
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (c >= n_chunks) return;
    const int f = warm_f[c];
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (f >= 0) {
        const real *x = warm_x + size_t(c) * (3 + PR + nd);
        for (int i = lane; i < PR; i += 32) {
            const float d = fabsf(float(x[3 + i] - pose[size_t(f) * PR + i]));
            if (i < body) v[0] = fmaxf(v[0], d); else v[1] = fmaxf(v[1], d);
        }
        if (lane < 3) v[2] = fabsf(float(x[lane] - trans[size_t(f) * 3 + lane]));
        for (int i = lane; i < nd; i += 32) v[3] = fmaxf(v[3], fabsf(float(x[3 + PR + i] - dmpls[size_t(f) * nd + i])));
    }
    for (int q = 0; q < 4; ++q) {
        for (int o = 16; o > 0; o >>= 1) v[q] = fmaxf(v[q], __shfl_xor_sync(0xffffffffu, v[q], o));
        if (lane == 0) out[4 * c + q] = v[q];
    }
}

// Mocap input adapter on the device (tools/mocap_interface.py:186,223-225,254-279; chmosh.py:582-594): from the raw marker
// table of a capture file [file frame][file column][xyz] (file units, float64) to the job's observations [frame][marker][xyz]
// (metres, compute precision) and visibility.  A sample is missing when a coordinate is NaN or all three are exactly zero
// (:277); such samples -- and markers whose label the file does not have (col < 0) -- are invisible and stored as zero.
template <class real>
__global__ void gather_markers_kernel(const double *__restrict__ raw, int n_cols, const int *__restrict__ col_of_marker, int M,
                                      int n_frames, int frame_step, double unit_per_metre, const double *__restrict__ rot,
                                      real *__restrict__ obs, uint8_t *__restrict__ vis) {
    const size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= size_t(n_frames) * M) return;
    const int f = int(i / M), mk = int(i - size_t(f) * M), col = col_of_marker[mk];
    double x = 0, y = 0, z = 0;
    bool ok = false;
    if (col >= 0) {
        const double *p = raw + (size_t(f) * frame_step * n_cols + col) * 3;
        x = p[0]; y = p[1]; z = p[2];
        ok = !(isnan(x) || isnan(y) || isnan(z)) && !(x == 0.0 && y == 0.0 && z == 0.0);
    }
    if (!ok) { x = y = z = 0; }
    else {
        if (rot) {      // mocap.rotate: the points turned by Rz Ry Rx before the unit conversion (mocap_interface.py:218-221)
            const double rx = rot[0] * x + rot[1] * y + rot[2] * z, ry = rot[3] * x + rot[4] * y + rot[5] * z, rz = rot[6] * x + rot[7] * y + rot[8] * z;
            x = rx; y = ry; z = rz;
        }
        x = x / unit_per_metre; y = y / unit_per_metre; z = z / unit_per_metre;
    }
    obs[3 * i] = real(x); obs[3 * i + 1] = real(y); obs[3 * i + 2] = real(z);
    vis[i] = ok ? 1 : 0;
}

// Host copy of a model description: the caller's buffers need not outlive mosh2_model_create, and the device copy of a
// precision is only built when the first job of that precision is created.
struct HostDesc {
    mosh2_model_desc d{};
    std::vector<int32_t> parents, w_joint, free1, free2, prior_ids, jangles_ids;
    std::vector<double> jangles_signs;
    std::vector<double> hand_comps, hands_mean, v0, sd, pd, w_val, j0, jd, coefs, prior_means, prior_Q, prior_neglogw;
    template <class T> static const T *keep(std::vector<T> &dst, const T *src, size_t n) {
        dst.assign(src, src + n);
        if (dst.empty()) dst.resize(1);
        return dst.data();
    }
    void copy_from(const mosh2_model_desc &s) {
        d = s;
        const size_t nJ = s.n_joints, S = size_t(3) * s.n_markers, nd = s.n_dmpl, K = s.prior_k, D = s.prior_d;
        d.parents = keep(parents, s.parents, nJ);
        d.w_joint = keep(w_joint, s.w_joint, S * s.kw);
        d.free1 = keep(free1, s.free1, s.n_free1);
        d.free2 = keep(free2, s.free2, s.n_free2);
        if (s.prior_ids) d.prior_ids = keep(prior_ids, s.prior_ids, D);
        if (s.n_jangles > 0) { d.jangles_ids = keep(jangles_ids, s.jangles_ids, s.n_jangles); d.jangles_signs = keep(jangles_signs, s.jangles_signs, s.n_jangles); }
        d.hand_comps = keep(hand_comps, s.hand_comps, size_t(s.n_hand_red) * s.n_hand_full);
        d.hands_mean = keep(hands_mean, s.hands_mean, s.n_hand_full);
        d.v0 = keep(v0, s.v0, S * 3);
        d.sd = keep(sd, s.sd, S * 3 * nd);
        d.pd = keep(pd, s.pd, (nJ - 1) * 3 * S * 9);
        d.w_val = keep(w_val, s.w_val, S * s.kw);
        d.j0 = keep(j0, s.j0, nJ * 3);
        d.jd = keep(jd, s.jd, nJ * 3 * nd);
        d.coefs = keep(coefs, s.coefs, size_t(s.n_markers) * 3);
        d.prior_means = keep(prior_means, s.prior_means, K * D);
        d.prior_Q = keep(prior_Q, s.prior_Q, K * D * D);
        d.prior_neglogw = keep(prior_neglogw, s.prior_neglogw, K);
    }
};

struct mosh2_model {
    int device = 0;
    HostDesc host;
    DevModel<float> f32;
    DevModel<double> f64;
    bool have_f32 = false, have_f64 = false;
    int n_joints = 0, n_markers = 0, p_red = 0, n_dmpl = 0;
    int ensure(int precision) {
        if (precision == MOSH2_F64) {
            if (!have_f64) { f64.device = device; const int rc = f64.build(host.d); if (rc) return rc; have_f64 = true; }
        } else if (!have_f32) { f32.device = device; const int rc = f32.build(host.d); if (rc) return rc; have_f32 = true; }
        return 0;
    }
};

struct mosh2_job {
    mosh2_model *model = nullptr;
    int precision = MOSH2_F32;
    int n_frames = 0, n_chunks = 1;
    int *d_chunk_tab = nullptr, *d_chunk_ids = nullptr, *d_warm_f = nullptr;
    void *d_warm_x = nullptr;
    float *d_delta = nullptr;
    std::vector<int> tab, tab0;       // host copy of the chunk table (tab0: as created; repairs edit tab)
    bool tab_dirty = false;
    double merge_tol = 0;
    int launch_blocks = 0;            // blocks of the next launch (all chunks, or the subset in d_chunk_ids)
    bool subset = false;
    mosh2::Options opt{};
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_in = nullptr;
    size_t esz = 4;                 // element size of the compute type
    size_t smem = 0, gws_stride = 0;
    int big_in_global = 0;
    // device buffers
    void *d_obs = nullptr, *d_out = nullptr, *d_gws = nullptr;
    uint8_t *d_vis = nullptr;
    int *d_status = nullptr, *d_counters = nullptr, *d_totals = nullptr;
    long long *d_prof = nullptr;
    // pinned staging
    void *h_obs = nullptr, *h_out = nullptr;
    uint8_t *h_vis = nullptr;
    void *d_lin = nullptr;                       // linearise mode: states in, normal equations / Jacobian rows / residuals out
    size_t lin_bytes = 0;
    int lin_mode = 0, lin_step = 1;
    void *h_raw = nullptr, *d_raw = nullptr;     // raw marker table of mosh2_job_upload_markers (pinned staging, device copy)
    int *d_cols = nullptr;
    size_t raw_bytes = 0;
    int *h_status = nullptr, *h_counters = nullptr;
    size_t n_obs = 0, n_out = 0;
    size_t o_fullpose = 0, o_pose = 0, o_trans = 0, o_dmpls = 0, o_mk = 0, o_errs = 0;   // element offsets in d_out
};

namespace {

template <class real, bool BIG>
cudaError_t launch_kernel(mosh2_job *j, const mosh2::Model<real> &m, const mosh2::Job<real> &job, int threads) {
    const mosh2::Dims d = mosh2::make_dims(m);
    mosh2::Work<real, BIG> w{};
    mosh2::Arena S{mosh2::kSmemHeader}, G{0};
    mosh2::carve<real, BIG>(w, d, m, S, G);
    w.tc = (w.tc_ok && threads >= 128) ? 1 : 0;
    const cudaError_t e = cudaFuncSetAttribute(mosh2_stageii_kernel<real, BIG>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(j->smem));
    if (e != cudaSuccess) return e;
    mosh2_stageii_kernel<real, BIG><<<j->launch_blocks, threads, j->smem, j->stream>>>(m, job, w, d);
    return cudaGetLastError();
}

template <class real>
int launch(mosh2_job *j, const mosh2::Model<real> &m) {
    mosh2::Job<real> job{};
    job.n_frames = j->n_frames; job.n_chunks = j->n_chunks;
    job.chunk_tab = j->d_chunk_tab; job.chunk_ids = j->subset ? j->d_chunk_ids : nullptr;
    job.warm_x = static_cast<real *>(j->d_warm_x); job.warm_f = j->d_warm_f; job.merge_tol = j->merge_tol;
    job.obs = static_cast<const real *>(j->d_obs);
    job.vis = j->d_vis;
    real *out = static_cast<real *>(j->d_out);
    job.fullpose = out + j->o_fullpose; job.pose = out + j->o_pose; job.trans = out + j->o_trans;
    job.dmpls = j->model->n_dmpl ? out + j->o_dmpls : nullptr;
    job.markers_sim = out + j->o_mk; job.errs = out + j->o_errs;
    job.status = j->d_status; job.counters = j->d_counters; job.totals = j->d_totals; job.prof = j->d_prof;
    job.gws = static_cast<char *>(j->d_gws); job.gws_stride = j->gws_stride;
    job.lin_mode = j->lin_mode; job.lin_step = j->lin_step;
    if (j->lin_mode) {      // layout of d_lin (reals): x [F][NX] | A [F][n][n] | g [F][n] | J [F][3M][n] | r [F][3M] | vp [F][9M]
        const size_t F = j->n_frames, M = j->model->n_markers, NX = 3 + j->model->p_red + j->model->n_dmpl;
        const size_t n = j->lin_step == 2 ? m.n2 : m.n1;
        real *p = static_cast<real *>(j->d_lin);
        job.lin_x = p; p += F * NX;
        job.lin_A = p; p += F * n * n;
        job.lin_g = p; p += F * n;
        job.lin_J = p; p += F * 3 * M * n;
        job.lin_r = p; p += F * 3 * M;
        job.lin_vp = p;
    }
    job.opt = j->opt;
    int threads = threads_for<real>();
    if (const char *e = getenv("MOSH2_DEV_THREADS")) {      // development aid: any multiple of 32 from 128 up to the launch bound
        const int t = atoi(e);
        if (t >= 128 && t <= threads && t % 32 == 0) threads = t;
    }
    CU(cudaEventRecord(j->ev0, j->stream));
    if (j->big_in_global) CU((launch_kernel<real, true>(j, m, job, threads)));
    else CU((launch_kernel<real, false>(j, m, job, threads)));
    CU(cudaGetLastError());
    CU(cudaEventRecord(j->ev1, j->stream));
    return 0;
}

template <class real>
void plan_workspace(mosh2::Model<real> &m, size_t *smem, size_t *gws, int *big) {
    // preference order: 20-marker tiles, then 10-marker tiles, while the workspace fits the shared-memory budget; the
    // f64 / oversized case moves A, its factor and the Jacobian tiles to a per-CTA global workspace
    const int tries[3][2] = {{20, 0}, {10, 0}, {10, 1}};   // markers per tile (a warp owns ten), big
    const char *dev_tile = getenv("MOSH2_DEV_TILE");      // development aid: 10 = skip the 20-marker tile
    const bool dev_big = getenv("MOSH2_DEV_BIG") != nullptr;   // development aid: force the global-workspace layout
    for (int pass = dev_big ? 2 : ((dev_tile && atoi(dev_tile) == 10) ? 1 : 0); pass < 3; ++pass) {
        m.tile_markers = tries[pass][0];
        m.dev_no_tc = getenv("MOSH2_DEV_NO_TC") ? 1 : 0;      // development aid: J^T J on the CUDA cores
        const bool in_global = tries[pass][1] != 0;
        const mosh2::Dims d = mosh2::make_dims(m);
        mosh2::Arena S{mosh2::kSmemHeader}, G{0};
        if (in_global) { mosh2::Work<real, true> w{}; mosh2::carve<real, true>(w, d, m, S, G); }
        else { mosh2::Work<real, false> w{}; mosh2::carve<real, false>(w, d, m, S, G); }
        *big = in_global ? 1 : 0;
        *smem = (S.off + 15) & ~size_t(15);
        *gws = (G.off + 255) & ~size_t(255);
        if (S.off <= kMaxSmem) return;
    }
}

}  // namespace

extern "C" {

int mosh2_version(void) { return MOSH2_VERSION; }
const char *mosh2_last_error(void) { return g_err.c_str(); }

int mosh2_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

void mosh2_default_options(mosh2_options *o) {
    if (!o) return;
    // support_data/conf/moshpp_conf.yaml:99,118-125; chmosh.py:460,653,671,697
    o->wt_data = 400; o->wt_poseB = 1.6; o->wt_poseH = 1.0; o->wt_velo = 2.5; o->wt_dmpl = 1.0;
    o->wt_annealing = 2.5; o->wt_extrap_dmpl = 6.0; o->num_train_markers = 46;
    o->delta_0 = 0.5; o->e3_first = 1e-3; o->e3 = 1e-2; o->maxiter = 100;
    o->optimize_fingers = 0; o->optimize_dynamics = 0;
    o->wt_poseF = 1.0; o->wt_expr = 1.0; o->optimize_face = 0;
}

int mosh2_model_create(const mosh2_model_desc *d, int device, mosh2_model **out) {
    if (!d || !out) return fail(MOSH2_E_INVALID, "null argument");
    *out = nullptr;
    if (d->n_joints < 1 || d->n_markers < 1 || d->kw < 1 || d->kw > 8 || d->n_free1 < 1 || d->n_free2 < d->n_free1)
        return fail(MOSH2_E_INVALID, "inconsistent model sizes");
    if (d->n_expr < 0 || d->n_expr > d->n_dmpl || d->face_lo < 0 || d->face_hi < d->face_lo || d->face_hi > d->p_red)
        return fail(MOSH2_E_INVALID, "inconsistent face description: n_expr=%d of %d linear coefficients, jaw ids [%d, %d)", d->n_expr,
                    d->n_dmpl, d->face_lo, d->face_hi);
    if (d->n_joints > 254) return fail(MOSH2_E_TOO_LARGE, "%d joints (max 254)", d->n_joints);
    if (d->n_jangles < 0 || d->n_jangles > mosh2::kMaxJangles || (d->n_jangles > 0 && (!d->jangles_ids || !d->jangles_signs)))
        return fail(MOSH2_E_INVALID, "joint-angle term: %d entries (max %d)", d->n_jangles, mosh2::kMaxJangles);
    for (int i = 0; i < d->n_jangles; ++i)
        if (d->jangles_ids[i] < 0 || d->jangles_ids[i] >= d->p_red) return fail(MOSH2_E_INVALID, "joint-angle entry %d refers to pose id %d of %d", i, d->jangles_ids[i], d->p_red);
    for (int i = 0; i < d->prior_d; ++i) {
        const int id = d->prior_ids ? d->prior_ids[i] : d->prior_off + i;
        if (id < 0 || id >= d->p_red) return fail(MOSH2_E_INVALID, "prior dimension %d refers to pose id %d of %d", i, id, d->p_red);
    }
    for (int j = 0; j < d->n_joints; ++j) {
        int depth = 1;
        for (int a = d->parents[j]; a >= 0; a = d->parents[a]) {
            if (a >= d->n_joints || ++depth > d->n_joints) return fail(MOSH2_E_INVALID, "parents[] is not a forest (joint %d)", j);
        }
        if (depth > mosh2::kMaxDepth) return fail(MOSH2_E_TOO_LARGE, "kinematic chain of joint %d is %d levels deep (max %d)", j, depth, mosh2::kMaxDepth);
    }
    if (d->body_dof + d->n_hand_full != 3 * d->n_joints || d->body_dof + d->n_hand_red != d->p_red)
        return fail(MOSH2_E_INVALID, "pose layout mismatch: body_dof=%d hand_full=%d hand_red=%d p_red=%d joints=%d",
                    d->body_dof, d->n_hand_full, d->n_hand_red, d->p_red, d->n_joints);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(MOSH2_E_NO_DEVICE, "no CUDA device: libmosh2 has no CPU path");
    }
    if (device < 0 || device >= ndev) return fail(MOSH2_E_INVALID, "device %d out of range (%d devices)", device, ndev);
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return fail(MOSH2_E_NO_DEVICE, "device %d is sm_%d%d; libmosh2 is built for sm_100a only", device, prop.major, prop.minor);
    mosh2_model *m = new (std::nothrow) mosh2_model;
    if (!m) return fail(MOSH2_E_INVALID, "out of host memory");
    m->device = device; m->n_joints = d->n_joints; m->n_markers = d->n_markers; m->p_red = d->p_red; m->n_dmpl = d->n_dmpl;
    m->host.copy_from(*d);      // the device copy of a precision is built by the first job that asks for it
    *out = m;
    return 0;
}

void mosh2_model_destroy(mosh2_model *m) {
    if (!m) return;
    cudaSetDevice(m->device);
    delete m;
}

int mosh2_job_create(mosh2_model *m, const mosh2_options *opt, int32_t n_frames, const mosh2_schedule *sched,
                     int32_t precision, mosh2_job **out) {
    return mosh2_job_create_batch(m, opt, 1, &n_frames, sched, precision, out);
}

int mosh2_job_create_batch(mosh2_model *m, const mosh2_options *opt, int32_t n_seq, const int32_t *frame_counts,
                           const mosh2_schedule *sched, int32_t precision, mosh2_job **out) {
    if (!m || !opt || !out || n_seq < 1 || !frame_counts) return fail(MOSH2_E_INVALID, "bad argument");
    long long total = 0;
    for (int q = 0; q < n_seq; ++q) {
        if (frame_counts[q] < 1) return fail(MOSH2_E_INVALID, "sequence %d has %d frames", q, frame_counts[q]);
        total += frame_counts[q];
    }
    if (total > 0x3fffffff) return fail(MOSH2_E_TOO_LARGE, "%lld frames in one job", total);
    const int32_t n_frames = int32_t(total);
    if (precision != MOSH2_F32 && precision != MOSH2_F64) return fail(MOSH2_E_INVALID, "precision must be MOSH2_F32 or MOSH2_F64");
    *out = nullptr;
    CU(cudaSetDevice(m->device));
    if (const int rc = m->ensure(precision)) return rc;
    mosh2_job *j = new (std::nothrow) mosh2_job;
    if (!j) return fail(MOSH2_E_INVALID, "out of host memory");
    j->model = m; j->precision = precision; j->n_frames = n_frames;
    const mosh2_host::Schedule s = mosh2_host::schedule(sched);
    j->tab = mosh2_host::chunk_table(frame_counts, n_seq, s.chunk_len, s.warmup, s.warm_full, s.first_extra);
    j->tab0 = j->tab;
    const std::vector<int> &tab = j->tab;
    j->n_chunks = int(tab.size() / mosh2::kChunkRec);
    j->launch_blocks = j->n_chunks;
    j->esz = precision == MOSH2_F64 ? 8 : 4;
    j->opt = mosh2_host::options(opt);

    size_t gws = 0;
    if (precision == MOSH2_F64) plan_workspace(m->f64.m, &j->smem, &gws, &j->big_in_global);
    else plan_workspace(m->f32.m, &j->smem, &gws, &j->big_in_global);
    if (j->smem > kMaxSmem) {
        const size_t need = j->smem;
        delete j;
        return fail(MOSH2_E_TOO_LARGE, "model needs %zu bytes of shared memory per block (max %zu)", need, kMaxSmem);
    }
    j->gws_stride = j->big_in_global ? gws : 0;

    const size_t F = n_frames, M = m->n_markers, PF = size_t(3) * m->n_joints, PR = m->p_red, nd = m->n_dmpl;
    j->n_obs = F * M * 3;
    size_t off = 0;
    j->o_fullpose = off; off += F * PF;
    j->o_pose = off; off += F * PR;
    j->o_trans = off; off += F * 3;
    j->o_dmpls = off; off += F * nd;
    j->o_mk = off; off += F * M * 3;
    j->o_errs = off; off += F * mosh2::N_ERR;
    j->n_out = off;
    cudaError_t e = cudaSuccess;
    auto chk = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
    chk(cudaStreamCreateWithFlags(&j->stream, cudaStreamNonBlocking));
    chk(cudaEventCreate(&j->ev0));
    chk(cudaEventCreate(&j->ev1));
    chk(cudaEventCreateWithFlags(&j->ev_in, cudaEventDisableTiming));
    chk(g_blocks.get(m->device, j->n_obs * j->esz, reinterpret_cast<void **>(&j->d_obs)));
    chk(g_blocks.get(m->device, j->n_out * j->esz, reinterpret_cast<void **>(&j->d_out)));
    chk(g_blocks.get(m->device, F * M, reinterpret_cast<void **>(&j->d_vis)));
    chk(g_blocks.get(m->device, F * sizeof(int), reinterpret_cast<void **>(&j->d_status)));
    chk(g_blocks.get(m->device, F * 4 * sizeof(int), reinterpret_cast<void **>(&j->d_counters)));
    chk(g_blocks.get(m->device, 8 * sizeof(int), reinterpret_cast<void **>(&j->d_totals)));
    chk(g_blocks.get(m->device, tab.size() * sizeof(int), reinterpret_cast<void **>(&j->d_chunk_tab)));
    chk(g_blocks.get(m->device, size_t(j->n_chunks) * sizeof(int), reinterpret_cast<void **>(&j->d_chunk_ids)));
    chk(g_blocks.get(m->device, size_t(j->n_chunks) * sizeof(int), reinterpret_cast<void **>(&j->d_warm_f)));
    chk(g_blocks.get(m->device, size_t(j->n_chunks) * 4 * sizeof(float), reinterpret_cast<void **>(&j->d_delta)));
    chk(g_blocks.get(m->device, size_t(j->n_chunks) * (3 + m->p_red + m->n_dmpl) * j->esz, reinterpret_cast<void **>(&j->d_warm_x)));
    if (e == cudaSuccess) chk(cudaMemcpy(j->d_chunk_tab, tab.data(), tab.size() * sizeof(int), cudaMemcpyHostToDevice));
    chk(g_blocks.get(m->device, 32 * sizeof(long long), reinterpret_cast<void **>(&j->d_prof)));
    if (j->gws_stride) chk(g_blocks.get(m->device, j->gws_stride * j->n_chunks, reinterpret_cast<void **>(&j->d_gws)));
    chk(g_blocks.get(-1, j->n_obs * j->esz, reinterpret_cast<void **>(&j->h_obs)));
    chk(g_blocks.get(-1, j->n_out * j->esz, reinterpret_cast<void **>(&j->h_out)));
    chk(g_blocks.get(-1, F * M, reinterpret_cast<void **>(&j->h_vis)));
    chk(g_blocks.get(-1, F * sizeof(int), reinterpret_cast<void **>(&j->h_status)));
    chk(g_blocks.get(-1, F * 4 * sizeof(int), reinterpret_cast<void **>(&j->h_counters)));
    if (e != cudaSuccess) {
        mosh2_job_destroy(j);
        return fail(MOSH2_E_CUDA, "job allocation failed: %s", cudaGetErrorString(e));
    }
    *out = j;
    return 0;
}

int mosh2_job_upload(mosh2_job *j, const double *obs, const uint8_t *vis) {
    if (!j || !obs || !vis) return fail(MOSH2_E_INVALID, "null argument");
    CU(cudaSetDevice(j->model->device));
    if (j->precision == MOSH2_F64) memcpy(j->h_obs, obs, j->n_obs * sizeof(double));
    else {
        float *h = static_cast<float *>(j->h_obs);
        for (size_t i = 0; i < j->n_obs; ++i) h[i] = float(obs[i]);
    }
    const size_t nv = size_t(j->n_frames) * j->model->n_markers;
    memcpy(j->h_vis, vis, nv);
    CU(cudaMemcpyAsync(j->d_obs, j->h_obs, j->n_obs * j->esz, cudaMemcpyHostToDevice, j->stream));
    CU(cudaMemcpyAsync(j->d_vis, j->h_vis, nv, cudaMemcpyHostToDevice, j->stream));
    return 0;
}

int mosh2_job_upload_markers(mosh2_job *j, const double *markers, int32_t n_file_frames, int32_t n_cols, const int32_t *col_of_marker,
                             int32_t frame_start, int32_t frame_step, double unit_per_metre, const double *rot3x3) {
    if (!j || !markers || !col_of_marker) return fail(MOSH2_E_INVALID, "null argument");
    const int F = j->n_frames, M = j->model->n_markers;
    if (n_cols < 1 || frame_step < 1 || frame_start < 0 || !(unit_per_metre > 0) ||
        size_t(frame_start) + size_t(F - 1) * frame_step >= size_t(n_file_frames))
        return fail(MOSH2_E_INVALID, "frames %d + k*%d (k < %d) do not fit a file of %d frames", frame_start, frame_step, F, n_file_frames);
    for (int i = 0; i < M; ++i)
        if (col_of_marker[i] >= n_cols) return fail(MOSH2_E_INVALID, "marker %d: column %d of %d", i, col_of_marker[i], n_cols);
    CU(cudaSetDevice(j->model->device));
    const int dv = j->model->device;
    // the rows [frame_start, last used frame] of the table, whole (all columns), through pinned staging
    const size_t rows = size_t(F - 1) * frame_step + 1, bytes = rows * n_cols * 3 * sizeof(double), extra = 16 * sizeof(double);
    if (bytes + extra > j->raw_bytes) {
        g_blocks.put(-1, j->h_raw); g_blocks.put(dv, j->d_raw);
        j->h_raw = j->d_raw = nullptr; j->raw_bytes = 0;
        CU(g_blocks.get(-1, bytes + extra, &j->h_raw));
        CU(g_blocks.get(dv, bytes + extra, &j->d_raw));
        j->raw_bytes = bytes + extra;
    }
    if (!j->d_cols) CU(g_blocks.get(dv, size_t(M) * sizeof(int), reinterpret_cast<void **>(&j->d_cols)));
    CU(cudaStreamSynchronize(j->stream));          // (the staging buffers may still feed an earlier upload)
    char *h = static_cast<char *>(j->h_raw);
    memcpy(h, markers + size_t(frame_start) * n_cols * 3, bytes);
    if (rot3x3) memcpy(h + bytes, rot3x3, 9 * sizeof(double));
    CU(cudaMemcpyAsync(j->d_raw, h, bytes + (rot3x3 ? 9 * sizeof(double) : 0), cudaMemcpyHostToDevice, j->stream));
    CU(cudaMemcpyAsync(j->d_cols, col_of_marker, size_t(M) * sizeof(int), cudaMemcpyHostToDevice, j->stream));
    const size_t n = size_t(F) * M;
    const int blocks = int((n + 255) / 256);
    const double *d_raw = static_cast<const double *>(j->d_raw);
    const double *d_rot = rot3x3 ? reinterpret_cast<const double *>(static_cast<const char *>(j->d_raw) + bytes) : nullptr;
    if (j->precision == MOSH2_F64)
        gather_markers_kernel<double><<<blocks, 256, 0, j->stream>>>(d_raw, n_cols, j->d_cols, M, F, frame_step, unit_per_metre, d_rot, static_cast<double *>(j->d_obs), j->d_vis);
    else
        gather_markers_kernel<float><<<blocks, 256, 0, j->stream>>>(d_raw, n_cols, j->d_cols, M, F, frame_step, unit_per_metre, d_rot, static_cast<float *>(j->d_obs), j->d_vis);
    CU(cudaGetLastError());
    return 0;
}

int mosh2_job_linearize(mosh2_job *j, const mosh2_options *opt, int32_t step, int32_t build, const double *x, const mosh2_lin_out *out) {
    if (!j || !x || !out || (step != 1 && step != 2)) return fail(MOSH2_E_INVALID, "bad argument");
    if (j->precision != MOSH2_F64) return fail(MOSH2_E_INVALID, "mosh2_job_linearize needs a float64 job");
    if (j->n_chunks < j->n_frames) return fail(MOSH2_E_INVALID, "mosh2_job_linearize needs a job of one-frame chunks (chunk_len = 1)");
    CU(cudaSetDevice(j->model->device));
    const mosh2::Model<double> &m = j->model->f64.m;
    const size_t F = j->n_frames, M = j->model->n_markers, NX = 3 + j->model->p_red + j->model->n_dmpl;
    const size_t n = step == 2 ? m.n2 : m.n1, n2 = m.n2 > m.n1 ? m.n2 : m.n1;
    const size_t words = F * (NX + n2 * n2 + n2 + 3 * M * n2 + 3 * M + 9 * M);
    if (words * sizeof(double) > j->lin_bytes) {
        g_blocks.put(j->model->device, j->d_lin);
        j->d_lin = nullptr; j->lin_bytes = 0;
        CU(g_blocks.get(j->model->device, words * sizeof(double), &j->d_lin));
        j->lin_bytes = words * sizeof(double);
    }
    if (opt) {      // the weights of this evaluation (Stage I anneals them between minimisations)
        mosh2::Options &o = j->opt;
        o.wt_data = opt->wt_data; o.wt_poseB = opt->wt_poseB; o.wt_poseH = opt->wt_poseH; o.optimize_fingers = opt->optimize_fingers;
    }
    CU(cudaMemcpyAsync(j->d_lin, x, F * NX * sizeof(double), cudaMemcpyHostToDevice, j->stream));
    CU(cudaMemsetAsync(j->d_out, 0, j->n_out * j->esz, j->stream));
    j->lin_mode = build ? 2 : 1;
    j->lin_step = step;
    j->subset = false;
    j->launch_blocks = int(F);
    const int rc = launch<double>(j, m);
    j->lin_mode = 0;
    j->launch_blocks = j->n_chunks;
    if (rc) return rc;
    const double *p = static_cast<const double *>(j->d_lin) + F * NX;
    const double *dA = p; p += F * n * n;
    const double *dg = p; p += F * n;
    const double *dJ = p; p += F * 3 * M * n;
    const double *dr = p; p += F * 3 * M;
    const double *dvp = p;
    const double *dout = static_cast<const double *>(j->d_out);
    auto back = [&](double *dst, const double *src, size_t cnt) { return dst ? cudaMemcpyAsync(dst, src, cnt * sizeof(double), cudaMemcpyDeviceToHost, j->stream) : cudaSuccess; };
    if (build) { CU(back(out->A, dA, F * n * n)); CU(back(out->g, dg, F * n)); CU(back(out->J, dJ, F * 3 * M * n)); }
    CU(back(out->r, dr, F * 3 * M));
    CU(back(out->vp, dvp, F * 9 * M));
    CU(back(out->errs, dout + j->o_errs, F * mosh2::N_ERR));
    CU(back(out->markers_sim, dout + j->o_mk, F * 3 * M));
    CU(cudaStreamSynchronize(j->stream));
    return 0;
}

int mosh2_job_launch(mosh2_job *j) {
    if (!j) return fail(MOSH2_E_INVALID, "null job");
    CU(cudaSetDevice(j->model->device));
    CU(cudaMemsetAsync(j->d_out, 0, j->n_out * j->esz, j->stream));
    CU(cudaMemsetAsync(j->d_status, 0, size_t(j->n_frames) * sizeof(int), j->stream));
    CU(cudaMemsetAsync(j->d_counters, 0, size_t(j->n_frames) * 4 * sizeof(int), j->stream));
    CU(cudaMemsetAsync(j->d_totals, 0, 8 * sizeof(int), j->stream));
    CU(cudaMemsetAsync(j->d_prof, 0, 32 * sizeof(long long), j->stream));
    if (j->tab_dirty) {               // a full launch runs the schedule the job was created with
        j->tab = j->tab0;
        CU(cudaMemcpyAsync(j->d_chunk_tab, j->tab.data(), j->tab.size() * sizeof(int), cudaMemcpyHostToDevice, j->stream));
        j->tab_dirty = false;
    }
    j->subset = false;
    j->launch_blocks = j->n_chunks;
    if (j->precision == MOSH2_F64) return launch<double>(j, j->model->f64.m);
    return launch<float>(j, j->model->f32.m);
}

int mosh2_job_relaunch_chunks(mosh2_job *j, int32_t n, const int32_t *chunk_ids, int32_t chunk_warmup, int32_t warmup_full, double merge_tol) {
    if (!j || n < 1 || !chunk_ids || !(merge_tol >= 0)) return fail(MOSH2_E_INVALID, "bad argument");
    j->merge_tol = merge_tol;
    CU(cudaSetDevice(j->model->device));
    const int wf = chunk_warmup < 0 ? 0 : mosh2_host::clamp_warm_full(chunk_warmup, warmup_full);
    for (int k = 0; k < n; ++k) {
        const int c = chunk_ids[k];
        if (c < 0 || c >= j->n_chunks) return fail(MOSH2_E_INVALID, "chunk %d out of range (%d chunks)", c, j->n_chunks);
        j->tab[size_t(c) * mosh2::kChunkRec + 3] = chunk_warmup;
        j->tab[size_t(c) * mosh2::kChunkRec + 4] = wf;
    }
    j->tab_dirty = true;
    CU(cudaStreamSynchronize(j->stream));
    CU(cudaMemcpy(j->d_chunk_tab, j->tab.data(), j->tab.size() * sizeof(int), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(j->d_chunk_ids, chunk_ids, size_t(n) * sizeof(int), cudaMemcpyHostToDevice));
    // the rows of the frames these chunks emit are rewritten by the kernel; everything else of the last launch stays
    j->subset = true;
    j->launch_blocks = n;
    if (j->precision == MOSH2_F64) return launch<double>(j, j->model->f64.m);
    return launch<float>(j, j->model->f32.m);
}

int mosh2_job_boundary_deltas(mosh2_job *j, int32_t body_ids, float *out) {
    if (!j || !out || body_ids < 0) return fail(MOSH2_E_INVALID, "bad argument");
    CU(cudaSetDevice(j->model->device));
    const int PR = j->model->p_red, nd = j->model->n_dmpl, blocks = (j->n_chunks + 3) / 4;
    if (j->precision == MOSH2_F64) {
        const double *o = static_cast<const double *>(j->d_out);
        boundary_delta_kernel<double><<<blocks, 128, 0, j->stream>>>(static_cast<const double *>(j->d_warm_x), j->d_warm_f, o + j->o_pose, o + j->o_trans, o + j->o_dmpls, j->d_delta, j->n_chunks, PR, nd, body_ids);
    } else {
        const float *o = static_cast<const float *>(j->d_out);
        boundary_delta_kernel<float><<<blocks, 128, 0, j->stream>>>(static_cast<const float *>(j->d_warm_x), j->d_warm_f, o + j->o_pose, o + j->o_trans, o + j->o_dmpls, j->d_delta, j->n_chunks, PR, nd, body_ids);
    }
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(out, j->d_delta, size_t(j->n_chunks) * 4 * sizeof(float), cudaMemcpyDeviceToHost, j->stream));
    CU(cudaStreamSynchronize(j->stream));
    return 0;
}

int mosh2_job_warm_states(mosh2_job *j, double *x, int32_t *frames) {
    if (!j || !x || !frames) return fail(MOSH2_E_INVALID, "null argument");
    CU(cudaSetDevice(j->model->device));
    CU(cudaStreamSynchronize(j->stream));
    const size_t nx = size_t(3) + j->model->p_red + j->model->n_dmpl, n = size_t(j->n_chunks) * nx;
    CU(cudaMemcpy(frames, j->d_warm_f, size_t(j->n_chunks) * sizeof(int), cudaMemcpyDeviceToHost));
    if (j->precision == MOSH2_F64) CU(cudaMemcpy(x, j->d_warm_x, n * sizeof(double), cudaMemcpyDeviceToHost));
    else {
        std::vector<float> tmp(n);
        CU(cudaMemcpy(tmp.data(), j->d_warm_x, n * sizeof(float), cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < n; ++i) x[i] = double(tmp[i]);
    }
    return 0;
}

int mosh2_job_sync(mosh2_job *j) {
    if (!j) return fail(MOSH2_E_INVALID, "null job");
    CU(cudaSetDevice(j->model->device));
    CU(cudaStreamSynchronize(j->stream));
    return 0;
}

int mosh2_job_kernel_ms(mosh2_job *j, float *ms) {
    if (!j || !ms) return fail(MOSH2_E_INVALID, "null argument");
    CU(cudaSetDevice(j->model->device));
    CU(cudaEventElapsedTime(ms, j->ev0, j->ev1));
    return 0;
}

void mosh2_release_cached_memory(void) { g_blocks.release_all(); }

int mosh2_job_span_ms(mosh2_job *first, mosh2_job *last, float *ms) {
    if (!first || !last || !ms) return fail(MOSH2_E_INVALID, "null argument");
    if (first->model->device != last->model->device) return fail(MOSH2_E_INVALID, "jobs live on different devices");
    CU(cudaSetDevice(first->model->device));
    CU(cudaEventElapsedTime(ms, first->ev0, last->ev1));
    return 0;
}

int mosh2_job_num_chunks(mosh2_job *j) { return j ? j->n_chunks : 0; }

int mosh2_job_chunk_ranges(mosh2_job *j, int32_t *out) {
    if (!j || !out) return fail(MOSH2_E_INVALID, "null argument");
    for (int c = 0; c < j->n_chunks; ++c) {
        out[2 * c] = j->tab0[size_t(c) * mosh2::kChunkRec];
        out[2 * c + 1] = j->tab0[size_t(c) * mosh2::kChunkRec + 1];
    }
    return 0;
}

// development builds (-DMOSH2_PROFILE) only: 32 phase clock sums of the last launch; not part of mosh2.h
int mosh2_dev_phase_clocks(mosh2_job *j, long long *out32) {
    if (!j || !out32) return fail(MOSH2_E_INVALID, "null argument");
    CU(cudaSetDevice(j->model->device));
    CU(cudaStreamSynchronize(j->stream));
    CU(cudaMemcpy(out32, j->d_prof, 32 * sizeof(long long), cudaMemcpyDeviceToHost));
    return 0;
}

int mosh2_job_totals(mosh2_job *j, int32_t *out8) {
    if (!j || !out8) return fail(MOSH2_E_INVALID, "null argument");
    CU(cudaSetDevice(j->model->device));
    CU(cudaStreamSynchronize(j->stream));
    CU(cudaMemcpy(out8, j->d_totals, 8 * sizeof(int), cudaMemcpyDeviceToHost));
    return 0;
}

int mosh2_job_upload_device(mosh2_job *j, const void *d_obs, int32_t obs_f64, const uint8_t *d_vis, void *producer_stream) {
    if (!j) return fail(MOSH2_E_INVALID, "null argument");
    return mosh2_job_upload_device_range(j, 0, j->n_frames, d_obs, obs_f64, d_vis, producer_stream);
}

int mosh2_job_upload_device_range(mosh2_job *j, int32_t frame0, int32_t nfr, const void *d_obs, int32_t obs_f64,
                                  const uint8_t *d_vis, void *producer_stream) {
    if (!j || !d_obs || !d_vis) return fail(MOSH2_E_INVALID, "null argument");
    if (frame0 < 0 || nfr < 1 || frame0 + nfr > j->n_frames) return fail(MOSH2_E_INVALID, "frame range [%d, %d) outside the job's %d frames", frame0, frame0 + nfr, j->n_frames);
    CU(cudaSetDevice(j->model->device));
    CU(cudaEventRecord(j->ev_in, static_cast<cudaStream_t>(producer_stream)));
    CU(cudaStreamWaitEvent(j->stream, j->ev_in, 0));
    const size_t M = j->model->n_markers, n = size_t(nfr) * M * 3, nv = size_t(nfr) * M, o0 = size_t(frame0) * M * 3;
    const bool dst64 = j->precision == MOSH2_F64;
    char *dst = static_cast<char *>(j->d_obs) + o0 * j->esz;
    if (dst64 == (obs_f64 != 0)) CU(cudaMemcpyAsync(dst, d_obs, n * j->esz, cudaMemcpyDeviceToDevice, j->stream));
    else {
        const int blocks = int((n + 255) / 256);
        if (dst64) convert_kernel<float, double><<<blocks, 256, 0, j->stream>>>(static_cast<const float *>(d_obs), reinterpret_cast<double *>(dst), n);
        else convert_kernel<double, float><<<blocks, 256, 0, j->stream>>>(static_cast<const double *>(d_obs), reinterpret_cast<float *>(dst), n);
        CU(cudaGetLastError());
    }
    CU(cudaMemcpyAsync(j->d_vis + size_t(frame0) * M, d_vis, nv, cudaMemcpyDeviceToDevice, j->stream));
    return 0;
}

int mosh2_job_row_width(mosh2_job *j) { return j ? 3 * j->model->n_joints + 3 + j->model->n_dmpl + mosh2::N_ERR + 2 : 0; }

int mosh2_job_download_device(mosh2_job *j, float *d_rows) {
    if (!j || !d_rows) return fail(MOSH2_E_INVALID, "null argument");
    CU(cudaSetDevice(j->model->device));
    const int PF = 3 * j->model->n_joints, nd = j->model->n_dmpl, width = mosh2_job_row_width(j);
    const size_t total = size_t(j->n_frames) * width;
    const int blocks = int((total + 255) / 256);
    if (j->precision == MOSH2_F64) {
        const double *o = static_cast<const double *>(j->d_out);
        pack_rows_kernel<double><<<blocks, 256, 0, j->stream>>>(o + j->o_fullpose, o + j->o_trans, o + j->o_dmpls, o + j->o_errs, j->d_status, j->d_counters, d_rows, j->n_frames, PF, nd);
    } else {
        const float *o = static_cast<const float *>(j->d_out);
        pack_rows_kernel<float><<<blocks, 256, 0, j->stream>>>(o + j->o_fullpose, o + j->o_trans, o + j->o_dmpls, o + j->o_errs, j->d_status, j->d_counters, d_rows, j->n_frames, PF, nd);
    }
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(j->stream));
    return 0;
}

int mosh2_job_download(mosh2_job *j, const mosh2_result *r) {
    if (!j || !r) return fail(MOSH2_E_INVALID, "null argument");
    CU(cudaSetDevice(j->model->device));
    const size_t F = j->n_frames;
    CU(cudaMemcpyAsync(j->h_out, j->d_out, j->n_out * j->esz, cudaMemcpyDeviceToHost, j->stream));
    CU(cudaMemcpyAsync(j->h_status, j->d_status, F * sizeof(int), cudaMemcpyDeviceToHost, j->stream));
    CU(cudaMemcpyAsync(j->h_counters, j->d_counters, F * 4 * sizeof(int), cudaMemcpyDeviceToHost, j->stream));
    CU(cudaStreamSynchronize(j->stream));
    const size_t M = j->model->n_markers, PF = size_t(3) * j->model->n_joints, PR = j->model->p_red, nd = j->model->n_dmpl;
    auto conv = [&](double *dst, size_t off, size_t n) {
        if (!dst) return;
        if (j->precision == MOSH2_F64) memcpy(dst, static_cast<double *>(j->h_out) + off, n * sizeof(double));
        else {
            const float *s = static_cast<float *>(j->h_out) + off;
            for (size_t i = 0; i < n; ++i) dst[i] = double(s[i]);
        }
    };
    conv(r->fullpose, j->o_fullpose, F * PF);
    conv(r->pose, j->o_pose, F * PR);
    conv(r->trans, j->o_trans, F * 3);
    if (nd) conv(r->dmpls, j->o_dmpls, F * nd);
    conv(r->markers_sim, j->o_mk, F * M * 3);
    conv(r->errs, j->o_errs, F * mosh2::N_ERR);
    if (r->status) memcpy(r->status, j->h_status, F * sizeof(int));
    if (r->counters) memcpy(r->counters, j->h_counters, F * 4 * sizeof(int));
    return 0;
}

void mosh2_job_destroy(mosh2_job *j) {
    if (!j) return;
    cudaSetDevice(j->model->device);
    if (j->stream) cudaStreamSynchronize(j->stream);
    const int dv = j->model->device;
    for (void *p : {static_cast<void *>(j->d_chunk_tab), static_cast<void *>(j->d_chunk_ids), static_cast<void *>(j->d_warm_f), j->d_warm_x,
                    static_cast<void *>(j->d_delta), j->d_obs, j->d_out, static_cast<void *>(j->d_vis), static_cast<void *>(j->d_status),
                    static_cast<void *>(j->d_counters), static_cast<void *>(j->d_totals), static_cast<void *>(j->d_prof), j->d_gws})
        g_blocks.put(dv, p);
    g_blocks.put(dv, j->d_raw);
    g_blocks.put(dv, j->d_lin);
    g_blocks.put(dv, j->d_cols);
    for (void *p : {j->h_obs, j->h_out, static_cast<void *>(j->h_vis), static_cast<void *>(j->h_status), static_cast<void *>(j->h_counters), j->h_raw})
        g_blocks.put(-1, p);
    if (j->ev0) cudaEventDestroy(j->ev0);
    if (j->ev1) cudaEventDestroy(j->ev1);
    if (j->ev_in) cudaEventDestroy(j->ev_in);
    if (j->stream) cudaStreamDestroy(j->stream);
    delete j;
}

int mosh2_solve(mosh2_model *m, const mosh2_options *opt, int32_t n_frames, const double *obs, const uint8_t *vis,
                const mosh2_schedule *sched, int32_t precision, const mosh2_result *res) {
    mosh2_job *j = nullptr;
    int rc = mosh2_job_create(m, opt, n_frames, sched, precision, &j);
    if (rc) return rc;
    rc = mosh2_job_upload(j, obs, vis);
    if (!rc) rc = mosh2_job_launch(j);
    if (!rc) rc = mosh2_job_download(j, res);
    mosh2_job_destroy(j);
    return rc;
}

// ---- Stage-I surface term: point-to-triangle-mesh distance with derivatives (mesh_distance.cuh) ----------------------------
int mosh2_mesh_distance(int32_t device, int32_t kind, double sigma, int32_t n_samples, const double *samples, int32_t n_verts,
                        const double *verts, int32_t n_tris, const int32_t *tris, const int32_t *nearest_tri,
                        const int32_t *nearest_part, const mosh2_mesh_distance_out *out, float *kernel_ms) {
    if (!samples || !verts || !tris || !out || n_samples < 1 || n_verts < 1 || n_tris < 1 || kind < 0 || kind > 2)
        return fail(MOSH2_E_INVALID, "bad argument");
    if ((nearest_tri == nullptr) != (nearest_part == nullptr)) return fail(MOSH2_E_INVALID, "nearest_tri and nearest_part go together");
    if (n_tris >= (1 << 28)) return fail(MOSH2_E_TOO_LARGE, "%d triangles (the search packs the index into 29 bits)", n_tris);
    for (int64_t i = 0; i < int64_t(3) * n_tris; ++i)
        if (tris[i] < 0 || tris[i] >= n_verts) return fail(MOSH2_E_INVALID, "triangle %lld refers to vertex %d of %d", (long long)(i / 3), tris[i], n_verts);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return fail(MOSH2_E_NO_DEVICE, "no CUDA device: libmosh2 has no CPU path"); }
    if (device < 0 || device >= ndev) return fail(MOSH2_E_INVALID, "device %d out of range (%d devices)", device, ndev);
    CU(cudaSetDevice(device));
    const size_t S = n_samples, V = n_verts, T = n_tris;
    struct Buf { int dev; void *p = nullptr; ~Buf() { g_blocks.put(dev, p); } };
    Buf d_s{device}, d_sf{device}, d_v{device}, d_f{device}, d_soup{device}, d_best{device}, d_tri{device}, d_part{device}, d_val{device}, d_ds{device}, d_dt{device};
    CU(g_blocks.get(device, S * 3 * sizeof(double), &d_s.p));
    CU(g_blocks.get(device, S * 3 * sizeof(float), &d_sf.p));
    CU(g_blocks.get(device, V * 3 * sizeof(double), &d_v.p));
    CU(g_blocks.get(device, T * 3 * sizeof(int), &d_f.p));
    CU(g_blocks.get(device, T * mosh2_md::kSoupFloats * sizeof(float), &d_soup.p));
    CU(g_blocks.get(device, S * sizeof(unsigned long long), &d_best.p));
    CU(g_blocks.get(device, S * sizeof(int), &d_tri.p));
    CU(g_blocks.get(device, S * sizeof(int), &d_part.p));
    CU(g_blocks.get(device, S * sizeof(double), &d_val.p));
    CU(g_blocks.get(device, S * 3 * sizeof(double), &d_ds.p));
    CU(g_blocks.get(device, S * 9 * sizeof(double), &d_dt.p));
    cudaStream_t st = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    CU(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    auto cleanup = [&]() { cudaEventDestroy(e0); cudaEventDestroy(e1); cudaStreamDestroy(st); };
    cudaError_t e = cudaSuccess;
    auto chk = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
    chk(cudaMemcpyAsync(d_s.p, samples, S * 3 * sizeof(double), cudaMemcpyHostToDevice, st));
    chk(cudaMemcpyAsync(d_v.p, verts, V * 3 * sizeof(double), cudaMemcpyHostToDevice, st));
    chk(cudaMemcpyAsync(d_f.p, tris, T * 3 * sizeof(int), cudaMemcpyHostToDevice, st));
    chk(cudaEventRecord(e0, st));
    if (nearest_tri) {
        chk(cudaMemcpyAsync(d_tri.p, nearest_tri, S * sizeof(int), cudaMemcpyHostToDevice, st));
        chk(cudaMemcpyAsync(d_part.p, nearest_part, S * sizeof(int), cudaMemcpyHostToDevice, st));
    } else {
        convert_kernel<double, float><<<int((S * 3 + 255) / 256), 256, 0, st>>>(static_cast<const double *>(d_s.p), static_cast<float *>(d_sf.p), S * 3);
        mosh2_md::soup_kernel<<<int((T + 255) / 256), 256, 0, st>>>(static_cast<const double *>(d_v.p), static_cast<const int *>(d_f.p), int(T), static_cast<float *>(d_soup.p));
        chk(cudaMemsetAsync(d_best.p, 0xff, S * sizeof(unsigned long long), st));
        // triangle ranges: enough blocks to fill the GPU (148 SMs, several blocks each), whole tiles per block
        const int sblocks = int((S + mosh2_md::kSamplesPerBlock - 1) / mosh2_md::kSamplesPerBlock);
        int splits = (4 * 148 + sblocks - 1) / sblocks;
        const int tiles = int((T + mosh2_md::kTileTris - 1) / mosh2_md::kTileTris);
        if (splits > tiles) splits = tiles;
        if (splits < 1) splits = 1;
        const int per = ((tiles + splits - 1) / splits) * mosh2_md::kTileTris;
        splits = int((T + per - 1) / per);
        mosh2_md::nearest_kernel<<<dim3(sblocks, splits), mosh2_md::kSamplesPerBlock, 0, st>>>(
            static_cast<const float *>(d_sf.p), int(S), static_cast<const float *>(d_soup.p), int(T), per, static_cast<unsigned long long *>(d_best.p));
        mosh2_md::unpack_kernel<<<int((S + 255) / 256), 256, 0, st>>>(static_cast<const unsigned long long *>(d_best.p), int(S), static_cast<int *>(d_tri.p), static_cast<int *>(d_part.p));
    }
    mosh2_md::evaluate_kernel<<<int((S + 127) / 128), 128, 0, st>>>(kind, sigma, static_cast<const double *>(d_s.p), int(S), static_cast<const double *>(d_v.p),
                                                                   static_cast<const int *>(d_f.p), static_cast<const int *>(d_tri.p), static_cast<const int *>(d_part.p),
                                                                   static_cast<double *>(d_val.p), static_cast<double *>(d_ds.p), static_cast<double *>(d_dt.p));
    chk(cudaGetLastError());
    chk(cudaEventRecord(e1, st));
    if (out->value) chk(cudaMemcpyAsync(out->value, d_val.p, S * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (out->tri) chk(cudaMemcpyAsync(out->tri, d_tri.p, S * sizeof(int), cudaMemcpyDeviceToHost, st));
    if (out->part) chk(cudaMemcpyAsync(out->part, d_part.p, S * sizeof(int), cudaMemcpyDeviceToHost, st));
    if (out->d_sample) chk(cudaMemcpyAsync(out->d_sample, d_ds.p, S * 3 * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (out->d_tri) chk(cudaMemcpyAsync(out->d_tri, d_dt.p, S * 9 * sizeof(double), cudaMemcpyDeviceToHost, st));
    chk(cudaStreamSynchronize(st));
    if (e == cudaSuccess && kernel_ms) chk(cudaEventElapsedTime(kernel_ms, e0, e1));
    cleanup();
    if (e != cudaSuccess) return fail(MOSH2_E_CUDA, "mosh2_mesh_distance: %s", cudaGetErrorString(e));
    return 0;
}

}  // extern "C"
