// mosh2_emu.cpp -- TEST-ONLY host build of the CTA program (moshpp_b200/csrc/mosh2_device.cuh).
//
// Compiles the device source with MOSH2_EMU: one "thread" (tid 0 of 1), barriers are no-ops.  The CPU
// test-suite runs it against the oracle to validate index math and control flow of the exact code that
// nvcc compiles for sm_100a.  It is never linked into libmosh2.so and never loaded by moshpp_b200.
#define MOSH2_EMU 1
#include "../../include/mosh2.h"
#include "../../moshpp_b200/csrc/mosh2_device.cuh"
#include "../../moshpp_b200/csrc/mosh2_host.h"

#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <vector>

namespace {

// One job on the single "thread block": the model tables as libmosh2.so builds them (mosh2_host::build_model), kept in host
// memory, the job's output rows, and the shared-memory buffer each chunk runs on.
template <class real>
struct Emu {
    mosh2::Model<real> m{};
    mosh2::Job<real> job{};
    std::vector<std::vector<char>> tables;
    std::vector<real> fullpose, pose, trans, dmpls, mk, errs;
    std::vector<int> status, counters;
    mosh2::Dims d{};
    mosh2::Work<real, false> w{};
    size_t smem_bytes = 0;
    std::vector<char> smem_raw;

    template <class T, class U>
    int up(const U *src, size_t n, const T **dst) {
        tables.emplace_back((n + 1) * sizeof(T) + 32);
        char *raw = tables.back().data();
        T *p = reinterpret_cast<T *>(raw + ((32 - (reinterpret_cast<uintptr_t>(raw) & 31)) & 31));
        for (size_t i = 0; i < n; ++i) p[i] = static_cast<T>(src[i]);
        *dst = p;
        return 0;
    }

    Emu(const mosh2_model_desc &desc, const mosh2_options *opt, int n_frames) {
        mosh2_host::build_model(desc, m, [this](const auto *src, size_t n, auto **dst) { return up(src, n, dst); });
        if (std::getenv("MOSH2_EMU_PLAN")) {        // development aid: shared-memory footprint of this model
            for (int tile : {20, 10}) {
                m.tile_markers = tile;
                m.dev_no_tc = sizeof(real) == 4 ? 0 : 1;   // what the GPU launch would lay out
                const mosh2::Dims dd = mosh2::make_dims(m);
                mosh2::Work<real, false> ww{};
                mosh2::Arena Sa{mosh2::kSmemHeader}, Ga{0};
                mosh2::carve<real, false>(ww, dd, m, Sa, Ga);
                std::fprintf(stderr, "plan: sizeof(real)=%zu tile=%d smem=%zu bytes (limit %d)\n", sizeof(real), tile, Sa.off, 227 * 1024);
                std::fprintf(stderr, "      A=%u Lm=%u Xhi=%u Xlo=%u Jt=%u Jf=%u Loc=%u MtR=%u u=%u dtg=%u Linv=%u tc_ok=%d\n", ww.A.ofs, ww.Lm.ofs, ww.Xhi.ofs,
                             ww.Xlo.ofs, ww.Jt.ofs, ww.Jf.ofs, ww.Loc.ofs, ww.MtR.ofs, ww.u.ofs, ww.dtg.ofs, ww.Linv.ofs, ww.tc_ok);
            }
        }
        m.tile_markers = 20;
        m.dev_no_tc = 1;                             // the host build runs the CUDA-core formulation
        d = mosh2::make_dims(m);
        mosh2::Arena S{mosh2::kSmemHeader}, G{0};
        mosh2::carve<real, false>(w, d, m, S, G);
        smem_bytes = S.off;
        smem_raw.resize(S.off + 128);

        const size_t F = n_frames, M = desc.n_markers, nd = desc.n_dmpl;
        fullpose.resize(F * 3 * desc.n_joints); pose.resize(F * desc.p_red); trans.resize(F * 3); dmpls.resize(F * nd + 1);
        mk.resize(F * M * 3); errs.resize(F * mosh2::N_ERR); status.resize(F); counters.resize(F * 4);
        job.n_frames = n_frames;
        job.fullpose = fullpose.data(); job.pose = pose.data(); job.trans = trans.data();
        job.dmpls = nd ? dmpls.data() : nullptr; job.markers_sim = mk.data(); job.errs = errs.data();
        job.status = status.data(); job.counters = counters.data();
        job.opt = mosh2_host::options(opt);
    }

    // chunks [c0, c1) one after the other, each on a zeroed shared-memory buffer
    void run_chunks(int c0, int c1) {
        char *smem_base = smem_raw.data() + ((32 - (reinterpret_cast<uintptr_t>(smem_raw.data()) & 31)) & 31);
        mosh2::m2_smem_ref() = reinterpret_cast<unsigned char *>(smem_base);
        for (int c = c0; c < c1; ++c) {
            std::memset(smem_base, 0, smem_bytes + 64);
            mosh2::Cta cta{0, 1};
            mosh2::Solver<real, false> s(m, job, w, d, cta);
            s.run_chunk(c);
        }
    }
};

template <class real>
int run(const mosh2_model_desc *desc, const mosh2_options *opt, int n_frames, const double *obs, const uint8_t *vis,
        const mosh2_schedule *sched, const mosh2_result *res, int n_seq = 1, const int *seq_counts = nullptr, bool resume_all = false) {
    if (!seq_counts) seq_counts = &n_frames;
    Emu<real> e(*desc, opt, n_frames);
    const size_t F = n_frames, M = desc->n_markers, PF = size_t(3) * desc->n_joints, PR = desc->p_red, nd = desc->n_dmpl;
    std::vector<real> o(F * M * 3);
    for (size_t i = 0; i < o.size(); ++i) o[i] = real(obs[i]);
    const mosh2_host::Schedule s = mosh2_host::schedule(sched);
    std::vector<int> tab = mosh2_host::chunk_table(seq_counts, n_seq, s.chunk_len, s.warmup, s.warm_full, s.first_extra);
    int totals[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    mosh2::Job<real> &job = e.job;
    job.n_chunks = int(tab.size() / mosh2::kChunkRec);
    job.chunk_tab = tab.data();
    job.obs = o.data(); job.vis = vis;
    job.totals = totals;
    e.run_chunks(0, job.n_chunks);
    if (resume_all) {       // boundary repair of every chunk, in order: chunk c continues from the rows chunk c-1 emitted
        for (int c = 1; c < job.n_chunks; ++c) {
            tab[size_t(c) * mosh2::kChunkRec + 3] = -1;
            e.run_chunks(c, c + 1);
        }
    }
    auto conv = [](double *dst, const std::vector<real> &src, size_t n) {
        if (dst) for (size_t i = 0; i < n; ++i) dst[i] = double(src[i]);
    };
    conv(res->fullpose, e.fullpose, F * PF);
    conv(res->pose, e.pose, F * PR);
    conv(res->trans, e.trans, F * 3);
    if (nd) conv(res->dmpls, e.dmpls, F * nd);
    conv(res->markers_sim, e.mk, F * M * 3);
    conv(res->errs, e.errs, F * mosh2::N_ERR);
    if (res->status) std::memcpy(res->status, e.status.data(), F * sizeof(int));
    if (res->counters) std::memcpy(res->counters, e.counters.data(), F * 4 * sizeof(int));
    return 0;
}

// linearise mode (mosh2_job_linearize): every frame evaluated / linearised at the caller's state, float64
int run_lin(const mosh2_model_desc *desc, const mosh2_options *opt, int n_frames, const double *obs, const uint8_t *vis,
            int step, int build, const double *x, const mosh2_lin_out *out) {
    Emu<double> e(*desc, opt, n_frames);
    const size_t F = n_frames, M = desc->n_markers, n = step == 2 ? desc->n_free2 : desc->n_free1;
    std::vector<double> A(F * n * n), g(F * n), J(F * 3 * M * n), r(F * 3 * M), vp(F * 9 * M);
    mosh2::Job<double> &job = e.job;
    job.n_chunks = n_frames;
    job.obs = obs; job.vis = vis;
    job.lin_mode = build ? 2 : 1; job.lin_step = step; job.lin_x = x;
    job.lin_A = A.data(); job.lin_g = g.data(); job.lin_J = J.data(); job.lin_r = r.data(); job.lin_vp = vp.data();
    e.run_chunks(0, n_frames);
    auto back = [](double *dst, const std::vector<double> &src) { if (dst) std::memcpy(dst, src.data(), src.size() * sizeof(double)); };
    back(out->errs, e.errs); back(out->markers_sim, e.mk); back(out->r, r); back(out->vp, vp);
    if (build) { back(out->A, A); back(out->g, g); back(out->J, J); }
    return 0;
}

}  // namespace

extern "C" int mosh2_emu_linearize(const mosh2_model_desc *desc, const mosh2_options *opt, int32_t n_frames, const double *obs,
                                   const uint8_t *vis, int32_t step, int32_t build, const double *x, const mosh2_lin_out *out) {
    return run_lin(desc, opt, n_frames, obs, vis, step, build, x, out);
}

extern "C" int mosh2_emu_solve(const mosh2_model_desc *desc, const mosh2_options *opt, int32_t n_frames,
                               const double *obs, const uint8_t *vis, const mosh2_schedule *sched,
                               int32_t precision, const mosh2_result *res) {
    if (precision == MOSH2_F64) return run<double>(desc, opt, n_frames, obs, vis, sched, res);
    return run<float>(desc, opt, n_frames, obs, vis, sched, res);
}

// several sequences of one subject back to back on the frame axis (mosh2_job_create_batch)
extern "C" int mosh2_emu_solve_batch(const mosh2_model_desc *desc, const mosh2_options *opt, int32_t n_seq, const int32_t *frame_counts,
                                     const double *obs, const uint8_t *vis, const mosh2_schedule *sched,
                                     int32_t precision, const mosh2_result *res) {
    int total = 0;
    for (int q = 0; q < n_seq; ++q) total += frame_counts[q];
    if (precision == MOSH2_F64) return run<double>(desc, opt, total, obs, vis, sched, res, n_seq, frame_counts);
    return run<float>(desc, opt, total, obs, vis, sched, res, n_seq, frame_counts);
}

// chunked solve followed by a resume (mosh2_job_relaunch_chunks with chunk_warmup < 0) of every chunk in order
extern "C" int mosh2_emu_solve_resumed(const mosh2_model_desc *desc, const mosh2_options *opt, int32_t n_frames,
                                       const double *obs, const uint8_t *vis, const mosh2_schedule *sched,
                                       int32_t precision, const mosh2_result *res) {
    if (precision == MOSH2_F64) return run<double>(desc, opt, n_frames, obs, vis, sched, res, 1, nullptr, true);
    return run<float>(desc, opt, n_frames, obs, vis, sched, res, 1, nullptr, true);
}
