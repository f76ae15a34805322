// mosh2_host.h -- host-side layout helpers shared by libmosh2.so and the test-only host build.
#pragma once
#include <algorithm>
#include <vector>

#include "../../include/mosh2.h"
#include "mosh2_device.cuh"

namespace mosh2_host {

// Splits the hand-PCA matrix C (n_red x n_full, row-major) into dense blocks of consecutive rows that
// share one non-zero column range (SMPL-H / SMPL-X: left and right hand; MANO: one block) and stores each
// block transposed, rows padded to a multiple of four: hct[ct_off + (q-q0)*rw4 + (r-r0)] = C[r][q].
// Falls back to a single dense block when the structure is irregular.
inline int hand_blocks(const double *C, int n_red, int n_full, mosh2::HandBlock *out, std::vector<double> &hct) {
    hct.clear();
    if (n_red == 0) return 0;
    std::vector<int> lo(n_red), hi(n_red);
    for (int r = 0; r < n_red; ++r) {
        int a = n_full, b = 0;
        for (int c = 0; c < n_full; ++c)
            if (C[size_t(r) * n_full + c] != 0.0) { if (c < a) a = c; b = c + 1; }
        if (b <= a) { a = 0; b = 0; }
        lo[r] = a; hi[r] = b;
    }
    int nb = 0;
    bool regular = true;
    for (int r = 0; r < n_red && regular;) {
        int e = r + 1;
        while (e < n_red && lo[e] == lo[r] && hi[e] == hi[r]) ++e;
        if (nb == mosh2::kMaxHandBlocks) { regular = false; break; }
        out[nb].r0 = r; out[nb].r1 = e; out[nb].q0 = lo[r]; out[nb].q1 = hi[r];
        ++nb;
        r = e;
    }
    for (int a = 0; a < nb && regular; ++a)          // column ranges of different blocks must not overlap
        for (int b = a + 1; b < nb; ++b)
            if (out[a].q0 < out[b].q1 && out[b].q0 < out[a].q1) regular = false;
    if (!regular) { nb = 1; out[0].r0 = 0; out[0].r1 = n_red; out[0].q0 = 0; out[0].q1 = n_full; }
    for (int b = 0; b < nb; ++b) {
        mosh2::HandBlock &h = out[b];
        h.rw4 = ((h.r1 - h.r0) + 3) & ~3;
        h.ct_off = int(hct.size());
        hct.resize(hct.size() + size_t(h.q1 - h.q0) * h.rw4, 0.0);
        for (int q = h.q0; q < h.q1; ++q)
            for (int r = h.r0; r < h.r1; ++r) hct[h.ct_off + size_t(q - h.q0) * h.rw4 + (r - h.r0)] = C[size_t(r) * n_full + q];
    }
    return nb;
}

// Fills `m` from a model description: its sizes and every table the kernel reads, among them the derived ones -- the joints
// in FK order, the hand-PCA blocks, the pose-blend table in its two layouts, the prior precisions padded to D4 and the image
// of the staged shared-memory tables.  `store(src, n, &dst)` keeps the n elements at src (int, double or unsigned char),
// converted to the type of *dst (int, real or unsigned char), where the kernel reads them, and points dst there; an empty
// array must still get a valid pointer.  The first nonzero return of `store` ends the build and is returned.
template <class real, class Store>
int build_model(const mosh2_model_desc &d, mosh2::Model<real> &m, Store store) {
    int rc = 0;
    auto put = [&](const auto *src, size_t n, auto **dst) { if (rc == 0) rc = store(src, n, dst); };
    const size_t nJ = d.n_joints, S = size_t(3) * d.n_markers, nd = d.n_dmpl;
    m.nJ = d.n_joints; m.M = d.n_markers; m.body_dof = d.body_dof; m.p_red = d.p_red;
    m.n_hand_red = d.n_hand_red; m.n_hand_full = d.n_hand_full; m.nd = d.n_dmpl; m.kw = d.kw;
    m.prior_k = d.prior_k; m.prior_d = d.prior_d;
    m.n1 = d.n_free1; m.n2 = d.n_free2; m.finger_lo = d.finger_lo; m.finger_hi = d.finger_hi;
    m.n_expr = d.n_expr; m.face_lo = d.face_lo; m.face_hi = d.face_hi;
    m.n_jang = d.n_jangles;
    for (int i = 0; i < d.n_jangles && i < mosh2::kMaxJangles; ++i) { m.jang_id[i] = d.jangles_ids[i]; m.jang_sign[i] = real(d.jangles_signs[i]); }
    put(d.parents, nJ, &m.parents);
    std::vector<int> order(nJ), ids(d.prior_d);
    {   // joints sorted by depth (stable): parents before children
        std::vector<int> depth(nJ, 0);
        for (size_t j = 0; j < nJ; ++j) { int dj = 0; for (int a = d.parents[j]; a >= 0; a = d.parents[a]) ++dj; depth[j] = dj; }
        for (size_t j = 0; j < nJ; ++j) order[j] = int(j);
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return depth[a] < depth[b]; });
        put(order.data(), nJ, &m.fk_order);
    }
    put(d.w_joint, S * d.kw, &m.w_joint);
    std::vector<double> hct;
    {   // dense blocks of the hand-PCA matrix (rows with the same non-zero column range), stored transposed
        mosh2::HandBlock blocks[mosh2::kMaxHandBlocks];
        m.hb_n = hand_blocks(d.hand_comps, d.n_hand_red, d.n_hand_full, blocks, hct);
        for (int b = 0; b < m.hb_n; ++b) m.hb[b] = blocks[b];
        m.hct_size = int(hct.size());
        put(hct.data(), hct.size(), &m.hct);
    }
    put(d.hands_mean, size_t(d.n_hand_full), &m.hands_mean);
    put(d.v0, S * 3, &m.v0);
    put(d.sd, S * 3 * nd, &m.sd);
    {   // pose-blend table twice: [(nJ-1)][9 e][3 c][Sp] (eval: four slots per 16-byte load, no padding) and
        // [(nJ-1)][9 e][3M slots][x y z -] (build: one slot per 16-byte load)
        const size_t S3 = size_t(3) * d.n_markers;
        const size_t Sp = (S3 + 3) & ~size_t(3);
        std::vector<double> pdc((nJ - 1) * 27 * Sp, 0.0), pd4((nJ - 1) * 9 * S3 * 4, 0.0);
        for (size_t j = 0; j + 1 < nJ; ++j)
            for (size_t sl = 0; sl < S3; ++sl)
                for (int c = 0; c < 3; ++c)
                    for (int e = 0; e < 9; ++e) {
                        const double v = d.pd[(j * 3 * S3 + 3 * sl + c) * 9 + e];
                        pdc[((j * 9 + e) * 3 + c) * Sp + sl] = v;
                        pd4[((j * 9 + e) * S3 + sl) * 4 + c] = v;
                    }
        put(pdc.data(), pdc.size(), &m.pdc);
        put(pd4.data(), pd4.size(), &m.pd4);
    }
    put(d.w_val, S * d.kw, &m.w_val);
    put(d.j0, nJ * 3, &m.j0);
    put(d.jd, nJ * 3 * nd, &m.jd);
    put(d.coefs, size_t(d.n_markers) * 3, &m.coefs);
    put(d.prior_means, size_t(d.prior_k) * d.prior_d, &m.prior_means);
    {   // prior precisions padded to D4 columns, as stored ([K][D i][D4 l]) and transposed per component ([K][D l][D4 i])
        const size_t K = d.prior_k, D = d.prior_d, D4 = (D + 3) & ~size_t(3);
        m.prior_d4 = int(D4);
        std::vector<double> q4(K * D * D4, 0.0), qt(K * D * D4, 0.0);
        for (size_t k = 0; k < K; ++k)
            for (size_t i = 0; i < D; ++i)
                for (size_t l = 0; l < D; ++l) {
                    q4[(k * D + i) * D4 + l] = d.prior_Q[(k * D + i) * D + l];
                    qt[(k * D + l) * D4 + i] = d.prior_Q[(k * D + i) * D + l];
                }
        put(q4.data(), q4.size(), &m.prior_Q4);
        put(qt.data(), qt.size(), &m.prior_Qt);
    }
    put(d.prior_neglogw, size_t(d.prior_k), &m.prior_nlw);
    for (int i = 0; i < d.prior_d; ++i) ids[i] = d.prior_ids ? d.prior_ids[i] : d.prior_off + i;
    put(ids.data(), ids.size(), &m.prior_ids);
    put(d.free1, size_t(d.n_free1), &m.free1);
    put(d.free2, size_t(d.n_free2), &m.free2);
    {   // image of the staged shared-memory tables (mosh2::carve / stage_image): what a chunk fetches with one bulk copy.  It
        // is built from the host arrays: the stored m.* may be device pointers.
        const mosh2::Dims dd = mosh2::make_dims(m);
        mosh2::Work<real, false> w{};
        mosh2::Arena Sa{mosh2::kSmemHeader}, Ga{0};
        mosh2::carve<real, false>(w, dd, m, Sa, Ga);
        std::vector<unsigned char> img(w.stage_bytes, 0);
        const int *isrc[6] = {d.parents, order.data(), d.w_joint, d.free1, d.free2, ids.data()};
        const double *rsrc[9] = {d.w_val, d.v0, d.coefs, d.j0, d.hands_mean, d.prior_means, d.prior_neglogw, d.jd, hct.data()};
        mosh2::stage_image(w, dd, m.hct_size, m.n_hand_full, [&](uint32_t ofs, int id, size_t n) {
            if (id < 6) { int *o = reinterpret_cast<int *>(img.data() + ofs); for (size_t i = 0; i < n; ++i) o[i] = isrc[id][i]; }
            else { real *o = reinterpret_cast<real *>(img.data() + ofs); for (size_t i = 0; i < n; ++i) o[i] = real(rsrc[id - 6][i]); }
        });
        put(img.data(), img.size(), &m.stage_blob);
    }
    return rc;
}

// The kernel's options of a job from the caller's.
inline mosh2::Options options(const mosh2_options *opt) {
    mosh2::Options q{};
    q.wt_data = opt->wt_data; q.wt_poseB = opt->wt_poseB; q.wt_poseH = opt->wt_poseH; q.wt_velo = opt->wt_velo;
    q.wt_dmpl = opt->wt_dmpl; q.wt_annealing = opt->wt_annealing; q.wt_extrap = opt->wt_extrap_dmpl;
    q.num_train_markers = opt->num_train_markers; q.delta_0 = opt->delta_0; q.e3_first = opt->e3_first; q.e3 = opt->e3;
    q.maxiter = opt->maxiter; q.optimize_fingers = opt->optimize_fingers; q.optimize_dynamics = opt->optimize_dynamics;
    q.wt_poseF = opt->wt_poseF; q.wt_expr = opt->wt_expr; q.optimize_face = opt->optimize_face;
    return q;
}

// Fully solved frames of a warm-up of `warmup` >= 0 frames: all of them unless 0 <= warmup_full < warmup.
inline int clamp_warm_full(int warmup, int warmup_full) { return (warmup_full < 0 || warmup_full > warmup) ? warmup : warmup_full; }

// The schedule a job runs (the arguments of chunk_table) from the caller's, which may be null (one chunk per sequence): a
// negative chunk length or warm-up counts as none, and the longer first chunk needs both.
struct Schedule {
    int chunk_len, warmup, warm_full, first_extra;
};
inline Schedule schedule(const mosh2_schedule *sched) {
    Schedule s{0, 0, 0, 0};
    if (!sched) return s;
    s.chunk_len = sched->chunk_len > 0 ? sched->chunk_len : 0;
    s.warmup = sched->chunk_warmup > 0 ? sched->chunk_warmup : 0;
    s.warm_full = clamp_warm_full(s.warmup, sched->warmup_full);
    s.first_extra = (sched->first_extra > 0 && s.chunk_len > 0 && s.warmup > 0) ? sched->first_extra : 0;
    return s;
}

// Chunk table of a job that holds n_seq sequences back to back on its frame axis: kChunkRec ints per chunk -- first
// emitted frame, end of the emitted range, first frame of the chunk's sequence, warm-up length (solved frames), number of
// fully solved warm-up frames.  chunk_len <= 0: one chunk per sequence (the reference's sequential pass).  Chunks never
// straddle a sequence boundary.  first_extra > 0: the FIRST chunk of every sequence emits chunk_len + first_extra frames --
// it has no warm-up to solve, so with first_extra = the cost of a warm-up every chunk of the sequence finishes at the same
// time, and no later chunk starts so close to the sequence start that its walk-back is cut short.
inline std::vector<int> chunk_table(const int *frame_counts, int n_seq, int chunk_len, int warmup, int warm_full, int first_extra = 0) {
    std::vector<int> tab;
    int s0 = 0;
    for (int q = 0; q < n_seq; ++q) {
        const int F = frame_counts[q];
        const int L = (chunk_len > 0 && chunk_len < F) ? chunk_len : F;
        const int E = (first_extra > 0 && L < F) ? first_extra : 0;
        for (int f = 0; f < F;) {
            long long e = (long long)f + L + (f == 0 ? E : 0);
            if (e > F) e = F;
            const int rec[mosh2::kChunkRec] = {s0 + f, s0 + int(e), s0, warmup, warm_full};
            tab.insert(tab.end(), rec, rec + mosh2::kChunkRec);
            f = int(e);
        }
        s0 += F;
    }
    return tab;
}

}  // namespace mosh2_host
