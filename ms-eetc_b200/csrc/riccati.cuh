// Search direction of one interior-point iteration: Riccati recursion over the shooting intervals.
//
// The Newton system of the reference NLP (all rows of ocp.py:183-241 linearised, bound and slack multipliers
// condensed by cell_eval) is a linear-quadratic OCP in (d t, d b, d Fel_{k-1} | d Fel, d Fpb, d s); cell_eval also
// eliminates d s, whose pivot does not depend on the value function, so the sweeps carry two controls.  It replaces
// IPOPT's sparse LDL^T (MUMPS) behind ocp.py:359:
//   riccati_backward   value functions P_k, p_k and feedback K_k, k_k; positive-definiteness of every reduced
//                      control Hessian is the inertia test (IPOPT Alg. IC regularises when it fails); a plain variant
//                      and one for delta_w != 0 so that the rarely needed correction stays out of the hot loop
//   riccati_forward    d Fel, d Fpb, d t, d b -- nothing else is sequential
//   cell_step          (interval-parallel) d s, the new coupling-row multipliers (costates of the stepped state), slack
//                      and inequality-multiplier steps, fraction-to-boundary limits, directional derivative of the barrier
//                      function; recomputes the row gradients / residuals bit for bit instead of reading them back
//   inst_alpha         deterministic per-instance reduction of those limits -> first trial step size
// The two sweeps are sequential in k for one instance; their stage data are prefetched DEPTH intervals ahead
// into a shared-memory ring with cp.async (one column per lane: no block-level synchronisation needed).
#pragma once
#include "core.cuh"
#if defined(__CUDACC__)
#include <cuda_pipeline_primitives.h>
#endif

namespace mseetc {

// ---- which planes a sweep consumes per interval ------------------------------------------------------------
// With the tiled layout every field of interval k of one instance is  record(k) + compile-time offset, and the record
// of k+1 follows at a compile-time stride, so the address arithmetic of a sweep is one pointer bump per interval.
enum { REC_STRIDE = WS_FIELDS * 32 };
struct BwdFields {   // condensed stage Hessian (9), linearised coupling rows (6), condensed gradient parts (4 + 4)
    enum { NF = QP_SWEEP_N };
    static MS_HD constexpr int off(int f) { return (WS_QP + f) * 32; }
};
struct FwdFields {   // feedback rows of Fel, Fpb (6 + 2) | linearised coupling rows (6)
    enum { NF = 14 };
    static MS_HD constexpr int off(int f) { return f < 8 ? (WS_RIC + RIC_K + f) * 32 : (WS_QP + QP_TAU_B + (f - 8)) * 32; }
};
enum { RING_NF_MAX = QP_SWEEP_N };

// direct loads (host emulation, and the device when no ring is configured)
template <class FL>
struct DirectFetch {
    MS_HD void start(const Ctx&, int, int, int, int) {}
    MS_HD void get(const Ctx& c, int k, int s, double* v) {
        const double* rec = &c.W(0, k, s);
#pragma unroll
        for (int f = 0; f < FL::NF; ++f) v[f] = rec[FL::off(f)];
    }
};

#if defined(__CUDACC__)
// cp.async ring in shared memory with DEPTH + 1 slots, column = thread: stage k + DEPTH*dir is requested as soon as
// stage k has been copied to registers, into the slot that was consumed one iteration earlier.  Slot indices and the
// global record pointer are running counters (no division, one pointer bump per interval).
// PF > 0: the record PF intervals further on is pulled into L2 at the same time (prefetch.global.L2: no shared memory, no
// registers), so that a shallow ring sees L2 latency instead of DRAM latency
template <class FL, int BS, int DEPTH, int PF = 0>
struct RingFetch {
    double* sm;          // this thread's column of slot 0
    const double* next;  // record of the next interval to request
    int left;            // intervals not yet requested
    int head, tail;      // slot to consume next / slot to fill next
    long step;           // +-REC_STRIDE
    __device__ void issue() {
        if (left > 0) {
            double* dst = sm + tail * (FL::NF * BS);
#pragma unroll
            for (int f = 0; f < FL::NF; ++f) __pipeline_memcpy_async(dst + f * BS, next + FL::off(f), 8);
            if (PF > 0 && left > PF) {
                const double* far = next + PF * step;
#pragma unroll
                for (int f = 0; f < FL::NF; ++f) asm volatile("prefetch.global.L2 [%0];" ::"l"(far + FL::off(f)));
            }
            next += step;
            --left;
        }
        __pipeline_commit();
        tail = (tail == DEPTH) ? 0 : tail + 1;
    }
    __device__ void start(const Ctx& c, int s, int kFirst, int kLast, int direction) {
        // a sweep that was left early (failed inertia test) still has copies in flight into these slots: drain them before the
        // slots are requested again, otherwise a stale copy can land after the new one
        asm volatile("cp.async.wait_all;" ::: "memory");
        next = &c.W(0, kFirst, s);
        step = (long)direction * REC_STRIDE;
        left = (direction < 0 ? kFirst - kLast : kLast - kFirst) + 1;
        head = tail = 0;
#pragma unroll
        for (int d = 0; d < DEPTH; ++d) issue();
    }
    __device__ void get(const Ctx&, int, int, double* v) {
        asm volatile("cp.async.wait_group %0;" ::"n"(DEPTH - 1) : "memory");      // (__pipeline_wait_prior caps its argument at 8)
        const double* src = sm + head * (FL::NF * BS);
#pragma unroll
        for (int f = 0; f < FL::NF; ++f) v[f] = src[f * BS];
        head = (head == DEPTH) ? 0 : head + 1;
        issue();
    }
};
#endif

// ---- one interval of the stage QP in registers --------------------------------------------------------------
struct StageQP {
    double M[6][6], m[6];     // Hessian / gradient over (t,b,f | Fel,Fpb,sl), delta_w included
    double G[3][6], r[3];     // next state = G (x;u) + r
    double pb, pF, rb;        // Phi_b, Phi_F, b residual (needed by the terminal-speed elimination)
};

// column of s of interval k (see QpField)
MS_HD void load_scol(const Ctx& c, int k, int s, double* vs) {
    const double* q = &c.W(WS_QP + QP_H_BSL, k, s);
    for (int i = 0; i < 6; ++i) vs[i] = q[i * 32];
}

// dense stage QP over (t,b,f | Fel,Fpb,s): the condensation of s is undone (v holds the condensed entries, vs the column of s)
MS_HD void stage_build(const double* v, const double* vs, double mu, double delta, double pn, bool last, StageQP& q) {
    for (int i = 0; i < 6; ++i) for (int j = 0; j < 6; ++j) q.M[i][j] = 0.0;
    const double hb = vs[0], hF = vs[1], hQ = vs[2], hss = vs[3], mS = vs[4] + mu * vs[5];
    const double is = rcp(hss);
    q.M[0][0] = v[QP_H_TT] + delta;
    q.M[1][1] = v[QP_H_BB] + hb * hb * is + delta;
    q.M[1][3] = q.M[3][1] = v[QP_H_BFEL] + hb * hF * is;
    q.M[1][4] = q.M[4][1] = v[QP_H_BFPB] + hb * hQ * is;
    q.M[1][5] = q.M[5][1] = hb;
    q.M[2][2] = v[QP_H_FF];
    q.M[2][3] = q.M[3][2] = v[QP_H_FFEL];
    q.M[3][3] = v[QP_H_FELFEL] + hF * hF * is + delta;
    q.M[3][4] = q.M[4][3] = v[QP_H_FELFPB] + hF * hQ * is;
    q.M[3][5] = q.M[5][3] = hF;
    q.M[4][4] = v[QP_H_FPBFPB] + hQ * hQ * is + delta;
    q.M[4][5] = q.M[5][4] = hQ;
    q.M[5][5] = hss + delta;
    q.m[0] = mu * v[QP_G1_T];
    q.m[1] = v[QP_G0_B] + mu * v[QP_G1_B] + hb * is * mS;
    q.m[2] = v[QP_G0_F];
    q.m[3] = v[QP_G0_FEL] + mu * v[QP_G1_FEL] + hF * is * mS;
    q.m[4] = v[QP_G0_FPB] + mu * v[QP_G1_FPB] + hQ * is * mS;
    q.m[5] = mS;
    const double tb = v[QP_TAU_B], tF = v[QP_TAU_F];
    q.pb = v[QP_PHI_B]; q.pF = v[QP_PHI_F]; q.rb = v[QP_RB];
    // G = [A B]: rows t, b, f of the next state
    const double G0[6] = {1.0, tb, 0.0, tF, pn * tF, 0.0};
    const double G1[6] = {0.0, q.pb, 0.0, q.pF, pn * q.pF, 0.0};
    const double G2[6] = {0.0, 0.0, 0.0, 1.0, 0.0, 0.0};
    for (int j = 0; j < 6; ++j) { q.G[0][j] = G0[j]; q.G[1][j] = last ? 0.0 : G1[j]; q.G[2][j] = G2[j]; }
    q.r[0] = v[QP_RT]; q.r[1] = last ? 0.0 : v[QP_RB]; q.r[2] = 0.0;   // d b_N = 0 is handled by elimination
}

// One backward Riccati step: (P, p) of the next node in, (P, p) of this node out, feedback K, kf.
// Returns false when the reduced control Hessian is not positive definite (wrong inertia of the KKT matrix).
MS_HD bool stage_riccati(StageQP& q, bool last, double pn, double P[3][3], double p[3], double K[3][3], double kf[3]) {
    double (*M)[6] = q.M;
    double* m = q.m;
    // M += G' P G ; m += G' (P r + p)
    double Y[3][6], pr[3];
    for (int a = 0; a < 3; ++a) {
        pr[a] = p[a] + P[a][0] * q.r[0] + P[a][1] * q.r[1] + P[a][2] * q.r[2];
        for (int j = 0; j < 6; ++j) Y[a][j] = P[a][0] * q.G[0][j] + P[a][1] * q.G[1][j] + P[a][2] * q.G[2][j];
    }
    for (int i = 0; i < 6; ++i) {
        m[i] += q.G[0][i] * pr[0] + q.G[1][i] * pr[1] + q.G[2][i] * pr[2];
        for (int j = i; j < 6; ++j) {
            const double x = M[i][j] + q.G[0][i] * Y[0][j] + q.G[1][i] * Y[1][j] + q.G[2][i] * Y[2][j];
            M[i][j] = x; M[j][i] = x;
        }
    }
    double eB = 0.0, ePn = 0.0, e0 = 0.0;
    if (last) {
        // terminal speed fixed: Phi_b db + Phi_F (dFel + dFpb) + rb = 0  ->  dFel = eB db + ePn dFpb + e0
        const double ipF = rcp(q.pF);
        eB = -q.pb * ipF; ePn = -pn; e0 = -q.rb * ipF;
        double colF[6];
        for (int i = 0; i < 6; ++i) colF[i] = M[i][3];
        const double mFF = M[3][3];
        for (int i = 0; i < 6; ++i) m[i] += colF[i] * e0;
        const double mF = m[3];
        const double ev[6] = {0.0, eB, 0.0, 0.0, ePn, 0.0};
        for (int i = 0; i < 6; ++i) m[i] += ev[i] * mF;
        for (int i = 0; i < 6; ++i)
            for (int j = 0; j < 6; ++j) M[i][j] += colF[i] * ev[j] + ev[i] * colF[j] + mFF * ev[i] * ev[j];
        for (int i = 0; i < 6; ++i) { M[i][3] = 0.0; M[3][i] = 0.0; }
        M[3][3] = 1.0; m[3] = 0.0;      // Fel of the last interval is now a dummy control
    }
    // Cholesky of the control block (indices 3..5), reciprocals of the pivots kept
    const double d0 = M[3][3];
    if (!(d0 > 0.0) || !isfinite(d0)) return false;
    const double i00 = rcp(sqrt(d0));
    const double l10 = M[4][3] * i00, l20 = M[5][3] * i00;
    const double d1 = M[4][4] - l10 * l10;
    if (!(d1 > 0.0) || !isfinite(d1)) return false;
    const double i11 = rcp(sqrt(d1));
    const double l21 = (M[5][4] - l20 * l10) * i11;
    const double d2 = M[5][5] - l20 * l20 - l21 * l21;
    if (!(d2 > 0.0) || !isfinite(d2)) return false;
    const double i22 = rcp(sqrt(d2));
    // solve Muu X = [Mux mu]  (4 right-hand sides)
    for (int j = 0; j < 4; ++j) {
        const double r0 = (j < 3) ? M[3][j] : m[3], r1 = (j < 3) ? M[4][j] : m[4], r2 = (j < 3) ? M[5][j] : m[5];
        const double y0 = r0 * i00, y1 = (r1 - l10 * y0) * i11, y2 = (r2 - l20 * y0 - l21 * y1) * i22;
        const double x2 = y2 * i22, x1 = (y1 - l21 * x2) * i11, x0 = (y0 - l10 * x1 - l20 * x2) * i00;
        if (j < 3) { K[0][j] = -x0; K[1][j] = -x1; K[2][j] = -x2; }
        else { kf[0] = -x0; kf[1] = -x1; kf[2] = -x2; }
    }
    // P = Mxx + Mxu K ; p = mx + Mxu kf
    double Pn[3][3], pnv[3];
    for (int i = 0; i < 3; ++i) {
        pnv[i] = m[i] + M[i][3] * kf[0] + M[i][4] * kf[1] + M[i][5] * kf[2];
        for (int j = 0; j < 3; ++j) Pn[i][j] = M[i][j] + M[i][3] * K[0][j] + M[i][4] * K[1][j] + M[i][5] * K[2][j];
    }
    for (int i = 0; i < 3; ++i) { p[i] = pnv[i]; for (int j = 0; j < 3; ++j) P[i][j] = 0.5 * (Pn[i][j] + Pn[j][i]); }
    if (last) {   // feedback row of the eliminated control
        for (int j = 0; j < 3; ++j) K[0][j] = ePn * K[1][j];
        K[0][1] += eB;
        kf[0] = e0 + ePn * kf[1];
    }
    return true;
}

// Backward Riccati step of a regular interval (k < N-1), exploiting the structure of the stage QP:
//   t+ = t + tau_b b + tau_F w + rt,   b+ = phi_b b + phi_F w + rb,   f+ = Fel,     w = Fel + pn Fpb
// the sparsity of the folded Hessian (QpField lists its non-zero entries) and the condensation of s.  The 2x2 control block
// is inverted through its leading entry and its determinant (no square roots); their signs -- together with the pivot of s,
// H_ss + delta > 0 -- are the inertia test.  `vs` (column of s) is only needed when delta_w != 0: the condensed entries were formed with delta = 0 and are corrected
// by (1/H_ss - 1/(H_ss + delta)) h h', which keeps IPOPT's "delta on every primal variable" exact.
// x = C^{-1} r for the 2x2 control block C = [[a, b], [b, d]] with i0 = 1/a and idet = 1/(a d - b^2): the two reciprocals do
// not depend on each other (shorter dependent chain than pivot-after-pivot), a > 0 and det > 0 are the inertia test
MS_HD void sym2_solve(double a, double b, double i0, double idet, double r0, double r1, double& x0, double& x1) {
    x1 = (a * r1 - b * r0) * idet;
    x0 = (r0 - b * x1) * i0;
}

// `cb` (optional): reduced control block of this stage, (M_FF, M_FQ, 1/M_FF, 1/det), for the chunk elements of pit.cuh
MS_HD bool stage_riccati_sparse(const double* v, const double* vs, double mu, double delta, double pn,
                                double P[3][3], double p[3], double K[3][3], double kf[3], double* cb = nullptr) {
    const double tb = v[QP_TAU_B], tF = v[QP_TAU_F], pb = v[QP_PHI_B], pF = v[QP_PHI_F], rt = v[QP_RT], rb = v[QP_RB];
    const double P00 = P[0][0], P01 = P[0][1], P02 = P[0][2], P11 = P[1][1], P12 = P[1][2], P22 = P[2][2];
    double Hbb = v[QP_H_BB], HbF = v[QP_H_BFEL], HbQ = v[QP_H_BFPB], HFF = v[QP_H_FELFEL], HFQ = v[QP_H_FELFPB], HQQ = v[QP_H_FPBFPB];
    double gb = v[QP_G0_B] + mu * v[QP_G1_B], gF = v[QP_G0_FEL] + mu * v[QP_G1_FEL], gQ = v[QP_G0_FPB] + mu * v[QP_G1_FPB];
    if (vs) {
        const double hb = vs[0], hF = vs[1], hQ = vs[2], hss = vs[3], mS = vs[4] + mu * vs[5];
        if (!(hss + delta > 0.0)) return false;
        const double cf = rcp(hss) - rcp(hss + delta);
        Hbb += hb * hb * cf; HbF += hb * hF * cf; HbQ += hb * hQ * cf;
        HFF += hF * hF * cf; HFQ += hF * hQ * cf; HQQ += hQ * hQ * cf;
        gb += hb * mS * cf; gF += hF * mS * cf; gQ += hQ * mS * cf;
    }
    // P times the b- and w-columns of the transition
    const double y0b = P00 * tb + P01 * pb, y1b = P01 * tb + P11 * pb, y2b = P02 * tb + P12 * pb;
    const double y0w = P00 * tF + P01 * pF, y1w = P01 * tF + P11 * pF, y2w = P02 * tF + P12 * pF;
    const double ww = tF * y0w + pF * y1w, bw = tb * y0w + pb * y1w;
    // stage Hessian + G' P G, non-zero entries only (t, b, f | F = Fel, Q = Fpb)
    const double Mtt = v[QP_H_TT] + delta + P00;
    const double Mtb = y0b;
    const double MtF = y0w + P02;
    const double MtQ = pn * y0w;
    const double Mbb = Hbb + delta + (tb * y0b + pb * y1b);
    const double MbF = HbF + (bw + y2b);
    const double MbQ = HbQ + pn * bw;
    const double Mff = v[QP_H_FF];
    const double MfF = v[QP_H_FFEL];
    const double MFF = ww + (2.0 * y2w + (P22 + (HFF + delta)));
    const double MFQ = HFQ + pn * (ww + y2w);
    const double MQQ = HQQ + delta + pn * (pn * ww);
    // gradient + G' (P r + p)
    const double pr0 = p[0] + P00 * rt + P01 * rb, pr1 = p[1] + P01 * rt + P11 * rb, pr2 = p[2] + P02 * rt + P12 * rb;
    const double gw = tF * pr0 + pF * pr1;
    const double mt = mu * v[QP_G1_T] + pr0;
    const double mb = gb + (tb * pr0 + pb * pr1);
    const double mf = v[QP_G0_F];
    const double mF = gF + (gw + pr2);
    const double mQ = gQ + pn * gw;
    // control block: positive definite <=> MFF > 0 and det > 0 (the second pivot of L D L' is det / MFF)
    const double det = MFF * MQQ - MFQ * MFQ;
    if (!(MFF > 0.0) || !(det > 0.0) || !isfinite(MFF) || !isfinite(det)) return false;
    const double i0 = rcp(MFF), idet = rcp(det);
    if (cb) { cb[0] = MFF; cb[1] = MFQ; cb[2] = i0; cb[3] = idet; }
    // feedback: Muu [K kf] = -[Mux mu]
    double x0, x1;
    sym2_solve(MFF, MFQ, i0, idet, MtF, MtQ, x0, x1);
    K[0][0] = -x0; K[1][0] = -x1;
    sym2_solve(MFF, MFQ, i0, idet, MbF, MbQ, x0, x1);
    K[0][1] = -x0; K[1][1] = -x1;
    sym2_solve(MFF, MFQ, i0, idet, MfF, 0.0, x0, x1);
    K[0][2] = -x0; K[1][2] = -x1;
    sym2_solve(MFF, MFQ, i0, idet, mF, mQ, x0, x1);
    kf[0] = -x0; kf[1] = -x1;
    K[2][0] = K[2][1] = K[2][2] = 0.0; kf[2] = 0.0;     // d s is recovered interval-parallel (cell_step)
    // value function of this node (upper triangle, mirrored)
    P[0][0] = Mtt + MtF * K[0][0] + MtQ * K[1][0];
    P[0][1] = P[1][0] = Mtb + MtF * K[0][1] + MtQ * K[1][1];
    P[0][2] = P[2][0] = MtF * K[0][2] + MtQ * K[1][2];
    P[1][1] = Mbb + MbF * K[0][1] + MbQ * K[1][1];
    P[1][2] = P[2][1] = MbF * K[0][2] + MbQ * K[1][2];
    P[2][2] = Mff + MfF * K[0][2];
    p[0] = mt + MtF * kf[0] + MtQ * kf[1];
    p[1] = mb + MbF * kf[0] + MbQ * kf[1];
    p[2] = mf + MfF * kf[0];
    return true;
}

MS_HD void stage_store(const Ctx& c, int k, int s, const double K[3][3], const double kf[3], const double P[3][3], const double p[3]) {
    double* r = &c.W(WS_RIC, k, s);
    for (int i = 0; i < 2; ++i) {      // feedback rows of Fel and Fpb
        for (int j = 0; j < 3; ++j) r[(RIC_K + 3 * i + j) * 32] = K[i][j];
        r[(RIC_KF + i) * 32] = kf[i];
    }
    for (int i = 0; i < 3; ++i) r[(RIC_PV + i) * 32] = p[i];
    r[(RIC_P + 0) * 32] = P[0][0]; r[(RIC_P + 1) * 32] = P[0][1]; r[(RIC_P + 2) * 32] = P[0][2];
    r[(RIC_P + 3) * 32] = P[1][1]; r[(RIC_P + 4) * 32] = P[1][2]; r[(RIC_P + 5) * 32] = P[2][2];
}

// terminal value function: only t_N is free (b_N fixed, Fel_{N-1} costless)
MS_HD void terminal_value(const Ctx& c, int s, int N, double mu, double delta, double P[3][3], double p[3]) {
    for (int i = 0; i < 3; ++i) { p[i] = 0.0; for (int j = 0; j < 3; ++j) P[i][j] = 0.0; }
    P[0][0] = c.W(WS_QP + QP_H_TT, N, s) + delta;
    p[0] = (c.cfg.energy ? 0.0 : rcp_slack(c.P(P_SCALE, s))) + mu * c.W(WS_QP + QP_G1_T, N, s);
    for (int i = 0; i < 6; ++i) c.W(WS_RIC + RIC_P + i, N, s) = 0.0;
    c.W(WS_RIC + RIC_P + 0, N, s) = P[0][0];
    c.W(WS_RIC + RIC_PV + 0, N, s) = p[0];
    c.W(WS_RIC + RIC_PV + 1, N, s) = 0.0;
    c.W(WS_RIC + RIC_PV + 2, N, s) = 0.0;
}

// ---- backward sweep over the intervals kHi-1 .. kLo, starting from (P, p) of node kHi ------------------------
// Optionally accumulates the closed-loop transition of the range: x_{kHi} = Mc x_{kLo} + mc.
MS_HD void closed_loop_compose(double* Mc, double* mc, const double* Mk, const double* mk) {
    // closed loop of one interval: x+ = (A + B K) x + (B kf + r) = Mk x + mk; compose: acc <- acc o this
    double Mn[9], mn[3];
    for (int i = 0; i < 3; ++i) {
        mn[i] = mc[i] + Mc[3 * i] * mk[0] + Mc[3 * i + 1] * mk[1] + Mc[3 * i + 2] * mk[2];
        for (int j = 0; j < 3; ++j) Mn[3 * i + j] = Mc[3 * i] * Mk[j] + Mc[3 * i + 1] * Mk[3 + j] + Mc[3 * i + 2] * Mk[6 + j];
    }
    for (int i = 0; i < 9; ++i) Mc[i] = Mn[i];
    for (int i = 0; i < 3; ++i) mc[i] = mn[i];
}

// REG: the regularised variant (delta_w != 0: the column of s is loaded and the condensed entries corrected); the plain
// variant keeps that rarely needed code out of the hot loop
template <bool REG, class Fetch>
MS_HD bool riccati_backward_range_t(const Ctx& c, int s, int N, int kLo, int kHi, double mu, double delta, Fetch& fetch,
                                    double P[3][3], double p[3], double* Mc, double* mc, bool storeAll) {
    const double pn = c.cfg.withPn ? 1.0 : 0.0;
    if (kHi <= kLo) return true;
    fetch.start(c, s, kHi - 1, kLo, -1);
    int k = kHi - 1;
    // a failed inertia test leaves the sweep at once (copies still in flight are drained by the next fetch.start)
    double v[BwdFields::NF], K[3][3], kf[3];
    if (k == N - 1) {
        // last interval: terminal speed fixed, Fel eliminated (dense algebra, once per sweep)
        fetch.get(c, k, s, v);
        double vs[6];
        load_scol(c, k, s, vs);
        StageQP q;
        stage_build(v, vs, mu, delta, pn, true, q);
        if (!stage_riccati(q, true, pn, P, p, K, kf)) return false;
        if (storeAll || k == kLo) stage_store(c, k, s, K, kf, P, p);
        if (Mc) {
            double Mk[9], mk[3];
            for (int i = 0; i < 3; ++i) {
                mk[i] = q.r[i] + q.G[i][3] * kf[0] + q.G[i][4] * kf[1] + q.G[i][5] * kf[2];
                for (int j = 0; j < 3; ++j) Mk[3 * i + j] = q.G[i][j] + q.G[i][3] * K[0][j] + q.G[i][4] * K[1][j] + q.G[i][5] * K[2][j];
            }
            closed_loop_compose(Mc, mc, Mk, mk);
        }
        --k;
    }
    for (; k >= kLo; --k) {
        fetch.get(c, k, s, v);
        double vs[6];
        if (REG) load_scol(c, k, s, vs);
        if (!stage_riccati_sparse(v, REG ? vs : nullptr, mu, delta, pn, P, p, K, kf)) return false;
        if (storeAll || k == kLo) stage_store(c, k, s, K, kf, P, p);
        if (Mc) {
            const double tb = v[QP_TAU_B], tF = v[QP_TAU_F], pb = v[QP_PHI_B], pF = v[QP_PHI_F];
            const double kfw = kf[0] + pn * kf[1];
            double Mk[9], mk[3];
            mk[0] = v[QP_RT] + tF * kfw; mk[1] = v[QP_RB] + pF * kfw; mk[2] = kf[0];
            for (int j = 0; j < 3; ++j) {
                const double kw = K[0][j] + pn * K[1][j];
                Mk[j] = (j == 0 ? 1.0 : j == 1 ? tb : 0.0) + tF * kw;
                Mk[3 + j] = (j == 1 ? pb : 0.0) + pF * kw;
                Mk[6 + j] = K[0][j];
            }
            closed_loop_compose(Mc, mc, Mk, mk);
        }
    }
    return true;
}

template <class Fetch>
MS_HD bool riccati_backward_range(const Ctx& c, int s, int N, int kLo, int kHi, double mu, double delta, Fetch& fetch,
                                  double P[3][3], double p[3], double* Mc, double* mc, bool storeAll = true) {
    if (delta > 0.0) return riccati_backward_range_t<true>(c, s, N, kLo, kHi, mu, delta, fetch, P, p, Mc, mc, storeAll);
    return riccati_backward_range_t<false>(c, s, N, kLo, kHi, mu, delta, fetch, P, p, Mc, mc, storeAll);
}

template <class Fetch>
MS_HD bool riccati_backward(const Ctx& c, int s, int N, double mu, double delta, Fetch& fetch) {
    double P[3][3], p[3];
    terminal_value(c, s, N, mu, delta, P, p);
    return riccati_backward_range(c, s, N, 0, N, mu, delta, fetch, P, p, nullptr, nullptr);
}

// ---- forward sweep over the intervals kLo .. kHi-1 from d x_{kLo}: primal step ---------------------------------
// Writes d Fel, d Fpb of interval k and d t, d b of node k+1 into the step planes.  d s and the new coupling-row multipliers
// (costates of the stepped state) need nothing sequential and are evaluated by the interval-parallel cell_step.
template <class Fetch>
MS_HD void riccati_forward_range(const Ctx& c, int s, int N, int kLo, int kHi, double mu, double delta, Fetch& fetch, double dx[3]) {
    const Config& g = c.cfg;
    (void)mu; (void)delta;
    if (kHi <= kLo) return;
    fetch.start(c, s, kLo, kHi - 1, +1);
    double* st = &c.W(WS_ST, kLo, s);
    for (int k = kLo; k < kHi; ++k, st += REC_STRIDE) {
        double v[FwdFields::NF];
        fetch.get(c, k, s, v);
        const double du0 = v[6] + v[0] * dx[0] + v[1] * dx[1] + v[2] * dx[2];
        const double du1 = g.withPn ? v[7] + v[3] * dx[0] + v[4] * dx[1] + v[5] * dx[2] : 0.0;
        const double tb = v[8], tF = v[9], pb = v[10], pF = v[11], rt = v[12], rb = v[13];
        const double dF = du0 + du1;
        const double dtn = dx[0] + tb * dx[1] + tF * dF + rt;
        const double dbn = (k + 1 < N) ? pb * dx[1] + pF * dF + rb : 0.0;
        st[ST_FEL * 32] = du0;
        st[ST_FPB * 32] = du1;
        st[ST_T * 32 + REC_STRIDE] = dtn;
        st[ST_B * 32 + REC_STRIDE] = dbn;
        dx[0] = dtn; dx[1] = dbn; dx[2] = du0;
    }
}

template <class Fetch>
MS_HD void riccati_forward(const Ctx& c, int s, int N, double mu, double delta, Fetch& fetch) {
    double dx[3] = {0.0, 0.0, 0.0};
    c.W(WS_ST + ST_T, 0, s) = 0.0;
    c.W(WS_ST + ST_B, 0, s) = 0.0;
    riccati_forward_range(c, s, N, 0, N, mu, delta, fetch, dx);
}

// ---- KKT error of the current iterate: partial reduction over k = w, w+W, ... ------------------------------
struct KktAcc {
    double th, fo, slog, sdamp, zsum, ysum;   // sums
    double dinf, pinf, cmin, cmax;            // max / min
};
MS_HD void kkt_init(KktAcc& a) {
    a.th = a.fo = a.slog = a.sdamp = a.zsum = a.ysum = 0.0;
    a.dinf = a.pinf = a.cmax = 0.0; a.cmin = 1e300;
}
// 14 planes per interval: MS_KKT_U intervals per group, all loads of a group in flight together (the blocks of the reduction
// clusters have 128 threads, so the 56 values of four intervals stay in registers)
#ifndef MS_KKT_U
#define MS_KKT_U 4
#endif
MS_HD void kkt_partials(const Ctx& c, int s, int N, int it, int w, int W, KktAcc& a) {
    kkt_init(a);
    for (int k0 = w; k0 <= N; k0 += MS_KKT_U * W) {
        double v[MS_KKT_U][14];
#pragma unroll
        for (int u = 0; u < MS_KKT_U; ++u) {
            const int k = k0 + u * W;
            if (k <= N) {
                const double* q = &c.W(WS_PART, k, s);
                v[u][0] = q[PC_TH * 32]; v[u][1] = q[PC_F * 32]; v[u][2] = q[PC_SLOG * 32]; v[u][3] = q[PC_SDAMP * 32];
                v[u][4] = q[PC_ZSUM * 32]; v[u][5] = q[PC_YSUM * 32]; v[u][6] = q[PC_DINF * 32]; v[u][7] = q[PC_PINF * 32];
                v[u][8] = q[PC_CMIN * 32]; v[u][9] = q[PC_CMAX * 32];
                if (k >= 1) {   // stationarity w.r.t. the node variables couples interval k-1 and k
                    v[u][10] = q[PC_OWN_T * 32]; v[u][11] = c.W(it + IT_YT, k - 1, s);
                    if (k < N) { v[u][12] = q[PC_OWN_B * 32]; v[u][13] = c.W(WS_PART + PC_CN_B, k - 1, s); }
                }
            }
        }
#pragma unroll
        for (int u = 0; u < MS_KKT_U; ++u) {
            const int k = k0 + u * W;
            if (k <= N) {
                a.th += v[u][0]; a.fo += v[u][1]; a.slog += v[u][2]; a.sdamp += v[u][3]; a.zsum += v[u][4]; a.ysum += v[u][5];
                a.dinf = fmax(a.dinf, v[u][6]);
                a.pinf = fmax(a.pinf, v[u][7]);
                a.cmin = fmin(a.cmin, v[u][8]);
                a.cmax = fmax(a.cmax, v[u][9]);
                if (k >= 1) {
                    a.dinf = fmax(a.dinf, fabs(v[u][10] + v[u][11]));
                    if (k < N) a.dinf = fmax(a.dinf, fabs(v[u][12] + v[u][13]));
                }
            }
        }
    }
}
MS_HD void kkt_combine(KktAcc& a, const KktAcc& b) {
    a.th += b.th; a.fo += b.fo; a.slog += b.slog; a.sdamp += b.sdamp; a.zsum += b.zsum; a.ysum += b.ysum;
    a.dinf = fmax(a.dinf, b.dinf); a.pinf = fmax(a.pinf, b.pinf); a.cmin = fmin(a.cmin, b.cmin); a.cmax = fmax(a.cmax, b.cmax);
}

// ---- per-instance: KKT error, termination, barrier update                      (IPOPT Alg. A, steps A-1..A-3)
MS_HD void inst_kkt(const Ctx& c, int s, const KktAcc& a) {
    const Config& g = c.cfg;
    if (s >= g.nInst || c.I(SI_PHASE, s) != PH_EVAL) return;
    const int N = c.I(SI_N_INT, s);
    count_cells(c, 1, N + 1);
    // screening against a minimum trip duration that may arrive while the batch is running (computed concurrently by a
    // time-optimal solve on another stream): terminalTime is an upper bound on t_N (ocp.py:260-261)
    if (c.tmin) {
        const double tm = c.tmin[c.I(SI_ORIG, s)];
        if (tm > 0.0 && (c.P(P_T, s) - c.P(P_T0, s)) < tm * (1.0 - MS_TMIN_MARGIN)) { finish(c, s, ST_INFEASIBLE); return; }
    }
    const double th = a.th, fo = a.fo, dinf = a.dinf, pinf = a.pinf, cmin = a.cmin, cmax = a.cmax, zsum = a.zsum, ysum = a.ysum;
    // counts for the IPOPT error scaling s_d, s_c (eq. 6)
    const int nrow = (g.withPower ? 2 : 0) + 1 + (g.energy ? 2 : 0);
    const int nbRow = (g.withPower ? 4 : 0) + 2 + (g.energy ? 2 : 0);
    const int nb = N * (2 + (g.withPn ? 2 : 0) + 1 + nbRow) + (N - 1) * 4 + 2;
    const int mrows = N * (nrow + 2);
    const double sd = fmax(100.0, (ysum + zsum) / (mrows + nb)) / 100.0;
    const double sc = fmax(100.0, zsum / nb) / 100.0;
    const double E0 = fmax(fmax(dinf / sd, pinf), cmax / sc);
    c.D(SD_THETA, s) = th; c.D(SD_FOBJ, s) = fo; c.D(SD_SLOG, s) = a.slog; c.D(SD_SDAMP, s) = a.sdamp;
    c.D(SD_KKT, s) = E0; c.D(SD_DINF, s) = dinf; c.D(SD_PINF, s) = pinf; c.D(SD_CINF, s) = cmax;
    if (c.D(SD_THETA_MAX, s) < 0.0) {
        c.D(SD_THETA_MAX, s) = 1e4 * fmax(1.0, th);
        c.D(SD_THETA_MIN, s) = 1e-4 * fmax(1.0, th);
    }
    if (!isfinite(E0) || !isfinite(fo)) { finish(c, s, ST_INVALID_NUMBER); return; }
    if (E0 <= g.tol) { finish(c, s, ST_SOLVE_SUCCEEDED); return; }
    // acceptable level for MS_ACCEPTABLE_ITER consecutive iterations (IPOPT default acceptable_iter 15)
    if (acceptable_point(c, s)) {
        if (++c.I(SI_NACC, s) >= MS_ACCEPTABLE_ITER) { finish(c, s, ST_ACCEPTABLE); return; }
    } else c.I(SI_NACC, s) = 0;
    if (c.I(SI_ITERS, s) >= g.maxIter) { finish(c, s, ST_MAXITER); return; }
    // stall watchdog (batch throughput): an instance that cycles around a kink of a non-smooth loss map would otherwise hold
    // the whole lock-step batch until max_iter; it ends with the status it would end with anyway
    if (g.stallIters > 0) {
        const double best = c.D(SD_KKT_BEST, s);
        // counted in trial evaluations (lock-step ticks), which is what a straggler costs the batch
        if (best <= 0.0 || E0 < 0.9 * best) { c.D(SD_KKT_BEST, s) = E0; c.I(SI_LAST_GAIN, s) = c.I(SI_TICKS, s); }
        else if (c.I(SI_TICKS, s) - c.I(SI_LAST_GAIN, s) > g.stallIters) { finish(c, s, acceptable_point(c, s) ? ST_ACCEPTABLE : ST_MAXITER); return; }
    }
    // ---- monotone barrier update (eq. 7), filter reset
    double mu = c.D(SD_MU, s);
    for (;;) {
        const double cinf = fmax(cmax - mu, mu - cmin);
        const double Emu = fmax(fmax(dinf / sd, pinf), cinf / sc);
        if (Emu <= 10.0 * mu && mu > g.tol / 10.0 * (1.0 + 1e-12)) {
            mu = fmax(g.tol / 10.0, fmin(0.2 * mu, pow(mu, 1.5)));
            c.I(SI_NFILT, s) = 0;
        } else break;
    }
    c.D(SD_MU, s) = mu; c.D(SD_TAU, s) = fmax(0.99, 1.0 - mu);
    c.I(SI_PHASE, s) = PH_FACTOR;
}

// ---- per-instance: search direction with inertia correction                     (IPOPT Alg. A step A-4, Alg. IC)
template <class FetchB, class FetchF>
MS_HD void inst_step(const Ctx& c, int s, FetchB& fb, FetchF& ff) {
    const Config& g = c.cfg;
    if (s >= g.nInst || c.I(SI_PHASE, s) != PH_FACTOR) return;
    const int N = c.I(SI_N_INT, s);
    const double mu = c.D(SD_MU, s);
    double delta = 0.0;
    const double dlast = c.D(SD_DELTA_LAST, s);
    bool ok = false;
    for (int tries = 0; tries < 40; ++tries) {
        count_cells(c, 2, N);
        if (riccati_backward(c, s, N, mu, delta, fb)) { ok = true; break; }
        c.I(SI_NREG, s) += 1;
        if (delta == 0.0) delta = (dlast == 0.0) ? 1e-4 : fmax(1e-20, dlast / 3.0);
        else delta *= (dlast == 0.0) ? 100.0 : 8.0;
        if (delta > 1e40) break;
    }
    if (!ok) { finish(c, s, ST_STEP_FAILED); return; }
    if (delta > 0.0) c.D(SD_DELTA_LAST, s) = delta;
    c.D(SD_DELTA, s) = delta;
    count_cells(c, 3, N);
    riccati_forward(c, s, N, mu, delta, ff);
    c.I(SI_FACT, s) = 1;
    c.I(SI_PHASE, s) = PH_STEPPED;
}

// ---- interval-parallel part of the step --------------------------------------------------------------------
// fraction-to-boundary limits of one cell, kept as fractions: the smallest ratio slack / (-d slack) (and z / (-d z)) of the bounds
// seen so far is nP / dP (nZ / dZ), compared by cross-multiplication -- one division per cell instead of one per bound
struct Ftb {
    double nP, dP, nZ, dZ, gphid;
};
MS_HD void ftb_bound(Ftb& f, double tau, double mu, double z, double slack, double dvSigned, bool oneSided) {
    // dvSigned = change of the slack; primal fraction-to-boundary (eq. 15a), dual step (eq. 15b), barrier slope
    (void)tau;
    if (dvSigned < 0.0 && slack * f.dP < f.nP * (-dvSigned)) { f.nP = slack; f.dP = -dvSigned; }
    const double r = rcp_slack(slack);
    const double dz = mu * r - z - (z * r) * dvSigned;
    if (dz < 0.0 && z * f.dZ < f.nZ * (-dz)) { f.nZ = z; f.dZ = -dz; }
    f.gphid += (-mu * r + (oneSided ? MS_KAPPA_D * mu : 0.0)) * dvSigned;
}

// DYN = false (no or constant-efficiency loss rows): the gradients and residuals of the inequality rows are cheap functions
// of the iterate this kernel loads anyway, so they are recomputed here -- bit for bit, see mul_rn -- instead of being stored
// by cell_eval and read back (16 planes less traffic in each of the two kernels); with the spline loss map they come from
// the stage-QP record.
template <bool DYN, bool INTL = false>
MS_HD void cell_step(const Ctx& c, int k, int s) {
    const Config& g = c.cfg;
    if (s >= g.nInst || c.I(SI_PHASE, s) != PH_STEPPED) return;
    const int N = c.I(SI_N_INT, s);
    if (k > N) return;
    const int it = c.I(SI_PARITY, s) ? WS_IT1 : WS_IT0;
    // ---- all loads first, then arithmetic, then all stores (loads must not queue behind stores through the same base)
    const int kn = (k < N) ? k + 1 : N, km = (k > 0) ? k - 1 : 0;
    double CI[IT_N], CS[ST_N], RP[9];
    constexpr int NQJ = DYN ? (QP_N - QP_H_BSL) : (QP_J_P0_B - QP_H_BSL);      // planes read from the stage-QP record
    double QJ[NQJ];
    {
        const double* ip = &c.W(it, k, s);
        const double* sp = &c.W(WS_ST, k, s);
        const double* qp = &c.W(WS_QP + QP_H_BSL, k, s);
        const double* rp = &c.W(WS_RIC + RIC_P, kn, s);       // value function of the next node: P (tt,tb,tf,bb,bf,ff), p
#pragma unroll
        for (int f = 0; f < IT_N; ++f) CI[f] = ip[f * 32];
#pragma unroll
        for (int f = 0; f < ST_N; ++f) CS[f] = sp[f * 32];
#pragma unroll
        for (int f = 0; f < NQJ; ++f) QJ[f] = qp[f * 32];
#pragma unroll
        for (int f = 0; f < 9; ++f) RP[f] = rp[f * 32];
    }
    const double dbn = c.W(WS_ST + ST_B, kn, s), dtn = c.W(WS_ST + ST_T, kn, s);
    const double bNext = DYN ? 0.0 : c.W(it + IT_B, kn, s);
    IntervalCoef q;
    if (!DYN) q = load_coef(c, (k < N) ? k : km, s);
    // last interval only: b_N is fixed, the multiplier of its row follows from stationarity w.r.t. Fel (see below)
    double LQ[8] = {0, 0, 0, 0, 0, 0, 0, 1.0};
    if (k == N - 1) {
        const double* q = &c.W(WS_QP, k, s);
        LQ[0] = q[QP_G0_FEL * 32]; LQ[1] = q[QP_G1_FEL * 32]; LQ[2] = q[QP_H_BFEL * 32]; LQ[3] = q[QP_H_FFEL * 32];
        LQ[4] = q[QP_H_FELFEL * 32]; LQ[5] = q[QP_H_FELFPB * 32]; LQ[6] = q[QP_TAU_F * 32]; LQ[7] = q[QP_PHI_F * 32];
    }
    const double pFel = c.W(it + IT_FEL, km, s), pDFel = c.W(WS_ST + ST_FEL, km, s);
    const double dsk = c.W(WS_TRK + TRK_DS, k, s);
    const Bnd B = load_bounds(c, k, s);
    const double mu = c.D(SD_MU, s), tauF = c.D(SD_TAU, s), iscale = rcp_slack(c.P(P_SCALE, s));
#define MS_QJ(F) QJ[(F) - QP_H_BSL]
    Ftb f{1.0, tauF, 1.0, tauF, 0.0};          // ratio 1 / tau: alpha = tau * ratio = 1 unless a bound is closer
    double OW[NROW], OYD[NROW], oyt = 0.0, oyb = 0.0, ods = 0.0;
#pragma unroll
    for (int j = 0; j < NROW; ++j) { OW[j] = 0.0; OYD[j] = 0.0; }
    const double dt = CS[ST_T], db = CS[ST_B];
    if (k >= 1) {
        const double t = CI[IT_T];
        ftb_bound(f, tauF, mu, CI[IT_Z + Z_T_L], t - B.tL, dt, false);
        ftb_bound(f, tauF, mu, CI[IT_Z + Z_T_U], B.tU - t, -dt, false);
        if (k < N) {
            const double b = CI[IT_B];
            ftb_bound(f, tauF, mu, CI[IT_Z + Z_B_L], b - B.bL, db, false);
            ftb_bound(f, tauF, mu, CI[IT_Z + Z_B_U], B.bU - b, -db, false);
        }
    }
    if (k < N) {
        const double du0 = CS[ST_FEL], du1 = CS[ST_FPB];
        // d s from its own stationarity row (s was eliminated from the stage QP before the sweep):
        //   (H_ss + delta) ds + H_bs db + H_Fs dFel + H_Qs dFpb + g_s = 0
        const double delta = c.D(SD_DELTA, s);
        const double sX = MS_QJ(QP_G0_SL) + mu * MS_QJ(QP_G1_SL) + MS_QJ(QP_H_BSL) * db + MS_QJ(QP_H_FELSL) * du0 + MS_QJ(QP_H_FPBSL) * du1;
        const double isd = rcp(MS_QJ(QP_H_SLSL) + delta);
        const double du2 = -sX * isd;
        ods = du2;
        const double fel = CI[IT_FEL], fpb = CI[IT_FPB], sl = CI[IT_SL];
        // gradients and residuals of the inequality rows: from the stage-QP record (DYN) or recomputed with the expressions of
        // cell_eval (ocp.py:189,199,225-226 with constant efficiencies)
        double jP0b, jP0f, jP1f, jP1n, jAccb, jLtrF, jLtrB, jLtrN, jLrgF, jLrgB, jLrgN, rres[NROW];
        if (DYN) {
            jP0b = MS_QJ(QP_J_P0_B); jP0f = MS_QJ(QP_J_P0_FEL); jP1f = MS_QJ(QP_J_P1_FEL); jP1n = MS_QJ(QP_J_P1_BN);
            jAccb = MS_QJ(QP_J_ACC_B);
            jLtrF = MS_QJ(QP_J_LTR_FEL); jLtrB = MS_QJ(QP_J_LTR_B); jLtrN = MS_QJ(QP_J_LTR_BN);
            jLrgF = MS_QJ(QP_J_LRG_FEL); jLrgB = MS_QJ(QP_J_LRG_B); jLrgN = MS_QJ(QP_J_LRG_BN);
#pragma unroll
            for (int j = 0; j < NROW; ++j) rres[j] = MS_QJ(QP_RES + j);
        } else {
            const double bk = CI[IT_B];
            double v0, v1, iv0, iv1;
            sqrt_inv(bk, v0, iv0);
            sqrt_inv(bNext, v1, iv1);
            double dval[NROW];
            ineq_values<false>(c, s, fel, fpb, sl, bk, bNext, q, dval);
            jP0b = 0.5 * fel * iv0; jP0f = v0; jP1f = v1; jP1n = 0.5 * fel * iv1;
            jAccb = -(0.5 * q.sr1 * iv0 + q.sr2);
            jLtrF = -c.P(P_CT, s); jLtrB = 0.0; jLtrN = 0.0;
            jLrgF = c.P(P_CR, s); jLrgB = 0.0; jLrgN = 0.0;
#pragma unroll
            for (int j = 0; j < NROW; ++j) rres[j] = row_on(g, j) ? sub_rn(dval[j], CI[IT_W + j]) : 0.0;
        }
        // new coupling-row multipliers = minus the costates of the stepped state: gradient of the value function of the
        // backward sweep at node k+1, plus the terms of this interval that depend on b_{k+1} directly
        const double pit = RP[6] + RP[0] * dtn + RP[1] * dbn + RP[2] * du0;
        double pib;
        if (k + 1 < N) {
            pib = RP[7] + RP[1] * dtn + RP[3] * dbn + RP[4] * du0
                + MS_QJ(QP_HC_B) * db + MS_QJ(QP_HC_FEL) * du0 + MS_QJ(QP_HC_FPB) * du1 + MS_QJ(QP_HC_SL) * du2
                + MS_QJ(QP_HPP) * dbn + MS_QJ(QP_GP0) + mu * MS_QJ(QP_GP1);
        } else {
            const double dfk = (k >= 1) ? pDFel : 0.0;        // d f_k = d Fel_{k-1}
            // stationarity w.r.t. Fel in the condensed entries; the last term vanishes unless delta_w != 0
            const double gF = LQ[0] + mu * LQ[1] + LQ[2] * db + LQ[3] * dfk + (LQ[4] + delta) * du0 + LQ[5] * du1
                            + MS_QJ(QP_H_FELSL) * sX * (rcp(MS_QJ(QP_H_SLSL)) - isd);
            pib = -(gF + LQ[6] * pit) / LQ[7];
        }
        oyt = -pit - CI[IT_YT];
        oyb = -pib - CI[IT_YB];
        ftb_bound(f, tauF, mu, CI[IT_Z + Z_FEL_L], fel - B.felL, du0, false);
        ftb_bound(f, tauF, mu, CI[IT_Z + Z_FEL_U], B.felU - fel, -du0, false);
        if (g.withPn) {
            ftb_bound(f, tauF, mu, CI[IT_Z + Z_FPB_L], fpb - B.fpbL, du1, false);
            ftb_bound(f, tauF, mu, CI[IT_Z + Z_FPB_U], B.fpbU - fpb, -du1, false);
        }
        ftb_bound(f, tauF, mu, CI[IT_Z + Z_SL_L], sl - B.slL, du2, true);
        // objective part of the barrier directional derivative
        if (g.energy) {
            f.gphid += (dsk * du0 + (INTL ? 1.0 : dsk) * du2) * iscale;
            if (k >= 1) f.gphid += (2e-3 * iscale) * (fel - pFel) * (du0 - pDFel);
        } else {
            f.gphid += (2e-4 * iscale) * (fel * du0 + fpb * du1);
        }
        // inequality rows: slack step d w = J d + (d(x) - w), multiplier step from the condensed equations
#pragma unroll
        for (int j = 0; j < NROW; ++j) {
            if (!row_on(g, j)) continue;
            double jd;
            if (j == R_P0) jd = jP0b * db + jP0f * du0;
            else if (j == R_P1) jd = jP1f * du0 + jP1n * dbn;
            else if (j == R_ACC) jd = jAccb * db + du0 + du1;
            else if (j == R_LTR) jd = du2 + jLtrF * du0 + jLtrB * db + jLtrN * (INTL ? du1 : dbn);      // INTL: coefficient of Fpb_k
            else jd = du2 + jLrgF * du0 + jLrgB * db + jLrgN * (INTL ? du1 : dbn);
            const double dw = jd + rres[j];
            double L, U; bool hasU;
            row_bounds(B, j, L, U, hasU);
            const int zl = (j == R_P0) ? Z_P0_L : (j == R_P1) ? Z_P1_L : (j == R_ACC) ? Z_ACC_L : (j == R_LTR) ? Z_LTR_L : Z_LRG_L;
            const double w = CI[IT_W + j];
            const double vL = CI[IT_Z + zl], sL = w - L;
            const double rL = rcp_slack(sL);
            double sig = vL * rL, gw = -mu * rL + (hasU ? 0.0 : MS_KAPPA_D * mu);
            ftb_bound(f, tauF, mu, vL, sL, dw, !hasU);
            if (hasU) {
                const double vU = CI[IT_Z + zl + 1], sU = U - w;
                const double rU = rcp_slack(sU);
                sig += vU * rU; gw += mu * rU;
                ftb_bound(f, tauF, mu, vU, sU, -dw, false);
            }
            OW[j] = dw;
            OYD[j] = sig * dw + gw - CI[IT_YD + j];
        }
    } else if (!g.energy) {
        f.gphid += dt * iscale;
    }
#undef MS_QJ
    if (k < N) {
        c.W(WS_ST + ST_SL, k, s) = ods;
        c.W(WS_ST + ST_YT, k, s) = oyt;
        c.W(WS_ST + ST_YB, k, s) = oyb;
#pragma unroll
        for (int j = 0; j < NROW; ++j) { c.W(WS_ST + ST_W + j, k, s) = OW[j]; c.W(WS_ST + ST_YD + j, k, s) = OYD[j]; }
    }
    c.W(WS_PART + PS_AP, k, s) = fmin(1.0, tauF * f.nP / f.dP);
    c.W(WS_PART + PS_AZ, k, s) = fmin(1.0, tauF * f.nZ / f.dZ);
    c.W(WS_PART + PS_GPHID, k, s) = f.gphid;
}

// ---- step-size limits of one instance and the first trial step size ----------------------------------------
MS_HD void alpha_partials(const Ctx& c, int s, int N, int w, int W, double* acc) {
    acc[0] = 1.0; acc[1] = 1.0; acc[2] = 0.0;
    for (int k0 = w; k0 <= N; k0 += MS_RED_U * W) {
        double v[MS_RED_U][3];
#pragma unroll
        for (int u = 0; u < MS_RED_U; ++u) {
            const int k = k0 + u * W;
            if (k <= N) {
                const double* q = &c.W(WS_PART + PS_AP, k, s);
                v[u][0] = q[0]; v[u][1] = q[32]; v[u][2] = q[64];
            }
        }
#pragma unroll
        for (int u = 0; u < MS_RED_U; ++u)
            if (k0 + u * W <= N) { acc[0] = fmin(acc[0], v[u][0]); acc[1] = fmin(acc[1], v[u][1]); acc[2] += v[u][2]; }
    }
}

MS_HD void inst_alpha(const Ctx& c, int s, const double* red) {
    const Config& g = c.cfg;
    if (s >= g.nInst || c.I(SI_PHASE, s) != PH_STEPPED) return;
    const double aP = red[0], aZ = red[1], gphid = red[2];
    if (!isfinite(gphid) || !isfinite(aP) || !isfinite(aZ)) { finish(c, s, ST_STEP_FAILED); return; }
    const double th = c.D(SD_THETA, s);
    double amin;
    if (gphid < 0.0) {                                   // eq. (23)
        amin = 1e-5;
        if (th > 0.0) amin = fmin(amin, 1e-8 * th / (-gphid));
        if (th <= c.D(SD_THETA_MIN, s)) amin = fmin(amin, pow(th, 1.1) / pow(-gphid, 2.3));
        amin *= 0.05;
    } else amin = 0.05 * 1e-5;
    c.D(SD_GPHID, s) = gphid;
    c.D(SD_ALPHA, s) = aP;
    c.D(SD_ALPHA_Z, s) = aZ;
    c.D(SD_ALPHA_MIN, s) = amin;
    c.I(SI_NLS, s) = 0;
    c.I(SI_PHASE, s) = PH_TRIAL;
}

}  // namespace mseetc
