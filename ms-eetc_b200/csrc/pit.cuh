// Parallel-in-time Riccati sweeps: G lanes per instance, each lane owns a contiguous chunk of shooting intervals.
//
// A chunk of consecutive intervals [kLo, kHi) maps the value function (Pi, pi) at its end node to the value function at its
// start node by a linear-fractional transformation (Sarkka & Garcia-Fernandez, "Temporal parallelization of dynamic
// programming and linear quadratic control", IEEE TAC 2023).  Here its coefficients are what a Riccati recursion from a
// REFERENCE terminal value (Pref, pref) produces anyway -- value function (Pbar, pbar) at the chunk start, closed-loop
// transition x_e = Phi x_a + phi under the reference gains -- plus the closed-loop controllability Gramian
//     W = sum_j Phi_{e<-j+1} B Rt_j^{-1} B' Phi_{e<-j+1}'            (Rt_j: reduced control Hessian of interval j)
// With dPi = Pi - Pref, dpi = pi - pref:
//     P_a = Pbar + Phi' T Phi,     T = (I + dPi W)^{-1} dPi = (dPi^{-1} + W)^{-1}     (symmetric)
//     p_a = pbar + Phi' (dpi + T (phi - W dpi))
// The reference is the value function the previous interior-point iteration left at the chunk-end node (zero before the
// first factorisation): the element then comes from a recursion that is as well conditioned as the sequential sweep (a zero
// terminal value is not: with free controls and next to no control cost the zero-terminal problem of a chunk is nearly
// singular and its element loses 6-7 digits), and the correction shrinks as the iteration converges -- exactly when the
// direction has to be accurate.  Elements are accumulated by the structure-exploiting stage recursion of riccati.cuh and only
// ever applied to a value function (never combined with each other):
//   phase A   every chunk but the first and the last: reference recursion -> element (27 numbers); the last chunk runs the
//             ordinary recursion from the terminal node (exact) and keeps its factors
//   chain     the value functions at the chunk ends follow one after the other, last chunk first: G - 2 applications of an
//             element (3x3 elimination with row pivoting each)
//   phase C   ordinary recursion inside every chunk from its end value: gains, value functions, exact inertia test; closed-loop
//             transition of the chunk
//   chain     state step at the chunk starts (G affine maps applied one after the other)
//   phase F   forward sweep inside every chunk
// Measured on the host emulation (tests/hostsim): identical iteration counts and statuses to the sequential sweeps for
// 8 / 16 / 32 lanes on every parity case; the directions agree to ~1e-13 relative.
#pragma once
#include "riccati.cuh"
#if !defined(__CUDACC__)
#include <vector>
#endif

namespace mseetc {

MS_HD void sym_to_full(const double* s, double F[3][3]) {
    F[0][0] = s[0]; F[0][1] = F[1][0] = s[1]; F[0][2] = F[2][0] = s[2];
    F[1][1] = s[3]; F[1][2] = F[2][1] = s[4]; F[2][2] = s[5];
}
MS_HD void full_to_sym(const double F[3][3], double* s) {
    s[0] = F[0][0]; s[1] = 0.5 * (F[0][1] + F[1][0]); s[2] = 0.5 * (F[0][2] + F[2][0]);
    s[3] = F[1][1]; s[4] = 0.5 * (F[1][2] + F[2][1]); s[5] = F[2][2];
}

// chunk geometry: the generic intervals 0 .. N-2 are split over G lanes; interval N-1 (terminal-speed elimination)
// belongs to lane G-1 in addition to its chunk
MS_HD void pit_chunk(int N, int G, int lane, int& kLo, int& kHi) {
    const int Ng = N - 1;
    const int L = (Ng + G - 1) / G;
    kLo = lane * L; if (kLo > Ng) kLo = Ng;
    kHi = kLo + L; if (kHi > Ng) kHi = Ng;
}

// affine map x -> M x + m
struct Aff {
    double M[9], m[3];
};
MS_HD void aff_identity(Aff& a) {
    for (int i = 0; i < 9; ++i) a.M[i] = 0.0;
    a.M[0] = a.M[4] = a.M[8] = 1.0;
    a.m[0] = a.m[1] = a.m[2] = 0.0;
}

struct ChunkElem {
    double P[6], p[3], Phi[9], phi[3], W[6];      // P, W symmetric: (00,01,02,11,12,22)
};

template <bool REG, class Fetch>
MS_HD bool chunk_element_t(const Ctx& c, int s, int kLo, int kHi, double mu, double delta, Fetch& fetch, const double* refP, const double* refp,
                           ChunkElem& E) {
    const double pn = c.cfg.withPn ? 1.0 : 0.0;
    double P[3][3], p[3];
    sym_to_full(refP, P);
    for (int i = 0; i < 3; ++i) p[i] = refp[i];
    for (int i = 0; i < 9; ++i) E.Phi[i] = 0.0;
    E.Phi[0] = E.Phi[4] = E.Phi[8] = 1.0;
    for (int i = 0; i < 3; ++i) E.phi[i] = 0.0;
    for (int i = 0; i < 6; ++i) E.W[i] = 0.0;
    if (kHi > kLo) {
        fetch.start(c, s, kHi - 1, kLo, -1);
        for (int k = kHi - 1; k >= kLo; --k) {
            double v[BwdFields::NF], vs[6], K[3][3], kf[3], cb[4];
            fetch.get(c, k, s, v);
            if (REG) load_scol(c, k, s, vs);
            if (!stage_riccati_sparse(v, REG ? vs : nullptr, mu, delta, pn, P, p, K, kf, cb)) return false;
            const double tb = v[QP_TAU_B], tF = v[QP_TAU_F], pb = v[QP_PHI_B], pF = v[QP_PHI_F];
            // Gramian: W += Y Rt^{-1} Y',  Y = Phi_{e<-k+1} B,  B = [(tF, pF, 1)  pn (tF, pF, 0)]
            double yF[3], yQ[3], xF[3], xQ[3];
            for (int i = 0; i < 3; ++i) {
                const double g = E.Phi[3 * i] * tF + E.Phi[3 * i + 1] * pF;
                yF[i] = g + E.Phi[3 * i + 2]; yQ[i] = pn * g;
                sym2_solve(cb[0], cb[1], cb[2], cb[3], yF[i], yQ[i], xF[i], xQ[i]);
            }
            E.W[0] += yF[0] * xF[0] + yQ[0] * xQ[0]; E.W[1] += yF[0] * xF[1] + yQ[0] * xQ[1]; E.W[2] += yF[0] * xF[2] + yQ[0] * xQ[2];
            E.W[3] += yF[1] * xF[1] + yQ[1] * xQ[1]; E.W[4] += yF[1] * xF[2] + yQ[1] * xQ[2]; E.W[5] += yF[2] * xF[2] + yQ[2] * xQ[2];
            // closed loop of this interval under the zero-terminal gains, composed onto the transition of the intervals behind it
            const double kfw = kf[0] + pn * kf[1];
            double Mk[9], mk[3];
            mk[0] = v[QP_RT] + tF * kfw; mk[1] = v[QP_RB] + pF * kfw; mk[2] = kf[0];
            for (int j = 0; j < 3; ++j) {
                const double kw = K[0][j] + pn * K[1][j];
                Mk[j] = (j == 0 ? 1.0 : j == 1 ? tb : 0.0) + tF * kw;
                Mk[3 + j] = (j == 1 ? pb : 0.0) + pF * kw;
                Mk[6 + j] = K[0][j];
            }
            closed_loop_compose(E.Phi, E.phi, Mk, mk);
        }
    }
    full_to_sym(P, E.P);
    for (int i = 0; i < 3; ++i) E.p[i] = p[i];
    return true;
}
template <class Fetch>
MS_HD bool chunk_element(const Ctx& c, int s, int kLo, int kHi, double mu, double delta, Fetch& fetch, const double* refP, const double* refp,
                         ChunkElem& E) {
    if (delta > 0.0) return chunk_element_t<true>(c, s, kLo, kHi, mu, delta, fetch, refP, refp, E);
    return chunk_element_t<false>(c, s, kLo, kHi, mu, delta, fetch, refP, refp, E);
}

// Value function at the start of a chunk from the one at its end, given as a difference to the reference value the element was
// accumulated with:   T = (I + dPi W)^{-1} dPi   (dPi symmetric, not necessarily definite; T symmetrised).
MS_HD bool chunk_apply_diff(const ChunkElem& E, const double dPi[3][3], const double dpi[3], double P[3][3], double p[3]) {
    double W[3][3];
    sym_to_full(E.W, W);
    // X = I + dPi W, equilibrated and inverted through its adjugate: four independent reciprocals and a short dependent chain --
    // this routine is the step of a sequential chain over the chunks.  The equilibrated X is moderately conditioned whenever the
    // reference and the true terminal value both give the right inertia; a tiny determinant fails the instance over to the
    // sequential sweeps.
    double X[3][3], D[3][3];
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j) X[i][j] = (i == j ? 1.0 : 0.0) + dPi[i][0] * W[0][j] + dPi[i][1] * W[1][j] + dPi[i][2] * W[2][j];
        // rows of very different size (a barrier term of 1e9 next to O(1) entries): equilibrate X T = dPi row by row
        const double big = fmax(fmax(fabs(X[i][0]), fabs(X[i][1])), fabs(X[i][2]));
        if (!(big > 0.0) || !isfinite(big)) return false;
        const double r = rcp(big);
        for (int j = 0; j < 3; ++j) { X[i][j] *= r; D[i][j] = dPi[i][j] * r; }
    }
    double A[3][3];
    A[0][0] = X[1][1] * X[2][2] - X[1][2] * X[2][1]; A[0][1] = X[0][2] * X[2][1] - X[0][1] * X[2][2]; A[0][2] = X[0][1] * X[1][2] - X[0][2] * X[1][1];
    A[1][0] = X[1][2] * X[2][0] - X[1][0] * X[2][2]; A[1][1] = X[0][0] * X[2][2] - X[0][2] * X[2][0]; A[1][2] = X[0][2] * X[1][0] - X[0][0] * X[1][2];
    A[2][0] = X[1][0] * X[2][1] - X[1][1] * X[2][0]; A[2][1] = X[0][1] * X[2][0] - X[0][0] * X[2][1]; A[2][2] = X[0][0] * X[1][1] - X[0][1] * X[1][0];
    const double det = X[0][0] * A[0][0] + X[0][1] * A[1][0] + X[0][2] * A[2][0];
    if (!(fabs(det) > 1e-9) || !isfinite(det)) return false;
    const double idet = rcp(det);
    double T[3][3];
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) T[i][j] = (A[i][0] * D[0][j] + A[i][1] * D[1][j] + A[i][2] * D[2][j]) * idet;
    for (int i = 0; i < 3; ++i)
        for (int j = i + 1; j < 3; ++j) { const double x = 0.5 * (T[i][j] + T[j][i]); T[i][j] = x; T[j][i] = x; }
    // P = Pbar + Phi' T Phi ;  p = pbar + Phi' (dpi + T (phi - W dpi))
    double TP[3][3], w[3], u[3];
    for (int i = 0; i < 3; ++i) {
        w[i] = E.phi[i] - (W[i][0] * dpi[0] + W[i][1] * dpi[1] + W[i][2] * dpi[2]);
        for (int j = 0; j < 3; ++j) TP[i][j] = T[i][0] * E.Phi[j] + T[i][1] * E.Phi[3 + j] + T[i][2] * E.Phi[6 + j];
    }
    for (int i = 0; i < 3; ++i) u[i] = dpi[i] + T[i][0] * w[0] + T[i][1] * w[1] + T[i][2] * w[2];
    double Pb[3][3];
    sym_to_full(E.P, Pb);
    for (int i = 0; i < 3; ++i) {
        p[i] = E.p[i] + (E.Phi[i] * u[0] + E.Phi[3 + i] * u[1] + E.Phi[6 + i] * u[2]);
        for (int j = i; j < 3; ++j) {
            const double x = Pb[i][j] + (E.Phi[i] * TP[0][j] + E.Phi[3 + i] * TP[1][j] + E.Phi[6 + i] * TP[2][j]);
            P[i][j] = x; P[j][i] = x;
        }
    }
    for (int i = 0; i < 3; ++i) { if (!isfinite(p[i])) return false; for (int j = 0; j < 3; ++j) if (!isfinite(P[i][j])) return false; }
    return true;
}

// ---- the lanes of one instance exchange elements, chunk-end values, chunk transitions and chunk-start states through a small
// buffer (shared memory on the device, a plain array in the host emulation): SH_N doubles per (chunk, instance)
enum PitShareField {
    SH_E = 0,                 // element of the chunk (27 numbers)
    SH_TR = SH_E + 12,        // later, in the same slot: closed-loop transition of the chunk (12)
    SH_REF = SH_E + 27,       // reference terminal value of the chunk (P 6, p 3); later the state step at the chunk start (3)
    SH_N = SH_REF + 9
};
// The value function at the END of chunk l (P 6, p 3) lives in the first 9 numbers of the element slot of chunk l + 1: the chain
// writes it there when it has consumed that element (the last chunk has no element: its slot takes the exact value of its start).
#define SH_PE_AT(sh, i, l, col) (sh).at(SH_E + (i), (l) + 1, col)
enum {
    PIT_BAD_INERTIA = 1,       // exact inertia test of an in-chunk recursion failed: regularise (delta_w ladder) and retry
    PIT_ELEM_FAILED = 2,       // reference recursion of a chunk not positive definite
    PIT_APPLY_FAILED = 4,      // I + dPi W numerically singular
    PIT_INCONSISTENT = 8,      // chain and recursion disagree on a chunk-end value function
    PIT_SCAN_FAILED = PIT_ELEM_FAILED | PIT_APPLY_FAILED | PIT_INCONSISTENT      // any of them: sequential sweeps
};
struct PitShare {
    double* base;      // [chunk][SH_N][width]
    int* flags;        // [width]: PIT_BAD_INERTIA | PIT_SCAN_FAILED
    int width;         // instances that share the buffer (a block's SL; 1 in the host emulation)
    MS_HD double& at(int field, int chunk, int col) const { return base[((size_t)chunk * SH_N + field) * width + col]; }
#if defined(__CUDA_ARCH__)
    __device__ void raise(int col, int bit) const { atomicOr(flags + col, bit); }
#else
    void raise(int col, int bit) const { flags[col] |= bit; }
#endif
};
// value functions agree when chain and recursion differ by less than this (relative to the largest entry); beyond it the
// instance is handed to the sequential sweeps
#define PIT_CONSISTENCY_TOL 1e-6

struct PitLane {
    int s, col, l, G, N, kLo, kHi;
    double mu, delta;
    double refP[6], refp[3];
};

// phase 0: reference terminal value of the chunk = what the previous factorisation left at its end node
MS_HD void pit_read_reference(const Ctx& c, PitLane& t) {
    const bool have = c.I(SI_FACT, t.s) != 0 && t.l >= 1 && t.l <= t.G - 2;
    for (int i = 0; i < 6; ++i) t.refP[i] = have ? c.W(WS_RIC + RIC_P + i, t.kHi, t.s) : 0.0;
    for (int i = 0; i < 3; ++i) t.refp[i] = have ? c.W(WS_RIC + RIC_PV + i, t.kHi, t.s) : 0.0;
}

// phase A: element of an inner chunk; the last chunk runs the ordinary recursion from the terminal node
template <class Fetch>
MS_HD void pit_phase_a(const Ctx& c, const PitLane& t, const PitShare& sh, Fetch& fb) {
    if (t.l >= 1 && t.l <= t.G - 2) {
        ChunkElem E;
        if (!chunk_element(c, t.s, t.kLo, t.kHi, t.mu, t.delta, fb, t.refP, t.refp, E)) { sh.raise(t.col, PIT_ELEM_FAILED); return; }
        const double* e = (const double*)&E;
        for (int i = 0; i < 27; ++i) sh.at(SH_E + i, t.l, t.col) = e[i];
        for (int i = 0; i < 6; ++i) sh.at(SH_REF + i, t.l, t.col) = t.refP[i];
        for (int i = 0; i < 3; ++i) sh.at(SH_REF + 6 + i, t.l, t.col) = t.refp[i];
    } else if (t.l == t.G - 1) {
        double P[3][3], p[3];
        Aff T;
        aff_identity(T);
        terminal_value(c, t.s, t.N, t.mu, t.delta, P, p);
        if (!riccati_backward_range(c, t.s, t.N, t.kLo, t.N, t.mu, t.delta, fb, P, p, T.M, T.m)) { sh.raise(t.col, PIT_BAD_INERTIA); return; }
        if (t.G >= 2) {
            double sy[6];
            full_to_sym(P, sy);
            for (int i = 0; i < 6; ++i) SH_PE_AT(sh, i, t.G - 2, t.col) = sy[i];
            for (int i = 0; i < 3; ++i) SH_PE_AT(sh, 6 + i, t.G - 2, t.col) = p[i];
        }
    }
}

// chain of value functions at the chunk ends (one lane per instance), last chunk first
MS_HD void pit_value_chain(const PitShare& sh, int col, int G) {
    if (sh.flags[col]) return;
    double Pn[3][3], pn[3];
    {
        double sy[6];
        for (int i = 0; i < 6; ++i) sy[i] = SH_PE_AT(sh, i, G - 2, col);
        sym_to_full(sy, Pn);
        for (int i = 0; i < 3; ++i) pn[i] = SH_PE_AT(sh, 6 + i, G - 2, col);
    }
    for (int l = G - 3; l >= 0; --l) {
        ChunkElem E;
        double* e = (double*)&E;
        for (int i = 0; i < 27; ++i) e[i] = sh.at(SH_E + i, l + 1, col);
        double R[3][3], sy[6], dP[3][3], dp[3];
        for (int i = 0; i < 6; ++i) sy[i] = sh.at(SH_REF + i, l + 1, col);
        sym_to_full(sy, R);
        for (int i = 0; i < 3; ++i) { dp[i] = pn[i] - sh.at(SH_REF + 6 + i, l + 1, col); for (int j = 0; j < 3; ++j) dP[i][j] = Pn[i][j] - R[i][j]; }
        double P[3][3], p[3];
        if (!chunk_apply_diff(E, dP, dp, P, p)) { sh.raise(col, PIT_APPLY_FAILED); return; }
        full_to_sym(P, sy);
        for (int i = 0; i < 6; ++i) SH_PE_AT(sh, i, l, col) = sy[i];
        for (int i = 0; i < 3; ++i) { SH_PE_AT(sh, 6 + i, l, col) = p[i]; pn[i] = p[i]; for (int j = 0; j < 3; ++j) Pn[i][j] = P[i][j]; }
    }
}

// phase C: ordinary recursion inside the chunk from its end value; closed-loop transition of the chunk; the value function it
// arrives at must be the one the chain predicted for the end of the previous chunk
template <class Fetch>
MS_HD void pit_phase_c(const Ctx& c, const PitLane& t, const PitShare& sh, Fetch& fb) {
    if (t.l > t.G - 2 || sh.flags[t.col]) return;
    double P[3][3], p[3], sy[6];
    for (int i = 0; i < 6; ++i) sy[i] = SH_PE_AT(sh, i, t.l, t.col);
    sym_to_full(sy, P);
    for (int i = 0; i < 3; ++i) p[i] = SH_PE_AT(sh, 6 + i, t.l, t.col);
    Aff T;
    aff_identity(T);
    if (!riccati_backward_range(c, t.s, t.N, t.kLo, t.kHi, t.mu, t.delta, fb, P, p, T.M, T.m)) { sh.raise(t.col, PIT_BAD_INERTIA); return; }
    for (int i = 0; i < 9; ++i) sh.at(SH_TR + i, t.l, t.col) = T.M[i];
    for (int i = 0; i < 3; ++i) sh.at(SH_TR + 9 + i, t.l, t.col) = T.m[i];
    if (t.l >= 1 && t.kHi > t.kLo) {
        double num = 0.0, den = 1e-300, pnum = 0.0, pden = 1e-300;
        full_to_sym(P, sy);
        for (int i = 0; i < 6; ++i) { const double q = SH_PE_AT(sh, i, t.l - 1, t.col); num = fmax(num, fabs(sy[i] - q)); den = fmax(den, fabs(q)); }
        for (int i = 0; i < 3; ++i) { const double q = SH_PE_AT(sh, 6 + i, t.l - 1, t.col); pnum = fmax(pnum, fabs(p[i] - q)); pden = fmax(pden, fabs(q)); }
        if (!(num <= PIT_CONSISTENCY_TOL * den) || !(pnum <= PIT_CONSISTENCY_TOL * pden + 1e-12)) sh.raise(t.col, PIT_INCONSISTENT);
    }
}

// chain of chunk-start states (one lane per instance): d x at the start of chunk l into SH_REF of chunk l
MS_HD void pit_state_chain(const PitShare& sh, int col, int G) {
    double dx[3] = {0.0, 0.0, 0.0};
    for (int l = 0; l < G; ++l) {
        for (int i = 0; i < 3; ++i) sh.at(SH_REF + i, l, col) = dx[i];
        if (l == G - 1) break;
        double nx[3];
        for (int i = 0; i < 3; ++i)
            nx[i] = sh.at(SH_TR + 9 + i, l, col) + sh.at(SH_TR + 3 * i, l, col) * dx[0] + sh.at(SH_TR + 3 * i + 1, l, col) * dx[1] + sh.at(SH_TR + 3 * i + 2, l, col) * dx[2];
        for (int i = 0; i < 3; ++i) dx[i] = nx[i];
    }
}

// phase F: forward sweep inside the chunk (the last lane also does interval N-1)
template <class Fetch>
MS_HD void pit_phase_f(const Ctx& c, const PitLane& t, const PitShare& sh, Fetch& ff) {
    double dx[3];
    for (int i = 0; i < 3; ++i) dx[i] = sh.at(SH_REF + i, t.l, t.col);
    if (t.l == 0) { c.W(WS_ST + ST_T, 0, t.s) = 0.0; c.W(WS_ST + ST_B, 0, t.s) = 0.0; }
    riccati_forward_range(c, t.s, t.N, t.kLo, (t.l == t.G - 1) ? t.N : t.kHi, t.mu, t.delta, ff, dx);
}

// inertia-correction ladder (IPOPT Alg. IC), one rung
MS_HD double pit_next_delta(double delta, double dlast) {
    if (delta == 0.0) return (dlast == 0.0) ? 1e-4 : fmax(1e-20, dlast / 3.0);
    return delta * ((dlast == 0.0) ? 100.0 : 8.0);
}

// ---- host emulation of the lane-parallel driver (tests/hostsim): the lanes of one instance in a loop, the same phases ----
#if !defined(__CUDACC__)
template <class FetchB, class FetchF>
inline void inst_step_pit_emulated(const Ctx& c, int s, int G, FetchB& fb, FetchF& ff, long* fallbacks) {
    const Config& g = c.cfg;
    if (s >= g.nInst || c.I(SI_PHASE, s) != PH_FACTOR) return;
    const int N = c.I(SI_N_INT, s);
    const double dlast = c.D(SD_DELTA_LAST, s);
    std::vector<double> buf((size_t)G * SH_N, 0.0);
    int flag = 0;
    PitShare sh{buf.data(), &flag, 1};
    std::vector<PitLane> lanes(G);
    for (int l = 0; l < G; ++l) {
        PitLane& t = lanes[l];
        t.s = s; t.col = 0; t.l = l; t.G = G; t.N = N; t.mu = c.D(SD_MU, s); t.delta = 0.0;
        pit_chunk(N, G, l, t.kLo, t.kHi);
        pit_read_reference(c, t);
    }
    double delta = 0.0;
    bool ok = false;
    for (int tries = 0; tries < 40; ++tries) {
        count_cells(c, 2, N);
        flag = 0;
        for (int l = 0; l < G; ++l) { lanes[l].delta = delta; pit_phase_a(c, lanes[l], sh, fb); }
        pit_value_chain(sh, 0, G);
        for (int l = 0; l < G; ++l) pit_phase_c(c, lanes[l], sh, fb);
        if (flag & PIT_SCAN_FAILED) { if (fallbacks) *fallbacks += 1; inst_step(c, s, fb, ff); return; }
        if (!(flag & PIT_BAD_INERTIA)) { ok = true; break; }
        c.I(SI_NREG, s) += 1;
        delta = pit_next_delta(delta, dlast);
        if (delta > 1e40) break;
    }
    if (!ok) { finish(c, s, ST_STEP_FAILED); return; }
    if (delta > 0.0) c.D(SD_DELTA_LAST, s) = delta;
    c.D(SD_DELTA, s) = delta;
    count_cells(c, 3, N);
    pit_state_chain(sh, 0, G);
    for (int l = 0; l < G; ++l) pit_phase_f(c, lanes[l], sh, ff);
    c.I(SI_FACT, s) = 1;
    c.I(SI_PHASE, s) = PH_STEPPED;
}
#endif

}  // namespace mseetc
