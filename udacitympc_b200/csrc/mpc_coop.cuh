// b200mpc cooperative solver: ONE PROBLEM PER WARP, lane <-> horizon stage.  The latency path.
//
// The throughput path (mpc_core.cuh, one problem per thread) amortises everything over 65 536 problems but a single
// problem advances at ~0.2 ms per interior-point iteration there.  Whenever only a few problems are left -- the thin tail
// of a batch, >24-iteration stragglers, or a small batch such as the reference's own one-problem MPC::Solve call -- this
// kernel takes over: every sweep is split into per-stage work that all lanes do in parallel (derivative blocks,
// residuals, trig, barrier terms, step-size candidates, error norms) and the short recurrences that are inherently
// sequential over the horizon (Riccati recursion, dx roll-out, lambda^+ back-substitution), which lane 0 runs on operands
// staged in shared memory.  The algorithm, the workspace layout and the control logic (Solver::forward_logic,
// step_logic, top_of_loop) are the thread version's; only the execution shape differs, so a problem can be handed from
// one to the other at any round boundary.
//
// The code is written against three primitives so that tests/hostsim can run it on the CPU:
//   for_stages(n, f)  device: each lane runs f(t) for t = lane, lane+32, ... < n     host: a plain loop
//   sync()            device: __syncwarp()                                            host: nothing
//   lane0()           device: lane == 0                                               host: true
#pragma once
#include "mpc_core.cuh"

namespace b200mpc {

// per-stage scratch in shared memory (doubles)
struct CoopStage {
  double A[10];            // Lin at the current iterate: a1,a2,a3,a4,a5,beta,pp,kap,sed,vce
  double H[6];             // Hes: xx,pp,vp,ee,ev,m
  double rb[5], cc, gc;    // -c(x,y,psi,v,epsi), c_cte, cte-fold linear coefficient
  double r0, r1, ru0, ru1; // control Hessian diagonal (with Sigma, dw) and control right-hand side
  double rs[5];            // state right-hand side
  double KF[13];           // K (2x4), Lambda^-1 (3), k (2)
  double ds[6], du[2];     // search direction of time t
  double sl[4], z[4];      // slacks (sl0,su0,sl1,su1) and multipliers (zl0,zu0,zl1,zu1) of u_t at the current iterate
  double s[6], u[2], lam[6], tr[4];   // current iterate of time t and its trig values
  double sn[6], un[2], zn[4], trn[4];   // trial iterate of time t
  double bl[6], lp[6], ln[6];  // lambda^+ recurrence offset, lambda^+_t, lambda_trial_t
  double red[12];          // per-stage partial reductions
};
constexpr int kCoopStageDoubles = sizeof(CoopStage) / sizeof(double);

struct CoopPub {   // scalars lane 0 publishes to the other lanes before a parallel phase
  double mu, tau, df, dw, alpha, alpha_du, alpha_lam;
  int cur, ls, use_csoc, phase, lskeep, resto_step;
};

template <int LANES, class Exec>
struct CoopSolver {
  Solver<LANES>& S;     // lane 0's scalar state + control logic (every lane holds an object; only lane 0's is meaningful)
  CoopStage* st;        // N entries
  CoopPub* pub;
  Exec ex;
  const Params& P;
  const int N, M;

  MPC_HD CoopSolver(Solver<LANES>& s, CoopStage* stages, CoopPub* p, Exec e) : S(s), st(stages), pub(p), ex(e), P(s.P), N(s.N), M(s.M) {}

  MPC_HD void publish() {
    if (ex.lane0()) {
      pub->mu = S.mu; pub->tau = S.tau; pub->df = S.df; pub->dw = S.dw_curr; pub->alpha = S.alpha; pub->alpha_du = S.alpha_du; pub->alpha_lam = S.fl(F_SOFTFIX) ? S.soft_alpha : S.alpha;
      pub->cur = S.cur; pub->ls = S.fl(F_LS) ? 1 : 0; pub->use_csoc = S.fl(F_INSOC) ? 1 : 0; pub->phase = S.phase; pub->lskeep = S.fl(F_LSKEEP) ? 1 : 0; pub->resto_step = S.fl(F_RESTO) ? 1 : 0;
    }
    ex.sync();
  }
  MPC_HD Lin lin_of(const CoopStage& c) const {
    Lin L;
    L.a1 = c.A[0]; L.a2 = c.A[1]; L.a3 = c.A[2]; L.a4 = c.A[3]; L.a5 = c.A[4]; L.beta = c.A[5]; L.pp = c.A[6]; L.kap = c.A[7];
    L.sed = c.A[8]; L.vce = c.A[9];
    return L;
  }
  MPC_HD double grad_u(double df, int j, int t, double u, double um, double up) const {
    const double wq = j == 0 ? P.w_delta : P.w_a, wd = j == 0 ? P.w_ddelta : P.w_da;
    double g = wq * u;
    if (t > 0) g += wd * (u - um);
    if (t < M - 1) g -= wd * (up - u);
    return (2.0 * df) * g;
  }
  MPC_HD double hess_u(double df, int j, int t) const {
    const double wq = j == 0 ? P.w_delta : P.w_a, wd = j == 0 ? P.w_ddelta : P.w_da;
    const double nd = (t > 0 ? 1.0 : 0.0) + (t < M - 1 ? 1.0 : 0.0);
    return 2.0 * df * (wq + nd * wd);
  }

  // ------------------------------------------------------------------------------------------
  // FACTOR, parallel part: load the current iterate of stage t and build everything the Riccati recursion, the dx
  // roll-out and the lambda^+ back-substitution need from it.  Needs s,u,lam of the neighbours: phase A loads, phase B uses.
  MPC_HD void load_iterate(int t) {
    const int r = S.rec(t) + kX * pub->cur;
    CoopStage& c = st[t];
    const bool ls = pub->ls != 0;
    for (int k = 0; k < 6; ++k) { c.s[k] = S.w(r + xS + k); c.lam[k] = ls ? 0.0 : S.w(r + xLAM + k); }
    if (t < M) {
      c.u[0] = S.w(r + xU); c.u[1] = S.w(r + xU + 1);
      c.z[0] = S.w(r + xZL); c.z[1] = S.w(r + xZU); c.z[2] = S.w(r + xZL + 1); c.z[3] = S.w(r + xZU + 1);
    }
  }
  MPC_HD void prep_factor(int t) {   // t < M
    CoopStage& c = st[t];
    const CoopStage& cn = st[t + 1];
    const bool ls = pub->ls != 0;
    const double df = pub->df, mu = pub->mu, dw = pub->dw;
    const double qc = ls ? 1.0 : 2.0 * P.w_cte * df + dw;
    const double gv2 = 2.0 * P.w_v * df, ge2 = 2.0 * P.w_epsi * df, gc2 = 2.0 * P.w_cte * df;
    const int r = S.rec(t) + kX * pub->cur;
    double sp, cp, se, ce, p0, p1, p2, p3;
    S.trig_of(r, sp, cp, se, ce);
    c.tr[0] = sp; c.tr[1] = cp; c.tr[2] = se; c.tr[3] = ce;
    poly_eval(S.cf, c.s[0], p0, p1, p2, p3);
    const Lin A = make_lin(P, c.s[3], c.u[0], sp, cp, se, ce, p1, p2);
    c.A[0] = A.a1; c.A[1] = A.a2; c.A[2] = A.a3; c.A[3] = A.a4; c.A[4] = A.a5; c.A[5] = A.beta; c.A[6] = A.pp; c.A[7] = A.kap;
    c.A[8] = A.sed; c.A[9] = A.vce;
    Hes H;
    if (ls) { H.xx = H.pp = H.vp = H.ee = H.ev = H.m = 0.0; }
    else H = make_hes(P, cn.lam, c.s[3], sp, cp, se, ce, p1, p2, p3);
    c.H[0] = H.xx; c.H[1] = H.pp; c.H[2] = H.vp; c.H[3] = H.ee; c.H[4] = H.ev; c.H[5] = H.m;
    if (ls) { c.rb[0] = c.rb[1] = c.rb[2] = c.rb[3] = c.rb[4] = 0.0; c.cc = 0.0; }
    else {
      double cres[6];
      if (pub->use_csoc) { for (int k = 0; k < 6; ++k) cres[k] = S.w(S.rec(t + 1) + oCSOC + k); }
      else S.residual(c.s, c.u, cn.s, sp, cp, se, p0, atan(p1), cres);
      c.rb[0] = -cres[0]; c.rb[1] = -cres[1]; c.rb[2] = -cres[2]; c.rb[3] = -cres[3]; c.cc = cres[4]; c.rb[4] = -cres[5];
    }
    const double rc_next = gc2 * cn.s[4] + cn.lam[4];
    c.gc = rc_next - qc * c.cc;
    const double um0 = t > 0 ? st[t - 1].u[0] : 0.0, um1 = t > 0 ? st[t - 1].u[1] : 0.0;
    const double up0 = t < M - 1 ? cn.u[0] : 0.0, up1 = t < M - 1 ? cn.u[1] : 0.0;
    const double gu0 = grad_u(df, 0, t, c.u[0], um0, up0), gu1 = grad_u(df, 1, t, c.u[1], um1, up1);
    const double zl0 = c.z[0], zu0 = c.z[1], zl1 = c.z[2], zu1 = c.z[3];
    if (ls) {
      c.r0 = 1.0; c.r1 = 1.0;
      c.ru0 = gu0 - zl0 + zu0; c.ru1 = gu1 - zl1 + zu1;
      c.sl[0] = c.sl[1] = c.sl[2] = c.sl[3] = 1.0;
    } else {
      c.sl[0] = safe_slack(c.u[0] - P.xl[0], mu, zl0, P.xl[0]); c.sl[1] = safe_slack(P.xu[0] - c.u[0], mu, zu0, P.xu[0]);
      c.sl[2] = safe_slack(c.u[1] - P.xl[1], mu, zl1, P.xl[1]); c.sl[3] = safe_slack(P.xu[1] - c.u[1], mu, zu1, P.xu[1]);
      const double isl0 = drcp(c.sl[0]), isu0 = drcp(c.sl[1]), isl1 = drcp(c.sl[2]), isu1 = drcp(c.sl[3]);
      const double bl0 = A.beta * (cn.lam[2] + cn.lam[5]), bl1 = P.dt * cn.lam[3];
      c.r0 = hess_u(df, 0, t) + dw + zl0 * isl0 + zu0 * isu0;
      c.r1 = hess_u(df, 1, t) + dw + zl1 * isl1 + zu1 * isu1;
      c.ru0 = gu0 - bl0 - mu * isl0 + mu * isu0;
      c.ru1 = gu1 - bl1 - mu * isl1 + mu * isu1;
    }
    double ATl[6];
    applyAT6(A, cn.lam, ATl);
    c.rs[0] = c.lam[0] - ATl[0];
    c.rs[1] = c.lam[1] - ATl[1];
    c.rs[2] = c.lam[2] - ATl[2];
    c.rs[3] = gv2 * (c.s[3] - P.ref_v) + c.lam[3] - ATl[3];
    c.rs[4] = ge2 * c.s[5] + c.lam[5] - ATl[5];
  }

  // FACTOR, sequential part (lane 0): the Riccati recursion on the staged blocks; same arithmetic as Solver::factor.
  MPC_HD bool seq_factor() {
    const bool ls = pub->ls != 0;
    const double df = pub->df, dw = pub->dw;
    const double qv = ls ? 1.0 : 2.0 * P.w_v * df + dw, qe = ls ? 1.0 : 2.0 * P.w_epsi * df + dw,
                 qc = ls ? 1.0 : 2.0 * P.w_cte * df + dw, q0 = ls ? 1.0 : dw;
    const double gv2 = 2.0 * P.w_v * df, ge2 = 2.0 * P.w_epsi * df;
#define PS(i, j) pss[((i) >= (j)) ? ((i) * ((i) + 1) / 2 + (j)) : ((j) * ((j) + 1) / 2 + (i))]
    double pss[15], psu[4][2], puu00 = 0.0, puu10 = 0.0, puu11 = 0.0, pv[5], pu0 = 0.0, pu1 = 0.0;
    for (int i = 0; i < 15; ++i) pss[i] = 0.0;
    for (int i = 0; i < 4; ++i) psu[i][0] = psu[i][1] = 0.0;
    {
      const CoopStage& cT = st[M];
      PS(0, 0) = q0; PS(1, 1) = q0; PS(2, 2) = q0; PS(3, 3) = qv; PS(4, 4) = qe;
      pv[0] = cT.lam[0]; pv[1] = cT.lam[1]; pv[2] = cT.lam[2];
      pv[3] = gv2 * (cT.s[3] - P.ref_v) + cT.lam[3];
      pv[4] = ge2 * cT.s[5] + cT.lam[5];
    }
    bool ok = true;
    for (int t = M - 1; t >= 0; --t) {
      CoopStage& c = st[t];
      const Lin A = lin_of(c);
      const double* rb = c.rb;
      double wv[5], wu0 = pu0, wu1 = pu1;
#pragma unroll
      for (int i = 0; i < 5; ++i) {
        double a = pv[i];
#pragma unroll
        for (int j = 0; j < 5; ++j) a += PS(i, j) * rb[j];
        wv[i] = a;
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) { wu0 += psu[i][0] * rb[i]; wu1 += psu[i][1] * rb[i]; }
      double T0[5], T1[5];
#pragma unroll
      for (int j = 0; j < 5; ++j) {
        T0[j] = A.beta * (PS(2, j) + PS(4, j)) + (j < 4 ? psu[j < 4 ? j : 0][0] : 0.0);
        T1[j] = P.dt * PS(3, j) + (j < 4 ? psu[j < 4 ? j : 0][1] : 0.0);
      }
      const double Tu00 = A.beta * psu[2][0] + puu00, Tu10 = P.dt * psu[3][0] + puu10, Tu11 = P.dt * psu[3][1] + puu11;
      const double L00 = c.r0 + A.beta * (T0[2] + T0[4]) + Tu00;
      const double L10 = A.beta * (T1[2] + T1[4]) + Tu10;
      const double L11 = c.r1 + P.dt * T1[3] + Tu11;
      const double det = L00 * L11 - L10 * L10;
      if (!(L00 > 0.0) || !(det > 0.0)) ok = false;
      const double idet = drcp(det);
      const double i00 = L11 * idet, i10 = -L10 * idet, i11 = L00 * idet;
      double G0[4], G1[4];
      applyA(A, T0[0], T0[1], T0[2], T0[3], T0[4], G0[0], G0[1], G0[2], G0[3]);
      applyA(A, T1[0], T1[1], T1[2], T1[3], T1[4], G1[0], G1[1], G1[2], G1[3]);
      G0[3] += c.H[5];
      const double h0 = c.ru0 + A.beta * (wv[2] + wv[4]) + wu0, h1 = c.ru1 + P.dt * wv[3] + wu1;
      double K0[4], K1[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) { K0[j] = i00 * G0[j] + i10 * G1[j]; K1[j] = i10 * G0[j] + i11 * G1[j]; }
      const double k0 = i00 * h0 + i10 * h1, k1 = i10 * h0 + i11 * h1;
#pragma unroll
      for (int j = 0; j < 4; ++j) { c.KF[j] = K0[j]; c.KF[4 + j] = K1[j]; }
      c.KF[8] = i00; c.KF[9] = i10; c.KF[10] = i11; c.KF[11] = k0; c.KF[12] = k1;
      double Y[5][4];
#pragma unroll
      for (int i = 0; i < 5; ++i) applyA(A, PS(i, 0), PS(i, 1), PS(i, 2), PS(i, 3), PS(i, 4), Y[i][0], Y[i][1], Y[i][2], Y[i][3]);
      double Sm[4][4];
#pragma unroll
      for (int j = 0; j < 4; ++j) applyA(A, Y[0][j], Y[1][j], Y[2][j], Y[3][j], Y[4][j], Sm[0][j], Sm[1][j], Sm[2][j], Sm[3][j]);
      double aw[4];
      applyA(A, wv[0], wv[1], wv[2], wv[3], wv[4], aw[0], aw[1], aw[2], aw[3]);
      const double ac[4] = {A.pp, -1.0, 0.0, A.sed};
      double nss[15];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j)
          nss[i * (i + 1) / 2 + j] = Sm[i][j] + qc * ac[i] * ac[j] - (G0[i] * K0[j] + G1[i] * K1[j]);
      nss[0] += q0 + c.H[0];
      nss[2] += q0;
      nss[5] += q0 + c.H[1];
      nss[8] += c.H[2];
      nss[9] += qv;
      const double qvce = qc * A.vce;
#pragma unroll
      for (int j = 0; j < 4; ++j) nss[10 + j] = qvce * ac[j];
      nss[13] += c.H[4];
      nss[14] = qe + c.H[3] + qvce * A.vce;
      double d0 = 0.0, d1 = 0.0;
      if (t > 0 && !ls) { d0 = 2.0 * df * P.w_ddelta; d1 = 2.0 * df * P.w_da; }
#pragma unroll
      for (int i = 0; i < 4; ++i) { psu[i][0] = K0[i] * d0; psu[i][1] = K1[i] * d1; }
      puu00 = -d0 * d0 * i00; puu10 = -d0 * d1 * i10; puu11 = -d1 * d1 * i11;
#pragma unroll
      for (int i = 0; i < 4; ++i) pv[i] = c.rs[i] + aw[i] + c.gc * ac[i] - (G0[i] * k0 + G1[i] * k1);
      pv[4] = c.rs[4] + c.gc * A.vce;
      pu0 = d0 * k0; pu1 = d1 * k1;
#pragma unroll
      for (int i = 0; i < 15; ++i) pss[i] = nss[i];
    }
#undef PS
    return ok;
  }

  // FORWARD, sequential part (lane 0): dx roll-out.  DS/DU also go to the workspace (the thread version may take over).
  MPC_HD void seq_forward() {
    const bool ls = pub->ls != 0;
    const double df = pub->df;
    double ds[6] = {0, 0, 0, 0, 0, 0}, dup0 = 0.0, dup1 = 0.0;
    for (int k = 0; k < 6; ++k) { st[0].ds[k] = 0.0; S.w(S.rec(0) + oDS + k) = 0.0; }
    for (int t = 0; t < M; ++t) {
      CoopStage& c = st[t];
      const Lin A = lin_of(c);
      const double* K = c.KF;
      double d0 = 0.0, d1 = 0.0;
      if (t > 0 && !ls) { d0 = 2.0 * df * P.w_ddelta; d1 = 2.0 * df * P.w_da; }
      const double e0 = d0 * dup0, e1 = d1 * dup1;
      const double du0 = -(K[0] * ds[0] + K[1] * ds[1] + K[2] * ds[2] + K[3] * ds[3] + K[11]) + (K[8] * e0 + K[9] * e1);
      const double du1 = -(K[4] * ds[0] + K[5] * ds[1] + K[6] * ds[2] + K[7] * ds[3] + K[12]) + (K[9] * e0 + K[10] * e1);
      c.du[0] = du0; c.du[1] = du1;
      S.w(S.rec(t) + oDU) = du0; S.w(S.rec(t) + oDU + 1) = du1;
      double dn[6];
      dn[0] = ds[0] + A.a1 * ds[2] + A.a3 * ds[3] + c.rb[0];
      dn[1] = ds[1] + A.a2 * ds[2] + A.a4 * ds[3] + c.rb[1];
      dn[2] = ds[2] + A.a5 * ds[3] + A.beta * du0 + c.rb[2];
      dn[3] = ds[3] + P.dt * du1 + c.rb[3];
      dn[4] = A.pp * ds[0] - ds[1] + A.sed * ds[3] + A.vce * ds[5] - c.cc;
      dn[5] = -A.kap * ds[0] + ds[2] + A.a5 * ds[3] + A.beta * du0 + c.rb[4];
      for (int k = 0; k < 6; ++k) { ds[k] = dn[k]; st[t + 1].ds[k] = dn[k]; S.w(S.rec(t + 1) + oDS + k) = dn[k]; }
      dup0 = du0; dup1 = du1;
    }
  }
  // FORWARD, parallel part: step-size candidates, barrier slope and tiny-step test of stage t (t < N; t == M: terminal state only)
  MPC_HD void post_forward(int t) {
    CoopStage& c = st[t];
    const double df = pub->df, mu = pub->mu, tau = pub->tau;
    const double gv2 = 2.0 * P.w_v * df, ge2 = 2.0 * P.w_epsi * df, gc2 = 2.0 * P.w_cte * df;
    const double tinytol = 10.0 * DBL_EPSILON;
    double a_pr = 1.0, a_du = 1.0, gbd = 0.0;
    bool nottiny = false;
    gbd += gv2 * (c.s[3] - P.ref_v) * c.ds[3] + gc2 * c.s[4] * c.ds[4] + ge2 * c.s[5] * c.ds[5];
    for (int k = 0; k < 6; ++k) nottiny = nottiny || fabs(c.ds[k]) > tinytol * (fabs(c.s[k]) + 1.0);
    if (t < M) {
      const double u0 = c.u[0], u1 = c.u[1], du0 = c.du[0], du1 = c.du[1];
      const double um0 = t > 0 ? st[t - 1].u[0] : 0.0, um1 = t > 0 ? st[t - 1].u[1] : 0.0;
      const double up0 = t < M - 1 ? st[t + 1].u[0] : 0.0, up1 = t < M - 1 ? st[t + 1].u[1] : 0.0;
      const double sl0 = c.sl[0], su0 = c.sl[1], sl1 = c.sl[2], su1 = c.sl[3];
      const double zl0 = c.z[0], zu0 = c.z[1], zl1 = c.z[2], zu1 = c.z[3];
      const double isl0 = drcp(sl0), isu0 = drcp(su0), isl1 = drcp(sl1), isu1 = drcp(su1);
      gbd += (grad_u(df, 0, t, u0, um0, up0) - mu * isl0 + mu * isu0) * du0 + (grad_u(df, 1, t, u1, um1, up1) - mu * isl1 + mu * isu1) * du1;
      if (du0 < 0.0) a_pr = dmin(a_pr, -ddiv(tau, du0) * sl0);
      if (du0 > 0.0) a_pr = dmin(a_pr, ddiv(tau, du0) * su0);
      if (du1 < 0.0) a_pr = dmin(a_pr, -ddiv(tau, du1) * sl1);
      if (du1 > 0.0) a_pr = dmin(a_pr, ddiv(tau, du1) * su1);
      const double dzl0 = (mu - sl0 * zl0 - zl0 * du0) * isl0, dzu0 = (mu - su0 * zu0 + zu0 * du0) * isu0;
      const double dzl1 = (mu - sl1 * zl1 - zl1 * du1) * isl1, dzu1 = (mu - su1 * zu1 + zu1 * du1) * isu1;
      if (dzl0 < 0.0) a_du = dmin(a_du, -ddiv(tau, dzl0) * zl0);
      if (dzu0 < 0.0) a_du = dmin(a_du, -ddiv(tau, dzu0) * zu0);
      if (dzl1 < 0.0) a_du = dmin(a_du, -ddiv(tau, dzl1) * zl1);
      if (dzu1 < 0.0) a_du = dmin(a_du, -ddiv(tau, dzu1) * zu1);
      nottiny = nottiny || fabs(du0) > tinytol * (fabs(u0) + 1.0) || fabs(du1) > tinytol * (fabs(u1) + 1.0);
    }
    c.red[0] = a_pr; c.red[1] = a_du; c.red[2] = gbd; c.red[3] = nottiny ? 1.0 : 0.0;
  }
  MPC_HD void reduce_forward() {   // lane 0
    double a_pr = 1.0, a_du = 1.0, gbd = 0.0;
    bool nottiny = false;
    for (int t = 0; t < N; ++t) {
      a_pr = dmin(a_pr, st[t].red[0]); a_du = dmin(a_du, st[t].red[1]); gbd += st[t].red[2]; nottiny = nottiny || st[t].red[3] != 0.0;
    }
    S.fw_alpha_pr = a_pr; S.fw_alpha_du = a_du; S.fw_gbd = gbd; S.fw_tiny = !nottiny;
  }

  // ------------------------------------------------------------------------------------------
  // STEP, parallel part 1: trial point, trial z (kappa_sigma reset), barrier / complementarity partials, and the
  // offset of the lambda^+ back-substitution of stage t.
  MPC_HD void step1(int t) {   // t < N
    CoopStage& c = st[t];
    // least-square multiplier pass (ls): H = I, the iterate does not move and nothing is written to the trial copy
    const bool ls = pub->ls != 0;
    const double a = ls ? 0.0 : pub->alpha, a_du = ls ? 0.0 : pub->alpha_du, mu = pub->mu, df = pub->df, dw = pub->dw;
    const double qv = ls ? 1.0 : 2.0 * P.w_v * df + dw, qe = ls ? 1.0 : 2.0 * P.w_epsi * df + dw, qc = ls ? 1.0 : 2.0 * P.w_cte * df + dw,
                 q0 = ls ? 1.0 : dw;
    const double gv2 = 2.0 * P.w_v * df, ge2 = 2.0 * P.w_epsi * df, gc2 = 2.0 * P.w_cte * df;
    const int rN = S.rec(t) + kX * (pub->cur ^ 1);
    double xm = 0.0, zz1 = 0.0, szmx = 0.0, szmn = 1e300, slog = 0.0;
    for (int k = 0; k < 6; ++k) { c.sn[k] = c.s[k] + a * c.ds[k]; if (!ls) S.w(rN + xS + k) = c.sn[k]; xm = dmax(xm, fabs(c.sn[k])); }
    const double* ds = c.ds;
    if (t == M) {
      c.lp[0] = -q0 * ds[0]; c.lp[1] = -q0 * ds[1]; c.lp[2] = -q0 * ds[2];
      c.lp[3] = -qv * ds[3] - gv2 * (c.s[3] - P.ref_v);
      c.lp[4] = -qc * ds[4] - gc2 * c.s[4];
      c.lp[5] = -qe * ds[5] - ge2 * c.s[5];
    } else {
      const double du0 = c.du[0], du1 = c.du[1];
      c.un[0] = c.u[0] + a * du0; c.un[1] = c.u[1] + a * du1;
      if (!ls) { S.w(rN + xU) = c.un[0]; S.w(rN + xU + 1) = c.un[1]; }
      xm = dmax(xm, dmax(fabs(c.un[0]), fabs(c.un[1])));
      const double sl0 = c.sl[0], su0 = c.sl[1], sl1 = c.sl[2], su1 = c.sl[3];
      double zl0 = c.z[0], zu0 = c.z[1], zl1 = c.z[2], zu1 = c.z[3];
      const double b0 = safe_slack(c.un[0] - P.xl[0], mu, zl0, P.xl[0]) * safe_slack(P.xu[0] - c.un[0], mu, zu0, P.xu[0]);
      const double b1 = safe_slack(c.un[1] - P.xl[1], mu, zl1, P.xl[1]) * safe_slack(P.xu[1] - c.un[1], mu, zu1, P.xu[1]);
      slog = log(b0 * b1);
      if (!ls) {
        zl0 += a_du * ddiv(mu - sl0 * zl0 - zl0 * du0, sl0);
        zu0 += a_du * ddiv(mu - su0 * zu0 + zu0 * du0, su0);
        zl1 += a_du * ddiv(mu - sl1 * zl1 - zl1 * du1, sl1);
        zu1 += a_du * ddiv(mu - su1 * zu1 + zu1 * du1, su1);
      }
      const double nsl0 = safe_slack(c.un[0] - P.xl[0], mu, zl0, P.xl[0]), nsu0 = safe_slack(P.xu[0] - c.un[0], mu, zu0, P.xu[0]);
      const double nsl1 = safe_slack(c.un[1] - P.xl[1], mu, zl1, P.xl[1]), nsu1 = safe_slack(P.xu[1] - c.un[1], mu, zu1, P.xu[1]);
      if (!ls) {
        const double m0 = mu / nsl0, m1 = mu / nsu0, m2 = mu / nsl1, m3 = mu / nsu1;
        zl0 = dclamp(zl0, 1e-10 * m0, 1e10 * m0);
        zu0 = dclamp(zu0, 1e-10 * m1, 1e10 * m1);
        zl1 = dclamp(zl1, 1e-10 * m2, 1e10 * m2);
        zu1 = dclamp(zu1, 1e-10 * m3, 1e10 * m3);
        S.w(rN + xZL) = zl0; S.w(rN + xZL + 1) = zl1; S.w(rN + xZU) = zu0; S.w(rN + xZU + 1) = zu1;
      }
      c.zn[0] = zl0; c.zn[1] = zu0; c.zn[2] = zl1; c.zn[3] = zu1;
      zz1 = zl0 + zl1 + zu0 + zu1;
      const double c0 = nsl0 * zl0, c1 = nsl1 * zl1, c2 = nsu0 * zu0, c3 = nsu1 * zu1;
      szmx = dmax(dmax(c0, c1), dmax(c2, c3));
      szmn = dmin(dmin(c0, c1), dmin(c2, c3));
      // trig of the trial point
      if (ls) { c.trn[0] = c.tr[0]; c.trn[1] = c.tr[1]; c.trn[2] = c.tr[2]; c.trn[3] = c.tr[3]; }
      else {
        double spn, cpn, sen, cen;
        sincos(c.sn[2], &spn, &cpn);
        sincos(c.sn[5], &sen, &cen);
        c.trn[0] = spn; c.trn[1] = cpn; c.trn[2] = sen; c.trn[3] = cen;
        S.w(rN + xTR) = spn; S.w(rN + xTR + 1) = cpn; S.w(rN + xTR + 2) = sen; S.w(rN + xTR + 3) = cen;
      }
      // offset of lambda^+_t = A_t^T lambda^+_{t+1} + bl_t (current linearisation, staged by prep_factor)
      c.bl[0] = -(q0 + c.H[0]) * ds[0];
      c.bl[1] = -q0 * ds[1];
      c.bl[2] = -((q0 + c.H[1]) * ds[2] + c.H[2] * ds[3]);
      c.bl[3] = -(c.H[2] * ds[2] + qv * ds[3] + c.H[4] * ds[5] + c.H[5] * du0) - gv2 * (c.s[3] - P.ref_v);
      c.bl[4] = -qc * ds[4] - gc2 * c.s[4];
      c.bl[5] = -((qe + c.H[3]) * ds[5] + c.H[4] * ds[3]) - ge2 * c.s[5];
    }
    c.red[0] = xm; c.red[1] = zz1; c.red[2] = szmx; c.red[3] = szmn; c.red[4] = slog;
  }
  // STEP, sequential part (lane 0): lambda^+ back-substitution
  MPC_HD void seq_step() {
    for (int t = M - 1; t >= 0; --t) {
      CoopStage& c = st[t];
      const Lin A = lin_of(c);
      double at[6];
      applyAT6(A, st[t + 1].lp, at);
      c.lp[0] = at[0] + c.bl[0]; c.lp[1] = at[1] + c.bl[1]; c.lp[2] = at[2] + c.bl[2]; c.lp[3] = at[3] + c.bl[3];
      c.lp[4] = c.bl[4]; c.lp[5] = at[5] + c.bl[5];
    }
  }
  // STEP, parallel part 2: trial multipliers, residuals and objective of stage t
  MPC_HD void step2(int t) {   // t < N
    CoopStage& c = st[t];
    const bool ls = pub->ls != 0, keep = pub->lskeep != 0;
    const double a = pub->alpha_lam;
    const int rN = S.rec(t) + kX * (ls ? pub->cur : (pub->cur ^ 1));
    double l1 = 0.0, dlm = 0.0, th = 0.0, cm = 0.0, f = 0.0;
    for (int k = 0; k < 6; ++k) {
      // ls: lam is 0; the first pass evaluates the norms for lambda = 0, the second (keep) stores the estimate
      c.ln[k] = ls ? (keep ? c.lp[k] : 0.0) : c.lam[k] + a * (c.lp[k] - c.lam[k]);
      if (!ls || keep) S.w(rN + xLAM + k) = c.ln[k];
      l1 += fabs(c.ln[k]);
      dlm = dmax(dlm, fabs(c.lp[k] - c.lam[k]));
    }
    f = S.state_cost(c.sn);
    if (t < M && !ls) {
      double p0, p1, p2, p3, cres[6];
      poly_eval(S.cf, c.sn[0], p0, p1, p2, p3);
      const double psides = atan(p1);
      S.residual(c.sn, c.un, st[t + 1].sn, c.trn[0], c.trn[1], c.trn[2], p0, psides, cres);
      for (int k = 0; k < 6; ++k) { th += fabs(cres[k]); cm = dmax(cm, fabs(cres[k])); }
      f += P.w_delta * (c.un[0] * c.un[0]) + P.w_a * (c.un[1] * c.un[1]);
      if (t > 0) {
        const double e0 = c.un[0] - st[t - 1].un[0], e1 = c.un[1] - st[t - 1].un[1];
        f += P.w_ddelta * (e0 * e0) + P.w_da * (e1 * e1);
      }
    }
    c.red[5] = l1; c.red[6] = dlm; c.red[7] = th; c.red[8] = cm; c.red[9] = f;
  }
  // STEP, parallel part 3: grad_x L at the trial iterate
  MPC_HD void step3(int t) {   // t < N
    CoopStage& c = st[t];
    const double df = pub->df;
    const double gv2 = 2.0 * P.w_v * df, ge2 = 2.0 * P.w_epsi * df, gc2 = 2.0 * P.w_cte * df;
    double dinf = 0.0;
    if (t == M) {
      dinf = dmax(dinf, dmax(fabs(c.ln[0]), dmax(fabs(c.ln[1]), fabs(c.ln[2]))));
      dinf = dmax(dinf, fabs(gv2 * (c.sn[3] - P.ref_v) + c.ln[3]));
      dinf = dmax(dinf, fabs(gc2 * c.sn[4] + c.ln[4]));
      dinf = dmax(dinf, fabs(ge2 * c.sn[5] + c.ln[5]));
    } else {
      double p0, p1, p2, p3;
      poly_eval(S.cf, c.sn[0], p0, p1, p2, p3);
      const Lin A = make_lin(P, c.sn[3], c.un[0], c.trn[0], c.trn[1], c.trn[2], c.trn[3], p1, p2);
      const double* ln1 = st[t + 1].ln;
      double at[6];
      applyAT6(A, ln1, at);
      dinf = dmax(dinf, dmax(fabs(c.ln[0] - at[0]), dmax(fabs(c.ln[1] - at[1]), fabs(c.ln[2] - at[2]))));
      dinf = dmax(dinf, fabs(gv2 * (c.sn[3] - P.ref_v) + c.ln[3] - at[3]));
      dinf = dmax(dinf, fabs(gc2 * c.sn[4] + c.ln[4]));
      dinf = dmax(dinf, fabs(ge2 * c.sn[5] + c.ln[5] - at[5]));
      const double um0 = t > 0 ? st[t - 1].un[0] : 0.0, um1 = t > 0 ? st[t - 1].un[1] : 0.0;
      const double up0 = t < M - 1 ? st[t + 1].un[0] : 0.0, up1 = t < M - 1 ? st[t + 1].un[1] : 0.0;
      const double g0 = grad_u(df, 0, t, c.un[0], um0, up0) - A.beta * (ln1[2] + ln1[5]) - c.zn[0] + c.zn[1];
      const double g1 = grad_u(df, 1, t, c.un[1], um1, up1) - P.dt * ln1[3] - c.zn[2] + c.zn[3];
      dinf = dmax(dinf, dmax(fabs(g0), fabs(g1)));
    }
    c.red[10] = dinf;
  }
  MPC_HD void reduce_step() {   // lane 0
    double xm = 0.0, zz1 = 0.0, szmx = 0.0, szmn = 1e300, slog = 0.0, l1 = 0.0, dlm = 0.0, th = 0.0, cm = 0.0, f = 0.0, dinf = 0.0;
    for (int t = 0; t < N; ++t) {
      const double* r = st[t].red;
      xm = dmax(xm, r[0]); l1 += r[5]; dlm = dmax(dlm, r[6]); f += r[9]; dinf = dmax(dinf, r[10]);
      if (t < M) { zz1 += r[1]; szmx = dmax(szmx, r[2]); szmn = dmin(szmn, r[3]); slog += r[4]; th += r[7]; cm = dmax(cm, r[8]); }
    }
    S.dualinf = dinf; S.lam1 = l1; S.z1 = zz1; S.sz_max = szmx; S.sz_min = szmn; S.xmaxabs = xm; S.dlam_max = dlm;
    S.tr_f = pub->df * f; S.tr_theta = th; S.tr_priminf = cm; S.tr_sumlog = slog;
  }

  // ------------------------------------------------------------------------------------------
  // One round: the three phases a problem may be in, each followed by the thread version's control logic on lane 0.
  MPC_HD void round() {
    publish();
    if (pub->phase == PH_RESTO) {
      // failed line search (Solver::resto_entry).  Restoration step (Solver::do_resto, sequential over the horizon): lane 0
      // rewrites the current iterate in the workspace, then every lane re-stages its stage with a zero search direction
      // for the zero-length STEP that follows
      if (ex.lane0()) S.resto_entry();
      publish();
      if (pub->resto_step) {   // not a soft restoration step, which reuses the staged Newton direction
        ex.for_stages(N, [&](int t) {
          load_iterate(t);
          for (int k = 0; k < 6; ++k) st[t].ds[k] = 0.0;
          st[t].du[0] = st[t].du[1] = 0.0;
        });
        ex.sync();
        ex.for_stages(M, [&](int t) { prep_factor(t); });
        ex.sync();
      }
    }
    if (pub->phase == PH_FACTOR) {
      ex.for_stages(N, [&](int t) { load_iterate(t); });
      ex.sync();
      ex.for_stages(M, [&](int t) { prep_factor(t); });
      ex.sync();
      if (ex.lane0()) {
        if (seq_factor()) S.phase = PH_FORWARD;
        else S.factor_failed();
      }
      publish();
    }
    if (pub->phase == PH_FORWARD) {
      if (ex.lane0()) seq_forward();
      ex.sync();
      if (!pub->ls) {
        ex.for_stages(N, [&](int t) { post_forward(t); });
        ex.sync();
      }
      if (ex.lane0()) {
        if (!pub->ls) reduce_forward();
        S.forward_logic();
      }
      publish();
    }
    if (pub->phase == PH_STEP) {
      {
        ex.for_stages(N, [&](int t) { step1(t); });
        ex.sync();
        if (ex.lane0()) seq_step();
        ex.sync();
        ex.for_stages(N, [&](int t) { step2(t); });
        ex.sync();
        ex.for_stages(N, [&](int t) { step3(t); });
        ex.sync();
        if (ex.lane0()) { reduce_step(); S.step_logic(); }
      }
      publish();
    }
  }
  // start point of a fresh problem, stage-parallel (Solver::init)
  MPC_HD void init(const double* s0) {
    if (ex.lane0()) S.init_scalars(s0, S.cf, kMaxCoef);
    ex.for_stages(N, [&](int t) {
      double f, th, cm, sl;
      S.init_stage(t, s0, f, th, cm, sl);
      st[t].red[0] = f; st[t].red[1] = th; st[t].red[2] = cm; st[t].red[3] = sl;
    });
    ex.sync();
    if (ex.lane0()) {
      double f = 0.0, th = 0.0, cm = 0.0, sl = 0.0;
      for (int t = 0; t < N; ++t) { f += st[t].red[0]; th += st[t].red[1]; cm = dmax(cm, st[t].red[2]); sl += st[t].red[3]; }
      S.init_finish(f, th, cm, sl);
    }
    ex.sync();
  }
  // warm starts, stage-parallel (Solver::init_warm / init_guess; the partial sums are added in stage order, so the result
  // is bit-identical to the thread version)
  MPC_HD void init_warm(const double* s0, double mu0) {
    const int c = (int)S.w(iCUR);
    const double df_old = S.w(dDF);
    if (ex.lane0()) S.warm_shift(s0);
    ex.sync();
    warm_common(s0, c, mu0, df_old, true);
  }
  MPC_HD void init_guess(const double* s0, const double* x, size_t xs, const double* m, size_t ms, double mu0) {
    ex.for_stages(N, [&](int t) { S.guess_stage(t, s0, x, xs, m, ms); });
    ex.sync();
    warm_common(s0, 0, mu0, 1.0, m != nullptr);
    if (ex.lane0()) S.guess_check();
    ex.sync();
  }
  MPC_HD void warm_common(const double* s0, int c, double mu0, double df_old, bool have_mult) {
    static_assert(Solver<LANES>::kWarmRed <= sizeof(st->red) / sizeof(double), "warm-start partials must fit CoopStage::red");
    const int b = kX * c;
    ex.for_stages(M, [&](int t) { S.warm_push_stage(t, b); });
    ex.sync();
    ex.for_stages(N, [&](int t) { S.warm_stage(t, b, st[t].red); });
    ex.sync();
    if (ex.lane0()) {
      double f = 0.0, th = 0.0, cm = 0.0, sl = 0.0, gmax = 0.0;
      for (int t = 0; t < N; ++t) S.warm_add(t, st[t].red, f, th, cm, sl, gmax);
      S.warm_scalars(s0, c, mu0, gmax);
      S.warm_finish(f, th, cm, sl);
      pub->df = S.df; pub->mu = S.mu;
    }
    ex.sync();
    const double ratio = pub->df / df_old, mu = pub->mu;
    ex.for_stages(N, [&](int t) { S.warm_mult_stage(t, b, ratio, mu, have_mult); });
    ex.sync();
  }
  // A problem taken over in the middle of an iteration (phase FORWARD, or STEP during backtracking): re-stage what
  // the earlier sweeps of this iteration left in shared memory, without touching the control state.
  MPC_HD void rebuild() {
    ex.for_stages(N, [&](int t) { load_iterate(t); });
    ex.sync();
    ex.for_stages(M, [&](int t) { prep_factor(t); });
    ex.sync();
    if (ex.lane0()) {
      seq_factor();
      if (pub->phase == PH_STEP || pub->phase == PH_RESTO) seq_forward();
    }
    ex.sync();
  }
  // runs the problem to completion; lane 0's Solver holds the final state
  MPC_HD void run() {
    publish();
    if (pub->phase == PH_FORWARD || pub->phase == PH_STEP || pub->phase == PH_RESTO) rebuild();
    while (pub->phase != PH_DONE) round();
  }
};

}  // namespace b200mpc
