// orbit.cuh — Keplerian radial velocities per epoch (replaces psoap/orbit.py get_velocities()).
#pragma once
#include "common.cuh"

namespace psoap {

enum Model { SB1 = 1, SB2 = 2, ST1 = 3, ST2 = 4, ST3 = 5 };

__host__ __device__ inline int model_ncomp(int m) { return (m == SB1 || m == ST1) ? 1 : ((m == SB2 || m == ST2) ? 2 : 3); }
__host__ __device__ inline int model_norb(int m) {  // psoap/utils.py:14 (index of gamma + 1)
    return m == SB1 ? 6 : m == SB2 ? 7 : m == ST1 ? 11 : m == ST2 ? 12 : 13;
}

// Python float modulus (result carries the sign of the divisor), orbit.py:60.
__device__ __forceinline__ double py_mod(double a, double b) {
    double m = fmod(a, b);
    if (m != 0.0) {
        if ((b < 0.0) != (m < 0.0)) m += b;
    } else {
        m = copysign(0.0, b);
    }
    return m;
}

// True anomaly, orbit.py:47-72: t' = (t - T0) % P; solve E - e sin E = 2 pi t'/P; f = 2 atan(sqrt((1+e)/(1-e))
// tan(E/2)), + 2 pi when E >= pi.  The reference calls scipy fsolve from E0 = M (lands within 2.8e-13 rad of
// the root, SURVEY.md §7); here: Newton safeguarded by the bracket [0, 2 pi] (the function is monotone).
// E_out (may be null) receives the eccentric anomaly E, for the orbit Jacobian.
__device__ inline double true_anomaly(double t, double T0, double P, double e, double* E_out = nullptr) {
    const double PI = 3.141592653589793;
    const double tp = py_mod(t - T0, P);
    const double Mn = 2 * PI * tp / P;
    double lo = 0.0, hi = 2 * PI, E = Mn;
    for (int it = 0; it < 64; ++it) {
        const double f = E - e * sin(E) - Mn;
        if (f > 0.0) hi = E; else lo = E;
        double En = E - f / (1.0 - e * cos(E));
        if (!(En > lo && En < hi)) En = 0.5 * (lo + hi);
        const double dE = fabs(En - E);
        E = En;
        if (dE <= 4.5e-16 * fmax(1.0, fabs(E))) break;
    }
    if (E_out) *E_out = E;
    const double th = 2 * atan(sqrt((1 + e) / (1 - e)) * tan(E / 2.));
    return (E < PI) ? th : th + 2 * PI;
}

// K (cos(omega pi/180 + f) + e cos(omega pi/180)), orbit.py:81
__device__ __forceinline__ double rv(double K, double e, double omega_deg, double f) {
    const double PI = 3.141592653589793;
    const double w = omega_deg * PI / 180;
    return K * (cos(w + f) + e * cos(w));
}

// One block; threads stride over epochs.  vel: [ncomp, n_epochs].  flag[0] is (re)written by this block:
// 1 when any |v| >= c_kms (sample_parallel.py:186-187) or, with check_gp, when a GP hyper-parameter that
// follows the orbital ones in the farm's vector is negative (covariance.py:317,:339,:362); else 0.
__device__ inline void orbit_block(int model, const double* __restrict__ p, const double* __restrict__ dates,
                                   int n_epochs, double* __restrict__ vel, int* __restrict__ flag, int check_gp) {
    const int ncomp = model_ncomp(model);
    __shared__ int s_flag;
    if (threadIdx.x == 0) {
        int f = 0;
        if (check_gp) {
            const double* gp = p + model_norb(model);
            for (int c = 0; c < 2 * ncomp; ++c)
                if (gp[c] < 0.0) f = 1;
        }
        s_flag = f;
    }
    __syncthreads();
    for (int ep = threadIdx.x; ep < n_epochs; ep += blockDim.x) {
        const double t = dates[ep];
        double v[3] = {0, 0, 0};
        if (model == SB1 || model == SB2) {
            const int o = (model == SB2) ? 1 : 0;
            const double K = p[o + 0], e = p[o + 1], om = p[o + 2], P = p[o + 3], T0 = p[o + 4], gam = p[o + 5];
            const double f = true_anomaly(t, T0, P, e);
            v[0] = rv(K, e, om, f) + gam;                                  // orbit.py:83-91
            if (model == SB2) v[1] = rv(K / p[0], e, om + 180, f) + gam;   // orbit.py:134-146
        } else {
            const int o = (model == ST1) ? 0 : 1;                          // q_in first for ST2/ST3
            const double K_in = p[o + 0], e_in = p[o + 1], om_in = p[o + 2], P_in = p[o + 3], T0_in = p[o + 4];
            const int oo = o + 5 + ((model == ST3) ? 1 : 0);               // q_out before K_out for ST3
            const double K_out = p[oo + 0], e_out = p[oo + 1], om_out = p[oo + 2], P_out = p[oo + 3],
                         T0_out = p[oo + 4], gam = p[oo + 5];
            const double fi = true_anomaly(t, T0_in, P_in, e_in);
            const double fo = true_anomaly(t, T0_out, P_out, e_out);
            const double v3 = rv(K_out, e_out, om_out, fo);
            v[0] = rv(K_in, e_in, om_in, fi) + v3 + gam;                                    // orbit.py:265-275
            if (model != ST1) v[1] = rv(K_in / p[0], e_in, om_in + 180, fi) + v3 + gam;     // orbit.py:345-363
            if (model == ST3) v[2] = rv(K_out / p[o + 5], e_out, om_out + 180, fo) + gam;   // orbit.py:444-460
        }
        bool fast = false;
        for (int c = 0; c < ncomp; ++c) {
            vel[(int64_t)c * n_epochs + ep] = v[c];
            if (!(fabs(v[c]) < C_KMS)) fast = true;
        }
        if (fast) atomicExch(&s_flag, 1);
    }
    __syncthreads();
    if (threadIdx.x == 0 && flag) flag[0] = s_flag;
}

// Derivatives of rv(K, e, omega, f(t; T0, P, e)) with respect to (K, e, omega, P, T0) at true anomaly f and eccentric
// anomaly E.  M = 2 pi ((t - T0) mod P) / P: dM/dP = -2 pi (t - T0) / P^2, dM/dT0 = -2 pi / P (the modulus drops out);
// dE/dM = 1 / (1 - e cos E), dE/de|M = sin E / (1 - e cos E), df/dE = sqrt(1 - e^2) / (1 - e cos E),
// df/de|E = sin f / (1 - e^2).  The + 2 pi branch of true_anomaly changes no derivative.
__device__ inline void rv_grad(double K, double e, double omega_deg, double P, double T0, double t, double f, double E,
                               double g[5]) {
    const double PI = 3.141592653589793;
    const double w = omega_deg * PI / 180;
    const double swf = sin(w + f), cw = cos(w);
    const double den = 1.0 - e * cos(E);
    const double se = sqrt(1.0 - e * e);
    const double dfdM = se / (den * den);
    const double dfde = se * sin(E) / (den * den) + sin(f) / (1.0 - e * e);
    const double dvdf = -K * swf;
    g[0] = cos(w + f) + e * cw;
    g[1] = dvdf * dfde + K * cw;
    g[2] = -K * (swf + e * sin(w)) * (PI / 180);
    g[3] = dvdf * dfdM * (-2 * PI * (t - T0) / (P * P));
    g[4] = dvdf * dfdM * (-2 * PI / P);
}

// dv_c[ep] / dp_k for every model, as orbit_block computes v: jac [ncomp][n_epochs][norb] (p in utils.registered_params
// order).  The secondary of a pair uses K / q and omega + 180, the triples sum these terms.  One block; threads stride
// over epochs.
__device__ inline void orbit_jacobian_block(int model, const double* __restrict__ p, const double* __restrict__ dates,
                                            int n_epochs, double* __restrict__ jac) {
    const int ncomp = model_ncomp(model), norb = model_norb(model);
    for (int ep = threadIdx.x; ep < n_epochs; ep += blockDim.x) {
        const double t = dates[ep];
        for (int c = 0; c < ncomp; ++c) {
            double* Jc = jac + ((int64_t)c * n_epochs + ep) * norb;
            for (int k = 0; k < norb; ++k) Jc[k] = 0.0;
            Jc[norb - 1] = 1.0;                                              // gamma
        }
        double* J0 = jac + (int64_t)ep * norb;                               // rows of components 0, 1, 2
        double* J1 = J0 + (int64_t)n_epochs * norb;
        double* J2 = J1 + (int64_t)n_epochs * norb;
        // Kepler term with scale K / q (q = 1: primary): derivatives into J at K index ik (and q index iq >= 0)
        auto term = [&](double* Jc, int o, int iq, double q, double K, double e, double om, double P, double T0, double f,
                        double E) {
            double g[5];
            rv_grad(K / q, e, om, P, T0, t, f, E, g);
            Jc[o] += g[0] / q;
            if (iq >= 0) Jc[iq] += -K / (q * q) * g[0];
#pragma unroll
            for (int k = 1; k < 5; ++k) Jc[o + k] += g[k];
        };
        if (model == SB1 || model == SB2) {
            const int o = (model == SB2) ? 1 : 0;
            const double K = p[o + 0], e = p[o + 1], om = p[o + 2], P = p[o + 3], T0 = p[o + 4];
            double E;
            const double f = true_anomaly(t, T0, P, e, &E);
            term(J0, o, -1, 1.0, K, e, om, P, T0, f, E);
            if (model == SB2) term(J1, o, 0, p[0], K, e, om + 180, P, T0, f, E);
        } else {
            const int o = (model == ST1) ? 0 : 1;
            const double K_in = p[o + 0], e_in = p[o + 1], om_in = p[o + 2], P_in = p[o + 3], T0_in = p[o + 4];
            const int oo = o + 5 + ((model == ST3) ? 1 : 0);
            const double K_out = p[oo + 0], e_out = p[oo + 1], om_out = p[oo + 2], P_out = p[oo + 3], T0_out = p[oo + 4];
            double Ei, Eo;
            const double fi = true_anomaly(t, T0_in, P_in, e_in, &Ei);
            const double fo = true_anomaly(t, T0_out, P_out, e_out, &Eo);
            term(J0, o, -1, 1.0, K_in, e_in, om_in, P_in, T0_in, fi, Ei);
            term(J0, oo, -1, 1.0, K_out, e_out, om_out, P_out, T0_out, fo, Eo);
            if (model != ST1) {
                term(J1, o, 0, p[0], K_in, e_in, om_in + 180, P_in, T0_in, fi, Ei);
                term(J1, oo, -1, 1.0, K_out, e_out, om_out, P_out, T0_out, fo, Eo);
            }
            if (model == ST3) term(J2, oo, o + 5, p[o + 5], K_out, e_out, om_out + 180, P_out, T0_out, fo, Eo);
        }
    }
}

__global__ void orbit_kernel(int model, const double* __restrict__ p, const double* __restrict__ dates,
                             int n_epochs, double* __restrict__ vel, int* __restrict__ flag, int check_gp) {
    orbit_block(model, p, dates, n_epochs, vel, flag, check_gp);
}

// Chunk farm: block b evaluates chunk b's epochs (every chunk carries its own date vector, data.py:126).
// One descriptor per (chunk, proposal) work item; p_off selects the proposal's parameter vector.
struct OrbitDesc {
    const double* dates;
    double* vel;
    int* flag;
    int n_epochs;
    int p_off;
};
__global__ void orbit_farm_kernel(int model, const double* __restrict__ p, const OrbitDesc* __restrict__ descs) {
    const OrbitDesc d = descs[blockIdx.x];
    orbit_block(model, p + d.p_off, d.dates, d.n_epochs, d.vel, d.flag, 1);
}

}  // namespace psoap
