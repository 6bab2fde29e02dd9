/*
 * smenv_oracle.c -- CPU restatement (plain C, float64) of the reference's per-step environment path.
 *
 * TEST INFRASTRUCTURE ONLY.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
 * legs may load this library; the product path (safemotionsrisk_b200/) never does.
 *
 * PARITY UNPINNED: the arithmetic of the reference lives in two third-party native packages that are not vendored
 * in /root/reference and cannot be installed here (requirements.txt:9-10): klimits==1.1.3 (safe acceleration range)
 * and pybullet==3.1.6 (FK, GJK closest points, contact manifolds, motor tracking).  The reference has no tests or
 * golden vectors (SURVEY.md section 4).  This file therefore restates
 *   - the reference's own Python call sites line by line (cited below), and
 *   - the published semantics of the two libraries (SURVEY.md Appendix B; Kiemel & Kroeger, ICRA 2021 for klimits),
 * and is pinned by closed forms, invariants and brute-force cross-checks in tests/ instead of by reference outputs.
 *
 * Step order follows safe_motions_base.py:1043-1227 (step / process_step_outcome), :1229-1299 (24 sub-steps),
 * :1330-1365 (_process_action_outcome) and :1775-1799 (_check_termination).
 */
#include "../include/smenv.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

#define BIG 1.0e6

/* ------------------------------------------------------------------------------------------------------------
 * 1. Safe acceleration range  (actions.py:97-106, :206-211 -> klimits.PosVelJerkLimitation)
 *
 * Model (actions.py:468-487): acceleration is piecewise linear between knots spaced ts.  The range of the next
 * knot acceleration a1 is the intersection of
 *   jerk      [a0 - J ts, a0 + J ts]
 *   acc       [-A, A]
 *   velocity  the largest / smallest a1 from which the hardest admissible braking (a_{k+1} = max(a_k - J ts, -A))
 *             keeps the velocity peak at or below the limit
 *   position  the largest / smallest a1 from which the same braking keeps the position peak at or below the limit
 * i.e. the exact set of a1 for which a limit-respecting continuation exists forever (the property klimits
 * guarantees).  If a bound cannot be met inside the jerk/acc interval the range collapses onto the least violating
 * end and a violation code is set (used to reject sampled start states, ctlp.py:1513-1523).
 * ---------------------------------------------------------------------------------------------------------- */

/* Largest a1 such that the velocity never exceeds vmax.  J = |min jerk|, A = |min acceleration|. */
static double vel_upper(double v0, double a0, double vmax, double J, double A, double ts) {
    double c = v0 + a0 * ts * 0.5 - vmax;
    if (c > 0.0) {
        /* even a1 = 0 overshoots at the next knot: a1 < 0 and the peak lies inside the first interval */
        double den = vmax - v0;
        if (a0 <= 0.0 || den <= 0.0) return -BIG;
        return a0 - (a0 * a0 * ts) / (2.0 * den);
    }
    /* a1 >= 0: braking at full jerk through zero, peak = v1 + a1^2 / (2J) */
    double a1u = J * (sqrt(ts * ts * 0.25 - 2.0 * c / J) - ts * 0.5);
    double JT = J * ts;
    double delta = JT - A;
    if (delta <= 0.0) return a1u;
    double n = ceil(a1u / JT) - 1.0;
    if (n < 0.0) n = 0.0;
    double x = a1u - n * JT;
    if (x >= delta) return a1u;
    /* the last braking interval is clamped by the acceleration limit: slope (x + A) / ts instead of J */
    double C = c + JT * ts * n * (n + 1.0) * 0.5;
    double D = ts * (n + 0.5);
    double qa = D + ts * 0.5, qb = C + D * A, qc = C * A;
    x = (sqrt(qb * qb - 4.0 * qa * qc) - qb) / (2.0 * qa);
    return n * JT + x;
}

/* Highest position reached from (p, v, a) when the next knot acceleration is a1 and the hardest braking follows, and
 * (if dbest_out is given) its derivative with respect to a1: the state derivatives dp, dv, da ride along the
 * simulated profile; the derivative of an interior peak is taken at fixed tau (the peak is a stationary point of the
 * position, so the motion of tau does not contribute). */
static double pos_peak_d(double p, double v, double a, double a1, double J, double A, double ts, double* dbest_out) {
    double best = p, dbest = 0.0;
    double dp = 0.0, dv = 0.0, da = 0.0, dan = 1.0;
    double an = a1;
    for (int it = 0; it < 16; ++it) {
        double j = (an - a) / ts;
        double dj = (dan - da) / ts;
        /* local maximum inside the interval: downward zero crossing of v(tau) = v + a tau + j tau^2 / 2 */
        double tau = -1.0;
        if (j == 0.0) {
            if (a < 0.0 && v > 0.0) tau = -v / a;
        } else {
            double disc = a * a - 2.0 * j * v;
            if (disc >= 0.0) {
                double s = sqrt(disc);
                if (a <= 0.0) {
                    if (s - a > 0.0) tau = 2.0 * v / (s - a);
                } else {
                    tau = (-a - s) / j;
                }
            }
        }
        if (tau > 0.0 && tau <= ts) {
            double pk = p + v * tau + 0.5 * a * tau * tau + (j * tau * tau * tau) / 6.0;
            if (pk > best) {
                best = pk;
                dbest = dp + dv * tau + 0.5 * da * tau * tau + (dj * tau * tau * tau) / 6.0;
            }
        }
        double pn = p + v * ts + (a / 3.0 + an / 6.0) * ts * ts;
        double vn = v + (a + an) * ts * 0.5;
        double dpn = dp + dv * ts + (da / 3.0 + dan / 6.0) * ts * ts;
        double dvn = dv + (da + dan) * ts * 0.5;
        p = pn; v = vn; a = an;
        dp = dpn; dv = dvn; da = dan;
        if (p > best) { best = p; dbest = dp; }
        if (a <= -A) {
            if (v > 0.0) {
                double pk = p + (v * v) / (2.0 * A);
                if (pk > best) { best = pk; dbest = dp + (v * dv) / A; }
            }
            break;
        }
        if (v <= 0.0 && a <= 0.0) break;
        an = a - J * ts;
        if (an < -A) { an = -A; dan = 0.0; }
    }
    if (dbest_out) *dbest_out = dbest;
    return best;
}
static double pos_peak(double p, double v, double a, double a1, double J, double A, double ts) {
    return pos_peak_d(p, v, a, a1, J, A, ts, (double*)0);
}

/* Acceptance window of the position-bound solve: a safe a1 (peak <= pmax) whose peak comes within this many rad of
 * the limit ends the search. */
#define POS_SOLVE_TOL 1e-10
/* Largest a1 in [lo, hi] whose position peak stays <= pmax; +BIG if hi itself is fine, -BIG if not even lo is.
 * The peak is an increasing, piecewise smooth and mostly convex function of a1: safeguarded Newton with the exact
 * derivative, aimed at the middle of the acceptance window, started from the secant of the bracket; a step that leaves
 * the bracket (flat stretches where the peak is the start position itself, kinks) is replaced by a bisection.
 * Mean 5 evaluations, at most 11 in 10^5 random cases (a regula falsi needed 8 on average and up to 26: the kernel
 * solves 32 bounds per warp in lockstep, so the longest solve of a warp sets its time). */
static double pos_upper(double p, double v, double a, double pmax, double lo, double hi, double J, double A,
                        double ts) {
    double fr = pos_peak(p, v, a, hi, J, A, ts) - pmax;
    if (fr <= 0.0) return BIG;
    double fl = pos_peak(p, v, a, lo, J, A, ts) - pmax;
    if (fl > 0.0) return fl > 1e-6 ? -BIG : lo; /* 1e-6 rad: the braking model ignores the opposite velocity limit, which can shift a
                                                   landing that rides exactly on the position limit by < 1e-6 rad */
    double xl = lo, xr = hi;
    double x = xr - fr * (xr - xl) / (fr - fl);
    if (!(x > xl && x < xr)) x = 0.5 * (xl + xr);
    for (int it = 0; it < 40; ++it) {
        double df;
        double f = pos_peak_d(p, v, a, x, J, A, ts, &df) - pmax;
        if (f <= 0.0 && f > -POS_SOLVE_TOL) return x;
        if (f <= 0.0) xl = x; else xr = x;
        if (xr - xl <= 1e-9) break;
        double xn = xl;
        if (df > 0.0) xn = x - (f + 0.5 * POS_SOLVE_TOL) / df;
        if (!(xn > xl && xn < xr)) xn = 0.5 * (xl + xr);
        x = xn;
    }
    return xl;
}

enum { CODE_VEL_HI = 1, CODE_VEL_LO = 2, CODE_POS_HI = 4, CODE_POS_LO = 8, CODE_ACC = 16 };

static void clamp_range(double* lo, double* hi, double blo, double bhi, int code_hi, int code_lo, int* code) {
    double nhi = *hi < bhi ? *hi : bhi;
    double nlo = *lo > blo ? *lo : blo;
    /* a bound that misses the interval by more than 1e-6 rad/s^2 is a violation; less is rounding noise of a
     * trajectory that rides exactly on a limit */
    if (nhi < *lo) { if (*lo - nhi > 1e-6) *code |= code_hi; nhi = *lo; }
    if (nlo > *hi) { if (nlo - *hi > 1e-6) *code |= code_lo; nlo = *hi; }
    if (nlo > nhi) { if (nlo - nhi > 1e-6) *code |= code_hi | code_lo; nlo = nhi; }
    *lo = nlo; *hi = nhi;
}

/* test hook: the braking-profile peak and its derivative with respect to the next-knot acceleration */
double smo_pos_peak(double p, double v, double a, double a1, double J, double A, double ts, double* dpeak) {
    return pos_peak_d(p, v, a, a1, J, A, ts, dpeak);
}

/* range of one joint with limits (J, A, V, [plo, phi]) */
static void safe_range_limits(double ts, double J, double A, double V, double plo, double phi, int limit_velocity,
                              int limit_position, double p, double v, double a, double* out_lo, double* out_hi,
                              int32_t* out_code) {
    int code = 0;
    double lo = a - J * ts, hi = a + J * ts;
    if (lo < -A) lo = -A;
    if (hi > A) hi = A;
    if (lo > hi) { /* |a| beyond the acceleration limit */
        code |= CODE_ACC;
        if (a > 0.0) lo = hi; else hi = lo;
    }
    if (limit_velocity) {
        double bhi = vel_upper(v, a, V, J, A, ts);
        double blo = -vel_upper(-v, -a, V, J, A, ts);
        clamp_range(&lo, &hi, blo, bhi, CODE_VEL_HI, CODE_VEL_LO, &code);
    }
    if (limit_position) {
        double bhi = pos_upper(p, v, a, phi, lo, hi, J, A, ts);
        double blo = -pos_upper(-p, -v, -a, -plo, -hi, -lo, J, A, ts);
        clamp_range(&lo, &hi, blo, bhi, CODE_POS_HI, CODE_POS_LO, &code);
    }
    *out_lo = lo; *out_hi = hi; *out_code = code;
}

void smo_safe_range_joint(const SmScene* sc, int j, double p, double v, double a, double* out_lo, double* out_hi,
                          int32_t* out_code) {
    safe_range_limits(sc->ts, sc->jerk_max[j], sc->acc_max[j], sc->vel_max[j], sc->pos_lo[j], sc->pos_hi[j],
                      sc->limit_velocity, sc->limit_position, p, v, a, out_lo, out_hi, out_code);
}

void smo_safe_range(const SmScene* sc, const double* q, const double* v, const double* a, double* lo, double* hi,
                    int32_t* code) {
    for (int j = 0; j < sc->n_joints; ++j) smo_safe_range_joint(sc, j, q[j], v[j], a[j], &lo[j], &hi[j], &code[j]);
}

/* ------------------------------------------------------------------------------------------------------------
 * 2. Action mapping and interpolation  (actions.py:268-280, :412-443, :468-487)
 * ---------------------------------------------------------------------------------------------------------- */
void smo_map_action(const SmScene* sc, const double* u, const double* lo_in, const double* hi_in, double* a1) {
    for (int j = 0; j < sc->n_joints; ++j) {
        double lo = lo_in[j], hi = hi_in[j];
        if (sc->action_mapping_factor != 1.0) { /* actions.py:271-276 */
            double mf = 0.5 * (sc->action_mapping_factor + 1.0);
            double diff = hi - lo;
            hi = lo + mf * diff;
            lo = lo + (1.0 - mf) * diff;
        }
        a1[j] = lo + 0.5 * (u[j] + 1.0) * (hi - lo); /* klimits.denormalize == actions.py:496-498 */
    }
}

/* time of sub-step k (1-based) as np.linspace(ts / S, ts, S) produces it (actions.py:420-421) */
static double substep_time(const SmScene* sc, int k) {
    int S = sc->substeps;
    if (S <= 1 || k == S) return sc->ts;
    double start = sc->ts / S;
    double step = (sc->ts - start) / (double)(S - 1);
    return start + (double)(k - 1) * step;
}

static void interpolate(const SmScene* sc, double q0, double v0, double a0, double a1, double t, double* q,
                        double* v, double* a) {
    double jerk = (a1 - a0) / sc->ts;
    *a = a0 + jerk * t;                                                           /* actions.py:482-487 */
    *v = v0 + a0 * t + 0.5 * jerk * t * t;                                        /* actions.py:475-480 */
    *q = q0 + v0 * t + 0.5 * a0 * t * t + (1.0 / 6.0) * jerk * t * t * t;         /* actions.py:468-473 */
}

/* ------------------------------------------------------------------------------------------------------------
 * 3. Forward kinematics  (ctlp.py:2940-2988 + LinkBase.get_position :5163-5195 -> getLinkState[4:6])
 *    T_frame = T_parent * [R_fix | t_fix] * Rot(axis, q)          (Bullet: parent * origin * joint rotation)
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct { double R[9]; double t[3]; } Xf;

static void xf_identity(Xf* x) {
    memset(x, 0, sizeof(*x));
    x->R[0] = x->R[4] = x->R[8] = 1.0;
}
static void mat_mul(const double* A, const double* B, double* C) {
    for (int i = 0; i < 3; ++i)
        for (int k = 0; k < 3; ++k) C[3 * i + k] = A[3 * i] * B[k] + A[3 * i + 1] * B[3 + k] + A[3 * i + 2] * B[6 + k];
}
static void mat_vec(const double* A, const double* x, double* y) {
    for (int i = 0; i < 3; ++i) y[i] = A[3 * i] * x[0] + A[3 * i + 1] * x[1] + A[3 * i + 2] * x[2];
}
static void axis_angle(const double* ax, double ang, double* R) {
    double c = cos(ang), s = sin(ang), t = 1.0 - c, x = ax[0], y = ax[1], z = ax[2];
    R[0] = t * x * x + c;     R[1] = t * x * y - s * z; R[2] = t * x * z + s * y;
    R[3] = t * x * y + s * z; R[4] = t * y * y + c;     R[5] = t * y * z - s * x;
    R[6] = t * x * z - s * y; R[7] = t * y * z + s * x; R[8] = t * z * z + c;
}
void smo_fk(const SmScene* sc, const double* q, Xf* frames /* [1 + n_joints] */) {
    xf_identity(&frames[0]);
    for (int j = 0; j < sc->n_joints; ++j) {
        const Xf* P = &frames[sc->joint_parent[j]];
        double Rj[9], R1[9], tp[3];
        mat_mul(P->R, sc->joint_R[j], R1);
        mat_vec(P->R, sc->joint_t[j], tp);
        axis_angle(sc->joint_axis[j], q[j], Rj);
        mat_mul(R1, Rj, frames[1 + j].R);
        for (int i = 0; i < 3; ++i) frames[1 + j].t[i] = P->t[i] + tp[i];
    }
}
/* exported: 12 doubles per frame (R row major, t) */
void smo_fk_flat(const SmScene* sc, const double* q, double* out) {
    Xf fr[1 + SM_MAX_JOINTS];
    smo_fk(sc, q, fr);
    for (int f = 0; f <= sc->n_joints; ++f) {
        memcpy(out + 12 * f, fr[f].R, 9 * sizeof(double));
        memcpy(out + 12 * f + 9, fr[f].t, 3 * sizeof(double));
    }
}

static void quat_to_mat(const double* q /* xyzw */, double* R) {
    double x = q[0], y = q[1], z = q[2], w = q[3];
    double n = x * x + y * y + z * z + w * w;
    double s = n > 0.0 ? 2.0 / n : 0.0;
    R[0] = 1.0 - s * (y * y + z * z); R[1] = s * (x * y - w * z);       R[2] = s * (x * z + w * y);
    R[3] = s * (x * y + w * z);       R[4] = 1.0 - s * (x * x + z * z); R[5] = s * (y * z - w * x);
    R[6] = s * (x * z - w * y);       R[7] = s * (y * z + w * x);       R[8] = 1.0 - s * (x * x + y * y);
}
/* p.getQuaternionFromEuler: roll about x, pitch about y, yaw about z, R = Rz Ry Rx */
static void euler_to_mat(const double* e, double* R) {
    double cr = cos(e[0]), sr = sin(e[0]), cp = cos(e[1]), sp = sin(e[1]), cy = cos(e[2]), sy = sin(e[2]);
    R[0] = cy * cp; R[1] = cy * sp * sr - sy * cr; R[2] = cy * sp * cr + sy * sr;
    R[3] = sy * cp; R[4] = sy * sp * sr + cy * cr; R[5] = sy * sp * cr - cy * sr;
    R[6] = -sp;     R[7] = cp * sr;                R[8] = cp * cr;
}

/* ------------------------------------------------------------------------------------------------------------
 * 4. GJK distance between two convex vertex sets (restates what p.getClosestPoints computes on the margin-less
 *    cores, SURVEY Appendix B.2; call sites ctlp.py:3267, :3300, :3353).  Voronoi-region simplex solver.
 * ---------------------------------------------------------------------------------------------------------- */
static double dot3(const double* a, const double* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
static void sub3(const double* a, const double* b, double* c) { c[0] = a[0] - b[0]; c[1] = a[1] - b[1]; c[2] = a[2] - b[2]; }
static void cross3(const double* a, const double* b, double* c) {
    c[0] = a[1] * b[2] - a[2] * b[1]; c[1] = a[2] * b[0] - a[0] * b[2]; c[2] = a[0] * b[1] - a[1] * b[0];
}

/* support of the transformed vertex set in world direction d: returns world point */
static void support(const double* verts, int n, const Xf* T, const double* d, double* out) {
    double dl[3]; /* d in the local frame = R^T d */
    dl[0] = T->R[0] * d[0] + T->R[3] * d[1] + T->R[6] * d[2];
    dl[1] = T->R[1] * d[0] + T->R[4] * d[1] + T->R[7] * d[2];
    dl[2] = T->R[2] * d[0] + T->R[5] * d[1] + T->R[8] * d[2];
    int best = 0;
    double bv = -1e300;
    for (int i = 0; i < n; ++i) {
        double s = dot3(verts + 3 * i, dl);
        if (s > bv) { bv = s; best = i; }
    }
    double w[3];
    mat_vec(T->R, verts + 3 * best, w);
    out[0] = w[0] + T->t[0]; out[1] = w[1] + T->t[1]; out[2] = w[2] + T->t[2];
}

/* closest point to the origin on triangle abc; writes barycentric mask of the supporting sub-simplex */
static void closest_triangle(const double* a, const double* b, const double* c, double* out, int* mask) {
    double ab[3], ac[3], ap[3], bp[3], cp[3];
    sub3(b, a, ab); sub3(c, a, ac);
    ap[0] = -a[0]; ap[1] = -a[1]; ap[2] = -a[2];
    double d1 = dot3(ab, ap), d2 = dot3(ac, ap);
    if (d1 <= 0.0 && d2 <= 0.0) { memcpy(out, a, 24); *mask = 1; return; }
    bp[0] = -b[0]; bp[1] = -b[1]; bp[2] = -b[2];
    double d3 = dot3(ab, bp), d4 = dot3(ac, bp);
    if (d3 >= 0.0 && d4 <= d3) { memcpy(out, b, 24); *mask = 2; return; }
    double vc = d1 * d4 - d3 * d2;
    if (vc <= 0.0 && d1 >= 0.0 && d3 <= 0.0) {
        double v = d1 / (d1 - d3);
        for (int i = 0; i < 3; ++i) out[i] = a[i] + v * ab[i];
        *mask = 3; return;
    }
    cp[0] = -c[0]; cp[1] = -c[1]; cp[2] = -c[2];
    double d5 = dot3(ab, cp), d6 = dot3(ac, cp);
    if (d6 >= 0.0 && d5 <= d6) { memcpy(out, c, 24); *mask = 4; return; }
    double vb = d5 * d2 - d1 * d6;
    if (vb <= 0.0 && d2 >= 0.0 && d6 <= 0.0) {
        double w = d2 / (d2 - d6);
        for (int i = 0; i < 3; ++i) out[i] = a[i] + w * ac[i];
        *mask = 5; return;
    }
    double va = d3 * d6 - d5 * d4;
    if (va <= 0.0 && (d4 - d3) >= 0.0 && (d5 - d6) >= 0.0) {
        double w = (d4 - d3) / ((d4 - d3) + (d5 - d6));
        for (int i = 0; i < 3; ++i) out[i] = b[i] + w * (c[i] - b[i]);
        *mask = 6; return;
    }
    double denom = 1.0 / (va + vb + vc);
    double v = vb * denom, w = vc * denom;
    for (int i = 0; i < 3; ++i) out[i] = a[i] + ab[i] * v + ac[i] * w;
    *mask = 7;
}

/* simplex S (n points, newest last) -> closest point v to origin, reduced simplex. returns 1 if origin enclosed */
static int simplex_closest(double S[4][3], int* n, double* v) {
    if (*n == 1) { memcpy(v, S[0], 24); return 0; }
    if (*n == 2) {
        double ab[3];
        sub3(S[1], S[0], ab);
        double t = -dot3(S[0], ab);
        double den = dot3(ab, ab);
        if (t <= 0.0 || den <= 0.0) { memcpy(v, S[0], 24); *n = 1; return 0; }
        if (t >= den) { memcpy(v, S[1], 24); memcpy(S[0], S[1], 24); *n = 1; return 0; }
        t /= den;
        for (int i = 0; i < 3; ++i) v[i] = S[0][i] + t * ab[i];
        return 0;
    }
    if (*n == 3) {
        int mask;
        closest_triangle(S[0], S[1], S[2], v, &mask);
        int k = 0;
        double T[3][3];
        for (int i = 0; i < 3; ++i) if (mask & (1 << i)) memcpy(T[k++], S[i], 24);
        for (int i = 0; i < k; ++i) memcpy(S[i], T[i], 24);
        *n = k;
        return 0;
    }
    /* tetrahedron: test the four faces whose outside half-space contains the origin */
    static const int F[4][4] = {{0, 1, 2, 3}, {0, 1, 3, 2}, {0, 2, 3, 1}, {1, 2, 3, 0}};
    double best = 1e300, bv[3] = {0, 0, 0};
    int bmask = 0, bf = -1, outside_any = 0;
    for (int f = 0; f < 4; ++f) {
        const double *a = S[F[f][0]], *b = S[F[f][1]], *c = S[F[f][2]], *d = S[F[f][3]];
        double ab[3], ac[3], n[3], ad[3];
        sub3(b, a, ab); sub3(c, a, ac); cross3(ab, ac, n); sub3(d, a, ad);
        double sd = dot3(ad, n);   /* side of the opposite vertex */
        double so = -dot3(a, n);   /* side of the origin */
        /* degenerate (flat) tetrahedron: treat every face as candidate.  Flat to rounding counts as well: there the sign
         * of sd is noise, and the origin far off the plane could pass every face test and be taken as enclosed (a
         * converged search whose last support point closes a parallelogram with the simplex reported distance 0). */
        if (fabs(sd) <= 1e-10 * sqrt(dot3(ab, ab) * dot3(ac, ac) * dot3(ad, ad))) sd = 0.0;
        if (sd == 0.0) { outside_any = 1; }
        if (sd == 0.0 || so * sd < 0.0) {
            outside_any = 1;
            double p[3];
            int m;
            closest_triangle(a, b, c, p, &m);
            double dd = dot3(p, p);
            if (dd < best) { best = dd; memcpy(bv, p, 24); bmask = m; bf = f; }
        }
    }
    if (!outside_any || bf < 0) return 1;
    double T[3][3];
    int k = 0;
    for (int i = 0; i < 3; ++i) if (bmask & (1 << i)) memcpy(T[k++], S[F[bf][i]], 24);
    for (int i = 0; i < k; ++i) memcpy(S[i], T[i], 24);
    *n = k;
    memcpy(v, bv, 24);
    return 0;
}

typedef struct { long calls, iters, dots; } GjkStats;
static GjkStats g_stats;

/* distance between the convex hulls of A and B (core distance, >= 0; 0 if they overlap).
 * If upper > 0 the search stops early once the distance is proven >= upper, and returns a value >= upper. */
double smo_gjk(const double* vA, int nA, const Xf* TA, const double* vB, int nB, const Xf* TB, double upper) {
    double S[4][3], v[3], w[3], sa[3], sb[3], d[3];
    int n = 0;
    g_stats.calls++;
    /* initial direction: between the first vertices */
    d[0] = 1.0; d[1] = 0.0; d[2] = 0.0;
    support(vA, nA, TA, d, sa);
    d[0] = -1.0;
    support(vB, nB, TB, d, sb);
    sub3(sa, sb, v);
    memcpy(S[0], v, 24);
    n = 1;
    double vv = dot3(v, v);
    for (int it = 0; it < 64; ++it) {
        g_stats.iters++;
        g_stats.dots += nA + nB;
        if (vv <= 1e-24) return 0.0;
        d[0] = -v[0]; d[1] = -v[1]; d[2] = -v[2];
        support(vA, nA, TA, d, sa);
        d[0] = v[0]; d[1] = v[1]; d[2] = v[2];
        support(vB, nB, TB, d, sb);
        sub3(sa, sb, w);
        double vw = dot3(v, w);
        if (upper > 0.0 && vw > 0.0 && vw * vw >= upper * upper * vv) return sqrt(vv) > upper ? sqrt(vv) : upper;
        if (vv - vw <= 1e-14 * vv) break; /* converged: |v| - v.w/|v| <= 1e-14 |v| */
        int dup = 0;
        for (int i = 0; i < n; ++i) {
            double e[3];
            sub3(S[i], w, e);
            if (dot3(e, e) <= 1e-28) dup = 1;
        }
        if (dup) break;
        memcpy(S[n], w, 24);
        n++;
        double nv[3];
        if (simplex_closest(S, &n, nv)) return 0.0;
        double nvv = dot3(nv, nv);
        if (nvv >= vv) break; /* no progress (numerical floor) */
        memcpy(v, nv, 24);
        vv = nvv;
    }
    return sqrt(vv);
}

void smo_gjk_stats(long* out, int reset) {
    out[0] = g_stats.calls; out[1] = g_stats.iters; out[2] = g_stats.dots;
    if (reset) memset(&g_stats, 0, sizeof(g_stats));
}

/* flat entry for the tests: T = 12 doubles (R row major, t) */
double smo_gjk_flat(const double* vA, int nA, const double* TA, const double* vB, int nB, const double* TB,
                    double upper) {
    Xf a, b;
    memcpy(a.R, TA, 72); memcpy(a.t, TA + 9, 24);
    memcpy(b.R, TB, 72); memcpy(b.t, TB + 9, 24);
    return smo_gjk(vA, nA, &a, vB, nB, &b, upper);
}

/* ------------------------------------------------------------------------------------------------------------
 * 5. Obstacle kinematics  (Planet.update ctlp.py:4503-4531, Ball.update :4103-4131)
 * ---------------------------------------------------------------------------------------------------------- */
static void planet_pose(const SmScene* sc, int o, int index_one, Xf* T) {
    int idx = index_one;
    if (o == 1) { /* coupled planet: ctlp.py:4481-4485 */
        idx = (index_one + sc->planet_shift) % sc->planet_steps;
        if (idx < 0) idx += sc->planet_steps;
    }
    quat_to_mat(sc->planet_quat[o] + 4 * idx, T->R);
    memcpy(T->t, sc->planet_pos[o] + 3 * idx, 24);
}

static void ball_position(const double* ob, double t, double* p) {
    /* ctlp.py:4109-4110: base_pos + v0 t + 0.5 g t^2 */
    p[0] = ob[SM_OB_BALL_P0 + 0] + ob[SM_OB_BALL_V0 + 0] * t;
    p[1] = ob[SM_OB_BALL_P0 + 1] + ob[SM_OB_BALL_V0 + 1] * t;
    p[2] = (ob[SM_OB_BALL_P0 + 2] + ob[SM_OB_BALL_V0 + 2] * t) + (0.5 * -9.81) * (t * t);
}
static void ball_pose(const double* ob, double t, Xf* T) {
    double e[3];
    ball_position(ob, t, T->t);
    e[0] = ob[SM_OB_BALL_EULER0 + 0];
    e[1] = ob[SM_OB_BALL_EULER0 + 1] + t * ob[SM_OB_BALL_OMEGA]; /* ctlp.py:4112-4114 */
    e[2] = ob[SM_OB_BALL_EULER0 + 2];
    euler_to_mat(e, T->R);
}

static void shape_frame(const SmScene* sc, const SmShape* sh, const Xf* robot, const Xf* obst, Xf* out) {
    if (sh->frame >= 100) *out = obst[sh->frame - 100];
    else *out = robot[sh->frame];
    (void)sc;
}

static double pair_distance(const SmScene* sc, int ia, int ib, const Xf* robot, const Xf* obst, double upper) {
    const SmShape *A = &sc->shapes[ia], *B = &sc->shapes[ib];
    Xf TA, TB;
    shape_frame(sc, A, robot, obst, &TA);
    shape_frame(sc, B, robot, obst, &TB);
    double core = smo_gjk(sc->verts + 3 * A->vert_off, A->vert_cnt, &TA, sc->verts + 3 * B->vert_off, B->vert_cnt,
                          &TB, upper > 0.0 ? upper + A->margin + B->margin : 0.0);
    return core - A->margin - B->margin; /* Bullet: distance between cores minus both margins (Appendix B.2) */
}

/* ------------------------------------------------------------------------------------------------------------
 * 6. Distances  (get_minimum_distance ctlp.py:3282-3374, get_minimum_distance_to_moving_obstacles :3217-3280)
 * ---------------------------------------------------------------------------------------------------------- */
void smo_human_fk(const SmScene* sc, const double* hq, Xf* fr);
/* hq: joint angles of the human (Human scene), else NULL */
static void obstacle_poses_h(const SmScene* sc, const double* ob, const double* hq, Xf* obst) {
    for (int o = 0; o < sc->n_obstacles; ++o) {
        if (sc->obst_kind[o] == SM_OBST_HUMAN) { if (hq) smo_human_fk(sc, hq, obst); continue; }
        if (sc->obst_kind[o] == SM_OBST_PLANET) planet_pose(sc, o, (int)ob[SM_OB_INDEX], &obst[o]);
        else if (sc->obst_kind[o] == SM_OBST_BALL) ball_pose(ob, ob[SM_OB_BALL_T], &obst[o]);
        else xf_identity(&obst[o]);
    }
}


void smo_distances_h(const SmScene* sc, const double* q, const double* ob, const double* hq, double* d_static,
                     double* d_self, double* d_moving);
void smo_distances(const SmScene* sc, const double* q, const double* ob, double* d_static, double* d_self,
                   double* d_moving) {
    smo_distances_h(sc, q, ob, (const double*)0, d_static, d_self, d_moving);
}
/* hq: setpoint pose of the human (set_position_in_obstacle_client_to_setpoints, ctlp.py:3246-3251), else NULL */
void smo_distances_h(const SmScene* sc, const double* q, const double* ob, const double* hq, double* d_static,
                     double* d_self, double* d_moving) {
    Xf robot[1 + SM_MAX_JOINTS], obst[SM_MAX_OBST_FRAMES];
    smo_fk(sc, q, robot);
    obstacle_poses_h(sc, ob, hq, obst);
    /* static and self: start at the cap, points beyond the query distance are not returned (ctlp.py:3290-3320) */
    double ds = sc->static_cap, dself = sc->static_cap;
    for (int i = 0; i < sc->n_static_pairs; ++i) {
        double d = pair_distance(sc, sc->static_pairs[i][0], sc->static_pairs[i][1], robot, obst, sc->static_cap);
        if (d <= sc->static_cap && d < ds) ds = d;
    }
    for (int i = 0; i < sc->n_self_pairs; ++i) {
        double d = pair_distance(sc, sc->self_pairs[i][0], sc->self_pairs[i][1], robot, obst, sc->static_cap);
        if (d <= sc->static_cap && d < dself) dself = d;
    }
    *d_static = ds;
    *d_self = dself;
    /* moving (ctlp.py:3217-3280): latched contact -> 0; inactive ball that did not hit -> not in the list */
    double dm = sc->moving_query + 0.002;
    if (ob[SM_OB_LATCH] != 0.0) { *d_moving = 0.0; return; }
    for (int o = 0; o < sc->n_obstacles; ++o) {
        if (sc->obst_kind[o] == SM_OBST_BALL && ob[SM_OB_BALL_ACTIVE] == 0.0) continue;
        for (int r = 0; r < sc->n_mov_reward; ++r)
            for (int s = 0; s < sc->obst_shape_cnt[o]; ++s) {
                double d = pair_distance(sc, sc->mov_reward[r], sc->obst_shape_off[o] + s, robot, obst,
                                         sc->moving_query);
                if (d <= sc->moving_query && d < dm) {
                    dm = d;
                    if (dm <= 0.0) { *d_moving = 0.0; return; } /* ctlp.py:3277-3278 */
                }
            }
    }
    *d_moving = dm;
}

/* distance of every pair of the distance classes at robot pose q, margins subtracted, GJK without early stop (test
 * hook: the tests find the pair that holds a class minimum and how far the other pairs are).  Pairs in the order of the
 * device's pair table (smenv_create): static pairs, self pairs, then per obstacle, per mov_reward shape, per part.
 * Obstacle poses as in smo_distances_h (hq: the human's joint angles, else NULL); the class rules of smo_distances_h
 * (cap and query filters, inactive ball, latched contact) are not applied. */
void smo_plan_pair_distances(const SmScene* sc, const double* q, const double* ob, const double* hq, double* out) {
    Xf robot[1 + SM_MAX_JOINTS], obst[SM_MAX_OBST_FRAMES];
    smo_fk(sc, q, robot);
    obstacle_poses_h(sc, ob, hq, obst);
    int k = 0;
    for (int i = 0; i < sc->n_static_pairs; ++i)
        out[k++] = pair_distance(sc, sc->static_pairs[i][0], sc->static_pairs[i][1], robot, obst, 0.0);
    for (int i = 0; i < sc->n_self_pairs; ++i)
        out[k++] = pair_distance(sc, sc->self_pairs[i][0], sc->self_pairs[i][1], robot, obst, 0.0);
    for (int o = 0; o < sc->n_obstacles; ++o)
        for (int r = 0; r < sc->n_mov_reward; ++r)
            for (int s = 0; s < sc->obst_shape_cnt[o]; ++s)
                out[k++] = pair_distance(sc, sc->mov_reward[r], sc->obst_shape_off[o] + s, robot, obst, 0.0);
}

/* contact in the simulation client: any manifold point between obstacle o and the robot, i.e. some convex pair
 * closer than the manifold's contact breaking threshold (SURVEY Appendix B.5; ctlp.py:4570-4579, :4186-4194) */
static int contact_exists(const SmScene* sc, int o, const Xf* robot, const Xf* obst) {
    for (int r = 0; r < sc->n_mov_contact; ++r)
        for (int s = 0; s < sc->obst_shape_cnt[o]; ++s) {
            double th = sc->contact_thresh[o][r];
            double d = pair_distance(sc, sc->mov_contact[r], sc->obst_shape_off[o] + s, robot, obst, th + 1e-3);
            if (d <= th) return 1;
        }
    return 0;
}

/* ------------------------------------------------------------------------------------------------------------
 * 7. Observation  (observations.py:233-351; ctlp.py:2352-2391)
 * ---------------------------------------------------------------------------------------------------------- */
static float clip1(double x) {
    float f = (float)x; /* np.array(..., dtype=np.float32) then clip (observations.py:343-351) */
    if (f > 1.0f) f = 1.0f;
    if (f < -1.0f) f = -1.0f;
    return f;
}
void smo_observation_tp(const SmScene* sc, const double* kin, const double* ob, const double* tp, float* obs) {
    int nj = sc->n_joints, k = 0;
    const double *q = kin, *v = kin + 8, *a = kin + 16;
    for (int j = 0; j < nj; ++j) obs[k++] = clip1(-1.0 + 2.0 * (q[j] - sc->pos_lo[j]) / (sc->pos_hi[j] - sc->pos_lo[j]));
    for (int j = 0; j < nj; ++j) obs[k++] = clip1(v[j] / sc->vel_max[j]);
    for (int j = 0; j < nj; ++j) obs[k++] = clip1(a[j] / sc->acc_max[j]);
    if (sc->use_target_points && tp) { /* observations.py:326-340; ctlp.py:2247-2271 (the target point is active) */
        if (sc->obs_add_tp_pos)
            for (int i = 0; i < 3; ++i)
                obs[k++] = clip1(-1.0 + 2.0 * (tp[SM_TP_POS + i] - sc->tp_box_min[i]) / (sc->tp_box_max[i] - sc->tp_box_min[i]));
        if (sc->obs_add_tp_rel)
            for (int i = 0; i < 3; ++i) {
                double rel = tp[SM_TP_POS + i] - tp[SM_TP_LINK_POS + i];
                obs[k++] = clip1(-1.0 + 2.0 * (rel - sc->tp_rel_min[i]) / (sc->tp_rel_max[i] - sc->tp_rel_min[i]));
            }
    }
    for (int o = 0; o < sc->n_obstacles; ++o) {
        if (sc->obst_kind[o] == SM_OBST_BALL) { /* position then velocity, both normalised (ctlp.py:2364-2377) */
            double p[3], t = ob[SM_OB_BALL_T];
            ball_position(ob, t, p);
            for (int i = 0; i < 3; ++i)
                obs[k++] = clip1(-1.0 + 2.0 * (p[i] - sc->ball_obs_pos_min[i]) /
                                            (sc->ball_obs_pos_max[i] - sc->ball_obs_pos_min[i]));
            for (int i = 0; i < 3; ++i) {
                double vel = ob[SM_OB_BALL_V0 + i] + (i == 2 ? -9.81 : 0.0) * t; /* ctlp.py:4146-4152 */
                obs[k++] = clip1(-1.0 + 2.0 * (vel - sc->ball_obs_vel_min[i]) /
                                            (sc->ball_obs_vel_max[i] - sc->ball_obs_vel_min[i]));
            }
        }
    }
    if (sc->n_obstacles > 0 && sc->obst_kind[0] == SM_OBST_PLANET) { /* observations.py:262-288 */
        int idx = (int)ob[SM_OB_INDEX];
        if (sc->obs_planet_size == 1) {
            obs[k++] = clip1(-1.0 + 2.0 * ((double)idx - 0.0) / ((double)sc->planet_steps - 0.0));
        } else {
            for (int i = 0; i < 2; ++i) {
                double lo = -sc->planet_obs_half[i], hi = sc->planet_obs_half[i];
                obs[k++] = clip1(-1.0 + 2.0 * (sc->planet_local_xy[2 * idx + i] - lo) / (hi - lo));
            }
        }
    }
}

void smo_observation(const SmScene* sc, const double* kin, const double* ob, float* obs) {
    smo_observation_tp(sc, kin, ob, 0, obs);
}

/* target link point of a pose: frame of the last joint o fixed transform to the target link o target_link_offset
 * (LinkPointBase.get_position, ctlp.py:4962-5075) */
void smo_target_link_point(const SmScene* sc, const double* q, double* p) {
    Xf fr[1 + SM_MAX_JOINTS];
    smo_fk(sc, q, fr);
    double loc[3], w[3];
    mat_vec(sc->target_R, sc->target_offset, loc);
    for (int i = 0; i < 3; ++i) loc[i] += sc->target_t[i];
    mat_vec(fr[sc->n_joints].R, loc, w);
    for (int i = 0; i < 3; ++i) p[i] = w[i] + fr[sc->n_joints].t[i];
}

/* ------------------------------------------------------------------------------------------------------------
 * 7b. Human  (Human, ctlp.py:4647-4959): a nested SafeMotionsEnv(robot_scene = 9) moves the two arms of a human
 *     (description/urdf/human.urdf:140-416); configuration in trained_networks/human_network/params.json.
 *     Per step of the main env the nested env runs (ctlp.py:962-976, :4818-4882; safe_motions_base.py:1043-1227):
 *       step:     action of the human's policy -> end acceleration (actions.py:268-280) -> braking-trajectory
 *                 collision check (ctlp.py:3026-3207; utils/braking_trajectory_generator.py) -> setpoints
 *       24 x      prepare_sim_step (motor control), update (target point reached?), contact human <-> robot
 *       outcome:  new knot, target-point bookkeeping, observation (38 entries)
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct SmoHumanIO {
    double* hkin;              /* [SM_KIN_STRIDE] q v a q_act of the human */
    double* hstate;            /* [SM_HSTATE_STRIDE] */
    double* hbrake;            /* [SM_HBRAKE_STEPS][SM_HUMAN_JOINTS] */
    const double* uh;          /* [8] action of the human's policy for this step */
    const double* next_target; /* [3] target point for the arm that becomes active when a point is reached (the
                                  reference samples it by rejection, ctlp.py:1658-1720), or NULL */
    float* hobs;               /* [SM_HOBS_STRIDE] out: observation of the nested env */
    int32_t braked;            /* out: 1 if the stored braking trajectory was executed */
    int32_t brake_poses;       /* out: poses the braking-trajectory check visited */
    int32_t brake_collision;   /* out: 1-based index of the first pose in collision, 0 = none, -1 = timeout */
    double brake_margin;       /* out: smallest |d_min - brake_safety| over the poses the check visited (see
                                  smo_human_check_braking) */
    double a1[SM_HUMAN_JOINTS];/* out: end acceleration of the step */
} SmoHumanIO;

int smo_sizeof_human_io(void) { return (int)sizeof(SmoHumanIO); }

/* frames of the human: [0] = base, [1 + j] = child link of joint j (same convention as smo_fk) */
void smo_human_fk(const SmScene* sc, const double* hq, Xf* fr /* [SM_MAX_OBST_FRAMES] */) {
    const SmHuman* h = &sc->human;
    memcpy(fr[0].R, h->base_R, sizeof(h->base_R));
    memcpy(fr[0].t, h->base_t, sizeof(h->base_t));
    for (int j = 0; j < h->n_joints; ++j) {
        const Xf* P = &fr[h->joint_parent[j]];
        double Rj[9], R1[9], tp[3];
        mat_mul(P->R, h->joint_R[j], R1);
        mat_vec(P->R, h->joint_t[j], tp);
        axis_angle(h->joint_axis[j], hq[j], Rj);
        mat_mul(R1, Rj, fr[1 + j].R);
        for (int i = 0; i < 3; ++i) fr[1 + j].t[i] = P->t[i] + tp[i];
    }
}
void smo_human_fk_flat(const SmScene* sc, const double* hq, double* out) {
    Xf fr[SM_MAX_OBST_FRAMES];
    smo_human_fk(sc, hq, fr);
    for (int f = 0; f <= sc->human.n_joints; ++f) {
        memcpy(out + 12 * f, fr[f].R, 9 * sizeof(double));
        memcpy(out + 12 * f + 9, fr[f].t, 3 * sizeof(double));
    }
}

/* target link point of arm r ("hand" + target_link_offset, LinkPointBase.get_position ctlp.py:4962-5075) */
static void human_link_point(const SmScene* sc, const Xf* fr, int r, double* p) {
    const Xf* F = &fr[4 * (r + 1)];
    double w[3];
    mat_vec(F->R, sc->human.tp_local[r], w);
    for (int i = 0; i < 3; ++i) p[i] = w[i] + F->t[i];
}
void smo_human_link_points(const SmScene* sc, const double* hq, double* out /* [2][3] */) {
    Xf fr[SM_MAX_OBST_FRAMES];
    smo_human_fk(sc, hq, fr);
    human_link_point(sc, fr, 0, out);
    human_link_point(sc, fr, 1, out + 3);
}

void smo_human_safe_range(const SmScene* sc, const double* q, const double* v, const double* a, double* lo, double* hi,
                          int32_t* code) {
    const SmHuman* h = &sc->human;
    for (int j = 0; j < h->n_joints; ++j)
        safe_range_limits(sc->ts, h->jerk_max[j], h->acc_max[j], h->vel_max[j], h->pos_lo[j], h->pos_hi[j], 1, 1, q[j],
                          v[j], a[j], &lo[j], &hi[j], &code[j]);
}

/* get_minimum_distance as the braking-trajectory check uses it (ctlp.py:3282-3374): is some observed pair closer than
 * the safety distance?  (table x forearm / hand, self-collision link pairs with forearm or hand) */
int smo_human_pose_collides(const SmScene* sc, const double* hq) {
    const SmHuman* h = &sc->human;
    Xf world[1 + SM_MAX_JOINTS], fr[SM_MAX_OBST_FRAMES];
    xf_identity(&world[0]);
    smo_human_fk(sc, hq, fr);
    for (int i = 0; i < h->n_brake_pairs; ++i) {
        double d = pair_distance(sc, h->brake_pairs[i][0], h->brake_pairs[i][1], world, fr, h->brake_safety + 1e-3);
        if (d < h->brake_safety) return 1;
    }
    return 0;
}

/* smallest distance over the pairs of the braking check at pose hq: exact below brake_safety + 1e-3, above that a lower
 * bound (the GJK search of a pair stops once it is proven that far).  d_min < brake_safety exactly where
 * smo_human_pose_collides reports a collision (same pair distances). */
static double human_brake_dmin(const SmScene* sc, const double* hq) {
    const SmHuman* h = &sc->human;
    Xf world[1 + SM_MAX_JOINTS], fr[SM_MAX_OBST_FRAMES];
    xf_identity(&world[0]);
    smo_human_fk(sc, hq, fr);
    double dmin = INFINITY;
    for (int i = 0; i < h->n_brake_pairs; ++i) {
        double d = pair_distance(sc, h->brake_pairs[i][0], h->brake_pairs[i][1], world, fr, h->brake_safety + 1e-3);
        if (d < dmin) dmin = d;
    }
    return dmin;
}

/* distance of every pair of the braking check (human.brake_pairs order) at pose hq, GJK without early stop (test hook:
 * the tests find the pair and link-group pair that decide a pose, and its clearance d - brake_safety) */
void smo_human_brake_pair_distances(const SmScene* sc, const double* hq, double* out /* [n_brake_pairs] */) {
    const SmHuman* h = &sc->human;
    Xf world[1 + SM_MAX_JOINTS], fr[SM_MAX_OBST_FRAMES];
    xf_identity(&world[0]);
    smo_human_fk(sc, hq, fr);
    for (int i = 0; i < h->n_brake_pairs; ++i)
        out[i] = pair_distance(sc, h->brake_pairs[i][0], h->brake_pairs[i][1], world, fr, 0.0);
}

/* BrakingTrajectoryGenerator.get_braking_acceleration for one joint (utils/braking_trajectory_generator.py:44-78): a
 * second limiter with velocity limits [0, 0] picks the next acceleration that brings the joint to rest.  Restated as:
 * the next-knot acceleration a1 from which the acceleration can be ramped back to zero at full jerk, in whole time
 * steps, so that velocity AND acceleration reach zero together:
 *     a1, a1 + r, ..., 0  (n ramp intervals, r = J ts)   =>   v_end = v + a ts / 2 + n ts a1 + ts r n (n - 1) / 2 = 0
 * with the smallest n whose a1 needs no more than n ramp intervals; clipped to the jerk / acceleration interval like
 * every bound of the limiter. */
static double brake_target(double v, double a, double J, double A, double ts) {
    double s0 = v + a * ts * 0.5;
    double sg = s0 < 0.0 ? -1.0 : 1.0;
    double S = sg * s0, r = J * ts;
    double a1 = 0.0;
    for (int n = 1; n <= 8; ++n) {
        double dn = (double)n;
        a1 = (S + ts * r * dn * (dn - 1.0) * 0.5) / (dn * ts);
        if (a1 <= dn * r) break;
    }
    a1 = -sg * a1;
    double lo = a - J * ts, hi = a + J * ts;
    if (lo < -A) lo = -A;
    if (hi > A) hi = A;
    if (lo > hi) { if (a > 0.0) lo = hi; else hi = lo; }
    if (a1 < lo) a1 = lo;
    if (a1 > hi) a1 = hi;
    return a1;
}

/* _compute_braking_acceleration (ctlp.py:3495-3507) + get_clipped_braking_acceleration: returns robot_stopped */
static int human_braking_acceleration(const SmScene* sc, const double* q, const double* v, const double* a,
                                      double* a_end) {
    const SmHuman* h = &sc->human;
    int all_small = 1;
    for (int j = 0; j < h->n_joints; ++j)
        if (!(fabs(v[j]) < 0.01 && fabs(a[j]) < 0.01)) all_small = 0;
    if (all_small) {
        for (int j = 0; j < h->n_joints; ++j) a_end[j] = 0.0;
        return 1;
    }
    for (int j = 0; j < h->n_joints; ++j) {
        /* np.clip(end_acceleration, next_acc_min, next_acc_max) with the full safe range (_acc_range_function,
         * ctlp.py:3496-3499), evaluated lazily: clip to the jerk / acceleration / velocity part of the range first; if the
         * braking profile that follows the clipped value keeps both position limits, the position bounds cannot cut it
         * (they are the largest / smallest accelerations with that property) and the iterative solve is not needed */
        double J = h->jerk_max[j], A = h->acc_max[j], ts = sc->ts;
        double lo, hi;
        int32_t code;
        safe_range_limits(ts, J, A, h->vel_max[j], h->pos_lo[j], h->pos_hi[j], 1, 0, q[j], v[j], a[j], &lo, &hi, &code);
        double e = brake_target(v[j], a[j], J, A, ts);
        if (fabs(v[j]) < 0.01 && fabs(a[j]) < 0.01) e = 0.0;
        double ec = e;
        if (ec < lo) ec = lo;
        if (ec > hi) ec = hi;
        int ok_hi = pos_peak(q[j], v[j], a[j], ec, J, A, ts) - h->pos_hi[j] <= 0.0;
        int ok_lo = pos_peak(-q[j], -v[j], -a[j], -ec, J, A, ts) - (-h->pos_lo[j]) <= 0.0;
        if (!(ok_hi && ok_lo)) {
            safe_range_limits(ts, J, A, h->vel_max[j], h->pos_lo[j], h->pos_hi[j], 1, 1, q[j], v[j], a[j], &lo, &hi, &code);
            ec = e;
            if (ec < lo) ec = lo;
            if (ec > hi) ec = hi;
        }
        a_end[j] = ec;
    }
    return 0;
}

/* check_braking_trajectory_method / _check_if_braking_trajectory_is_collision_free (ctlp.py:3026-3053, :3155-3207):
 * execute the next step with a_target, then brake; every step is checked at brake_checks poses.  Returns 1 if the
 * braking trajectory has to be executed instead (collision or timeout).  brake_acc receives the braking accelerations
 * b_1 .. b_k that follow a_target (the part adapt_action keeps, ctlp.py:3096-3119), *k_out their number.
 * *margin_out (if not NULL) receives the smallest |d_min - brake_safety| over the poses visited, d_min the smallest pair
 * distance of a pose (human_brake_dmin: exact up to 1e-3 m, a lower bound beyond): how far the decision is from flipping
 * under a small error of the distances. */
int smo_human_check_braking(const SmScene* sc, const double* q0, const double* v0, const double* a0,
                            const double* a_target, double* brake_acc /* [SM_HBRAKE_STEPS][8] */, int* k_out,
                            int* poses_out, int* collision_out, double* margin_out) {
    const SmHuman* h = &sc->human;
    const int nj = h->n_joints, C = h->brake_checks;
    double ts = sc->ts;
    double q[SM_HUMAN_JOINTS], v[SM_HUMAN_JOINTS], as[SM_HUMAN_JOINTS], ae[SM_HUMAN_JOINTS];
    memcpy(q, q0, sizeof(q)); memcpy(v, v0, sizeof(v)); memcpy(as, a0, sizeof(as)); memcpy(ae, a_target, sizeof(ae));
    int k = 0, poses = 0;
    double margin = INFINITY;
    *collision_out = 0;
    if (margin_out) *margin_out = margin;
    for (;;) {
        /* np.linspace(ts / C, ts, C) */
        double pend[SM_HUMAN_JOINTS];
        for (int m = 1; m <= C; ++m) {
            double t;
            if (C <= 1 || m == C) t = ts;
            else { double start = ts / C, step = (ts - start) / (double)(C - 1); t = start + (double)(m - 1) * step; }
            double pm[SM_HUMAN_JOINTS];
            for (int j = 0; j < nj; ++j) { double vv, aa; interpolate(sc, q[j], v[j], as[j], ae[j], t, &pm[j], &vv, &aa); }
            ++poses;
            const double dmin = human_brake_dmin(sc, pm);
            if (fabs(dmin - h->brake_safety) < margin) margin = fabs(dmin - h->brake_safety);
            if (margin_out) *margin_out = margin;
            if (dmin < h->brake_safety) { *collision_out = poses; *k_out = k; *poses_out = poses; return 1; }
            if (m == C) memcpy(pend, pm, sizeof(pm));
        }
        /* _compute_next_braking_trajectory_time_step (ctlp.py:3467-3493) */
        if ((double)k * ts > h->brake_timeout) { *collision_out = -1; *k_out = k; *poses_out = poses; return 1; }
        double vend[SM_HUMAN_JOINTS], anext[SM_HUMAN_JOINTS];
        for (int j = 0; j < nj; ++j) { double qq, aa; interpolate(sc, q[j], v[j], as[j], ae[j], ts, &qq, &vend[j], &aa); }
        int stopped = human_braking_acceleration(sc, pend, vend, ae, anext);
        if (stopped) break;
        if (k < SM_HBRAKE_STEPS) memcpy(brake_acc + (size_t)k * SM_HUMAN_JOINTS, anext, sizeof(anext));
        ++k;
        memcpy(q, pend, sizeof(q)); memcpy(v, vend, sizeof(v)); memcpy(as, ae, sizeof(as)); memcpy(ae, anext, sizeof(ae));
    }
    *k_out = k; *poses_out = poses;
    return 0;
}

/* the nested env's step up to the setpoints: range, action mapping, braking-trajectory method (actions.py:282-376) */
static void human_pre_step(const SmScene* sc, SmoHumanIO* H) {
    const SmHuman* h = &sc->human;
    double *q = H->hkin, *v = H->hkin + 8, *a = H->hkin + 16;
    double lo[SM_HUMAN_JOINTS], hi[SM_HUMAN_JOINTS];
    int32_t code[SM_HUMAN_JOINTS];
    smo_human_safe_range(sc, q, v, a, lo, hi, code);
    for (int j = 0; j < h->n_joints; ++j) H->a1[j] = lo[j] + 0.5 * (H->uh[j] + 1.0) * (hi[j] - lo[j]);
    H->braked = 0; H->brake_poses = 0; H->brake_collision = 0; H->brake_margin = INFINITY;
    H->hstate[SM_HS_STEPS] += 1.0;
    if (!h->check_braking) return;
    double bacc[SM_HBRAKE_STEPS * SM_HUMAN_JOINTS];
    int k = 0, poses = 0, coll = 0;
    int execute = smo_human_check_braking(sc, q, v, a, H->a1, bacc, &k, &poses, &coll, &H->brake_margin);
    H->brake_poses = poses; H->brake_collision = coll;
    int count = (int)H->hstate[SM_HS_BRAKE_COUNT];
    if (execute) { /* get_braking_acceleration (ctlp.py:3000-3024): next acceleration of the stored trajectory */
        H->braked = 1;
        if (count > 0) {
            memcpy(H->a1, H->hbrake, SM_HUMAN_JOINTS * sizeof(double));
            memmove(H->hbrake, H->hbrake + SM_HUMAN_JOINTS, (size_t)(count - 1) * SM_HUMAN_JOINTS * sizeof(double));
            H->hstate[SM_HS_BRAKE_COUNT] = (double)(count - 1);
        } else {
            for (int j = 0; j < h->n_joints; ++j) H->a1[j] = 0.0;
        }
    } else { /* adapt_action: the checked trajectory becomes the valid one (ctlp.py:3096-3119) */
        if (k > SM_HBRAKE_STEPS) k = SM_HBRAKE_STEPS;
        memcpy(H->hbrake, bacc, (size_t)k * SM_HUMAN_JOINTS * sizeof(double));
        H->hstate[SM_HS_BRAKE_COUNT] = (double)k;
    }
    H->hstate[SM_HS_BRAKED] = (double)H->braked;
}

/* one 1/240 s sub-step of the human: setpoint, motor tracking (Human.prepare_sim_step ctlp.py:4850-4860), then the
 * nested wrapper's update: is the active target point reached? (ctlp.py:2787-2821) */
static void human_substep(const SmScene* sc, SmoHumanIO* H, double t, double dt) {
    const SmHuman* h = &sc->human;
    double *q = H->hkin, *v = H->hkin + 8, *a = H->hkin + 16, *qa = H->hkin + 24;
    double qset[SM_HUMAN_JOINTS];
    for (int j = 0; j < h->n_joints; ++j) {
        double qs, vs, as;
        interpolate(sc, q[j], v[j], a[j], H->a1[j], t, &qs, &vs, &as);
        qset[j] = qs;
        qa[j] = qa[j] + sc->track_kp * (qs - qa[j]) + (0.87 * dt) * vs; /* use_controller_target_velocities = true */
    }
    Xf fr[SM_MAX_OBST_FRAMES];
    smo_human_fk(sc, qset, fr);
    for (int r = 0; r < 2; ++r) human_link_point(sc, fr, r, H->hstate + 12 * r + SM_TP_LINK_POS);
    for (int r = 0; r < 2; ++r) {
        double* tp = H->hstate + 12 * r;
        if (tp[SM_TP_ACTIVE] == 0.0) continue;
        double dx = tp[SM_TP_LINK_POS] - tp[SM_TP_POS], dy = tp[SM_TP_LINK_POS + 1] - tp[SM_TP_POS + 1],
               dz = tp[SM_TP_LINK_POS + 2] - tp[SM_TP_POS + 2];
        if (sqrt(dx * dx + dy * dy + dz * dz) < h->tp_radius) {
            tp[SM_HTP_REACHED] = 1.0;
            tp[SM_TP_ACTIVE] = 0.0;
            tp[SM_TP_REACHED_N] += 1.0;
            H->hstate[12 * ((r + 1) % 2) + SM_HTP_SAMPLE_NEW] = 1.0; /* alternating target points (ctlp.py:2815-2817) */
        }
    }
}

/* observation of the nested env (observations.py:313-351 with two arms and alternating target points) */
void smo_human_observation(const SmScene* sc, const double* hkin, const double* hstate, float* hobs) {
    const SmHuman* h = &sc->human;
    int k = 0;
    for (int j = 0; j < 8; ++j) hobs[k++] = clip1(-1.0 + 2.0 * (hkin[j] - h->pos_lo[j]) / (h->pos_hi[j] - h->pos_lo[j]));
    for (int j = 0; j < 8; ++j) hobs[k++] = clip1(hkin[8 + j] / h->vel_max[j]);
    for (int j = 0; j < 8; ++j) hobs[k++] = clip1(hkin[16 + j] / h->acc_max[j]);
    for (int r = 0; r < 2; ++r) {
        const double* tp = hstate + 12 * r;
        for (int i = 0; i < 3; ++i)
            hobs[k++] = tp[SM_TP_ACTIVE] != 0.0
                            ? clip1(-1.0 + 2.0 * (tp[SM_TP_POS + i] - h->tp_box_min[i]) / (h->tp_box_max[i] - h->tp_box_min[i]))
                            : 0.0f;
    }
    for (int r = 0; r < 2; ++r) {
        const double* tp = hstate + 12 * r;
        for (int i = 0; i < 3; ++i) {
            double rel = tp[SM_TP_POS + i] - tp[SM_TP_LINK_POS + i];
            hobs[k++] = tp[SM_TP_ACTIVE] != 0.0
                            ? clip1(-1.0 + 2.0 * (rel - h->tp_rel_min[i]) / (h->tp_rel_max[i] - h->tp_rel_min[i])) : 0.0f;
        }
    }
    for (int r = 0; r < 2; ++r) hobs[k++] = hstate[12 * r + SM_TP_ACTIVE] != 0.0 ? 1.0f : 0.0f;
    while (k < SM_HOBS_STRIDE) hobs[k++] = 0.0f;
}

/* process_step_outcome of the nested env: new knot, target points (get_target_point_observation ctlp.py:2210-2271) */
static void human_post_step(const SmScene* sc, SmoHumanIO* H) {
    const SmHuman* h = &sc->human;
    double *q = H->hkin, *v = H->hkin + 8, *a = H->hkin + 16;
    for (int j = 0; j < h->n_joints; ++j) {
        double qs, vs, as;
        interpolate(sc, q[j], v[j], a[j], H->a1[j], substep_time(sc, sc->substeps), &qs, &vs, &as);
        q[j] = qs; v[j] = vs; a[j] = H->a1[j];
    }
    for (int r = 0; r < 2; ++r) {
        double* tp = H->hstate + 12 * r;
        tp[SM_HTP_REACHED] = 0.0;
        if (tp[SM_HTP_SAMPLE_NEW] != 0.0 && H->next_target) {
            memcpy(tp + SM_TP_POS, H->next_target, 3 * sizeof(double));
            tp[SM_HTP_SAMPLE_NEW] = 0.0;
            tp[SM_TP_ACTIVE] = 1.0;
            tp[SM_TP_INIT_DIST] = NAN;
            H->hstate[SM_HS_DRAWS] += 1.0;
        }
    }
    for (int r = 0; r < 2; ++r) {
        double* tp = H->hstate + 12 * r;
        if (tp[SM_TP_ACTIVE] == 0.0) continue;
        double dx = tp[SM_TP_POS] - tp[SM_TP_LINK_POS], dy = tp[SM_TP_POS + 1] - tp[SM_TP_LINK_POS + 1],
               dz = tp[SM_TP_POS + 2] - tp[SM_TP_LINK_POS + 2];
        tp[SM_TP_LAST_DIST] = sqrt(dx * dx + dy * dy + dz * dz);
        if (isnan(tp[SM_TP_INIT_DIST])) tp[SM_TP_INIT_DIST] = tp[SM_TP_LAST_DIST];
    }
    if (H->hobs) smo_human_observation(sc, H->hkin, H->hstate, H->hobs);
}

/* start of an episode of the nested env (ObstacleWrapperBase.reset, ctlp.py:1020-1048): one arm gets the first target
 * point, nothing is stored from earlier braking checks */
void smo_human_init(const SmScene* sc, double* hkin, double* hstate, const double* hq, const double* hv,
                    const double* ha, const double* first_target, int active_arm, float* hobs) {
    memset(hkin, 0, SM_KIN_STRIDE * sizeof(double));
    memset(hstate, 0, SM_HSTATE_STRIDE * sizeof(double));
    double dt = sc->ts / (double)sc->substeps;
    for (int j = 0; j < sc->human.n_joints; ++j) {
        hkin[j] = hq[j]; hkin[8 + j] = hv[j]; hkin[16 + j] = ha[j];
        hkin[24 + j] = hq[j] + (0.87 * dt) * hv[j]; /* as the robot: one stepSimulation with the start state as target */
    }
    double lp[6];
    smo_human_link_points(sc, hq, lp);
    for (int r = 0; r < 2; ++r) memcpy(hstate + 12 * r + SM_TP_LINK_POS, lp + 3 * r, 3 * sizeof(double));
    double* tp = hstate + 12 * active_arm;
    memcpy(tp + SM_TP_POS, first_target, 3 * sizeof(double));
    tp[SM_TP_ACTIVE] = 1.0;
    double dx = tp[SM_TP_POS] - tp[SM_TP_LINK_POS], dy = tp[SM_TP_POS + 1] - tp[SM_TP_LINK_POS + 1],
           dz = tp[SM_TP_POS + 2] - tp[SM_TP_LINK_POS + 2];
    tp[SM_TP_LAST_DIST] = tp[SM_TP_INIT_DIST] = sqrt(dx * dx + dy * dy + dz * dz);
    hstate[SM_HS_DRAWS] = 1.0;
    if (hobs) smo_human_observation(sc, hkin, hstate, hobs);
}

/* ObstacleWrapperBase.reset with compute_initial_braking_trajectory (ctlp.py:1120-1139): the stored braking trajectory
 * starts as the accelerations that brake from the start state.  As in the reference the position handed to the range
 * computation is not advanced along this trajectory (start_position = position[-1] is the previous step's start). */
void smo_human_initial_braking(const SmScene* sc, const double* hkin, double* hstate, double* hbrake) {
    const SmHuman* h = &sc->human;
    if (!h->check_braking || !h->initial_braking_trajectory) return;
    double q[SM_HUMAN_JOINTS], v[SM_HUMAN_JOINTS], a[SM_HUMAN_JOINTS], e[SM_HUMAN_JOINTS];
    memcpy(q, hkin, sizeof(q)); memcpy(v, hkin + 8, sizeof(v)); memcpy(a, hkin + 16, sizeof(a));
    int k = 0;
    for (;;) {
        if ((double)(k - 1) * sc->ts > h->brake_timeout || k >= SM_HBRAKE_STEPS) break;
        if (human_braking_acceleration(sc, q, v, a, e)) break;
        memcpy(hbrake + (size_t)k * SM_HUMAN_JOINTS, e, sizeof(e));
        ++k;
        for (int j = 0; j < h->n_joints; ++j) {
            double qq, vv, aa;
            interpolate(sc, q[j], v[j], a[j], e[j], sc->ts, &qq, &vv, &aa);
            v[j] = vv; a[j] = e[j];
        }
    }
    hstate[SM_HS_BRAKE_COUNT] = (double)k;
}

/* getContactPoints(bodyA = human, bodyB = robot) in the simulation client (ctlp.py:4888-4898): both at their
 * motor-tracked poses; every human link (also the body) against every robot link */
static int human_contact_exists(const SmScene* sc, const Xf* robot, const Xf* hfr) {
    const SmHuman* h = &sc->human;
    for (int r = 0; r < sc->n_mov_contact; ++r)
        for (int s = 0; s < h->n_shapes; ++s) {
            double th = h->contact_thresh[h->shape_link[s]][r];
            double d = pair_distance(sc, sc->mov_contact[r], h->shape_off + s, robot, hfr, th + 1e-3);
            if (d <= th) return 1;
        }
    return 0;
}

/* ------------------------------------------------------------------------------------------------------------
 * 8. One env step  (safe_motions_base.py:1043-1227)
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct SmoStepOut {
    float reward;
    int32_t done;
    int32_t term_reason;
    float info[SM_INFO_STRIDE];
    double range_lo[SM_MAX_JOINTS], range_hi[SM_MAX_JOINTS];
    double a1[SM_MAX_JOINTS];
    double d_static, d_self, d_moving; /* raw distances before the 1 mm clamp */
} SmoStepOut;

/* kin: [q8 v8 a8 qact8], ob: obstacle record, episode_length in/out.  u: n_joints actions as doubles. */
/* tp: target-point record (SM_TP_STRIDE doubles) or NULL; next_target: the target point that replaces a reached one
 * (drawn by the caller, like next_ball, because the reference samples it with data-dependent rejection sampling). */
static void step_core(const SmScene* sc, double* kin, double* ob, double* tp, SmoHumanIO* H, int32_t* episode_length,
                      double* ep_return, const double* u, const double* next_ball, const double* next_target, float* obs,
                      SmoStepOut* out) {
    int nj = sc->n_joints, S = sc->substeps;
    double *q = kin, *v = kin + 8, *a = kin + 16, *qa = kin + 24;
    int32_t code[SM_MAX_JOINTS];
    memset(out, 0, sizeof(*out));
    *episode_length += 1;                                        /* safe_motions_base.py:1044 */
    smo_safe_range(sc, q, v, a, out->range_lo, out->range_hi, code);
    smo_map_action(sc, u, out->range_lo, out->range_hi, out->a1); /* actions.py:291 */
    int rcode = 0;
    for (int j = 0; j < nj; ++j) rcode |= code[j];
    if (H) human_pre_step(sc, H); /* obstacle_wrapper.step() -> Human.step (ctlp.py:962-966, :4818-4840) */

    /* --- 24 sub-steps (safe_motions_base.py:1233-1277).  Inside sub-step k Bullet first detects collisions on the
     * poses left by sub-step k-1 (tracked robot pose, obstacle pose of the previous update), then integrates the
     * motor-controlled joints; afterwards obstacle_wrapper.update advances the obstacles and reads the manifolds. */
    double dt = sc->ts / (double)S;
    Xf robot[1 + SM_MAX_JOINTS], obst[SM_MAX_OBST_FRAMES];
    for (int k = 1; k <= S; ++k) {
        double t = substep_time(sc, k);
        int test_contacts = (sc->contact_stride > 0) && (k % sc->contact_stride == 0);
        int contact[SM_MAX_OBSTACLES] = {0, 0};
        if (test_contacts && ob[SM_OB_LATCH] == 0.0) {
            smo_fk(sc, qa, robot);
            obstacle_poses_h(sc, ob, H ? H->hkin + 24 : (const double*)0, obst); /* the human at its tracked pose */
            for (int o = 0; o < sc->n_obstacles; ++o) {
                if (sc->obst_kind[o] == SM_OBST_BALL && ob[SM_OB_BALL_ACTIVE] == 0.0) continue;
                if (sc->obst_kind[o] == SM_OBST_HUMAN) { contact[o] = H ? human_contact_exists(sc, robot, obst) : 0; continue; }
                contact[o] = contact_exists(sc, o, robot, obst);
            }
        }
        /* motor tracking: q+ = q + kp (q_set - q) + track_vel dt v_set  (SURVEY Appendix B.4) */
        double qset[SM_MAX_JOINTS];
        for (int j = 0; j < nj; ++j) {
            double qs, vs, as;
            interpolate(sc, q[j], v[j], a[j], out->a1[j], t, &qs, &vs, &as);
            qset[j] = qs;
            qa[j] = qa[j] + sc->track_kp * (qs - qa[j]) + (sc->track_vel * dt) * vs;
        }
        /* target point reached? (ctlp.py:2787-2821; target link point of the setpoint pose,
         * target_point_use_actual_position = False) */
        if (sc->use_target_points && tp) {
            smo_target_link_point(sc, qset, tp + SM_TP_LINK_POS);
            if (tp[SM_TP_ACTIVE] != 0.0) {
                double dx = tp[SM_TP_LINK_POS] - tp[SM_TP_POS], dy = tp[SM_TP_LINK_POS + 1] - tp[SM_TP_POS + 1],
                       dz = tp[SM_TP_LINK_POS + 2] - tp[SM_TP_POS + 2];
                if (sqrt(dx * dx + dy * dy + dz * dz) < sc->tp_radius) {
                    tp[SM_TP_REACHED] = 1.0;
                    tp[SM_TP_ACTIVE] = 0.0;
                    tp[SM_TP_REACHED_N] += 1.0;
                }
            }
        }
        /* obstacle_wrapper.update (ctlp.py:2590-2862) */
        for (int o = 0; o < sc->n_obstacles; ++o) {
            if (sc->obst_kind[o] == SM_OBST_HUMAN && H) { /* ctlp.py:2613-2615: Human.update, then the contact latch */
                human_substep(sc, H, t, dt);
                if (contact[o]) ob[SM_OB_LATCH] = 1.0;
            } else if (sc->obst_kind[o] == SM_OBST_PLANET) {
                if (o == 0) ob[SM_OB_INDEX] = (double)(((int)ob[SM_OB_INDEX] + 1) % sc->planet_steps);
                if (contact[o] && sc->terminate_moving) ob[SM_OB_LATCH] = 1.0; /* ctlp.py:2631-2637 */
            } else if (sc->obst_kind[o] == SM_OBST_BALL && ob[SM_OB_BALL_ACTIVE] != 0.0) {
                ob[SM_OB_INDEX] += 1.0;                       /* ctlp.py:4104-4105 */
                ob[SM_OB_BALL_T] = ob[SM_OB_BALL_T] + dt;
                double p[3];
                ball_position(ob, ob[SM_OB_BALL_T], p);
                if (ob[SM_OB_INDEX] > ob[SM_OB_BALL_NMAX] || ob[SM_OB_INDEX] >= ob[SM_OB_BALL_NHIT]) {
                    ob[SM_OB_BALL_ACTIVE] = 0.0;              /* missed robot / hit obstacle (ctlp.py:2840-2848) */
                } else if (sqrt(p[0] * p[0] + p[1] * p[1]) < sc->ball_active_xy) {
                    if (contact[o]) {                          /* ctlp.py:2853-2861 */
                        ob[SM_OB_BALL_ACTIVE] = 0.0;
                        ob[SM_OB_LATCH] = 1.0;
                    }
                }
            }
        }
    }
    /* --- process_step_outcome: new knot (safe_motions_base.py:1179-1185) */
    double jerk_rel = 0.0;
    for (int j = 0; j < nj; ++j) {
        double qs, vs, as;
        interpolate(sc, q[j], v[j], a[j], out->a1[j], substep_time(sc, S), &qs, &vs, &as);
        double jr = fabs((out->a1[j] - a[j]) / sc->ts) / sc->jerk_max[j]; /* rewards.py:181-186 */
        if (jr > jerk_rel) jerk_rel = jr;
        q[j] = qs; v[j] = vs; a[j] = out->a1[j];
    }
    if (H) human_post_step(sc, H); /* obstacle_wrapper.process_step_outcome -> Human.process_step_outcome */
    /* --- reward (rewards.py:95-169, :432-502) */
    smo_distances_h(sc, q, ob, H ? H->hkin : (const double*)0, &out->d_static, &out->d_self, &out->d_moving);
    double ds = out->d_static, dself = out->d_self, dm = out->d_moving;
    int c_static = 0, c_self = 0, c_moving = 0;
    if (ds < sc->collision_dist) { ds = 0.0; c_static = 1; }
    if (dself < sc->collision_dist) { dself = 0.0; c_self = 1; }
    if (dm < sc->collision_dist) { dm = 0.0; c_moving = 1; }
    double r_self = 0.0, r_static = 0.0, r_moving = 0.0;
    if (sc->w_self != 0.0) { double r = dself / sc->d_self; if (r > 1.0) r = 1.0; r_self = r * r; }
    if (sc->w_static != 0.0) { double r = ds / sc->d_static; if (r > 1.0) r = 1.0; r_static = r * r; }
    { double r = dm / sc->d_moving; if (r > 1.0) r = 1.0; r_moving = r * r; }
    double action_punishment = 1.0; /* rewards.py:436 */
    if (sc->punish_action) {
        double m = 0.0;
        for (int j = 0; j < nj; ++j) if (fabs(u[j]) > m) m = fabs(u[j]);
        double pu = (m - sc->action_thresh) / (1.0 - sc->action_thresh); /* rewards.py:18-21 */
        if (pu > 1.0) pu = 1.0;
        if (pu < 0.0) pu = 0.0;
        action_punishment = pu * pu;
    }
    double low_acc = 0.0, low_vel = 0.0;
    if (sc->w_low_acc != 0.0) { /* rewards.py:448-453 */
        double m = 0.0;
        for (int j = 0; j < nj; ++j) { double r = fabs(-1.0 + 2.0 * (a[j] + sc->acc_max[j]) / (2.0 * sc->acc_max[j])); if (r > m) m = r; }
        double rd = m / sc->thr_low_acc; if (rd > 1.0) rd = 1.0;
        low_acc = (rd - 1.0) * (rd - 1.0);
    }
    if (sc->w_low_vel != 0.0) {
        double m = 0.0;
        for (int j = 0; j < nj; ++j) { double r = fabs(-1.0 + 2.0 * (v[j] + sc->vel_max[j]) / (2.0 * sc->vel_max[j])); if (r > m) m = r; }
        double rd = m / sc->thr_low_vel; if (rd > 1.0) rd = 1.0;
        low_vel = (rd - 1.0) * (rd - 1.0);
    }
    int term_coll = (sc->terminate_self && c_self) || (sc->terminate_static && c_static) ||
                    (sc->terminate_moving && c_moving);
    int finished = *episode_length >= sc->episode_steps; /* trajectory_manager.py:187-192 */
    double bonus = (finished && !term_coll) ? sc->termination_bonus : 0.0;            /* rewards.py:465-472 */
    double punish = term_coll ? sc->early_termination_punishment : 0.0;               /* rewards.py:474-479 */
    double reward = (1.0 - action_punishment) * sc->action_max_punishment + r_self * sc->w_self +
                    r_static * sc->w_static + r_moving * sc->w_moving + low_acc * sc->w_low_acc +
                    low_vel * sc->w_low_vel + bonus + punish;                         /* rewards.py:481-488 */
    double tp_reward = 0.0;
    if (sc->use_target_points && tp) { /* TargetPointReachingReward (rewards.py:303-396; ctlp.py:2309-2350) */
        double norm = 1.0;
        if ((tp[SM_TP_ACTIVE] != 0.0 || tp[SM_TP_REACHED] != 0.0) && sc->tp_normalize) {
            norm = tp[SM_TP_INIT_DIST];
            if (norm == 0.0) norm += 0.0000001;
        }
        if (tp[SM_TP_ACTIVE] != 0.0) {
            double dx = tp[SM_TP_POS] - tp[SM_TP_LINK_POS], dy = tp[SM_TP_POS + 1] - tp[SM_TP_LINK_POS + 1],
                   dz = tp[SM_TP_POS + 2] - tp[SM_TP_LINK_POS + 2];
            tp_reward = (tp[SM_TP_LAST_DIST] - sqrt(dx * dx + dy * dy + dz * dz)) / (sc->ts * norm);
        } else if (tp[SM_TP_REACHED] != 0.0) {
            tp_reward = tp[SM_TP_LAST_DIST] / (sc->ts * norm) + sc->tp_bonus;
        }
        double pun = sc->punish_action ? action_punishment : 0.0; /* rewards.py:307, :317-318 */
        reward = tp_reward * sc->tp_reward_factor - pun * sc->action_max_punishment + r_self * sc->w_self +
                 r_static * sc->w_static + r_moving * sc->w_moving;               /* rewards.py:354-361 */
    }
    /* --- termination priority self -> static -> moving -> length (safe_motions_base.py:1775-1799) */
    int done = 0, reason = SM_TERM_UNSET;
    if (sc->terminate_self && c_self) { done = 1; reason = SM_TERM_SELF_COLLISION; }
    else if (sc->terminate_static && c_static) { done = 1; reason = SM_TERM_STATIC_COLLISION; }
    else if (sc->terminate_moving && c_moving) { done = 1; reason = SM_TERM_MOVING_COLLISION; }
    else if (finished) { done = 1; reason = SM_TERM_TRAJECTORY_LENGTH; }
    double reward_raw = reward;
    if (sc->reward_scale != 0.0) reward *= sc->reward_scale;                          /* rewards.py:172-176 */
    *ep_return += reward;
    out->reward = (float)reward;
    out->info[SM_INFO_REWARD_RAW] = (float)reward_raw;
    out->info[SM_INFO_FIRST_RISKY_STEP] = -1.0f; /* the gate is not part of the oracle step: tests apply it in NumPy */
    out->done = done;
    out->term_reason = reason;
    out->info[SM_INFO_D_STATIC] = (float)ds;
    out->info[SM_INFO_D_SELF] = (float)dself;
    out->info[SM_INFO_D_MOVING] = (float)dm;
    out->info[SM_INFO_COLL_STATIC] = (float)c_static;
    out->info[SM_INFO_COLL_SELF] = (float)c_self;
    out->info[SM_INFO_COLL_MOVING] = (float)c_moving;
    out->info[SM_INFO_ACTION_PUNISH] = (float)action_punishment;
    out->info[SM_INFO_R_STATIC] = (float)r_static;
    out->info[SM_INFO_R_SELF] = (float)r_self;
    out->info[SM_INFO_R_MOVING] = (float)r_moving;
    out->info[SM_INFO_EPISODE_LENGTH] = (float)*episode_length;
    out->info[SM_INFO_EPISODE_RETURN] = (float)*ep_return;
    out->info[SM_INFO_RANGE_CODE] = (float)rcode;
    out->info[SM_INFO_CONTACT_LATCH] = (float)(ob[SM_OB_LATCH] != 0.0);
    out->info[SM_INFO_MAX_JERK_REL] = (float)jerk_rel;
    out->info[SM_INFO_TP_REWARD] = (float)tp_reward;
    /* a ball that reached a final state is replaced when the next observation is taken (ctlp.py:2354-2360,
     * :2893-2895); the new launch (release point, speed vector, orientation, hit times) is an input here because
     * the reference draws it with data-dependent rejection sampling (ctlp.py:1723-1931). */
    if (next_ball && sc->n_obstacles > 0 && sc->obst_kind[0] == SM_OBST_BALL && ob[SM_OB_BALL_ACTIVE] == 0.0) {
        memcpy(ob + SM_OB_BALL_P0, next_ball, 10 * sizeof(double)); /* p0, v0, euler0, omega */
        ob[SM_OB_INDEX] = 0.0;
        ob[SM_OB_BALL_T] = 0.0;
        ob[SM_OB_BALL_ACTIVE] = 1.0;
        ob[SM_OB_LATCH] = 0.0;
        ob[SM_OB_BALL_NMAX] = next_ball[10];
        ob[SM_OB_BALL_NHIT] = next_ball[11];
    }
    /* get_target_point_observation (ctlp.py:2210-2271): a reached point is replaced, distances are recorded */
    if (sc->use_target_points && tp) {
        if (tp[SM_TP_REACHED] != 0.0 && next_target) {
            memcpy(tp + SM_TP_POS, next_target, 3 * sizeof(double));
            tp[SM_TP_ACTIVE] = 1.0;
            tp[SM_TP_INIT_DIST] = NAN;
            tp[SM_TP_DRAWS] += 1.0;
        }
        tp[SM_TP_REACHED] = 0.0;
        if (tp[SM_TP_ACTIVE] != 0.0) {
            double dx = tp[SM_TP_POS] - tp[SM_TP_LINK_POS], dy = tp[SM_TP_POS + 1] - tp[SM_TP_LINK_POS + 1],
                   dz = tp[SM_TP_POS + 2] - tp[SM_TP_LINK_POS + 2];
            tp[SM_TP_LAST_DIST] = sqrt(dx * dx + dy * dy + dz * dz);
            if (isnan(tp[SM_TP_INIT_DIST])) tp[SM_TP_INIT_DIST] = tp[SM_TP_LAST_DIST];
        }
    }
    if (obs) {
        smo_observation_tp(sc, kin, ob, tp, obs);
        if (H && H->hobs) /* Human.kinematic_observation: the first 3 x 8 entries of the nested env's observation */
            memcpy(obs + sc->obs_size - 3 * sc->human.n_joints, H->hobs, 3 * sc->human.n_joints * sizeof(float));
    }
}

void smo_step_tp(const SmScene* sc, double* kin, double* ob, double* tp, int32_t* episode_length, double* ep_return,
                 const double* u, const double* next_ball, const double* next_target, float* obs, SmoStepOut* out) {
    step_core(sc, kin, ob, tp, (SmoHumanIO*)0, episode_length, ep_return, u, next_ball, next_target, obs, out);
}

/* Human scene: one step of the main env including the nested env of the human */
void smo_step_human(const SmScene* sc, double* kin, double* ob, SmoHumanIO* H, int32_t* episode_length,
                    double* ep_return, const double* u, float* obs, SmoStepOut* out) {
    step_core(sc, kin, ob, (double*)0, H, episode_length, ep_return, u, (const double*)0, (const double*)0, obs, out);
}

/* batch driver of the Human scene.  hactions [n][8]; next_target [n][3] or NULL; hinfo [n][4] = braked, poses visited by
 * the braking-trajectory check, first colliding pose (0 none, -1 timeout), reserved; hmargin [n] or NULL: the check's
 * smallest |d_min - brake_safety| over the poses it visited (infinite if it did not run) */
void smo_step_batch_human(const SmScene* sc, int n, double* kin, double* ob, double* hkin, double* hstate, double* hbrake,
                          int32_t* episode, double* ep_return, const float* actions, const float* hactions,
                          const double* next_target, float* obs, float* hobs, float* reward, uint8_t* done,
                          int32_t* term, float* info, int32_t* hinfo, double* hmargin) {
    for (int e = 0; e < n; ++e) {
        double u[SM_MAX_JOINTS], uh[SM_HUMAN_JOINTS];
        SmoStepOut out;
        SmoHumanIO H;
        memset(&H, 0, sizeof(H));
        for (int j = 0; j < sc->n_joints; ++j) u[j] = (double)actions[e * sc->n_joints + j];
        for (int j = 0; j < SM_HUMAN_JOINTS; ++j) uh[j] = (double)hactions[e * SM_HUMAN_JOINTS + j];
        H.hkin = hkin + (size_t)e * SM_KIN_STRIDE;
        H.hstate = hstate + (size_t)e * SM_HSTATE_STRIDE;
        H.hbrake = hbrake + (size_t)e * SM_HBRAKE_STEPS * SM_HUMAN_JOINTS;
        H.uh = uh;
        H.next_target = next_target ? next_target + (size_t)e * 3 : 0;
        H.hobs = hobs + (size_t)e * SM_HOBS_STRIDE;
        smo_step_human(sc, kin + (size_t)e * SM_KIN_STRIDE, ob + (size_t)e * SM_OBST_STRIDE, &H, episode + 4 * e,
                       ep_return + e, u, obs ? obs + (size_t)e * sc->obs_size : 0, &out);
        reward[e] = out.reward;
        done[e] = (uint8_t)out.done;
        term[e] = out.term_reason;
        memcpy(info + (size_t)e * SM_INFO_STRIDE, out.info, sizeof(out.info));
        if (hmargin) hmargin[e] = H.brake_margin;
        if (hinfo) { hinfo[4 * e] = H.braked; hinfo[4 * e + 1] = H.brake_poses; hinfo[4 * e + 2] = H.brake_collision; hinfo[4 * e + 3] = 0; }
    }
}

void smo_step(const SmScene* sc, double* kin, double* ob, int32_t* episode_length, double* ep_return,
              const double* u, const double* next_ball, float* obs, SmoStepOut* out) {
    smo_step_tp(sc, kin, ob, 0, episode_length, ep_return, u, next_ball, 0, obs, out);
}

/* start of an episode with target points: the first target point and its distances (ctlp.py:2216-2245) */
void smo_target_init(const SmScene* sc, const double* kin, double* tp, const double* first_target) {
    memset(tp, 0, SM_TP_STRIDE * sizeof(double));
    smo_target_link_point(sc, kin, tp + SM_TP_LINK_POS);
    memcpy(tp + SM_TP_POS, first_target, 3 * sizeof(double));
    tp[SM_TP_ACTIVE] = 1.0;
    tp[SM_TP_DRAWS] = 1.0;
    double dx = tp[SM_TP_POS] - tp[SM_TP_LINK_POS], dy = tp[SM_TP_POS + 1] - tp[SM_TP_LINK_POS + 1],
           dz = tp[SM_TP_POS + 2] - tp[SM_TP_LINK_POS + 2];
    tp[SM_TP_LAST_DIST] = tp[SM_TP_INIT_DIST] = sqrt(dx * dx + dy * dy + dz * dz);
}

/* batch driver used by bench.py's CPU baseline and by the tests: steps n envs once. */
void smo_step_batch(const SmScene* sc, int n, double* kin, double* ob, int32_t* episode, double* ep_return,
                    const float* actions, const double* next_ball /* [n][12] or NULL */, float* obs, float* reward,
                    uint8_t* done, int32_t* term, float* info) {
    for (int e = 0; e < n; ++e) {
        double u[SM_MAX_JOINTS];
        SmoStepOut out;
        for (int j = 0; j < sc->n_joints; ++j) u[j] = (double)actions[e * sc->n_joints + j];
        smo_step(sc, kin + (size_t)e * SM_KIN_STRIDE, ob + (size_t)e * SM_OBST_STRIDE, episode + 4 * e,
                 ep_return + e, u, next_ball ? next_ball + (size_t)e * 12 : 0,
                 obs ? obs + (size_t)e * sc->obs_size : 0, &out);
        reward[e] = out.reward;
        done[e] = (uint8_t)out.done;
        term[e] = out.term_reason;
        memcpy(info + (size_t)e * SM_INFO_STRIDE, out.info, sizeof(out.info));
    }
}

void smo_step_batch_tp(const SmScene* sc, int n, double* kin, double* ob, double* tp, int32_t* episode,
                       double* ep_return, const float* actions, const double* next_ball, const double* next_target,
                       float* obs, float* reward, uint8_t* done, int32_t* term, float* info) {
    for (int e = 0; e < n; ++e) {
        double u[SM_MAX_JOINTS];
        SmoStepOut out;
        for (int j = 0; j < sc->n_joints; ++j) u[j] = (double)actions[e * sc->n_joints + j];
        smo_step_tp(sc, kin + (size_t)e * SM_KIN_STRIDE, ob + (size_t)e * SM_OBST_STRIDE,
                    tp ? tp + (size_t)e * SM_TP_STRIDE : 0, episode + 4 * e, ep_return + e, u,
                    next_ball ? next_ball + (size_t)e * 12 : 0, next_target ? next_target + (size_t)e * 3 : 0,
                    obs ? obs + (size_t)e * sc->obs_size : 0, &out);
        reward[e] = out.reward;
        done[e] = (uint8_t)out.done;
        term[e] = out.term_reason;
        memcpy(info + (size_t)e * SM_INFO_STRIDE, out.info, sizeof(out.info));
    }
}

int smo_sizeof_scene(void) { return (int)sizeof(SmScene); }
int smo_sizeof_stepout(void) { return (int)sizeof(SmoStepOut); }

/* Philox4x32-10 (Salmon et al., SC'11), the counter-based generator the device kernels use for pool picks and
 * random actions; restated so the tests can predict which pool entry an auto-reset loads. */
void smo_philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t* out) {
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
