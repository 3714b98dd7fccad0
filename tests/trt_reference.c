/*
 * trt_reference.c -- TEST INFRASTRUCTURE ONLY: the two-relaxation-time (TRT) collision on the CPU oracle.
 *
 * Compiled from this file by tests/trt_reference.py, with the flags oracle/Makefile uses, once per precision.
 * It includes oracle/lbm_oracle.c unchanged, so the state struct, the equilibrium forms, the wall gather and
 * the boundary sets are the oracle's own; only the collision of `update_fluid` and the relaxation factor of
 * `neq_extrap` differ, written here in literal form:
 *
 *   collision, for every opposite pair (q, qbar):
 *     n+ = (f_q + f_qbar)/2 - (feq_q + feq_qbar)/2      n- = (f_q - f_qbar)/2 - (feq_q - feq_qbar)/2
 *     f_q <- f_q - om_p n+ - om_m n-                    f_0 <- f_0 - om_p (f_0 - feq_0)
 *   inlet / outlet / lid link q of boundary node b, fluid neighbour nb = b + c_q, n_q = g_q(nb) - feq_q(nb):
 *     feq_q(bc) + (1 - om_p) (n_q + n_qbar)/2 + (1 - om_m) (n_q - n_qbar)/2
 *
 * with om_p = 1/tau and om_m = 1 / (1/2 + magic / (tau - 1/2)) (computed in double, as the library's host does).
 * An oracle handle stepped with trt_step_* instead of orc_step_* is the reference of the GPU's TRT kernels.
 */
#include "../oracle/lbm_oracle.c"

static void trt_update_fluid(FN(orc_state) *s, REAL om_p, REAL om_m) {
    const int nlat = s->nlat, nfl = s->nfl;
#pragma omp parallel for schedule(static)
    for (int j = 0; j < nfl; j++) {
        const int i = s->flist[j];
        REAL f[19], feq[19];
        for (int q = 0; q < 19; q++) {
            int n = s->pull[(size_t)q * nfl + j];
            f[q] = n >= 0 ? s->src[(size_t)q * nlat + n] : R(0.0);
        }
        REAL rho = R(0.0);
        for (int q = 0; q < 19; q++) rho = rho + f[q];
        REAL ux = (f[1] - f[2] + f[7] + f[8] - f[9] - f[10] + f[11] + f[12] - f[13] - f[14]) / rho;
        REAL uy = (f[3] - f[4] + f[7] - f[8] + f[9] - f[10] + f[15] - f[16] + f[17] - f[18]) / rho;
        REAL uz = (f[5] - f[6] + f[11] - f[12] + f[13] - f[14] + f[15] + f[16] - f[17] - f[18]) / rho;
        s->rho[i] = rho, s->ux[i] = ux, s->uy[i] = uy, s->uz[i] = uz;
        feq_all(rho, ux, uy, uz, feq);
        s->dst[i] = f[0] - om_p * (f[0] - feq[0]);
        for (int q = 1; q < 19; q++) {
            const int qb = OPP[q];
            REAL np = R(0.5) * (f[q] + f[qb]) - R(0.5) * (feq[q] + feq[qb]);
            REAL nm = R(0.5) * (f[q] - f[qb]) - R(0.5) * (feq[q] - feq[qb]);
            s->dst[(size_t)q * nlat + i] = f[q] - om_p * np - om_m * nm;
        }
    }
}

/* neq_extrap of lbm_oracle.c with the TRT relaxation of the extrapolated non-equilibrium */
static REAL trt_neq_extrap(const FN(orc_state) *s, int x, int y, int z, int q, int kind, int vaxis, REAL upresc,
                           REAL om_p, REAL om_m) {
    int n = nb_idx(s, x, y, z, CX[q], CY[q], CZ[q], 0);
    const int qb = OPP[q];
    REAL rho = R(0.0), ux = R(0.0), uy = R(0.0), uz = R(0.0), fnb = R(0.0), fnbb = R(0.0);
    if (n >= 0) {
        rho = s->rho[n], ux = s->ux[n], uy = s->uy[n], uz = s->uz[n];
        fnb = s->dst[(size_t)q * s->nlat + n], fnbb = s->dst[(size_t)qb * s->nlat + n];
    }
    REAL wden = q == 0 ? R(3.0) : (q < 7 ? R(18.0) : R(36.0));
    REAL feq = feq_q(q, rho / R(3.0), rho / R(18.0), rho / R(36.0), ux, uy, uz);
    REAL feqb = feq_q(qb, rho / R(3.0), rho / R(18.0), rho / R(36.0), ux, uy, uz);
    REAL tmp;
    if (kind == 1) {
        REAL one = R(1.0);
        tmp = feq_q(q, one / R(3.0), one / R(18.0), one / R(36.0), ux, uy, uz);
    } else {
        int cs = vaxis == 0 ? CX[q] : (vaxis == 1 ? CY[q] : CZ[q]);
        REAL rw = kind == 0 ? rho / wden : R(1.0) / wden;
        tmp = feq_bc_axis(rw, cs, upresc);
    }
    REAL nq = fnb - feq, nqb = fnbb - feqb;
    return tmp + ((R(1.0) - om_p) * (R(0.5) * (nq + nqb)) + (R(1.0) - om_m) * (R(0.5) * (nq - nqb)));
}

/* boundary_stream of lbm_oracle.c with trt_neq_extrap */
static void trt_boundary_stream(FN(orc_state) *s, REAL om_p, REAL om_m) {
    const int nlat = s->nlat, nb = s->nb;
    const int ywrap = (s->case_id == CASE_POS || s->case_id == CASE_BIF);
    double scale = 1.0;
    if (s->pulse_amp != 0.0) scale = 1.0 + s->pulse_amp * sin(2.0 * M_PI * (double)s->step_count / s->pulse_period);
#pragma omp parallel for schedule(static)
    for (int b = 0; b < nb; b++) {
        int i = s->blist[b];
        size_t c = (size_t)s->cart[i];
        int g = s->geo[c];
        int x = (int)(c % s->nx), y = (int)((c / s->nx) % s->ny), z = (int)(c / ((size_t)s->nx * s->ny));
        REAL *out = s->bscratch + (size_t)19 * b;
        for (int q = 0; q < 19; q++) out[q] = s->dst[(size_t)q * nlat + i];
        if (g == 1) {
            if (s->case_id != CASE_LDC) wall_gather(s, s->dst, x, y, z, ywrap, out);
            continue;
        }
        const int *set = NULL;
        int kind = 0, vaxis = 1;
        REAL up = R(0.0);
        switch (s->case_id) {
        case CASE_LDC:
            if (g == 2) set = SET_YM, kind = 0, vaxis = 2, up = s->u_bc;
            break;
        case CASE_POS:
            if (g == 3) set = SET_YM, kind = 0, vaxis = 1, up = parabola(s, s->u_bc, x, z);
            if (g == 2) set = SET_YP, kind = 0, vaxis = 1, up = parabola(s, s->u_bc, x, z);
            break;
        case CASE_BIF:
            if (g == 3) set = SET_YM, kind = 1;
            if (g == 2) set = SET_YP, kind = 0, vaxis = 1, up = (REAL)(s->inlety[x + z * s->nx] * (REAL)scale);
            break;
        default:
            if (g == 2) set = SET_XP, kind = 2, vaxis = 0, up = (REAL)(s->cor_uin * (REAL)scale);
            if (g == 3) set = SET_XM, kind = 0, vaxis = 0, up = s->cor_uout;
            if (g == 5 || g == 6 || g == 7) set = SET_ZM, kind = 0, vaxis = 2, up = s->cor_usub;
            break;
        }
        if (set)
            for (int k = 0; k < 5; k++) out[set[k]] = trt_neq_extrap(s, x, y, z, set[k], kind, vaxis, up, om_p, om_m);
    }
#pragma omp parallel for schedule(static)
    for (int b = 0; b < nb; b++) {
        int i = s->blist[b];
        const REAL *out = s->bscratch + (size_t)19 * b;
        for (int q = 0; q < 19; q++) s->dst[(size_t)q * nlat + i] = out[q];
    }
}

/* orc_step of lbm_oracle.c (defined LDC order) with the TRT collision */
void FN(trt_step)(FN(orc_state) *s, int nsteps, double magic) {
    const REAL om_p = R(1.0) / s->tau;
    const REAL om_m = (REAL)(1.0 / (0.5 + magic / ((double)s->tau - 0.5)));
    for (int it = 0; it < nsteps; it++) {
        if (s->case_id == CASE_LDC) ldc_wall_bounce_src(s, 0);
        trt_update_fluid(s, om_p, om_m);
        trt_boundary_stream(s, om_p, om_m);
        REAL *t = s->src;
        s->src = s->dst;
        s->dst = t;
        s->step_count++;
    }
}
