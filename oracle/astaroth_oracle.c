/* CPU oracle for the astaroth `solve<step>` substep (SURVEY.md 8 row a18) -- plain C (+OpenMP).
 *
 * TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  Restates, operation by operation and in the same
 * association order, the generated device code of the reference's astaroth extract:
 *   first/second/cross_derivative, der{x,y,z,xx,yy,zz,xy,xz,yz}   astaroth/user_kernels.h:36-183
 *   gradient / hessian / laplace / divergence / curl / ...         astaroth/user_kernels.h:194-288
 *   continuity, momentum, induction, lnT, heat_conduction, entropy  astaroth/user_kernels.h:376-428
 *   solve<step_number>                                              astaroth/user_kernels.h:437-469
 *   rk3_integrate (Williamson 1980)                                 astaroth/integration.cuh:14-52
 *   dot / mul / cross                                               astaroth/math_utils.h:164-187
 * Indexing is the reference's memory-offset indexing IDX(i,j,k) = i + j*mx + k*mx*my
 * (astaroth/kernels.cu:15, 27-29) over allocations that include the radius-3 ghost cells.
 *
 * Parity status: the reference holds NO test for these numerics (astaroth/astaroth.cu:538 "TODO"); the pin is
 * tests/golden/astaroth_solve_ref.npz, produced on a B200 by the reference's own solve<> kernels
 * (oracle/ref/ref_astaroth_solve.cu + oracle/ref/make_astaroth_golden.py).  Floating point: compiled with
 * -ffp-contract=off while nvcc contracts a*b+c into FMAs, so agreement is to rounding, not bit-exact.  The `f80`
 * instance (long double: 64-bit mantissa on x86-64) is the reference the FP32 and FP64 kernels are bounded against,
 * a few ulp of the field's magnitude (tests/astaroth_util.py).
 */
#include <math.h>
#include <stdint.h>

#ifdef _OPENMP
#include <omp.h>
#endif

/* the uniforms solve<> reads through DCONST (astaroth/user_kernels.h:389-427, astaroth.conf) */
typedef struct {
  double inv_dsx, inv_dsy, inv_dsz;
  double dt;
  double cs2_sound, gamma, cp_sound, lnrho0, lnT0;
  double mu0, nu_visc, zeta, eta;
} so_ac_params;

enum { LNRHO = 0, UUX, UUY, UUZ, AX, AY, AZ, ENTROPY, NFIELDS };

#define AC_TEMPLATE(R, SUF, EXP)                                                                                       \
  typedef struct {                                                                                                     \
    R x, y, z;                                                                                                         \
  } v3_##SUF;                                                                                                          \
  typedef struct {                                                                                                     \
    v3_##SUF row[3];                                                                                                   \
  } m3_##SUF;                                                                                                          \
  typedef struct {                                                                                                     \
    R value;                                                                                                           \
    v3_##SUF gradient;                                                                                                 \
    m3_##SUF hessian;                                                                                                  \
  } data_##SUF;                                                                                                        \
                                                                                                                       \
  static inline R first_derivative_##SUF(const R *p, R inv_ds) {                                                       \
    const R c[4] = {0, (R)3.0 / (R)4.0, -(R)3.0 / (R)20.0, (R)1.0 / (R)60.0};                                          \
    R res = 0;                                                                                                         \
    for (int i = 1; i <= 3; ++i) res += c[i] * (p[3 + i] - p[3 - i]);                                                  \
    return res * inv_ds;                                                                                               \
  }                                                                                                                    \
  static inline R second_derivative_##SUF(const R *p, R inv_ds) {                                                      \
    const R c[4] = {-(R)49.0 / (R)18.0, (R)3.0 / (R)2.0, -(R)3.0 / (R)20.0, (R)1.0 / (R)90.0};                         \
    R res = c[0] * p[3];                                                                                               \
    for (int i = 1; i <= 3; ++i) res += c[i] * (p[3 + i] + p[3 - i]);                                                  \
    return res * inv_ds * inv_ds;                                                                                      \
  }                                                                                                                    \
  static inline R cross_derivative_##SUF(const R *a, const R *b, R inv_a, R inv_b) {                                   \
    const R fac = (R)1.0 / (R)720.0;                                                                                   \
    const R c[4] = {(R)0.0 * fac, (R)270.0 * fac, -(R)27.0 * fac, (R)2.0 * fac};                                       \
    R res = 0;                                                                                                         \
    for (int i = 1; i <= 3; ++i) res += c[i] * (a[3 + i] + a[3 - i] - b[3 + i] - b[3 - i]);                            \
    return res * inv_a * inv_b;                                                                                        \
  }                                                                                                                    \
  /* pencil through (i,j,k) along direction (dx,dy,dz): offsets -3..3 */                                               \
  static inline void pencil_##SUF(R *p, const R *f, int64_t mx, int64_t mxy, int64_t i, int64_t j, int64_t k, int dx,  \
                                  int dy, int dz) {                                                                    \
    for (int o = 0; o < 7; ++o)                                                                                        \
      p[o] = f[(i + dx * (o - 3)) + (j + dy * (o - 3)) * mx + (k + dz * (o - 3)) * mxy];                               \
  }                                                                                                                    \
  static inline data_##SUF read_data_##SUF(const R *f, int64_t mx, int64_t mxy, int64_t i, int64_t j, int64_t k,       \
                                           const so_ac_params *P) {                                                    \
    const R ix = (R)P->inv_dsx, iy = (R)P->inv_dsy, iz = (R)P->inv_dsz;                                                \
    R px[7], py[7], pz[7], a[7], b[7];                                                                                 \
    data_##SUF d;                                                                                                      \
    d.value = f[i + j * mx + k * mxy];                                                                                 \
    pencil_##SUF(px, f, mx, mxy, i, j, k, 1, 0, 0);                                                                    \
    pencil_##SUF(py, f, mx, mxy, i, j, k, 0, 1, 0);                                                                    \
    pencil_##SUF(pz, f, mx, mxy, i, j, k, 0, 0, 1);                                                                    \
    d.gradient.x = first_derivative_##SUF(px, ix);                                                                     \
    d.gradient.y = first_derivative_##SUF(py, iy);                                                                     \
    d.gradient.z = first_derivative_##SUF(pz, iz);                                                                     \
    d.hessian.row[0].x = second_derivative_##SUF(px, ix);                                                              \
    pencil_##SUF(a, f, mx, mxy, i, j, k, 1, 1, 0);  /* derxy: (x+o, y+o) and (x+o, y-o), user_kernels.h:97-111 */      \
    pencil_##SUF(b, f, mx, mxy, i, j, k, 1, -1, 0);                                                                    \
    d.hessian.row[0].y = cross_derivative_##SUF(a, b, ix, iy);                                                         \
    pencil_##SUF(a, f, mx, mxy, i, j, k, 1, 0, 1);  /* derxz, :113-127 */                                              \
    pencil_##SUF(b, f, mx, mxy, i, j, k, 1, 0, -1);                                                                    \
    d.hessian.row[0].z = cross_derivative_##SUF(a, b, ix, iz);                                                         \
    d.hessian.row[1].x = d.hessian.row[0].y;                                                                           \
    d.hessian.row[1].y = second_derivative_##SUF(py, iy);                                                              \
    pencil_##SUF(a, f, mx, mxy, i, j, k, 0, 1, 1);  /* deryz, :149-163 */                                              \
    pencil_##SUF(b, f, mx, mxy, i, j, k, 0, 1, -1);                                                                    \
    d.hessian.row[1].z = cross_derivative_##SUF(a, b, iy, iz);                                                         \
    d.hessian.row[2].x = d.hessian.row[0].z;                                                                           \
    d.hessian.row[2].y = d.hessian.row[1].z;                                                                           \
    d.hessian.row[2].z = second_derivative_##SUF(pz, iz);                                                              \
    return d;                                                                                                          \
  }                                                                                                                    \
  static inline R dot_##SUF(v3_##SUF a, v3_##SUF b) { return a.x * b.x + a.y * b.y + a.z * b.z; }                      \
  static inline v3_##SUF mul_##SUF(m3_##SUF m, v3_##SUF x) {                                                           \
    v3_##SUF r = {dot_##SUF(m.row[0], x), dot_##SUF(m.row[1], x), dot_##SUF(m.row[2], x)};                             \
    return r;                                                                                                          \
  }                                                                                                                    \
  static inline v3_##SUF cross_##SUF(v3_##SUF a, v3_##SUF b) {                                                         \
    v3_##SUF c = {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};                                \
    return c;                                                                                                          \
  }                                                                                                                    \
  static inline v3_##SUF add_##SUF(v3_##SUF a, v3_##SUF b) {                                                           \
    v3_##SUF c = {a.x + b.x, a.y + b.y, a.z + b.z};                                                                    \
    return c;                                                                                                          \
  }                                                                                                                    \
  static inline v3_##SUF sub_##SUF(v3_##SUF a, v3_##SUF b) {                                                           \
    v3_##SUF c = {a.x - b.x, a.y - b.y, a.z - b.z};                                                                    \
    return c;                                                                                                          \
  }                                                                                                                    \
  static inline v3_##SUF neg_##SUF(v3_##SUF a) {                                                                       \
    v3_##SUF c = {-a.x, -a.y, -a.z};                                                                                   \
    return c;                                                                                                          \
  }                                                                                                                    \
  static inline v3_##SUF scale_##SUF(R s, v3_##SUF a) {                                                                \
    v3_##SUF c = {s * a.x, s * a.y, s * a.z};                                                                          \
    return c;                                                                                                          \
  }                                                                                                                    \
  static inline R laplace_##SUF(const data_##SUF *d) {                                                                 \
    return d->hessian.row[0].x + d->hessian.row[1].y + d->hessian.row[2].z;                                            \
  }                                                                                                                    \
  static inline v3_##SUF laplace_vec_##SUF(const data_##SUF *v) {                                                      \
    v3_##SUF r = {laplace_##SUF(&v[0]), laplace_##SUF(&v[1]), laplace_##SUF(&v[2])};                                   \
    return r;                                                                                                          \
  }                                                                                                                    \
  static inline R divergence_##SUF(const data_##SUF *v) { return v[0].gradient.x + v[1].gradient.y + v[2].gradient.z; }\
  static inline v3_##SUF curl_##SUF(const data_##SUF *v) {                                                             \
    v3_##SUF r = {v[2].gradient.y - v[1].gradient.z, v[0].gradient.z - v[2].gradient.x,                                \
                  v[1].gradient.x - v[0].gradient.y};                                                                  \
    return r;                                                                                                          \
  }                                                                                                                    \
  static inline v3_##SUF gradient_of_divergence_##SUF(const data_##SUF *v) {                                           \
    v3_##SUF r = {v[0].hessian.row[0].x + v[1].hessian.row[0].y + v[2].hessian.row[0].z,                               \
                  v[0].hessian.row[1].x + v[1].hessian.row[1].y + v[2].hessian.row[1].z,                               \
                  v[0].hessian.row[2].x + v[1].hessian.row[2].y + v[2].hessian.row[2].z};                              \
    return r;                                                                                                          \
  }                                                                                                                    \
  static inline m3_##SUF stress_tensor_##SUF(const data_##SUF *v) {                                                    \
    m3_##SUF S;                                                                                                        \
    S.row[0].x = ((R)2.0 / (R)3.0) * v[0].gradient.x - ((R)1.0 / (R)3.0) * (v[1].gradient.y + v[2].gradient.z);        \
    S.row[0].y = ((R)1.0 / (R)2.0) * (v[0].gradient.y + v[1].gradient.x);                                              \
    S.row[0].z = ((R)1.0 / (R)2.0) * (v[0].gradient.z + v[2].gradient.x);                                              \
    S.row[1].y = ((R)2.0 / (R)3.0) * v[1].gradient.y - ((R)1.0 / (R)3.0) * (v[0].gradient.x + v[2].gradient.z);        \
    S.row[1].z = ((R)1.0 / (R)2.0) * (v[1].gradient.z + v[2].gradient.y);                                              \
    S.row[2].z = ((R)2.0 / (R)3.0) * v[2].gradient.z - ((R)1.0 / (R)3.0) * (v[0].gradient.x + v[1].gradient.y);        \
    S.row[1].x = S.row[0].y;                                                                                           \
    S.row[2].x = S.row[0].z;                                                                                           \
    S.row[2].y = S.row[1].z;                                                                                           \
    return S;                                                                                                          \
  }                                                                                                                    \
  static inline R contract_##SUF(m3_##SUF m) {                                                                         \
    R res = 0;                                                                                                         \
    for (int i = 0; i < 3; ++i) res += dot_##SUF(m.row[i], m.row[i]);                                                  \
    return res;                                                                                                        \
  }                                                                                                                    \
  static inline R rk3_##SUF(int step, R prev, R curr, R roc, R dt) {                                                   \
    const R alpha[4] = {0, (R).0, (R)(-5. / 9.), (R)(-153. / 128.)};                                                   \
    const R beta[4] = {0, (R)(1. / 3.), (R)(15. / 16.), (R)(8. / 15.)};                                                \
    if (step == 0) return curr + beta[step + 1] * roc * dt;                                                            \
    return curr + beta[step + 1] * (alpha[step + 1] * ((R)1. / beta[step]) * (curr - prev) + roc * dt);                \
  }                                                                                                                    \
                                                                                                                       \
  /* one cell of solve<step> (user_kernels.h:437-469) */                                                               \
  static inline void solve_cell_##SUF(int step, const R *const *in, R *const *out, int64_t mx, int64_t mxy, int64_t i, \
                                      int64_t j, int64_t k, const so_ac_params *P) {                                   \
    const int64_t idx = i + j * mx + k * mxy;                                                                          \
    const R dt = (R)P->dt, gam = (R)P->gamma, cp = (R)P->cp_sound, lnrho0 = (R)P->lnrho0, mu0 = (R)P->mu0;             \
    const R nu = (R)P->nu_visc, zeta = (R)P->zeta, eta = (R)P->eta, cs2s = (R)P->cs2_sound, lnT0 = (R)P->lnT0;         \
    const data_##SUF lnrho = read_data_##SUF(in[LNRHO], mx, mxy, i, j, k, P);                                          \
    data_##SUF uu[3], aa[3];                                                                                           \
    for (int c = 0; c < 3; ++c) {                                                                                      \
      uu[c] = read_data_##SUF(in[UUX + c], mx, mxy, i, j, k, P);                                                       \
      aa[c] = read_data_##SUF(in[AX + c], mx, mxy, i, j, k, P);                                                        \
    }                                                                                                                  \
    const data_##SUF ss = read_data_##SUF(in[ENTROPY], mx, mxy, i, j, k, P);                                           \
    const v3_##SUF uval = {uu[0].value, uu[1].value, uu[2].value};                                                     \
    /* continuity, :383-385 */                                                                                         \
    const R cont = -dot_##SUF(uval, lnrho.gradient) - divergence_##SUF(uu);                                            \
    /* induction, :397-402 */                                                                                          \
    const v3_##SUF B = curl_##SUF(aa);                                                                                 \
    const v3_##SUF lap_a = laplace_vec_##SUF(aa);                                                                      \
    const v3_##SUF ind = add_##SUF(cross_##SUF(uval, B), scale_##SUF(eta, lap_a));                                     \
    /* momentum, :387-395 */                                                                                           \
    const m3_##SUF S = stress_tensor_##SUF(uu);                                                                        \
    const R cs2 = cs2s * EXP(gam * ss.value / cp + (gam - 1) * (lnrho.value - lnrho0));                                \
    const v3_##SUF jj = scale_##SUF((R)1.0 / mu0, sub_##SUF(gradient_of_divergence_##SUF(aa), lap_a));                 \
    const R inv_rho = (R)1.0 / EXP(lnrho.value);                                                                       \
    const m3_##SUF G = {{uu[0].gradient, uu[1].gradient, uu[2].gradient}};                                             \
    const v3_##SUF gdu = gradient_of_divergence_##SUF(uu);                                                             \
    v3_##SUF mom = neg_##SUF(mul_##SUF(G, uval));                                                                      \
    mom = sub_##SUF(mom, scale_##SUF(cs2, add_##SUF(scale_##SUF((R)1.0 / cp, ss.gradient), lnrho.gradient)));          \
    mom = add_##SUF(mom, scale_##SUF(inv_rho, cross_##SUF(jj, B)));                                                    \
    {                                                                                                                  \
      v3_##SUF visc = add_##SUF(laplace_vec_##SUF(uu), scale_##SUF((R)1.0 / (R)3.0, gdu));                             \
      visc = add_##SUF(visc, scale_##SUF((R)2.0, mul_##SUF(S, lnrho.gradient)));                                       \
      mom = add_##SUF(mom, scale_##SUF(nu, visc));                                                                     \
    }                                                                                                                  \
    mom = add_##SUF(mom, scale_##SUF(zeta, gdu));                                                                      \
    /* entropy, :403-428 */                                                                                            \
    const R lnT = lnT0 + gam * ss.value / cp + (gam - (R)1.0) * (lnrho.value - lnrho0);                                \
    const R inv_pT = (R)1.0 / (EXP(lnrho.value) * EXP(lnT));                                                           \
    const R divu = divergence_##SUF(uu);                                                                               \
    const R RHS = (0) - (0) + eta * (mu0)*dot_##SUF(jj, jj) + (R)2.0 * EXP(lnrho.value) * nu * contract_##SUF(S) +     \
                  zeta * EXP(lnrho.value) * divu * divu;                                                               \
    R heat;                                                                                                            \
    {                                                                                                                  \
      const R inv_cp = (R)1.0 / cp;                                                                                    \
      const v3_##SUF grad_ln_chi = neg_##SUF(lnrho.gradient);                                                          \
      const R first = gam * inv_cp * laplace_##SUF(&ss) + (gam - (R)1.0) * laplace_##SUF(&lnrho);                      \
      const v3_##SUF second =                                                                                          \
          add_##SUF(scale_##SUF(gam * inv_cp, ss.gradient), scale_##SUF(gam - (R)1.0, lnrho.gradient));                \
      const v3_##SUF third =                                                                                           \
          add_##SUF(scale_##SUF(gam, add_##SUF(scale_##SUF(inv_cp, ss.gradient), lnrho.gradient)), grad_ln_chi);       \
      const R chi = ((R)0.001) / (EXP(lnrho.value) * cp);                                                              \
      heat = cp * chi * (first + dot_##SUF(second, third));                                                            \
    }                                                                                                                  \
    const R ent = -dot_##SUF(uval, ss.gradient) + inv_pT * RHS + heat;                                                 \
    /* rk3 updates in the reference's order: lnrho, aa, uu, ss (:444-453) */                                           \
    const R o_lnrho = rk3_##SUF(step, out[LNRHO][idx], lnrho.value, cont, dt);                                         \
    const R o_ax = rk3_##SUF(step, out[AX][idx], aa[0].value, ind.x, dt);                                              \
    const R o_ay = rk3_##SUF(step, out[AY][idx], aa[1].value, ind.y, dt);                                              \
    const R o_az = rk3_##SUF(step, out[AZ][idx], aa[2].value, ind.z, dt);                                              \
    const R o_ux = rk3_##SUF(step, out[UUX][idx], uu[0].value, mom.x, dt);                                             \
    const R o_uy = rk3_##SUF(step, out[UUY][idx], uu[1].value, mom.y, dt);                                             \
    const R o_uz = rk3_##SUF(step, out[UUZ][idx], uu[2].value, mom.z, dt);                                             \
    const R o_ss = rk3_##SUF(step, out[ENTROPY][idx], ss.value, ent, dt);                                              \
    out[LNRHO][idx] = o_lnrho;                                                                                         \
    out[UUX][idx] = o_ux;                                                                                              \
    out[UUY][idx] = o_uy;                                                                                              \
    out[UUZ][idx] = o_uz;                                                                                              \
    out[AX][idx] = o_ax;                                                                                               \
    out[AY][idx] = o_ay;                                                                                               \
    out[AZ][idx] = o_az;                                                                                               \
    out[ENTROPY][idx] = o_ss;                                                                                          \
  }                                                                                                                    \
                                                                                                                       \
  /* integrate_substep (astaroth/kernels.cu:62-87): solve<step> on the box [lo, hi) in memory-offset coordinates.   */ \
  void so_astaroth_substep_##SUF(int step, const R *const *in, R *const *out, int64_t mx, int64_t my, const int64_t *lo,\
                                 const int64_t *hi, const so_ac_params *P) {                                           \
    const int64_t mxy = mx * my;                                                                                       \
    _Pragma("omp parallel for collapse(2) schedule(static)") for (int64_t k = lo[2]; k < hi[2]; ++k) {                 \
      for (int64_t j = lo[1]; j < hi[1]; ++j) {                                                                        \
        for (int64_t i = lo[0]; i < hi[0]; ++i) solve_cell_##SUF(step, in, out, mx, mxy, i, j, k, P);                  \
      }                                                                                                                \
    }                                                                                                                  \
  }

AC_TEMPLATE(double, f64, exp)
AC_TEMPLATE(float, f32, expf)
/* x87 extended precision (64-bit mantissa): the high-precision reference the GPU kernels are bounded against */
AC_TEMPLATE(long double, f80, expl)
