// Counts the algorithmic FLOPs of one physics substep by instantiating the kernel's own recursion templates
// (so100_mujoco_rl_b200/csrc/so100_dyn.cuh) with an operation-counting scalar.  Convention (SURVEY.md §8 d):
// add / sub / mul / div = 1, an FMA = 2 (it is written as mul + add here), sincos = 2, compares / selects / abs = 0.
//   g++ -O1 -std=c++17 -o /tmp/count_flops tools/count_flops.cpp && /tmp/count_flops
#include <cstdio>
#include "../so100_mujoco_rl_b200/csrc/so100_dyn.cuh"

struct C {
  double v;
  static long n;
  C() : v(0) {}
  C(double x) : v(x) {}
  C(int x) : v(x) {}
  explicit operator double() const { return v; }
  explicit operator float() const { return (float)v; }
};
long C::n = 0;
C operator+(C a, C b) { C::n++; return C(a.v + b.v); }
C operator-(C a, C b) { C::n++; return C(a.v - b.v); }
C operator*(C a, C b) { C::n++; return C(a.v * b.v); }
C operator/(C a, C b) { C::n++; return C(a.v / b.v); }
C operator-(C a) { return C(-a.v); }
C& operator+=(C& a, C b) { C::n++; a.v += b.v; return a; }
C& operator-=(C& a, C b) { C::n++; a.v -= b.v; return a; }
bool operator<(C a, C b) { return a.v < b.v; }
bool operator>(C a, C b) { return a.v > b.v; }
bool operator<=(C a, C b) { return a.v <= b.v; }
bool operator>=(C a, C b) { return a.v >= b.v; }
bool operator==(C a, C b) { return a.v == b.v; }
bool operator!=(C a, C b) { return a.v != b.v; }

int main() {
  DynC<C> D;
  ConC<C> K;
  for (int i = 0; i < SO_NJ; i++) {
    for (int k = 0; k < 9; k++) D.L[i].R[k] = (k % 4 == 0) ? 1.0 : 0.01 * (k + i);
    for (int k = 0; k < 3; k++) { D.L[i].p[k] = 0.1 * (k + 1); D.L[i].h[k] = 0.01 * (k + 1); }
    for (int k = 0; k < 6; k++) D.L[i].I[k] = k < 3 ? 1e-3 : 1e-5;
    D.L[i].m = 0.1; D.L[i].arm = 0.1;
    K.fr_D[i] = 1; K.fr_B[i] = 105; K.fr_loss[i] = 0.1; K.lo[i] = -10; K.hi[i] = 10; K.lim_B[i] = 105; K.lim_K[i] = 2770;
    K.invw[i] = 9; K.imp0[i] = 0.9; K.imp1[i] = 0.95; K.imp_w[i] = 0.001; K.imp_mid[i] = 0.5; K.imp_pow[i] = 2;
    K.imp_rw[i] = 1000; K.imp_rmid[i] = 2; K.imp_r1mid[i] = 2;
  }
  D.a0[0] = 0; D.a0[1] = 0; D.a0[2] = 9.81;
  C s[6], c[6], qd[6], q[6], bias[6], M[21], b[6], a[6];
  for (int j = 0; j < 6; j++) { s[j] = 0.3; c[j] = 0.95; qd[j] = 0.2; q[j] = 0.1; a[j] = 0; }
  long sincos = 6 * 2;
  C::n = 0;
  dyn_bias_mass<C>(D, s, c, qd, bias, M);
  long dyn = C::n;
  C::n = 0;
  for (int j = 0; j < 6; j++) { C f = C(50.0) * q[j] - C(50.0) * q[j] - C(5.0) * qd[j]; b[j] = f - bias[j]; }
  long act = C::n;
  C::n = 0;
  C zc[6]; for (int j = 0; j < 6; j++) zc[j] = 0;
  solve_qacc<C>(K, K.fr_loss, M, b, q, zc, qd, a, 12);  // converge first: the counted calls then run exactly their scheduled sweeps
  C::n = 0;
  solve_qacc<C>(K, K.fr_loss, M, b, q, zc, qd, a, 5);
  long solve5 = C::n;
  C::n = 0;
  solve_qacc<C>(K, K.fr_loss, M, b, q, zc, qd, a, 3);
  long solve3 = C::n;
  C::n = 0;
  for (int j = 0; j < 6; j++) { qd[j] += C(0.002) * a[j]; q[j] += C(0.002) * qd[j]; }
  long integ = C::n;
  long common = sincos + dyn + act + integ;
  // the shipped schedule (csrc/so100_b200.cu physics<>): 5 Gauss-Seidel sweeps on the first substep of an env step
  // (ctrl has just jumped), 3 on the other 15 (warm start within a few %)
  long step = 16 * common + solve5 + 15 * solve3;
  printf("per substep: sincos %ld  bias+mass %ld  actuation %ld  euler %ld  solve(5 sweeps) %ld  solve(3 sweeps) %ld\n", sincos, dyn, act, integ, solve5, solve3);
  printf("per env step: 16 x %ld + %ld + 15 x %ld = %ld FLOP (+ ~150 task logic, ~330 snapshot kinematics)\n", common, solve5, solve3, step);
  printf("(generic recursion, friction rows only; the model-specialised kernel executes fewer FLOP for the same result, and\n"
         " arm-floor contact adds data-dependent work that is not counted: bench.py's `frac` is useful work / FFMA peak)\n");
  return 0;
}
