// oracle_capi.cpp — C entry points over pbh_oracle.hpp (TEST INFRASTRUCTURE, NOT PRODUCT CODE).
//
// Built into oracle/liboracle.so by oracle/Makefile.  Used only by tests/, __graft_entry__.smoke()
// and bench.py's cpu_baseline / --impl reference legs, as the checker or as the timed CPU baseline.
// Batch entry points use the byte-plane wire layout of include/pbh_b200.h so that GPU and oracle
// outputs can be compared with memcmp.
#include "pbh_oracle.hpp"

#include <atomic>
#include <cstring>
#include <memory>
#include <thread>

using namespace pbh_oracle;

namespace {

// ---- circuit description shared with include/pbh_b200.h (kept layout-identical, see static_assert
// in the product's capi) ----
struct circuit_desc {
  uint8_t q_l[4], q_r[4], q_o[4], q_m[4], q_c[4];
  uint8_t c_a_wire[4], c_a_index[4], c_b_wire[4], c_b_index[4], c_c_wire[4], c_c_index[4];
};

Constrains to_constrains(const circuit_desc& d) {
  Constrains k;
  auto wire = [](uint8_t w) { return w == 0 ? 'A' : (w == 1 ? 'B' : 'C'); };
  for (int i = 0; i < 4; i++) {
    k.q_l.push_back(f17(d.q_l[i])); k.q_r.push_back(f17(d.q_r[i])); k.q_o.push_back(f17(d.q_o[i]));
    k.q_m.push_back(f17(d.q_m[i])); k.q_c.push_back(f17(d.q_c[i]));
    k.c_a.push_back({wire(d.c_a_wire[i]), d.c_a_index[i]});
    k.c_b.push_back({wire(d.c_b_wire[i]), d.c_b_index[i]});
    k.c_c.push_back({wire(d.c_c_wire[i]), d.c_c_index[i]});
  }
  return k;
}

struct Setup {
  Constrains constraints;
  std::unique_ptr<Plonk> plonk;
};

// returns nullptr when the reference's setup would panic
std::unique_ptr<Setup> make_setup(const circuit_desc* d, uint8_t s, uint32_t srs_n, uint8_t omega_pows) {
  try {
    auto st = std::make_unique<Setup>();
    st->constraints = to_constrains(*d);
    st->plonk = std::make_unique<Plonk>(SRS::create(f101(s), srs_n), f17(omega_pows));
    return st;
  } catch (const Panic&) {
    return nullptr;
  }
}

template <class Fn>
void parallel_for(size_t n, int threads, Fn fn) {
  if (threads <= 1 || n < 2) { fn(0, n); return; }
  std::vector<std::thread> pool;
  size_t chunk = (n + threads - 1) / threads;
  for (int t = 0; t < threads; t++) {
    size_t lo = std::min(n, (size_t)t * chunk), hi = std::min(n, lo + chunk);
    if (lo < hi) pool.emplace_back([=] { fn(lo, hi); });
  }
  for (auto& th : pool) th.join();
}

inline void put_point(uint8_t* proof, size_t pitch, size_t i, int k, const G1P& p) {
  proof[(2 * k) * pitch + i] = (uint8_t)p.x.v;
  proof[(2 * k + 1) * pitch + i] = (uint8_t)p.y.v;
  if (p.infinite) {
    if (k < 8) proof[18 * pitch + i] |= (uint8_t)(1u << k);
    else proof[19 * pitch + i] |= 1u;
  }
}
inline G1P get_point(const uint8_t* proof, size_t pitch, size_t i, int k) {
  G1P p;
  p.x.v = proof[(2 * k) * pitch + i];   // raw bytes: range-checked by the caller
  p.y.v = proof[(2 * k + 1) * pitch + i];
  p.infinite = k < 8 ? ((proof[18 * pitch + i] >> k) & 1) : (proof[19 * pitch + i] & 1);
  return p;
}

// one proof through the oracle; returns the status byte and fills `pr` when 0
int prove_one(const Setup& st, const uint8_t w[12], const uint8_t r[9], const uint8_t c[5], Proof& pr) {
  for (int k = 0; k < 12; k++) if (w[k] >= 17) return 32;
  for (int k = 0; k < 9; k++) if (r[k] >= 17) return 32;
  for (int k = 0; k < 5; k++) if (c[k] >= 17) return 32;
  Assigments as;
  for (int k = 0; k < 4; k++) { as.a.push_back(f17(w[k])); as.b.push_back(f17(w[4 + k])); as.c.push_back(f17(w[8 + k])); }
  F17 rand[9];
  for (int k = 0; k < 9; k++) rand[k] = f17(r[k]);
  Challange ch{f17(c[0]), f17(c[1]), f17(c[2]), f17(c[3]), f17(c[4])};
  try {
    pr = st.plonk->prove(st.constraints, as, ch, rand);
    return 0;
  } catch (const Panic& p) {
    return p.site;
  }
}

// Fiat-Shamir seed of a context (include/pbh_b200.h, "Fiat-Shamir transcript"): SHA-256 over a domain tag, omega_pows,
// the circuit description and the SRS
void fs_seed(const Setup& st, const circuit_desc& d, uint8_t omega_pows, uint8_t out[32]) {
  std::vector<uint8_t> m;
  const char* tag = "plonk-by-fingers/fiat-shamir/v1";
  for (const char* c = tag; *c; c++) m.push_back((uint8_t)*c);
  m.push_back(omega_pows);
  const uint8_t* sel[5] = {d.q_l, d.q_r, d.q_o, d.q_m, d.q_c};
  for (int k = 0; k < 5; k++) for (int i = 0; i < 4; i++) m.push_back((uint8_t)(sel[k][i] % 17));
  const uint8_t* cc[6] = {d.c_a_wire, d.c_a_index, d.c_b_wire, d.c_b_index, d.c_c_wire, d.c_c_index};
  for (int k = 0; k < 6; k++) for (int i = 0; i < 4; i++) m.push_back(cc[k][i]);
  const SRS& srs = st.plonk->srs;
  m.push_back((uint8_t)srs.g1s.size());
  for (const G1P& p : srs.g1s) FsTranscript::put_point(m, p);
  m.push_back((uint8_t)srs.g2_1.a.v); m.push_back((uint8_t)srs.g2_1.b.v);
  m.push_back((uint8_t)srs.g2_s.a.v); m.push_back((uint8_t)srs.g2_s.b.v);
  Sha256::hash(m, out);
}

// one proof with transcript-derived challenges; `derived` = alpha beta gamma z v u (those derived before a panic, 0 after)
int prove_one_fs(const Setup& st, const uint8_t seed[32], const uint8_t w[12], const uint8_t r[9], Proof& pr, uint8_t derived[6]) {
  for (int k = 0; k < 6; k++) derived[k] = 0;
  for (int k = 0; k < 12; k++) if (w[k] >= 17) return 32;
  for (int k = 0; k < 9; k++) if (r[k] >= 17) return 32;
  Assigments as;
  for (int k = 0; k < 4; k++) { as.a.push_back(f17(w[k])); as.b.push_back(f17(w[4 + k])); as.c.push_back(f17(w[8 + k])); }
  F17 rand[9];
  for (int k = 0; k < 9; k++) rand[k] = f17(r[k]);
  FsTranscript tr(seed);
  int status = 0;
  try {
    pr = st.plonk->prove_cs(st.constraints, as, tr, rand);
  } catch (const Panic& p) {
    status = p.site;
  }
  for (int k = 0; k < 6; k++) derived[k] = tr.derived[k];
  return status;
}

void store_proof(const Proof& pr, uint8_t* proof, size_t pitch, size_t i) {
  const G1P* pts[9] = {&pr.a_s, &pr.b_s, &pr.c_s, &pr.z_s, &pr.t_lo_s, &pr.t_mid_s, &pr.t_hi_s, &pr.w_z_s, &pr.w_z_omega_s};
  for (int k = 0; k < 9; k++) put_point(proof, pitch, i, k, *pts[k]);
  const F17 ev[7] = {pr.a_z, pr.b_z, pr.c_z, pr.s_sigma_1_z, pr.s_sigma_2_z, pr.r_z, pr.z_omega_z};
  for (int k = 0; k < 7; k++) proof[(20 + k) * pitch + i] = (uint8_t)ev[k].v;
}

// ---- synthetic input stream (SURVEY.md §8d); must match the device generator bit for bit ----
inline uint64_t splitmix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
inline uint32_t draw(uint64_t base, uint32_t j, uint32_t range) {
  uint64_t r = splitmix64(base + (uint64_t)j * 0xD1B54A32D192ED03ull);
  return (uint32_t)(((unsigned __int128)r * range) >> 64);
}
constexpr uint32_t kGenMaxAttempts = 4096;   // PBH_GEN_MAX_ATTEMPTS of include/pbh_b200.h
struct WitnessTable { uint8_t xyz[289][3]; };
const WitnessTable& witness_table() {
  static WitnessTable t = [] {
    WitnessTable w{};
    int n = 0;
    for (int x = 0; x < 17; x++)
      for (int y = 0; y < 17; y++)
        for (int z = 0; z < 17; z++)
          if ((x * x + y * y) % 17 == (z * z) % 17) { w.xyz[n][0] = x; w.xyz[n][1] = y; w.xyz[n][2] = z; n++; }
    return w;
  }();
  return t;
}
void sample_attempt(uint64_t seed, uint64_t index, uint32_t k, uint8_t w[12], uint8_t r[9], uint8_t c[5], uint8_t& u) {
  uint64_t base = splitmix64(seed ^ (index * 0x9E3779B97F4A7C15ull) ^ ((uint64_t)k * 0xC2B2AE3D27D4EB4Full));
  const uint8_t* s = witness_table().xyz[draw(base, 0, 289)];
  uint8_t x = s[0], y = s[1], z = s[2];
  uint8_t xx = (x * x) % 17, yy = (y * y) % 17, zz = (z * z) % 17;
  w[0] = x; w[1] = y; w[2] = z; w[3] = xx;      // a   (generalises src/pbh/mod.rs:70-75)
  w[4] = x; w[5] = y; w[6] = z; w[7] = yy;      // b
  w[8] = xx; w[9] = yy; w[10] = zz; w[11] = zz; // c
  for (int j = 0; j < 9; j++) r[j] = (uint8_t)draw(base, 1 + j, 17);
  for (int j = 0; j < 5; j++) c[j] = (uint8_t)draw(base, 10 + j, 17);
  u = (uint8_t)draw(base, 15, 17);
}

}  // namespace

extern "C" {

// ------------------------------------------------------------------------------------------------
// fine-grained operations, used to pin the oracle against the reference's own unit-test vectors
// ------------------------------------------------------------------------------------------------
#define DISPATCH_M(M, ...)                                           \
  switch (M) {                                                       \
    case 17: { using F = Fp<17>; __VA_ARGS__ } break;                \
    case 101: { using F = Fp<101>; __VA_ARGS__ } break;              \
    case 257: { using F = Fp<257>; __VA_ARGS__ } break;              \
    case 337: { using F = Fp<337>; __VA_ARGS__ } break;              \
    case 104729: { using F = Fp<104729>; __VA_ARGS__ } break;        \
    case 15485863: { using F = Fp<15485863>; __VA_ARGS__ } break;    \
    default: return -1;                                              \
  }

// op: 0 add, 1 sub, 2 mul, 3 div (returns 1 for None), 4 neg(a), 5 pow(a, b as exponent), 6 inv(a) (1 for None)
int oracle_field_op(uint64_t M, int op, uint64_t a, uint64_t b, uint64_t* out) {
  DISPATCH_M(M, {
    F x = F::from_u64(a), y = F::from_u64(b);
    switch (op) {
      case 0: *out = (x + y).v; return 0;
      case 1: *out = (x - y).v; return 0;
      case 2: *out = (x * y).v; return 0;
      case 3: { auto r = x / y; if (!r) return 1; *out = r->v; return 0; }
      case 4: *out = (-x).v; return 0;
      case 5: *out = x.pow(b).v; return 0;
      case 6: { auto r = x.inv(); if (!r) return 1; *out = r->v; return 0; }
      default: return -1;
    }
  })
  return -1;
}

// polynomials: coefficients as signed integers (Poly::from(&[i64]) semantics).
// op: 0 a+=b, 1 a-=b (Q1), 2 a*b, 3 a/b -> (out, out2), 4 eval(a, b[0]), 5 z(points=a), 6 normalize(a),
//     7 lagrange(xs=a, ys=b), 8 a * scalar b[0] (Q15)
int oracle_poly_op(uint64_t M, int op, const int64_t* a, size_t la, const int64_t* b, size_t lb, uint64_t* out,
                   size_t* lout, uint64_t* out2, size_t* lout2) {
  try {
    DISPATCH_M(M, {
      std::vector<F> va, vb;
      for (size_t i = 0; i < la; i++) va.push_back(F::from_i64(a[i]));
      for (size_t i = 0; i < lb; i++) vb.push_back(F::from_i64(b[i]));
      auto emit = [&](const Poly<F>& p, uint64_t* o, size_t* lo) {
        for (size_t i = 0; i < p.c.size(); i++) o[i] = p.c[i].v;
        *lo = p.c.size();
      };
      switch (op) {
        case 0: { Poly<F> p(va); p += Poly<F>(vb); emit(p, out, lout); return 0; }
        case 1: { Poly<F> p(va); p -= Poly<F>(vb); emit(p, out, lout); return 0; }
        case 2: { emit(Poly<F>(va) * Poly<F>(vb), out, lout); return 0; }
        case 3: { auto qr = poly_div(Poly<F>(va), Poly<F>(vb)); emit(qr.first, out, lout); emit(qr.second, out2, lout2); return 0; }
        case 4: { out[0] = Poly<F>(va).eval(vb[0]).v; *lout = 1; return 0; }
        case 5: { emit(Poly<F>::z(va), out, lout); return 0; }
        case 6: { emit(Poly<F>(va), out, lout); return 0; }
        case 7: {
          std::vector<std::pair<F, F>> pts;
          for (size_t i = 0; i < la; i++) pts.push_back({va[i], vb[i]});
          emit(Poly<F>::lagrange(pts), out, lout);
          return 0;
        }
        case 8: { emit(Poly<F>(va) * vb[0], out, lout); return 0; }
        default: return -1;
      }
    })
  } catch (const Panic&) {
    return 1;
  }
  return -1;
}

// matrices, row-major u64.  op: 0 a*b, 1 inv(a), 2 a+b, 3 a * poly(b as column of coefficients) -> poly
int oracle_matrix_op(uint64_t M, int op, const uint64_t* a, size_t am, size_t an, const uint64_t* b, size_t bm,
                     size_t bn, uint64_t* out, size_t* om, size_t* on) {
  try {
    DISPATCH_M(M, {
      Matrix<F> A = Matrix<F>::from_u64(std::vector<uint64_t>(a, a + am * an), am, an);
      auto emit = [&](const Matrix<F>& R) {
        for (size_t i = 0; i < R.v.size(); i++) out[i] = R.v[i].v;
        *om = R.m; *on = R.n;
      };
      switch (op) {
        case 0: { Matrix<F> B = Matrix<F>::from_u64(std::vector<uint64_t>(b, b + bm * bn), bm, bn); emit(A * B); return 0; }
        case 1: emit(A.inv()); return 0;
        case 2: { Matrix<F> B = Matrix<F>::from_u64(std::vector<uint64_t>(b, b + bm * bn), bm, bn); emit(A + B); return 0; }
        case 3: {
          std::vector<F> vb;
          for (size_t i = 0; i < bm * bn; i++) vb.push_back(F::from_u64(b[i]));
          Poly<F> p = A.mul_poly(Poly<F>(vb));
          for (size_t i = 0; i < p.c.size(); i++) out[i] = p.c[i].v;
          *om = p.c.size(); *on = 1;
          return 0;
        }
        default: return -1;
      }
    })
  } catch (const Panic&) {
    return 1;
  }
  return -1;
}

// src/fft.rs: which 0 = VandermondeMatrix, 1 = CooleyTurkey; inverse 0 = fft, 1 = fft_inv
int oracle_fft(uint64_t M, uint64_t omega, size_t size, int which, int inverse, const uint64_t* in, size_t n_in,
               uint64_t* out, size_t* n_out) {
  try {
    DISPATCH_M(M, {
      std::vector<F> v;
      for (size_t i = 0; i < n_in; i++) v.push_back(F::from_u64(in[i]));
      EvaluationDomainGenerator<F> d{F::from_u64(omega), size};
      std::vector<F> r;
      if (which == 0) { VandermondeFFT<F> f(d); r = inverse ? f.fft_inv(v) : f.fft(v); }
      else { CooleyTukeyFFT<F> f(d); r = inverse ? f.fft_inv(v) : f.fft(v); }
      for (size_t i = 0; i < r.size(); i++) out[i] = r[i].v;
      *n_out = r.size();
      return 0;
    })
  } catch (const Panic&) {
    return 1;
  }
  return -1;
}

int oracle_mul_ntt(uint64_t M, uint64_t omega, size_t size, int which, const uint64_t* a, size_t la, const uint64_t* b,
                   size_t lb, uint64_t* out, size_t* n_out) {
  try {
    DISPATCH_M(M, {
      std::vector<F> va, vb;
      for (size_t i = 0; i < la; i++) va.push_back(F::from_u64(a[i]));
      for (size_t i = 0; i < lb; i++) vb.push_back(F::from_u64(b[i]));
      EvaluationDomainGenerator<F> d{F::from_u64(omega), size};
      std::vector<F> r;
      if (which == 0) { VandermondeFFT<F> f(d); r = mul_ntt<F>(f, va, vb); }
      else { CooleyTukeyFFT<F> f(d); r = mul_ntt<F>(f, va, vb); }
      for (size_t i = 0; i < r.size(); i++) out[i] = r[i].v;
      *n_out = r.size();
      return 0;
    })
  } catch (const Panic&) {
    return 1;
  }
  return -1;
}

// G1 points as (x, y, infinite) triples of u8.  Return 1 when the reference would panic.
int oracle_g1_add(const uint8_t p[3], const uint8_t q[3], uint8_t out[3]) {
  try {
    G1P a = g1f(p[0], p[1]); a.infinite = p[2] != 0;
    G1P b = g1f(q[0], q[1]); b.infinite = q[2] != 0;
    G1P r = a + b;
    out[0] = (uint8_t)r.x.v; out[1] = (uint8_t)r.y.v; out[2] = r.infinite;
    return 0;
  } catch (const Panic&) { return 1; }
}
int oracle_g1_mul(const uint8_t p[3], uint8_t k, uint8_t out[3]) {
  try {
    G1P a = g1f(p[0], p[1]); a.infinite = p[2] != 0;
    G1P r = a * f101(k);
    out[0] = (uint8_t)r.x.v; out[1] = (uint8_t)r.y.v; out[2] = r.infinite;
    return 0;
  } catch (const Panic&) { return 1; }
}
int oracle_g1_neg(const uint8_t p[3], uint8_t out[3]) {
  G1P a = g1f(p[0], p[1]); a.infinite = p[2] != 0;
  G1P r = -a;
  out[0] = (uint8_t)r.x.v; out[1] = (uint8_t)r.y.v; out[2] = r.infinite;
  return 0;
}
int oracle_g1_in_curve(const uint8_t p[3]) {
  G1P a = g1f(p[0], p[1]); a.infinite = p[2] != 0;
  return a.in_curve() ? 1 : 0;
}
int oracle_g2_add(const uint8_t p[2], const uint8_t q[2], uint8_t out[2]) {
  try { G2P r = g2f(p[0], p[1]) + g2f(q[0], q[1]); out[0] = (uint8_t)r.a.v; out[1] = (uint8_t)r.b.v; return 0; }
  catch (const Panic&) { return 1; }
}
int oracle_g2_mul(const uint8_t p[2], uint8_t k, uint8_t out[2]) {
  try { G2P r = g2f(p[0], p[1]) * f101(k); out[0] = (uint8_t)r.a.v; out[1] = (uint8_t)r.b.v; return 0; }
  catch (const Panic&) { return 1; }
}
int oracle_gt_mul(const uint8_t p[2], const uint8_t q[2], uint8_t out[2]) {
  GTP r = GTP::make(f101(p[0]), f101(p[1])) * GTP::make(f101(q[0]), f101(q[1]));
  out[0] = (uint8_t)r.a.v; out[1] = (uint8_t)r.b.v; return 0;
}
int oracle_gt_pow(const uint8_t p[2], uint64_t n, uint8_t out[2]) {
  GTP r = GTP::make(f101(p[0]), f101(p[1])).pow(n);
  out[0] = (uint8_t)r.a.v; out[1] = (uint8_t)r.b.v; return 0;
}
int oracle_gt_neg(const uint8_t p[2], uint8_t out[2]) {
  GTP r = -GTP::make(f101(p[0]), f101(p[1]));
  out[0] = (uint8_t)r.a.v; out[1] = (uint8_t)r.b.v; return 0;
}
int oracle_pairing(const uint8_t p[3], const uint8_t q[2], uint8_t out[2]) {
  try {
    G1P a = g1f(p[0], p[1]); a.infinite = p[2] != 0;
    GTP r = pairing(a, g2f(q[0], q[1]));
    out[0] = (uint8_t)r.a.v; out[1] = (uint8_t)r.b.v; return 0;
  } catch (const Panic&) { return 1; }
}
// Miller value before the final exponentiation (pairing_f(17, p, q)); for SURVEY.md §9 cross-checks
int oracle_miller(const uint8_t p[3], const uint8_t q[2], uint8_t out[2]) {
  try {
    G1P a = g1f(p[0], p[1]); a.infinite = p[2] != 0;
    GTP r = pairing_f(17, a, g2f(q[0], q[1]));
    out[0] = (uint8_t)r.a.v; out[1] = (uint8_t)r.b.v; return 0;
  } catch (const Panic&) { return 1; }
}

// ------------------------------------------------------------------------------------------------
// setup read-back
// ------------------------------------------------------------------------------------------------
// g1s: (srs_n+1) triples; g2: g2_1.a g2_1.b g2_s.a g2_s.b; consts: 8 triples q_m_s q_l_s q_r_s q_o_s q_c_s s1 s2 s3
int oracle_setup(const void* circuit, uint8_t s, uint32_t srs_n, uint8_t omega_pows, uint8_t* g1s, uint8_t g2[4],
                 uint8_t consts[24]) {
  auto st = make_setup((const circuit_desc*)circuit, s, srs_n, omega_pows);
  if (!st) return 1;
  for (size_t i = 0; i < st->plonk->srs.g1s.size(); i++) {
    const G1P& p = st->plonk->srs.g1s[i];
    g1s[3 * i] = (uint8_t)p.x.v; g1s[3 * i + 1] = (uint8_t)p.y.v; g1s[3 * i + 2] = p.infinite;
  }
  g2[0] = (uint8_t)st->plonk->srs.g2_1.a.v; g2[1] = (uint8_t)st->plonk->srs.g2_1.b.v;
  g2[2] = (uint8_t)st->plonk->srs.g2_s.a.v; g2[3] = (uint8_t)st->plonk->srs.g2_s.b.v;
  try {
    const Plonk& pl = *st->plonk;
    const Constrains& k = st->constraints;
    std::vector<F17> s1 = pl.copy_constraints_to_roots(k.c_a), s2 = pl.copy_constraints_to_roots(k.c_b),
                     s3 = pl.copy_constraints_to_roots(k.c_c);
    const std::vector<F17>* vecs[8] = {&k.q_m, &k.q_l, &k.q_r, &k.q_o, &k.q_c, &s1, &s2, &s3};
    for (int i = 0; i < 8; i++) {
      G1P p = pl.srs.eval_at_s(pl.interpolate_at_h(*vecs[i]));
      consts[3 * i] = (uint8_t)p.x.v; consts[3 * i + 1] = (uint8_t)p.y.v; consts[3 * i + 2] = p.infinite;
    }
  } catch (const Panic&) { return 1; }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// batched prove / verify in the wire layout of include/pbh_b200.h
// ------------------------------------------------------------------------------------------------
int oracle_prove_batch(const void* circuit, uint8_t s, uint32_t srs_n, uint8_t omega_pows, size_t n, const uint8_t* wit,
                       size_t wit_pitch, const uint8_t* rnd, size_t rand_pitch, const uint8_t* chal, size_t chal_pitch,
                       uint8_t* proof, size_t proof_pitch, uint8_t* status, int threads) {
  auto st = make_setup((const circuit_desc*)circuit, s, srs_n, omega_pows);
  if (!st) return -2;
  parallel_for(n, threads, [&](size_t lo, size_t hi) {
    for (size_t i = lo; i < hi; i++) {
      uint8_t w[12], r[9], c[5];
      for (int k = 0; k < 12; k++) w[k] = wit[k * wit_pitch + i];
      for (int k = 0; k < 9; k++) r[k] = rnd[k * rand_pitch + i];
      for (int k = 0; k < 5; k++) c[k] = chal[k * chal_pitch + i];
      for (int k = 0; k < 27; k++) proof[k * proof_pitch + i] = 0;
      Proof pr;
      int stt = prove_one(*st, w, r, c, pr);
      status[i] = (uint8_t)stt;
      if (stt == 0) store_proof(pr, proof, proof_pitch, i);
    }
  });
  return 0;
}

// ---- Fiat-Shamir variants: challenges derived from the transcript instead of passed in ----
int oracle_sha256(const uint8_t* data, size_t len, uint8_t out[32]) {
  Sha256 h; h.update(data, len); h.finish(out);
  return 0;
}
int oracle_fs_seed(const void* circuit, uint8_t s, uint32_t srs_n, uint8_t omega_pows, uint8_t out[32]) {
  auto st = make_setup((const circuit_desc*)circuit, s, srs_n, omega_pows);
  if (!st) return -2;
  fs_seed(*st, *(const circuit_desc*)circuit, omega_pows, out);
  return 0;
}
// chal_out (nullable): 6 planes alpha beta gamma z v u.  partial = 0: zero for items whose status != 0 (the product's
// contract); partial = 1: the challenges derived before the panic are kept (test aid).
int oracle_prove_fs_batch(const void* circuit, uint8_t s, uint32_t srs_n, uint8_t omega_pows, size_t n, const uint8_t* wit,
                          size_t wit_pitch, const uint8_t* rnd, size_t rand_pitch, uint8_t* proof, size_t proof_pitch,
                          uint8_t* status, uint8_t* chal_out, size_t chal_pitch, int partial, int threads) {
  auto st = make_setup((const circuit_desc*)circuit, s, srs_n, omega_pows);
  if (!st) return -2;
  uint8_t seed[32];
  fs_seed(*st, *(const circuit_desc*)circuit, omega_pows, seed);
  parallel_for(n, threads, [&](size_t lo, size_t hi) {
    for (size_t i = lo; i < hi; i++) {
      uint8_t w[12], r[9], d[6];
      for (int k = 0; k < 12; k++) w[k] = wit[k * wit_pitch + i];
      for (int k = 0; k < 9; k++) r[k] = rnd[k * rand_pitch + i];
      for (int k = 0; k < 27; k++) proof[k * proof_pitch + i] = 0;
      Proof pr;
      int stt = prove_one_fs(*st, seed, w, r, pr, d);
      status[i] = (uint8_t)stt;
      if (stt == 0) store_proof(pr, proof, proof_pitch, i);
      if (chal_out) for (int k = 0; k < 6; k++) chal_out[k * chal_pitch + i] = (stt == 0 || partial) ? d[k] : 0;
    }
  });
  return 0;
}

int oracle_verify_batch(const void* circuit, uint8_t s, uint32_t srs_n, uint8_t omega_pows, size_t n,
                        const uint8_t* proof, size_t proof_pitch, const uint8_t* chal, size_t chal_pitch,
                        const uint8_t* u, uint8_t* result, uint8_t* gt, size_t gt_pitch, int threads);

// The verifier replays the transcript over the proof bytes (each point as x, y, infinite, 0; evaluations as they are)
// and then runs Plonk::verify with the derived Challange and rand[0] = u.  Items with a coordinate byte >= 101 or a
// stray flag bit answer 0x20 and get zero challenges.
int oracle_verify_fs_batch(const void* circuit, uint8_t s, uint32_t srs_n, uint8_t omega_pows, size_t n, const uint8_t* proof,
                           size_t proof_pitch, uint8_t* result, uint8_t* chal_out, size_t chal_pitch, uint8_t* gt,
                           size_t gt_pitch, int threads) {
  auto st = make_setup((const circuit_desc*)circuit, s, srs_n, omega_pows);
  if (!st) return -2;
  uint8_t seed[32];
  fs_seed(*st, *(const circuit_desc*)circuit, omega_pows, seed);
  std::vector<uint8_t> chal(6 * n, 0);
  parallel_for(n, threads, [&](size_t lo, size_t hi) {
    for (size_t i = lo; i < hi; i++) {
      bool bad = false;
      for (int k = 0; k < 18; k++) bad |= proof[k * proof_pitch + i] >= 101;
      bad |= (proof[19 * proof_pitch + i] & 0xFE) != 0;
      if (bad) continue;
      G1P pt[9];
      for (int k = 0; k < 9; k++) pt[k] = get_point(proof, proof_pitch, i, k);
      F17 ev[7];
      for (int k = 0; k < 7; k++) ev[k].v = proof[(20 + k) * proof_pitch + i];
      FsTranscript tr(seed);
      F17 beta, gamma;
      tr.beta_gamma(pt[0], pt[1], pt[2], beta, gamma);
      tr.alpha(pt[3]);
      tr.zeta(pt[4], pt[5], pt[6]);
      tr.v(ev);
      tr.u(pt[7], pt[8]);
      for (int k = 0; k < 6; k++) chal[k * n + i] = tr.derived[k];
    }
  });
  int rc = oracle_verify_batch(circuit, s, srs_n, omega_pows, n, proof, proof_pitch, chal.data(), n, chal.data() + 5 * n, result, gt,
                               gt_pitch, threads);
  if (chal_out) for (int k = 0; k < 6; k++) for (size_t i = 0; i < n; i++) chal_out[k * chal_pitch + i] = chal[k * n + i];
  return rc;
}

int oracle_verify_batch(const void* circuit, uint8_t s, uint32_t srs_n, uint8_t omega_pows, size_t n,
                        const uint8_t* proof, size_t proof_pitch, const uint8_t* chal, size_t chal_pitch,
                        const uint8_t* u, uint8_t* result, uint8_t* gt, size_t gt_pitch, int threads) {
  auto st = make_setup((const circuit_desc*)circuit, s, srs_n, omega_pows);
  if (!st) return -2;
  parallel_for(n, threads, [&](size_t lo, size_t hi) {
    for (size_t i = lo; i < hi; i++) {
      if (gt) for (int k = 0; k < 4; k++) gt[k * gt_pitch + i] = 0;
      bool bad = false;
      for (int k = 0; k < 18; k++) bad |= proof[k * proof_pitch + i] >= 101;
      bad |= (proof[19 * proof_pitch + i] & 0xFE) != 0;
      for (int k = 0; k < 5; k++) bad |= chal[k * chal_pitch + i] >= 17;
      bad |= u[i] >= 17;
      if (bad) { result[i] = 0x20; continue; }
      Proof pr;
      G1P* pts[9] = {&pr.a_s, &pr.b_s, &pr.c_s, &pr.z_s, &pr.t_lo_s, &pr.t_mid_s, &pr.t_hi_s, &pr.w_z_s, &pr.w_z_omega_s};
      for (int k = 0; k < 9; k++) *pts[k] = get_point(proof, proof_pitch, i, k);
      F17* ev[7] = {&pr.a_z, &pr.b_z, &pr.c_z, &pr.s_sigma_1_z, &pr.s_sigma_2_z, &pr.r_z, &pr.z_omega_z};
      // raw bytes: a value >= 17 models a U64Field that fails in_field() (src/plonk.rs:538-547)
      for (int k = 0; k < 7; k++) ev[k]->v = proof[(20 + k) * proof_pitch + i];
      Challange ch{f17(chal[0 * chal_pitch + i]), f17(chal[1 * chal_pitch + i]), f17(chal[2 * chal_pitch + i]),
                   f17(chal[3 * chal_pitch + i]), f17(chal[4 * chal_pitch + i])};
      F17 rr[1] = {f17(u[i])};
      VerifyTrace tr;
      try {
        bool ok = st->plonk->verify(st->constraints, pr, ch, rr, &tr);
        if (tr.reason == 1) result[i] = 0x02;
        else if (tr.reason == 2) result[i] = 0x04;
        else {
          result[i] = ok ? 0x01 : 0x00;
          if (gt) {
            gt[0 * gt_pitch + i] = (uint8_t)tr.e_1.a.v; gt[1 * gt_pitch + i] = (uint8_t)tr.e_1.b.v;
            gt[2 * gt_pitch + i] = (uint8_t)tr.e_2.a.v; gt[3 * gt_pitch + i] = (uint8_t)tr.e_2.b.v;
          }
        }
      } catch (const Panic& p) {
        result[i] = p.site == SITE_VERIFY_ZH0 ? 0x10 : 0x40;
      }
    }
  });
  return 0;
}

// golden-run intermediates for SURVEY.md §9: returns normalised coefficient vectors, each prefixed by its
// length, in the order f_a f_b f_c q_m q_l q_r q_o q_c s1 s2 s3 l1 a b c acc_x z z_omega numerator t r w_z w_zw
int oracle_prove_trace(const void* circuit, uint8_t s, uint32_t srs_n, uint8_t omega_pows, const uint8_t w[12],
                       const uint8_t r[9], const uint8_t c[5], uint8_t* out, size_t out_cap, size_t* out_len) {
  auto st = make_setup((const circuit_desc*)circuit, s, srs_n, omega_pows);
  if (!st) return -2;
  Assigments as;
  for (int k = 0; k < 4; k++) { as.a.push_back(f17(w[k])); as.b.push_back(f17(w[4 + k])); as.c.push_back(f17(w[8 + k])); }
  F17 rand[9];
  for (int k = 0; k < 9; k++) rand[k] = f17(r[k]);
  Challange ch{f17(c[0]), f17(c[1]), f17(c[2]), f17(c[3]), f17(c[4])};
  ProveTrace tr;
  int status = 0;
  try { st->plonk->prove(st->constraints, as, ch, rand, &tr); } catch (const Panic& p) { status = p.site; }
  const Poly<F17>* polys[23] = {&tr.f_a, &tr.f_b, &tr.f_c, &tr.q_m, &tr.q_l, &tr.q_r, &tr.q_o, &tr.q_c, &tr.s1, &tr.s2,
                                &tr.s3, &tr.l1, &tr.a, &tr.b, &tr.c, &tr.acc_x, &tr.z, &tr.z_omega, &tr.numerator,
                                &tr.t, &tr.r, &tr.w_z, &tr.w_z_omega};
  size_t pos = 0;
  for (auto* p : polys) {
    if (pos + 1 + p->c.size() > out_cap) return -1;
    out[pos++] = (uint8_t)p->c.size();
    for (auto& x : p->c) out[pos++] = (uint8_t)x.v;
  }
  *out_len = pos;
  return status;
}

// ------------------------------------------------------------------------------------------------
// sweep operations in plane layout (same signatures as the product's, minus the context)
// ------------------------------------------------------------------------------------------------
int oracle_intt4_batch(size_t n, const uint8_t* evals, size_t in_pitch, uint8_t* coeffs, size_t out_pitch) {
  Plonk pl(SRS::create(f101(2), 6), f17(4));
  for (size_t i = 0; i < n; i++) {
    std::vector<F17> v;
    for (int k = 0; k < 4; k++) v.push_back(f17(evals[k * in_pitch + i]));
    Poly<F17> p = pl.interpolate_at_h(v);
    for (int k = 0; k < 4; k++) coeffs[k * out_pitch + i] = k < (int)p.c.size() ? (uint8_t)p.c[k].v : 0;
  }
  return 0;
}
int oracle_ntt4_batch(size_t n, const uint8_t* coeffs, size_t in_pitch, uint8_t* evals, size_t out_pitch) {
  CooleyTukeyFFT<F17> f(EvaluationDomainGenerator<F17>{f17(4), 4});
  for (size_t i = 0; i < n; i++) {
    std::vector<F17> v;
    for (int k = 0; k < 4; k++) v.push_back(f17(coeffs[k * in_pitch + i]));
    std::vector<F17> r = f.fft(v);
    for (int k = 0; k < 4; k++) evals[k * out_pitch + i] = (uint8_t)r[k].v;
  }
  return 0;
}
int oracle_poly_mul_batch(size_t n, uint32_t la, uint32_t lb, const uint8_t* a, size_t a_pitch, const uint8_t* b,
                          size_t b_pitch, uint8_t* out, size_t out_pitch) {
  for (size_t i = 0; i < n; i++) {
    std::vector<F17> va, vb;
    for (uint32_t k = 0; k < la; k++) va.push_back(f17(a[k * a_pitch + i]));
    for (uint32_t k = 0; k < lb; k++) vb.push_back(f17(b[k * b_pitch + i]));
    Poly<F17> p = Poly<F17>(va) * Poly<F17>(vb);
    for (uint32_t k = 0; k < la + lb - 1; k++) out[k * out_pitch + i] = k < p.c.size() ? (uint8_t)p.c[k].v : 0;
  }
  return 0;
}
int oracle_poly_add_batch(size_t n, uint32_t len, int subtract, const uint8_t* a, size_t a_pitch, const uint8_t* b,
                          size_t b_pitch, uint8_t* out, size_t out_pitch) {
  for (size_t i = 0; i < n; i++) {
    // equal-length raw vectors (no normalisation before the operation, so Q1 cannot trigger)
    std::vector<F17> va, vb;
    for (uint32_t k = 0; k < len; k++) { va.push_back(f17(a[k * a_pitch + i])); vb.push_back(f17(b[k * b_pitch + i])); }
    Poly<F17> p = Poly<F17>::raw(va), q = Poly<F17>::raw(vb);
    if (subtract) p -= q; else p += q;
    for (uint32_t k = 0; k < len; k++) out[k * out_pitch + i] = k < p.c.size() ? (uint8_t)p.c[k].v : 0;
  }
  return 0;
}
int oracle_poly_div_zh_batch(size_t n, const uint8_t* p, size_t p_pitch, uint8_t* q, size_t q_pitch, uint8_t* r,
                             size_t r_pitch) {
  Poly<F17> zh = Poly<F17>::z({f17(1), f17(4), f17(16), f17(13)});
  for (size_t i = 0; i < n; i++) {
    std::vector<F17> v;
    for (int k = 0; k < 22; k++) v.push_back(f17(p[k * p_pitch + i]));
    auto qr = poly_div(Poly<F17>(v), zh);
    for (int k = 0; k < 18; k++) q[k * q_pitch + i] = k < (int)qr.first.c.size() ? (uint8_t)qr.first.c[k].v : 0;
    for (int k = 0; k < 4; k++) r[k * r_pitch + i] = k < (int)qr.second.c.size() ? (uint8_t)qr.second.c[k].v : 0;
  }
  return 0;
}
// in: len coefficient planes then one scalar plane
int oracle_poly_scale_batch(size_t n, uint32_t len, const uint8_t* in, size_t in_pitch, uint8_t* out, size_t out_pitch) {
  for (size_t i = 0; i < n; i++) {
    std::vector<F17> v;
    for (uint32_t k = 0; k < len; k++) v.push_back(f17(in[k * in_pitch + i]));
    Poly<F17> p = Poly<F17>(v) * f17(in[len * in_pitch + i]);                       // src/poly.rs:220-228 (Q15)
    for (uint32_t k = 0; k < len; k++) out[k * out_pitch + i] = k < p.c.size() ? (uint8_t)p.c[k].v : 0;
  }
  return 0;
}
// in: len coefficient planes then the point x; out: one plane
int oracle_poly_eval_batch(size_t n, uint32_t len, const uint8_t* in, size_t in_pitch, uint8_t* out) {
  for (size_t i = 0; i < n; i++) {
    std::vector<F17> v;
    for (uint32_t k = 0; k < len; k++) v.push_back(f17(in[k * in_pitch + i]));
    out[i] = (uint8_t)Poly<F17>(v).eval(f17(in[len * in_pitch + i])).v;             // src/poly.rs:71-79
  }
  return 0;
}
// in: len coefficient planes then c; out: len-1 quotient planes of p / (x - c), then the remainder plane
int oracle_poly_div_linear_batch(size_t n, uint32_t len, const uint8_t* in, size_t in_pitch, uint8_t* out, size_t out_pitch) {
  for (size_t i = 0; i < n; i++) {
    std::vector<F17> v;
    for (uint32_t k = 0; k < len; k++) v.push_back(f17(in[k * in_pitch + i]));
    F17 c = f17(in[len * in_pitch + i]);
    auto qr = poly_div(Poly<F17>(v), Poly<F17>({-c, F17::one()}));                  // src/poly.rs:230-247, src/plonk.rs:437-442
    for (uint32_t k = 0; k + 1 < len; k++) out[k * out_pitch + i] = k < qr.first.c.size() ? (uint8_t)qr.first.c[k].v : 0;
    out[(len - 1) * out_pitch + i] = qr.second.c.empty() ? 0 : (uint8_t)qr.second.c[0].v;
  }
  return 0;
}
// mul_ntt (src/fft.rs:109-132) with CooleyTurkey over F_M: a (la planes), b (lb planes), la + lb == size; out: size planes
int oracle_mul_ntt_batch(size_t n, uint64_t M, uint64_t omega, uint32_t size, uint32_t la, uint32_t lb, const uint16_t* a,
                         size_t a_pitch, const uint16_t* b, size_t b_pitch, uint16_t* out, size_t out_pitch) {
  try {
    DISPATCH_M(M, {
      EvaluationDomainGenerator<F> d{F::from_u64(omega), size};
      CooleyTukeyFFT<F> f(d);
      for (size_t i = 0; i < n; i++) {
        std::vector<F> va, vb;
        for (uint32_t k = 0; k < la; k++) va.push_back(F::from_u64(a[k * a_pitch + i]));
        for (uint32_t k = 0; k < lb; k++) vb.push_back(F::from_u64(b[k * b_pitch + i]));
        std::vector<F> r = mul_ntt<F>(f, va, vb);
        for (uint32_t k = 0; k < size; k++) out[k * out_pitch + i] = k < r.size() ? (uint16_t)r[k].v : 0;
      }
      return 0;
    })
  } catch (const Panic&) {
    return 1;
  }
  return -1;
}
int oracle_g1_smul_batch(size_t n, const uint8_t* in, size_t in_pitch, uint8_t* out, size_t out_pitch) {
  for (size_t i = 0; i < n; i++) {
    uint8_t p[3] = {in[i], in[in_pitch + i], in[2 * in_pitch + i]}, o[3];
    if (oracle_g1_mul(p, in[3 * in_pitch + i], o)) { o[0] = o[1] = 0; o[2] = 0xFF; }
    out[i] = o[0]; out[out_pitch + i] = o[1]; out[2 * out_pitch + i] = o[2];
  }
  return 0;
}
int oracle_g1_add_batch(size_t n, const uint8_t* in, size_t in_pitch, uint8_t* out, size_t out_pitch) {
  for (size_t i = 0; i < n; i++) {
    uint8_t p[3] = {in[i], in[in_pitch + i], in[2 * in_pitch + i]};
    uint8_t q[3] = {in[3 * in_pitch + i], in[4 * in_pitch + i], in[5 * in_pitch + i]}, o[3];
    if (oracle_g1_add(p, q, o)) { o[0] = o[1] = 0; o[2] = 0xFF; }
    out[i] = o[0]; out[out_pitch + i] = o[1]; out[2 * out_pitch + i] = o[2];
  }
  return 0;
}
int oracle_kzg_commit_batch(uint8_t s, uint32_t srs_n, size_t n, const uint8_t* coeffs, size_t in_pitch, uint8_t* out,
                            size_t out_pitch) {
  SRS srs;
  try { srs = SRS::create(f101(s), srs_n); } catch (const Panic&) { return -2; }
  for (size_t i = 0; i < n; i++) {
    std::vector<F17> v;
    for (int k = 0; k < 7; k++) v.push_back(f17(coeffs[k * in_pitch + i]));
    uint8_t o[3];
    try {
      G1P p = srs.eval_at_s(Poly<F17>(v));
      o[0] = (uint8_t)p.x.v; o[1] = (uint8_t)p.y.v; o[2] = p.infinite;
    } catch (const Panic&) { o[0] = o[1] = 0; o[2] = 0xFF; }
    out[i] = o[0]; out[out_pitch + i] = o[1]; out[2 * out_pitch + i] = o[2];
  }
  return 0;
}
int oracle_pairing_batch(size_t n, const uint8_t* in, size_t in_pitch, uint8_t* out, size_t out_pitch) {
  for (size_t i = 0; i < n; i++) {
    uint8_t p[3] = {in[i], in[in_pitch + i], in[2 * in_pitch + i]};
    uint8_t q[2] = {in[3 * in_pitch + i], in[4 * in_pitch + i]}, o[2];
    if (oracle_pairing(p, q, o)) { o[0] = o[1] = 0xFF; }
    out[i] = o[0]; out[out_pitch + i] = o[1];
  }
  return 0;
}

// ------------------------------------------------------------------------------------------------
// synthetic inputs, digests
// ------------------------------------------------------------------------------------------------
int oracle_generate_inputs(const void* circuit, uint8_t s, uint32_t srs_n, uint8_t omega_pows, size_t n,
                           uint64_t first_index, uint64_t seed, int dist, uint8_t* wit, size_t wit_pitch, uint8_t* rnd,
                           size_t rand_pitch, uint8_t* chal, size_t chal_pitch, uint8_t* u, uint8_t* attempt,
                           int threads) {
  auto st = make_setup((const circuit_desc*)circuit, s, srs_n, omega_pows);
  if (!st) return -2;
  parallel_for(n, threads, [&](size_t lo, size_t hi) {
    for (size_t i = lo; i < hi; i++) {
      uint8_t w[12], r[9], c[5], uu = 0;
      uint32_t k = 0;
      for (;; k++) {
        // past PBH_GEN_MAX_ATTEMPTS (include/pbh_b200.h): attempt 0's draw, reported as attempt 255
        sample_attempt(seed, first_index + i, k < kGenMaxAttempts ? k : 0, w, r, c, uu);
        if (dist == 0 || k == kGenMaxAttempts) break;
        Proof pr;
        if (prove_one(*st, w, r, c, pr) != 0) continue;
        const G1P* pts[9] = {&pr.a_s, &pr.b_s, &pr.c_s, &pr.z_s, &pr.t_lo_s, &pr.t_mid_s, &pr.t_hi_s, &pr.w_z_s, &pr.w_z_omega_s};
        bool any_inf = false;
        for (auto* p : pts) any_inf |= p->infinite;
        if (any_inf) continue;                         // verify would return false at in_curve (Q9)
        if (f17(c[3]).pow(4) == F17::one()) continue;  // verify would panic on Z_H(z) = 0 (Q4)
        break;
      }
      for (int j = 0; j < 12; j++) wit[j * wit_pitch + i] = w[j];
      for (int j = 0; j < 9; j++) rnd[j * rand_pitch + i] = r[j];
      for (int j = 0; j < 5; j++) chal[j * chal_pitch + i] = c[j];
      u[i] = uu;
      if (attempt) attempt[i] = (uint8_t)std::min<uint32_t>(k, 255);
    }
  });
  return 0;
}

static inline uint32_t rotl32(uint32_t x, int r) { return (x << r) | (x >> (32 - r)); }
static inline uint32_t fmix32(uint32_t h) { h ^= h >> 16; h *= 0x85EBCA6Bu; h ^= h >> 13; h *= 0xC2B2AE35u; h ^= h >> 16; return h; }
uint64_t oracle_digest(size_t n, uint64_t first_index, uint32_t planes, const uint8_t* data, size_t pitch) {
  uint64_t acc = 0;
  for (size_t i = 0; i < n; i++) {
    uint64_t idx = first_index + i;
    uint32_t a = (uint32_t)idx * 0x9E3779B1u + planes, b = (uint32_t)(idx >> 32) * 0x85EBCA77u + 0x27D4EB2Fu;
    for (uint32_t k = 0; k < planes; k += 4) {
      uint32_t wv = 0;
      for (uint32_t bb = 0; bb < 4 && k + bb < planes; bb++) wv |= (uint32_t)data[(size_t)(k + bb) * pitch + i] << (8 * bb);
      a = rotl32((a ^ wv) * 0xCC9E2D51u, 15);
      b = rotl32((b + wv) * 0x1B873593u, 13) ^ a;
    }
    acc += ((uint64_t)fmix32(a ^ rotl32(b, 16)) << 32) | fmix32(b + a);
  }
  return acc;
}
int oracle_pack_verdicts(size_t n, const uint8_t* result, uint8_t* bitmap) {
  std::memset(bitmap, 0, (n + 7) / 8);
  for (size_t i = 0; i < n; i++) if (result[i] & 1) bitmap[i / 8] |= (uint8_t)(1u << (i % 8));
  return 0;
}

int oracle_hardware_threads() { return (int)std::thread::hardware_concurrency(); }

}  // extern "C"
