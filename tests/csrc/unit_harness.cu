// unit_harness.cu -- test-only shared library (not part of libfibb200.so): evaluates the device
// functions of the arithmetic layer (fib_math.cuh) and the models' voltage-only intermediates
// elementwise over host arrays, so that tests/test_gpu_math_layer.py can compare each of them with a
// float64 reference on its own.  It includes the product headers unchanged and is compiled with the
// library's nvcc flags (fib_tf_b200.build.NVCC_FLAGS, -fmad=false), so every function rounds here as it
// does in the step kernels.
//
// Every entry point comes in two flavours: packed == 0 evaluates T = float, one element per thread;
// packed == 1 evaluates T = f2, elements 2i and 2i+1 are the two lanes of thread i (so the caller
// chooses which inputs share a pair; n must then be even).  Threads are numbered in array order, 128
// to a block: the 32 consecutive threads of a warp see consecutive elements (or pairs).
#include <stdio.h>

#include "model_br.cuh"
#include "model_court.cuh"
#include "model_fenton.cuh"

using namespace fib;

namespace {

enum Unary {
  U_EXP = 0, U_EXPM1, U_EXPM1_NEG, U_RCP, U_LOG, U_SQRT, U_HALF_1P_TANH, U_NEG, U_ABS
};
enum Binary { B_ADD = 0, B_SUB, B_MUL, B_DIV, B_MIN, B_MAX, B_SEL_LT, B_SEL_GT };

constexpr int kBlock = 128;

template <class T> __device__ __forceinline__ T load(const float* p, size_t i) {
  return from_lanes<T>(p + i * Lanes<T>::N);
}
template <class T> __device__ __forceinline__ void store(float* p, size_t i, T v) {
  to_lanes(v, p + i * Lanes<T>::N);
}
__device__ __forceinline__ size_t thread_index() { return (size_t)blockIdx.x * blockDim.x + threadIdx.x; }

template <class T>
__global__ void unary_kernel(int fn, const float* __restrict__ x, size_t m, float* __restrict__ out) {
  const size_t i = thread_index();
  if (i >= m) return;
  const T a = load<T>(x, i);
  T r = a;
  switch (fn) {
    case U_EXP: r = m_exp(a); break;
    case U_EXPM1: r = m_expm1(a); break;
    case U_EXPM1_NEG: r = m_expm1_neg(a); break;
    case U_RCP: r = m_rcp(a); break;
    case U_LOG: r = m_log(a); break;
    case U_SQRT: r = m_sqrt(a); break;
    case U_HALF_1P_TANH: r = m_half_1p_tanh(a); break;
    case U_NEG: r = -a; break;
    case U_ABS: r = vabs(a); break;
  }
  store(out, i, r);
}

template <class T>
__global__ void binary_kernel(int fn, const float* __restrict__ x, const float* __restrict__ y, size_t m,
                              float* __restrict__ out) {
  const size_t i = thread_index();
  if (i >= m) return;
  const T a = load<T>(x, i), b = load<T>(y, i);
  T r = a;
  switch (fn) {
    case B_ADD: r = a + b; break;
    case B_SUB: r = a - b; break;
    case B_MUL: r = a * b; break;
    case B_DIV: r = m_div(a, b); break;
    case B_MIN: r = vmin(a, b); break;
    case B_MAX: r = vmax(a, b); break;
    case B_SEL_LT: r = sel(lt(a, b), a, b); break;
    case B_SEL_GT: r = sel(gt(a, b), a, b); break;
  }
  store(out, i, r);
}

template <class T>
__global__ void fma_kernel(const float* __restrict__ x, const float* __restrict__ y, const float* __restrict__ z,
                           size_t m, float* __restrict__ out) {
  const size_t i = thread_index();
  if (i >= m) return;
  store(out, i, vfma(load<T>(x, i), load<T>(y, i), load<T>(z, i)));
}

template <class T>
__global__ void exp_affine_kernel(const float* __restrict__ x, size_t m, float c, float add, float* __restrict__ out) {
  const size_t i = thread_index();
  if (i >= m) return;
  store(out, i, m_exp_affine(load<T>(x, i), c, add));
}

template <bool US, bool RATES, class T>
__global__ void court_inter_kernel(const float* __restrict__ v, size_t m, float* __restrict__ out) {
  const size_t i = thread_index();
  if (i >= m) return;
  T q[kInterCols];
  court_inter_dev<US, RATES, T>(load<T>(v, i), q);
  constexpr int L = Lanes<T>::N;
  for (int l = 0; l < L; ++l)
    for (int k = 0; k < kInterCols; ++k) out[(i * L + l) * kInterCols + k] = lane(q[k], l);
}

template <class T>
__global__ void rush_larsen_kernel(const float* __restrict__ g, const float* __restrict__ gi,
                                   const float* __restrict__ tau, size_t m, float neg_dt, float* __restrict__ out) {
  const size_t i = thread_index();
  if (i >= m) return;
  store(out, i, rush_larsen(load<T>(g, i), load<T>(gi, i), load<T>(tau, i), neg_dt));
}

// one gate update of the exact BR gates, as BeelerReuter<0, true>::cell runs it; s and out are
// [n][7] in the model's order (C, M, H, J, D, F, XI)
template <class T>
__global__ void br_gates_kernel(const float* __restrict__ v, const float* __restrict__ s_in, size_t m, float neg_dt,
                                float neg_dt_slow, float* __restrict__ out) {
  const size_t i = thread_index();
  if (i >= m) return;
  constexpr int L = Lanes<T>::N;
  float lanes[L];
  T s[7];
  for (int k = 0; k < 7; ++k) {
    for (int l = 0; l < L; ++l) lanes[l] = s_in[(i * L + l) * 7 + k];
    s[k] = from_lanes<T>(lanes);
  }
  const T V0 = load<T>(v, i);
  const T k = m_exp(T(0.04f) * V0);
  const T rk = m_rcp(k);
  br_gates_exact<true>(V0, rk, s, neg_dt, neg_dt_slow);
  for (int k2 = 0; k2 < 7; ++k2)
    for (int l = 0; l < L; ++l) out[(i * L + l) * 7 + k2] = lane(s[k2], l);
}

// the readable statement of the exact gates: out [n][12] = (inf, rate) of gates 0..5 (xi m h j d f)
__global__ void br_inf_rate_kernel(const float* __restrict__ v, size_t m, float* __restrict__ out) {
  const size_t i = thread_index();
  if (i >= m) return;
  float* o = out + i * 12;
  br_inf_rate_exact<0>(v[i], o[0], o[1]);
  br_inf_rate_exact<1>(v[i], o[2], o[3]);
  br_inf_rate_exact<2>(v[i], o[4], o[5]);
  br_inf_rate_exact<3>(v[i], o[6], o[7]);
  br_inf_rate_exact<4>(v[i], o[8], o[9]);
  br_inf_rate_exact<5>(v[i], o[10], o[11]);
}

struct Poly { float c[9]; };   // a kernel parameter, as BeelerReuter::Params::poly is

template <class T>
__global__ void br_poly8_kernel(Poly p, const float* __restrict__ x, size_t m, float* __restrict__ out) {
  const size_t i = thread_index();
  if (i >= m) return;
  store(out, i, br_poly8(p.c, load<T>(x, i)));
}

// device buffers freed on every return path
struct Buf {
  float* p = nullptr;
  ~Buf() { cudaFree(p); }
};

int report(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return 0;
  fprintf(stderr, "unit_harness: %s: %s\n", what, cudaGetErrorString(e));
  return 1;
}
#define UT_CHECK(x) do { if (report((x), #x)) return 1; } while (0)

int upload(Buf& b, const float* host, size_t n) {
  UT_CHECK(cudaMalloc(&b.p, n * sizeof(float)));
  UT_CHECK(cudaMemcpy(b.p, host, n * sizeof(float), cudaMemcpyHostToDevice));
  return 0;
}
int download(float* host, const Buf& b, size_t n) {
  UT_CHECK(cudaGetLastError());
  UT_CHECK(cudaDeviceSynchronize());
  UT_CHECK(cudaMemcpy(host, b.p, n * sizeof(float), cudaMemcpyDeviceToHost));
  return 0;
}
// threads for n elements; 0 when a packed call has an odd n (caller error)
size_t threads(int packed, size_t n) { return packed ? ((n & 1) ? 0 : n / 2) : n; }
unsigned blocks(size_t m) { return (unsigned)((m + kBlock - 1) / kBlock); }

}  // namespace

#define UT_ARGS(m)                                         \
  if (n == 0) return 0;                                    \
  const size_t m = threads(packed, n);                     \
  if (m == 0) return 2;

extern "C" {

int ut_unary(int fn, int packed, const float* x, size_t n, float* out) {
  UT_ARGS(m)
  Buf a, o;
  if (upload(a, x, n)) return 1;
  UT_CHECK(cudaMalloc(&o.p, n * sizeof(float)));
  if (packed) unary_kernel<f2><<<blocks(m), kBlock>>>(fn, a.p, m, o.p);
  else unary_kernel<float><<<blocks(m), kBlock>>>(fn, a.p, m, o.p);
  return download(out, o, n);
}

int ut_binary(int fn, int packed, const float* x, const float* y, size_t n, float* out) {
  UT_ARGS(m)
  Buf a, b, o;
  if (upload(a, x, n) || upload(b, y, n)) return 1;
  UT_CHECK(cudaMalloc(&o.p, n * sizeof(float)));
  if (packed) binary_kernel<f2><<<blocks(m), kBlock>>>(fn, a.p, b.p, m, o.p);
  else binary_kernel<float><<<blocks(m), kBlock>>>(fn, a.p, b.p, m, o.p);
  return download(out, o, n);
}

int ut_fma(int packed, const float* x, const float* y, const float* z, size_t n, float* out) {
  UT_ARGS(m)
  Buf a, b, c, o;
  if (upload(a, x, n) || upload(b, y, n) || upload(c, z, n)) return 1;
  UT_CHECK(cudaMalloc(&o.p, n * sizeof(float)));
  if (packed) fma_kernel<f2><<<blocks(m), kBlock>>>(a.p, b.p, c.p, m, o.p);
  else fma_kernel<float><<<blocks(m), kBlock>>>(a.p, b.p, c.p, m, o.p);
  return download(out, o, n);
}

int ut_exp_affine(int packed, const float* x, size_t n, float c, float add, float* out) {
  UT_ARGS(m)
  Buf a, o;
  if (upload(a, x, n)) return 1;
  UT_CHECK(cudaMalloc(&o.p, n * sizeof(float)));
  if (packed) exp_affine_kernel<f2><<<blocks(m), kBlock>>>(a.p, m, c, add, o.p);
  else exp_affine_kernel<float><<<blocks(m), kBlock>>>(a.p, m, c, add, o.p);
  return download(out, o, n);
}

// out [n][32] in the CourtQ order (fib_tf_b200._capi.INTER_NAMES)
int ut_court_inter(int us, int rates, int packed, const float* v, size_t n, float* out) {
  UT_ARGS(m)
  Buf a, o;
  if (upload(a, v, n)) return 1;
  UT_CHECK(cudaMalloc(&o.p, n * kInterCols * sizeof(float)));
  const unsigned g = blocks(m);
  switch ((us ? 4 : 0) | (rates ? 2 : 0) | (packed ? 1 : 0)) {
    case 0: court_inter_kernel<false, false, float><<<g, kBlock>>>(a.p, m, o.p); break;
    case 1: court_inter_kernel<false, false, f2><<<g, kBlock>>>(a.p, m, o.p); break;
    case 2: court_inter_kernel<false, true, float><<<g, kBlock>>>(a.p, m, o.p); break;
    case 3: court_inter_kernel<false, true, f2><<<g, kBlock>>>(a.p, m, o.p); break;
    case 4: court_inter_kernel<true, false, float><<<g, kBlock>>>(a.p, m, o.p); break;
    case 5: court_inter_kernel<true, false, f2><<<g, kBlock>>>(a.p, m, o.p); break;
    case 6: court_inter_kernel<true, true, float><<<g, kBlock>>>(a.p, m, o.p); break;
    case 7: court_inter_kernel<true, true, f2><<<g, kBlock>>>(a.p, m, o.p); break;
  }
  return download(out, o, n * kInterCols);
}

int ut_rush_larsen(int packed, const float* g, const float* g_inf, const float* tau, size_t n, float neg_dt,
                   float* out) {
  UT_ARGS(m)
  Buf a, b, c, o;
  if (upload(a, g, n) || upload(b, g_inf, n) || upload(c, tau, n)) return 1;
  UT_CHECK(cudaMalloc(&o.p, n * sizeof(float)));
  if (packed) rush_larsen_kernel<f2><<<blocks(m), kBlock>>>(a.p, b.p, c.p, m, neg_dt, o.p);
  else rush_larsen_kernel<float><<<blocks(m), kBlock>>>(a.p, b.p, c.p, m, neg_dt, o.p);
  return download(out, o, n);
}

int ut_br_gates_exact(int packed, const float* v, const float* s, size_t n, float neg_dt, float neg_dt_slow,
                      float* out) {
  UT_ARGS(m)
  Buf a, b, o;
  if (upload(a, v, n) || upload(b, s, n * 7)) return 1;
  UT_CHECK(cudaMalloc(&o.p, n * 7 * sizeof(float)));
  if (packed) br_gates_kernel<f2><<<blocks(m), kBlock>>>(a.p, b.p, m, neg_dt, neg_dt_slow, o.p);
  else br_gates_kernel<float><<<blocks(m), kBlock>>>(a.p, b.p, m, neg_dt, neg_dt_slow, o.p);
  return download(out, o, n * 7);
}

int ut_br_inf_rate_exact(const float* v, size_t n, float* out) {
  const int packed = 0;
  UT_ARGS(m)
  Buf a, o;
  if (upload(a, v, n)) return 1;
  UT_CHECK(cudaMalloc(&o.p, n * 12 * sizeof(float)));
  br_inf_rate_kernel<<<blocks(m), kBlock>>>(a.p, m, o.p);
  return download(out, o, n * 12);
}

int ut_br_poly8(int packed, const float* c9, const float* x, size_t n, float* out) {
  UT_ARGS(m)
  Poly p;
  for (int i = 0; i < 9; ++i) p.c[i] = c9[i];
  Buf a, o;
  if (upload(a, x, n)) return 1;
  UT_CHECK(cudaMalloc(&o.p, n * sizeof(float)));
  if (packed) br_poly8_kernel<f2><<<blocks(m), kBlock>>>(p, a.p, m, o.p);
  else br_poly8_kernel<float><<<blocks(m), kBlock>>>(p, a.p, m, o.p);
  return download(out, o, n);
}

}  // extern "C"
