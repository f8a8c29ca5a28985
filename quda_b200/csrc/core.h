// Site-level building blocks of the B200 Wilson/clover Dslash engine: native field accessors,
// gauge reconstruction, spin projection, SU(3) algebra, checkerboard index math.
//
// Everything here is `B2_HD` (host + device) and free of CUDA-only constructs so that the very same
// site code can be compiled by g++ into the test-only "host twin" (tests/hosttwin/) and checked
// against the CPU oracle without a GPU.  The product only ever runs it inside CUDA kernels.
//
// Layout conventions follow the reference's native ("FloatN") orders so that fields produced by /
// handed to QUDA can be consumed unchanged (citations: /root/reference/include/...):
//   spinor  color_spinor_field_order.h:1191-1300   real r=(spin*3+colour)*2+reim, plane r/N, lane r%N,
//                                                  element (plane*volumeCB + x_cb)*N + lane ; N = 2 (fp64), 4 (fp32), 8 (half)
//                                                  half: int16 * per-site float norm, norm array after the 24*volumeCB shorts
//   gauge   gauge_field_order.h:1516-1588,2369-2443 element ((dir*M + i)*stride + x_cb)*N + lane, stride = volumeCB + pad,
//                                                  parity offset Bytes/2; ghost links of dim d at x_cb = volumeCB + face_idx
//   recon   gauge_field_order.h:964-1005 (18), :1071-1141 (12), :1267-1413 (8), timeBoundary :1019-1049
//   project color_spinor.h:290-392, reconstruct :693-812 (UKQCD / non-relativistic basis, no factor 1/2)
//   index   index_helper.cuh:250-302
#pragma once

#include <cmath>
#include <cstddef>
#include <cstdint>
#include <cstring>
#include <type_traits>
#include <utility>

#if defined(__CUDACC__)
#define B2_HD __host__ __device__ __forceinline__
#define B2_D __device__ __forceinline__
#else
#define B2_HD inline
#define B2_D inline
#endif

namespace b200
{

  // ------------------------------------------------------------------ small vector types (16-byte moves)
  struct alignas(16) f4 { float x, y, z, w; };
  struct alignas(16) d2 { double x, y; };
  struct alignas(8) f2 { float x, y; };
  struct alignas(16) s8 { short v[8]; };
  struct alignas(8) s4 { short v[4]; };
  struct alignas(4) s2 { short v[2]; };

  // Global-memory access policy hooks.  On the device these become cache-hinted PTX; on the host plain loads.
  // STREAM: read-once data (gauge links, clover) -- do not allocate in L1, evict-first in L2.
  // REUSE : neighbour spinors -- default caching (L1 + L2) so the 8-fold neighbour reuse is served on chip.
  // COHERENT: data another agent may write while this kernel is resident (ghost slabs filled by peer GPUs over NVLink,
  //            fields a kernel updates in place): ordinary coherent loads that do not allocate in L1 -- never the
  //            non-coherent (.nc) path, which requires the data to be read-only for the kernel's lifetime.
  enum class Cache { REUSE, STREAM, COHERENT };

  template <Cache c, typename V> B2_HD V ld(const V *p)
  {
#if defined(__CUDA_ARCH__)
    static_assert(sizeof(V) == 16 || sizeof(V) == 8 || sizeof(V) == 4, "vector width");
    if constexpr (sizeof(V) == 16) {
      uint4 r;
      if constexpr (c == Cache::COHERENT) {
        // weak coherent load: ordered after the flag acquire (thread 0, system scope) + CTA barrier by causality order;
        // L1::no_allocate so that no line of a ghost slab is ever kept in the (non-coherent) L1
#ifndef B2_GHOST_LD
#define B2_GHOST_LD "ld.global.L1::no_allocate"
#endif
        asm volatile(B2_GHOST_LD ".v4.u32 {%0,%1,%2,%3}, [%4];"
                     : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                     : "l"(p)
                     : "memory");
      } else if constexpr (c == Cache::STREAM) {
#ifdef B2_L2_HINTS
        // read-once data: additionally ask L2 to evict these lines first so they do not displace neighbour spinors
        unsigned long long pol;
        asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
        asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
                     : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                     : "l"(p), "l"(pol));
#else
        asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                     : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                     : "l"(p));
#endif
      } else
        asm volatile("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
      return *reinterpret_cast<V *>(&r);
    } else if constexpr (sizeof(V) == 8) {
      uint2 r;
      if constexpr (c == Cache::COHERENT)
        asm volatile(B2_GHOST_LD ".v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p) : "memory");
      else if constexpr (c == Cache::STREAM)
        asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
      else
        asm volatile("ld.global.nc.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
      return *reinterpret_cast<V *>(&r);
    } else {
      unsigned r;
      if constexpr (c == Cache::COHERENT)
        asm volatile(B2_GHOST_LD ".u32 %0, [%1];" : "=r"(r) : "l"(p) : "memory");
      else
        asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(r) : "l"(p));
      return *reinterpret_cast<V *>(&r);
    }
#else
    return *p;
#endif
  }

  // streaming store: the output spinor is not re-read by this kernel
  template <typename V> B2_HD void st_stream(V *p, const V &v)
  {
#if defined(__CUDA_ARCH__)
    if constexpr (sizeof(V) == 16) {
      const uint4 r = *reinterpret_cast<const uint4 *>(&v);
      asm volatile("st.global.cs.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(r.x), "r"(r.y), "r"(r.z), "r"(r.w) : "memory");
    } else if constexpr (sizeof(V) == 8) {
      const uint2 r = *reinterpret_cast<const uint2 *>(&v);
      asm volatile("st.global.cs.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(r.x), "r"(r.y) : "memory");
    } else {
      const unsigned r = *reinterpret_cast<const unsigned *>(&v);
      asm volatile("st.global.cs.u32 [%0], %1;" ::"l"(p), "r"(r) : "memory");
    }
#else
    *p = v;
#endif
  }

  // ------------------------------------------------------------------ precision traits
  constexpr float kFixedMax = 32767.0f;
  constexpr float kFixedInvMax = 3.0518509476e-5f; // convert.h:44-55

  struct PrecF64 {
    using real = double;
    using store = double;
    static constexpr int bytes = 8;
    static constexpr bool fixed = false;
    static constexpr int Ns = 2; // spinor vector length
    using svec = d2;
    using ghost_vec = d2; // ghost (half-spinor) vector: N_ghost = 2
    static constexpr int Ng = 2;
  };
  struct PrecF32 {
    using real = float;
    using store = float;
    static constexpr int bytes = 4;
    static constexpr bool fixed = false;
    static constexpr int Ns = 4;
    using svec = f4;
    using ghost_vec = f4;
    static constexpr int Ng = 4;
  };
  struct PrecH16 {
    using real = float;
    using store = short;
    static constexpr int bytes = 2;
    static constexpr bool fixed = true;
    static constexpr int Ns = 8;
    using svec = s8;
    using ghost_vec = s4; // color_spinor_field_order.h:1065-1148: half ghost uses N_ghost = 4
    static constexpr int Ng = 4;
  };

  // gauge vector length N per (precision, reconstruct): gauge_field_order.h:2369-2443
  template <class P, int recon> struct GaugeVec;
  template <int recon> struct GaugeVec<PrecF64, recon> { using vec = d2; static constexpr int N = 2; };
  template <> struct GaugeVec<PrecF32, 18> { using vec = f2; static constexpr int N = 2; };
  template <> struct GaugeVec<PrecF32, 12> { using vec = f4; static constexpr int N = 4; };
  template <> struct GaugeVec<PrecF32, 8> { using vec = f4; static constexpr int N = 4; };
  template <> struct GaugeVec<PrecH16, 18> { using vec = s2; static constexpr int N = 2; };
  template <> struct GaugeVec<PrecH16, 12> { using vec = s4; static constexpr int N = 4; };
  template <> struct GaugeVec<PrecH16, 8> { using vec = s8; static constexpr int N = 8; };

#ifndef B2_I2F_NATIVE
#define B2_I2F_NATIVE 1
#endif
  // int16 pair -> two floats.  The half-precision kernels are issue-bound, so the conversions are split between two
  // pipes (B2_I2F_NATIVE == 1, measured best on B200: half recon-12 49.6 us vs 55.7 all-magic vs 51.5 all-native): the low
  // half goes through the conversion unit (I2F.S16, one issue slot, slow pipe), the high half through the integer/FP32
  // pipes -- PRMT sign-extends it, adding it to the bit pattern of 1.5*2^23 puts the integer into the mantissa and one
  // FADD removes the bias (exact; the integer analogue of the reference's QUDA_ALTERNATIVE_I_TO_F path, convert.h:66-78).
  // B2_I2F_NATIVE == 3 (experimental): the conversion unit takes 7 of 8 values, the integer/FP32 pipes every 8th (the
  // high half of words with phase % 4 == 3).  Issue-slot model per site and SM (half recon-12, 272 conversions, I2F at
  // 16 lanes/clk/SM): split 50/50 -> 552 issue cycles vs 264 on the conversion unit; 7/8 -> ~500 vs ~476: balanced.
  template <int phase = 0> B2_HD void s16x2_to_f32(unsigned w, float &lo, float &hi)
  {
#if defined(__CUDA_ARCH__) && (B2_I2F_NATIVE == 3)
    short s0, s1;
    asm("mov.b32 {%0, %1}, %2;" : "=h"(s0), "=h"(s1) : "r"(w));
    lo = (float)s0;
    if constexpr (phase % 4 == 3) {
      unsigned b;
      asm("prmt.b32 %0, %1, 0, 0xbb32;" : "=r"(b) : "r"(w));
      hi = __int_as_float((int)(b + 0x4B400000u)) - 12582912.0f;
    } else {
      hi = (float)s1;
    }
#elif defined(__CUDA_ARCH__) && (B2_I2F_NATIVE == 2)
    // both halves through the conversion unit (I2F.S16 reads either half of a register directly: one issue slot each)
    short s0, s1;
    asm("mov.b32 {%0, %1}, %2;" : "=h"(s0), "=h"(s1) : "r"(w));
    lo = (float)s0;
    hi = (float)s1;
#elif defined(__CUDA_ARCH__) && (B2_I2F_NATIVE == 1)
    // split the work between the conversion unit (low half) and the integer/FP32 pipes (high half)
    short s0, s1;
    asm("mov.b32 {%0, %1}, %2;" : "=h"(s0), "=h"(s1) : "r"(w));
    lo = (float)s0;
    unsigned b;
    asm("prmt.b32 %0, %1, 0, 0xbb32;" : "=r"(b) : "r"(w));
    hi = __int_as_float((int)(b + 0x4B400000u)) - 12582912.0f;
#elif defined(__CUDA_ARCH__)
    unsigned a, b;
    asm("prmt.b32 %0, %1, 0, 0x9910;" : "=r"(a) : "r"(w));
    asm("prmt.b32 %0, %1, 0, 0xbb32;" : "=r"(b) : "r"(w));
    lo = __int_as_float((int)(a + 0x4B400000u)) - 12582912.0f;
    hi = __int_as_float((int)(b + 0x4B400000u)) - 12582912.0f;
#else
    lo = (float)(short)(w & 0xffffu);
    hi = (float)(short)(w >> 16);
#endif
  }

  // generic "vector of storage elements -> reals" used by every accessor
  // `phase`: position of the vector in its site record (only used to spread conversions over pipes, B2_I2F_NATIVE == 3)
  template <int phase = 0, typename real, typename V> B2_HD void vec_to_real(real *out, const V &v)
  {
    if constexpr (sizeof(V) == sizeof(short) * 8 && alignof(V) == 16 && std::is_same<V, struct s8>::value) {
      unsigned w[4];
      memcpy(w, &v, sizeof(w)); // (type punning through memcpy: folded to register moves, no aliasing UB on the host)
      float lo, hi;
      s16x2_to_f32<0>(w[0], lo, hi);
      out[0] = lo, out[1] = hi;
      s16x2_to_f32<1>(w[1], lo, hi);
      out[2] = lo, out[3] = hi;
      s16x2_to_f32<2>(w[2], lo, hi);
      out[4] = lo, out[5] = hi;
      s16x2_to_f32<3>(w[3], lo, hi);
      out[6] = lo, out[7] = hi;
    } else if constexpr (std::is_same<V, struct s4>::value) {
      unsigned w[2];
      memcpy(w, &v, sizeof(w));
      float lo, hi;
      s16x2_to_f32<2 * (phase % 2)>(w[0], lo, hi);
      out[0] = lo, out[1] = hi;
      s16x2_to_f32<2 * (phase % 2) + 1>(w[1], lo, hi);
      out[2] = lo, out[3] = hi;
    } else if constexpr (std::is_same<V, struct s2>::value) {
      float lo, hi;
      unsigned w;
      memcpy(&w, &v, sizeof(w));
      s16x2_to_f32<phase % 4>(w, lo, hi);
      out[0] = lo;
      out[1] = hi;
    } else if constexpr (std::is_same<V, struct f4>::value) {
      out[0] = v.x; out[1] = v.y; out[2] = v.z; out[3] = v.w;
    } else {
      out[0] = v.x; out[1] = v.y;
    }
  }

  // vec_to_real over an array of M vectors with the vector index as compile-time phase
  template <int N, typename real, typename V, int... I>
  B2_HD void vecs_to_real_impl(real *out, const V *v, std::integer_sequence<int, I...>)
  {
    (vec_to_real<I>(out + I * N, v[I]), ...);
  }
  template <int M, int N, typename real, typename V> B2_HD void vecs_to_real(real *out, const V *v)
  {
    vecs_to_real_impl<N>(out, v, std::make_integer_sequence<int, M> {});
  }

  // round-to-nearest-even float -> int16 as the reference's device path does (convert.h:84-107)
  B2_HD short f2s(float f)
  {
#if defined(__CUDA_ARCH__)
    return (short)__float_as_int(f + 12582912.0f); // magic-number round to nearest even: low 16 bits hold the integer
#else
    return (short)std::nearbyintf(f);
#endif
  }

  B2_HD float fast_div(float a, float b)
  {
#if defined(__CUDA_ARCH__)
    return __fdividef(a, b);
#else
    return a / b;
#endif
  }

  // ------------------------------------------------------------------ complex helpers on (re, im) pairs
  template <typename T> struct cplx {
    T re, im;
  };
  template <typename T> B2_HD cplx<T> cmul(const cplx<T> &a, const cplx<T> &b)
  {
    return {a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re};
  }
  template <typename T> B2_HD cplx<T> conj(const cplx<T> &a) { return {a.re, -a.im}; }

  // ------------------------------------------------------------------ paired FP32 (sm_100: FFMA2 / FADD2 / FMUL2)
  // One instruction does the same fp32 operation on both halves of a 64-bit register pair, each lane rounded exactly as the
  // scalar instruction.  The fp32 site code (fp32 storage, and half, which computes in fp32) runs its complex arithmetic on
  // (re, im) pairs through these helpers, keeping every lane's operation sequence and FMA contraction of the scalar code,
  // so the output is bit-identical to the scalar path (B2_PACKED_F32=0, also what the host twin and fp64 compile).
  //
  // What ptxas folds into operand modifiers at no cost: swapping the halves (`.LO_HI`), negating one half (`.NP`) or
  // both, and a scalar broadcast (`R.F32`) for the second factor when it is written as pack2(x, x) or pack2(-x, x).  So
  // multiplying by +-i is fma2(swap2(h), pack2(-x, x), acc): the sign pattern goes on the pair, the scalar is broadcast.
  // ptxas contracts a mul2 feeding an add2 into one FFMA2 despite the .rn, so a product that the scalar code rounds
  // before adding is only ever used as a multiplicand or as the addend of an fma2.
#ifndef B2_PACKED_F32
#define B2_PACKED_F32 1
#endif
#if defined(__CUDA_ARCH__) && B2_PACKED_F32
#define B2_F32X2 1
  using f32x2 = unsigned long long;
  B2_D f32x2 pack2(float lo, float hi)
  {
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
  }
  B2_D void unpack2(f32x2 p, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(p)); }
  B2_D f32x2 fma2(f32x2 a, f32x2 b, f32x2 c)
  {
    f32x2 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
  }
  B2_D f32x2 add2(f32x2 a, f32x2 b)
  {
    f32x2 d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
  }
  B2_D f32x2 sub2(f32x2 a, f32x2 b)
  {
    f32x2 d;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
  }
  B2_D f32x2 mul2(f32x2 a, f32x2 b)
  {
    f32x2 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
  }
  B2_D f32x2 swap2(f32x2 a)
  {
    float lo, hi;
    unpack2(a, lo, hi);
    return pack2(hi, lo);
  }
  B2_D f32x2 ld2(const float *p) { return pack2(p[0], p[1]); }
  B2_D void st2(float *p, f32x2 v) { unpack2(v, p[0], p[1]); }
#else
#define B2_F32X2 0
#endif

  // ------------------------------------------------------------------ lattice geometry + index math
  struct Geom {
    int X[4];    // local lattice extents (full sites), X[0] even
    int Xh0;     // X[0]/2
    int volume_cb;
    int face_cb[4]; // sites of one parity on a face orthogonal to d: prod_{e!=d} X[e] / 2
  };

  B2_HD void geom_init(Geom &g, const int *X)
  {
    for (int d = 0; d < 4; d++) g.X[d] = X[d];
    g.Xh0 = X[0] / 2;
    g.volume_cb = X[0] / 2 * X[1] * X[2] * X[3];
    for (int d = 0; d < 4; d++) g.face_cb[d] = g.volume_cb * 2 / X[d] / 2;
  }

  // checkerboard index -> coordinates (index_helper.cuh:284-302)
  B2_HD void coords_from_cb(int *x, const Geom &g, int x_cb, int parity)
  {
    const int za = x_cb / g.Xh0;
    const int zb = za / g.X[1];
    x[1] = za - zb * g.X[1];
    x[3] = zb / g.X[2];
    x[2] = zb - x[3] * g.X[2];
    x[0] = 2 * x_cb + ((x[1] + x[2] + x[3] + parity) & 1) - za * g.X[0];
  }

  B2_HD int cb_from_coords(const int *x, const Geom &g)
  {
    return (((x[3] * g.X[2] + x[2]) * g.X[1] + x[1]) * g.X[0] + x[0]) >> 1;
  }

  // Index (within the face of one parity) of the site with coordinates x on a face orthogonal to d:
  // the three remaining coordinates in x-fastest order, halved (index_helper.cuh:445-500, ghostFaceIndex, nFace=1).
  B2_HD int face_index(const int *x, const Geom &g, int d)
  {
    switch (d) {
    case 0: return ((x[3] * g.X[2] + x[2]) * g.X[1] + x[1]) >> 1;
    case 1: return ((x[3] * g.X[2] + x[2]) * g.X[0] + x[0]) >> 1;
    case 2: return ((x[3] * g.X[1] + x[1]) * g.X[0] + x[0]) >> 1;
    default: return ((x[2] * g.X[1] + x[1]) * g.X[0] + x[0]) >> 1;
    }
  }

  // Inverse of face_index: coordinates of face site `idx` (parity `parity`) on the slice x[d] = xd.
  B2_HD void coords_from_face(int *x, const Geom &g, int d, int xd, int idx, int parity)
  {
    // dims other than d in increasing order: a (fastest), b, c
    const int a = (d == 0) ? 1 : 0;
    const int b = (d <= 1) ? 2 : 1;
    const int c = (d <= 2) ? 3 : 2;
    const int Xa = g.X[a], Xb = g.X[b];
    const int ah = Xa / 2;
    const int row = idx / ah; // = xc*Xb + xb
    const int xc = row / Xb;
    const int xb = row - xc * Xb;
    const int xa = 2 * (idx - row * ah) + ((xb + xc + xd + parity) & 1);
    x[a] = xa;
    x[b] = xb;
    x[c] = xc;
    x[d] = xd;
  }

  // ------------------------------------------------------------------ native spinor accessor
  template <class P> struct SpinorView {
    using store = typename P::store;
    store *v;    // base of this parity block
    float *norm; // per-site scale (fixed point only)
    int stride;  // = volumeCB of the field

    // load planes [p0, p0+np) of N-vectors into out[(p - p0)*N + lane] (unscaled for fixed point)
    template <int p0, int np, Cache c = Cache::REUSE> B2_HD void load_planes(typename P::real *out, int x_cb) const
    {
      using V = typename P::svec;
      constexpr int N = P::Ns;
      const V *base = reinterpret_cast<const V *>(v);
#pragma unroll
      for (int i = 0; i < np; i++) {
        const V t = ld<c>(base + (size_t)(p0 + i) * stride + x_cb);
        vec_to_real(out + i * N, t);
      }
    }

    template <Cache c = Cache::REUSE> B2_HD float load_norm(int x_cb) const
    {
      if constexpr (P::fixed)
        return ld<c>(norm + x_cb);
      else
        return 1.0f;
    }

    // full 24-real load, scaled to real values
    template <Cache c = Cache::REUSE> B2_HD void load(typename P::real *out, int x_cb) const
    {
      load_planes<0, 24 / P::Ns, c>(out, x_cb);
      if constexpr (P::fixed) {
        const float n = load_norm<c == Cache::COHERENT ? Cache::COHERENT : Cache::REUSE>(x_cb);
#pragma unroll
        for (int i = 0; i < 24; i++) out[i] *= n;
      }
    }

    // store 24 reals (color_spinor_field_order.h:1254-1292: block-float with max-abs norm for fixed point)
    B2_HD void save(const typename P::real *in, int x_cb) const
    {
      using V = typename P::svec;
      constexpr int N = P::Ns;
      V *base = reinterpret_cast<V *>(v);
      typename P::real t[24];
#pragma unroll
      for (int i = 0; i < 24; i++) t[i] = in[i];
      if constexpr (P::fixed) {
        float mx = 0.0f;
#pragma unroll
        for (int i = 0; i < 24; i++) mx = fmaxf(mx, fabsf(t[i]));
        st_stream(norm + x_cb, mx * kFixedInvMax);
        const float sinv = fast_div(kFixedMax, mx);
#pragma unroll
        for (int i = 0; i < 24; i++) t[i] *= sinv;
      }
#pragma unroll
      for (int i = 0; i < 24 / N; i++) {
        V o;
        store *e = reinterpret_cast<store *>(&o);
#pragma unroll
        for (int j = 0; j < N; j++) {
          if constexpr (P::fixed)
            e[j] = f2s(t[i * N + j]);
          else
            e[j] = t[i * N + j];
        }
        st_stream(base + (size_t)i * stride + x_cb, o);
      }
    }
  };

  // ------------------------------------------------------------------ ghost (spin-projected, 12 reals) accessor
  // One face buffer: [M_ghost planes][face_cb] of N_ghost vectors (+ float norm[face_cb] for fixed point),
  // color_spinor_field_order.h:1065-1180.
  template <class P> struct GhostView {
    using store = typename P::store;
    store *v;
    float *norm;
    int face_cb;

    B2_HD void load(typename P::real *out, int idx) const
    {
      using V = typename P::ghost_vec;
      constexpr int N = P::Ng;
      const V *base = reinterpret_cast<const V *>(v);
#pragma unroll
      for (int i = 0; i < 12 / N; i++) {
        const V t = ld<Cache::COHERENT>(base + (size_t)i * face_cb + idx); // written by the neighbour while we are resident
        vec_to_real(out + i * N, t);
      }
      if constexpr (P::fixed) {
        const float n = ld<Cache::COHERENT>(norm + idx);
#pragma unroll
        for (int i = 0; i < 12; i++) out[i] *= n;
      }
    }

    B2_HD void save(const typename P::real *in, int idx) const
    {
      using V = typename P::ghost_vec;
      constexpr int N = P::Ng;
      V *base = reinterpret_cast<V *>(v);
      typename P::real t[12];
#pragma unroll
      for (int i = 0; i < 12; i++) t[i] = in[i];
      if constexpr (P::fixed) {
        float mx = 0.0f;
#pragma unroll
        for (int i = 0; i < 12; i++) mx = fmaxf(mx, fabsf(t[i]));
        norm[idx] = mx * kFixedInvMax;
        const float sinv = fast_div(kFixedMax, mx);
#pragma unroll
        for (int i = 0; i < 12; i++) t[i] *= sinv;
      }
#pragma unroll
      for (int i = 0; i < 12 / N; i++) {
        V o;
        store *e = reinterpret_cast<store *>(&o);
#pragma unroll
        for (int j = 0; j < N; j++) {
          if constexpr (P::fixed)
            e[j] = f2s(t[i * N + j]);
          else
            e[j] = t[i * N + j];
        }
        base[(size_t)i * face_cb + idx] = o; // plain store: may target a peer GPU's buffer over NVLink
      }
    }
  };

  // ------------------------------------------------------------------ gauge accessor + reconstruction
  struct GaugeMeta {
    double anisotropy;
    double link_max;     // fixed-point scale for recon-18 (LinkMax)
    int t_boundary;      // +1 periodic, -1 anti-periodic
    int first_time_slice; // this rank holds t = 0 of the global lattice
    int last_time_slice;  // this rank holds the last global time slice
    int t_bound_cb;      // (X3-1)*X0*X1*X2/2 : first checkerboard index of the last local time slice
    int volume_cb;
  };

  template <class P, int recon> struct GaugeView {
    using real = typename P::real;
    using store = typename P::store;
    using V = typename GaugeVec<P, recon>::vec;
    static constexpr int N = GaugeVec<P, recon>::N;
    static constexpr int M = recon / N;

    const store *g[2]; // base pointer per parity
    int stride;        // volumeCB + pad
    real aniso, tb, link_scale;
    int t_bound_cb, volume_cb, first_ts, last_ts;

    B2_HD void init(const void *base, size_t parity_offset_bytes, int stride_, const GaugeMeta &m)
    {
      g[0] = reinterpret_cast<const store *>(base);
      g[1] = reinterpret_cast<const store *>(reinterpret_cast<const char *>(base) + parity_offset_bytes);
      stride = stride_;
      aniso = (real)m.anisotropy;
      tb = (real)m.t_boundary;
      link_scale = (real)m.link_max;
      t_bound_cb = m.t_bound_cb;
      volume_cb = m.volume_cb;
      first_ts = m.first_time_slice;
      last_ts = m.last_time_slice;
    }

    // u0 factor of timeBoundary() (gauge_field_order.h:1019-1049, PAD ghost exchange); idx may be >= volume_cb (ghost)
    B2_HD real u0(int dir, int idx) const
    {
      if (dir < 3) return aniso;
      if (idx >= volume_cb) return first_ts ? tb : (real)1;
      if (idx >= t_bound_cb) return last_ts ? tb : (real)1;
      return (real)1;
    }

    // raw (still packed) link: M vectors straight from memory -- lets a kernel issue the loads of all its links first
    // and unpack each one only when its hop is computed
    struct Raw {
      V w[M];
    };

    // `c`: STREAM for the single-source kernels (each link is read once), REUSE where sibling warps of the CTA load the
    // same link (multi-RHS, CTA flavour) and L1 should serve the repeats
    template <Cache c = Cache::STREAM> B2_HD void load_raw(Raw &r, int dir, int x_cb, int parity) const
    {
      const V *base = reinterpret_cast<const V *>(g[parity]);
#pragma unroll
      for (int i = 0; i < M; i++) r.w[i] = ld<c>(base + (size_t)(dir * M + i) * stride + x_cb);
    }

    B2_HD void unpack(real *u, const Raw &r, int dir, int x_cb) const
    {
      real t[recon];
#pragma unroll
      for (int i = 0; i < M; i++) {
        vec_to_real(t + i * N, r.w[i]);
        if constexpr (P::fixed) {
#pragma unroll
          for (int j = 0; j < N; j++) t[i * N + j] *= kFixedInvMax;
        }
      }
      if constexpr (recon == 18) {
#pragma unroll
        for (int i = 0; i < 18; i++) u[i] = P::fixed ? link_scale * t[i] : t[i];
      } else if constexpr (recon == 12) {
#pragma unroll
        for (int i = 0; i < 12; i++) u[i] = t[i];
        row2(u, u0(dir, x_cb));
      } else {
        unpack8(u, t, u0(dir, x_cb));
      }
    }

    // Fixed-point links, scaling deferred: u = U / scale with the raw int16 values (exact in fp32) in rows 0,1, so that
    // the caller can fold `scale` (and the neighbour spinor's block-float norm) into the ONE multiply-add that
    // accumulates the hop -- removes the 12..18 per-link and 24 per-spinor scaling multiplies from the instruction-bound
    // half-precision kernels.  recon-12: row 2 = u0 * conj(row0 x row1) is quadratic in the raw values, so it gets
    // the missing power of 1/32767 here; recon-8 is not linear in its parameters and keeps the plain path (scale = 1).
    B2_HD void unpack_deferred(real *u, real &scale, const Raw &r, int dir, int x_cb) const
    {
      static_assert(P::fixed, "deferred scaling is for the fixed-point formats");
      if constexpr (recon == 8) {
        unpack(u, r, dir, x_cb);
        scale = (real)1;
      } else {
        real t[recon];
        vecs_to_real<M, N>(t, r.w);
        if constexpr (recon == 18) {
#pragma unroll
          for (int i = 0; i < 18; i++) u[i] = t[i];
          scale = link_scale * kFixedInvMax;
        } else {
#pragma unroll
          for (int i = 0; i < 12; i++) u[i] = t[i];
          row2(u, u0(dir, x_cb) * kFixedInvMax);
          scale = kFixedInvMax;
        }
      }
    }

    // recon-12: row 2 = s * conj(row0 x row1), rows 0 and 1 already in u[0..11]
    B2_HD static void row2(real *u, real s)
    {
#if B2_F32X2
      if constexpr (std::is_same<real, float>::value) {
        // cmul(a, b) as nvcc contracts it: re = fma(a.re, b.re, -(a.im*b.im)), im = fma(a.im, b.re, a.re*b.im)
        auto cmul2 = [](f32x2 a, const float *b) {
          return fma2(a, pack2(b[0], b[0]), mul2(swap2(a), pack2(-b[1], b[1])));
        };
        const f32x2 a0 = ld2(u), a1 = ld2(u + 2), a2 = ld2(u + 4);
        const float *b0 = u + 6, *b1 = u + 8, *b2 = u + 10;
        const f32x2 ss = pack2(s, -s);
        st2(u + 12, mul2(sub2(cmul2(a1, b2), cmul2(a2, b1)), ss));
        st2(u + 14, mul2(sub2(cmul2(a2, b0), cmul2(a0, b2)), ss));
        st2(u + 16, mul2(sub2(cmul2(a0, b1), cmul2(a1, b0)), ss));
        return;
      }
#endif
      const cplx<real> a0 {u[0], u[1]}, a1 {u[2], u[3]}, a2 {u[4], u[5]};
      const cplx<real> b0 {u[6], u[7]}, b1 {u[8], u[9]}, b2 {u[10], u[11]};
      cplx<real> c0 = cmul(a1, b2), c1 = cmul(a2, b0), c2 = cmul(a0, b1);
      const cplx<real> d0 = cmul(a2, b1), d1 = cmul(a0, b2), d2_ = cmul(a1, b0);
      u[12] = s * (c0.re - d0.re);
      u[13] = -s * (c0.im - d0.im);
      u[14] = s * (c1.re - d1.re);
      u[15] = -s * (c1.im - d1.im);
      u[16] = s * (c2.re - d2_.re);
      u[17] = -s * (c2.im - d2_.im);
    }

    // load link (dir, x_cb, parity) into row-major u[18] = U[row][col] (re, im)
    template <Cache c = Cache::STREAM> B2_HD void load(real *u, int dir, int x_cb, int parity) const
    {
      Raw r;
      load_raw<c>(r, dir, x_cb, parity);
      unpack(u, r, dir, x_cb);
    }

    // 8-parameter reconstruction (gauge_field_order.h:1303-1390); packed = [arg(U10)/pi, arg(-U20)/pi, U11, U12, U00]
    // with the roles of rows 0 and 1 swapped and row 2 negated relative to the "textbook" parametrisation.
    B2_HD static void unpack8(real *u, const real *in, real u0v)
    {
      const real u0_inv = rcp_((real)u0v);
      cplx<real> o[9];
      o[1] = {in[2], in[3]};
      o[2] = {in[4], in[5]};
      o[3] = {in[6], in[7]};
      real sn, cs;
      sincospi_(in[0], &sn, &cs);
      o[0] = {cs, sn};
      sincospi_(in[1], &sn, &cs);
      o[6] = {cs, sn};
      real row_sum = o[1].re * o[1].re;
      row_sum += o[1].im * o[1].im;
      row_sum += o[2].re * o[2].re;
      row_sum += o[2].im * o[2].im;
      const real row_sum_inv = rcp_(row_sum);
      real diff = u0_inv * u0_inv - row_sum;
      const real m00 = diff > 0 ? diff * rsqrt_(diff) : (real)0;
      o[0].re *= m00;
      o[0].im *= m00;
      real col_sum = o[0].re * o[0].re;
      col_sum += o[0].im * o[0].im;
      col_sum += o[3].re * o[3].re;
      col_sum += o[3].im * o[3].im;
      diff = u0_inv * u0_inv - col_sum;
      const real m20 = diff > 0 ? diff * rsqrt_(diff) : (real)0;
      o[6].re *= m20;
      o[6].im *= m20;
      const real r_inv2 = u0_inv * row_sum_inv;
      {
        cplx<real> A = cmul(conj(o[0]), o[3]);
        A.re *= u0v;
        A.im *= u0v;
        cplx<real> t4 = cmul(conj(o[6]), conj(o[2]));
        const cplx<real> a1 = cmul(A, o[1]);
        o[4] = {-r_inv2 * (t4.re + a1.re), -r_inv2 * (t4.im + a1.im)};
        cplx<real> t5 = cmul(conj(o[6]), conj(o[1]));
        const cplx<real> a2 = cmul(A, o[2]);
        o[5] = {r_inv2 * (t5.re - a2.re), r_inv2 * (t5.im - a2.im)};
      }
      {
        cplx<real> A = cmul(conj(o[0]), o[6]);
        A.re *= u0v;
        A.im *= u0v;
        cplx<real> t7 = cmul(conj(o[3]), conj(o[2]));
        const cplx<real> a1 = cmul(A, o[1]);
        o[7] = {r_inv2 * (t7.re - a1.re), r_inv2 * (t7.im - a1.im)};
        cplx<real> t8 = cmul(conj(o[3]), conj(o[1]));
        const cplx<real> a2 = cmul(A, o[2]);
        o[8] = {-r_inv2 * (t8.re + a2.re), -r_inv2 * (t8.im + a2.im)};
      }
      // undo the row permutation: {b, a, -c} -> {a, b, c}
#pragma unroll
      for (int i = 0; i < 3; i++) {
        u[2 * i] = o[i + 3].re;
        u[2 * i + 1] = o[i + 3].im;
        u[6 + 2 * i] = o[i].re;
        u[6 + 2 * i + 1] = o[i].im;
        u[12 + 2 * i] = -o[i + 6].re;
        u[12 + 2 * i + 1] = -o[i + 6].im;
      }
    }

    // single precision: hardware reciprocal / sin / cos (MUFU); |error| ~1e-6, far inside the 1e-4 gate
    B2_HD static float rcp_(float x)
    {
#if defined(__CUDA_ARCH__)
      return __frcp_rn(x);
#else
      return 1.0f / x;
#endif
    }
    B2_HD static double rcp_(double x) { return 1.0 / x; }
    B2_HD static void sincospi_(float x, float *s, float *c)
    {
#if defined(__CUDA_ARCH__)
      __sincosf(x * 3.14159265358979323846f, s, c);
#else
      *s = (float)std::sin(3.14159265358979323846 * (double)x);
      *c = (float)std::cos(3.14159265358979323846 * (double)x);
#endif
    }
    B2_HD static void sincospi_(double x, double *s, double *c)
    {
#if defined(__CUDA_ARCH__)
      ::sincospi(x, s, c);
#else
      *s = std::sin(3.14159265358979323846 * x);
      *c = std::cos(3.14159265358979323846 * x);
#endif
    }
    B2_HD static float rsqrt_(float x)
    {
#if defined(__CUDA_ARCH__)
      return ::rsqrtf(x);
#else
      return 1.0f / std::sqrt(x);
#endif
    }
    B2_HD static double rsqrt_(double x)
    {
#if defined(__CUDA_ARCH__)
      return ::rsqrt(x);
#else
      return 1.0 / std::sqrt(x);
#endif
    }
  };

  // ------------------------------------------------------------------ SU(3) x half-spinor
  // h: 2 spins x 3 colours (12 reals, (s*3+c)*2+reim); u row-major.  r = U h  or  r = U^dagger h.
  template <bool adjoint, typename real> B2_HD void su3_mul(real *r, const real *u, const real *h)
  {
#if B2_F32X2
    if constexpr (std::is_same<real, float>::value) { // per lane the chain below: (re, im) += ur (hr, hi) + ui (-hi, hr)
#pragma unroll
      for (int s = 0; s < 2; s++) {
#pragma unroll
        for (int i = 0; i < 3; i++) {
          f32x2 acc = pack2(0.0f, 0.0f);
#pragma unroll
          for (int j = 0; j < 3; j++) {
            const float ur = adjoint ? u[(j * 3 + i) * 2] : u[(i * 3 + j) * 2];
            const float ui = adjoint ? -u[(j * 3 + i) * 2 + 1] : u[(i * 3 + j) * 2 + 1];
            const f32x2 hv = ld2(h + (s * 3 + j) * 2);
            acc = fma2(hv, pack2(ur, ur), acc);
            acc = fma2(swap2(hv), pack2(-ui, ui), acc);
          }
          st2(r + (s * 3 + i) * 2, acc);
        }
      }
      return;
    }
#endif
#pragma unroll
    for (int s = 0; s < 2; s++) {
#pragma unroll
      for (int i = 0; i < 3; i++) {
        real re = 0, im = 0;
#pragma unroll
        for (int j = 0; j < 3; j++) {
          const real ur = adjoint ? u[(j * 3 + i) * 2] : u[(i * 3 + j) * 2];
          const real ui = adjoint ? -u[(j * 3 + i) * 2 + 1] : u[(i * 3 + j) * 2 + 1];
          const real hr = h[(s * 3 + j) * 2], hi = h[(s * 3 + j) * 2 + 1];
          re += ur * hr;
          re -= ui * hi;
          im += ur * hi;
          im += ui * hr;
        }
        r[(s * 3 + i) * 2] = re;
        r[(s * 3 + i) * 2 + 1] = im;
      }
    }
  }

  // ------------------------------------------------------------------ spin projection / reconstruction, UKQCD basis
  // P(mu, sign) = 1 + sign*gamma_mu.  project: 24 -> 12 reals.  For mu = 3 only half of the spinor is needed:
  // project_t takes the 12 reals of the upper (sign=+1) or lower (sign=-1) spin pair.
  template <typename real> B2_HD void project(real *h, const real *v, int mu, int sign)
  {
    const real sg = (real)sign;
#if B2_F32X2
    if constexpr (std::is_same<real, float>::value) { // the +-1 factors are exact: fma2 by them is the scalar FADD
      const f32x2 pi = pack2(-sg, sg), mi = pack2(sg, -sg), p1 = pack2(sg, sg), m1 = pack2(-sg, -sg); // +-s*i, +-s
#pragma unroll
      for (int c = 0; c < 3; c++) {
        const f32x2 v0 = ld2(v + (0 * 3 + c) * 2), v1 = ld2(v + (1 * 3 + c) * 2);
        const f32x2 v2 = ld2(v + (2 * 3 + c) * 2), v3 = ld2(v + (3 * 3 + c) * 2);
        f32x2 h0, h1;
        if (mu == 0) {
          h0 = fma2(swap2(v3), pi, v0);
          h1 = fma2(swap2(v2), pi, v1);
        } else if (mu == 1) {
          h0 = fma2(v3, p1, v0);
          h1 = fma2(v2, m1, v1);
        } else if (mu == 2) {
          h0 = fma2(swap2(v2), pi, v0);
          h1 = fma2(swap2(v3), mi, v1);
        } else {
          const f32x2 two = pack2(2.0f, 2.0f);
          h0 = mul2(sign > 0 ? v0 : v2, two);
          h1 = mul2(sign > 0 ? v1 : v3, two);
        }
        st2(h + (0 * 3 + c) * 2, h0);
        st2(h + (1 * 3 + c) * 2, h1);
      }
      return;
    }
#endif
#pragma unroll
    for (int c = 0; c < 3; c++) {
      const real v0r = v[(0 * 3 + c) * 2], v0i = v[(0 * 3 + c) * 2 + 1];
      const real v1r = v[(1 * 3 + c) * 2], v1i = v[(1 * 3 + c) * 2 + 1];
      const real v2r = v[(2 * 3 + c) * 2], v2i = v[(2 * 3 + c) * 2 + 1];
      const real v3r = v[(3 * 3 + c) * 2], v3i = v[(3 * 3 + c) * 2 + 1];
      real h0r, h0i, h1r, h1i;
      if (mu == 0) { // h0 = v0 + s*i*v3 ; h1 = v1 + s*i*v2
        h0r = v0r - sg * v3i;
        h0i = v0i + sg * v3r;
        h1r = v1r - sg * v2i;
        h1i = v1i + sg * v2r;
      } else if (mu == 1) { // h0 = v0 + s*v3 ; h1 = v1 - s*v2
        h0r = v0r + sg * v3r;
        h0i = v0i + sg * v3i;
        h1r = v1r - sg * v2r;
        h1i = v1i - sg * v2i;
      } else if (mu == 2) { // h0 = v0 + s*i*v2 ; h1 = v1 - s*i*v3
        h0r = v0r - sg * v2i;
        h0i = v0i + sg * v2r;
        h1r = v1r + sg * v3i;
        h1i = v1i - sg * v3r;
      } else {
        if (sign > 0) {
          h0r = 2 * v0r;
          h0i = 2 * v0i;
          h1r = 2 * v1r;
          h1i = 2 * v1i;
        } else {
          h0r = 2 * v2r;
          h0i = 2 * v2i;
          h1r = 2 * v3r;
          h1i = 2 * v3i;
        }
      }
      h[(0 * 3 + c) * 2] = h0r;
      h[(0 * 3 + c) * 2 + 1] = h0i;
      h[(1 * 3 + c) * 2] = h1r;
      h[(1 * 3 + c) * 2 + 1] = h1i;
    }
  }

#if B2_F32X2
  // acc += s * reconstruct(h) on (re, im) pairs: one FFMA2 per colour and spin, as the scalar forms below
  B2_D void reconstruct_add_x2(float *acc, const float *h, int mu, int sign, float s)
  {
    const float sg = (float)sign * s;
    const f32x2 p = pack2(s, s), ps = pack2(sg, sg), ms = pack2(-sg, -sg), pi = pack2(sg, -sg), mi = pack2(-sg, sg);
#pragma unroll
    for (int c = 0; c < 3; c++) {
      const f32x2 h0 = ld2(h + (0 * 3 + c) * 2), h1 = ld2(h + (1 * 3 + c) * 2);
      float *a0 = acc + (0 * 3 + c) * 2, *a1 = acc + (1 * 3 + c) * 2, *a2 = acc + (2 * 3 + c) * 2, *a3 = acc + (3 * 3 + c) * 2;
      if (mu == 3 && sign < 0) {
        st2(a2, fma2(h0, p, ld2(a2)));
        st2(a3, fma2(h1, p, ld2(a3)));
        continue;
      }
      st2(a0, fma2(h0, p, ld2(a0)));
      st2(a1, fma2(h1, p, ld2(a1)));
      if (mu == 0) { // rows 2,3: -s*i*h1, -s*i*h0
        st2(a2, fma2(swap2(h1), pi, ld2(a2)));
        st2(a3, fma2(swap2(h0), pi, ld2(a3)));
      } else if (mu == 1) { // rows 2,3: -s*h1, +s*h0
        st2(a2, fma2(h1, ms, ld2(a2)));
        st2(a3, fma2(h0, ps, ld2(a3)));
      } else if (mu == 2) { // rows 2,3: -s*i*h0, +s*i*h1
        st2(a2, fma2(swap2(h0), pi, ld2(a2)));
        st2(a3, fma2(swap2(h1), mi, ld2(a3)));
      }
    }
  }
#endif

  // h = 2 t (12 reals): the t-direction projection of a spin pair that is already loaded
  template <typename real> B2_HD void twice12(real *h, const real *t)
  {
#if B2_F32X2
    if constexpr (std::is_same<real, float>::value) {
#pragma unroll
      for (int i = 0; i < 12; i += 2) st2(h + i, mul2(ld2(t + i), pack2(2.0f, 2.0f)));
      return;
    }
#endif
#pragma unroll
    for (int i = 0; i < 12; i++) h[i] = 2 * t[i];
  }

  // acc += reconstruct(h) for P(mu, sign)
  template <typename real> B2_HD void reconstruct_add(real *acc, const real *h, int mu, int sign)
  {
    const real sg = (real)sign;
#if B2_F32X2
    if constexpr (std::is_same<real, float>::value) {
      reconstruct_add_x2(acc, h, mu, sign, 1.0f); // a += 1 * h is the scalar FADD
      return;
    }
#endif
#pragma unroll
    for (int c = 0; c < 3; c++) {
      const real h0r = h[(0 * 3 + c) * 2], h0i = h[(0 * 3 + c) * 2 + 1];
      const real h1r = h[(1 * 3 + c) * 2], h1i = h[(1 * 3 + c) * 2 + 1];
      real *a0 = acc + (0 * 3 + c) * 2, *a1 = acc + (1 * 3 + c) * 2, *a2 = acc + (2 * 3 + c) * 2, *a3 = acc + (3 * 3 + c) * 2;
      if (mu == 0) { // rows 2,3: -s*i*h1, -s*i*h0
        a0[0] += h0r; a0[1] += h0i; a1[0] += h1r; a1[1] += h1i;
        a2[0] += sg * h1i; a2[1] -= sg * h1r;
        a3[0] += sg * h0i; a3[1] -= sg * h0r;
      } else if (mu == 1) { // rows 2,3: -s*h1, +s*h0
        a0[0] += h0r; a0[1] += h0i; a1[0] += h1r; a1[1] += h1i;
        a2[0] -= sg * h1r; a2[1] -= sg * h1i;
        a3[0] += sg * h0r; a3[1] += sg * h0i;
      } else if (mu == 2) { // rows 2,3: -s*i*h0, +s*i*h1
        a0[0] += h0r; a0[1] += h0i; a1[0] += h1r; a1[1] += h1i;
        a2[0] += sg * h0i; a2[1] -= sg * h0r;
        a3[0] -= sg * h1i; a3[1] += sg * h1r;
      } else {
        if (sign > 0) {
          a0[0] += h0r; a0[1] += h0i; a1[0] += h1r; a1[1] += h1i;
        } else {
          a2[0] += h0r; a2[1] += h0i; a3[0] += h1r; a3[1] += h1i;
        }
      }
    }
  }

  // acc += s * reconstruct(h): the deferred-scaling form (one FFMA per component instead of FADD + earlier FMULs)
  template <typename real> B2_HD void reconstruct_add_scaled(real *acc, const real *h, int mu, int sign, real s)
  {
#if B2_F32X2
    if constexpr (std::is_same<real, float>::value) {
      reconstruct_add_x2(acc, h, mu, sign, s);
      return;
    }
#endif
    const real sg = (real)sign * s;
#pragma unroll
    for (int c = 0; c < 3; c++) {
      const real h0r = h[(0 * 3 + c) * 2], h0i = h[(0 * 3 + c) * 2 + 1];
      const real h1r = h[(1 * 3 + c) * 2], h1i = h[(1 * 3 + c) * 2 + 1];
      real *a0 = acc + (0 * 3 + c) * 2, *a1 = acc + (1 * 3 + c) * 2, *a2 = acc + (2 * 3 + c) * 2, *a3 = acc + (3 * 3 + c) * 2;
      if (mu == 0) {
        a0[0] += s * h0r; a0[1] += s * h0i; a1[0] += s * h1r; a1[1] += s * h1i;
        a2[0] += sg * h1i; a2[1] -= sg * h1r;
        a3[0] += sg * h0i; a3[1] -= sg * h0r;
      } else if (mu == 1) {
        a0[0] += s * h0r; a0[1] += s * h0i; a1[0] += s * h1r; a1[1] += s * h1i;
        a2[0] -= sg * h1r; a2[1] -= sg * h1i;
        a3[0] += sg * h0r; a3[1] += sg * h0i;
      } else if (mu == 2) {
        a0[0] += s * h0r; a0[1] += s * h0i; a1[0] += s * h1r; a1[1] += s * h1i;
        a2[0] += sg * h0i; a2[1] -= sg * h0r;
        a3[0] -= sg * h1i; a3[1] += sg * h1r;
      } else {
        if (sign > 0) {
          a0[0] += s * h0r; a0[1] += s * h0i; a1[0] += s * h1r; a1[1] += s * h1i;
        } else {
          a2[0] += s * h0r; a2[1] += s * h0i; a3[0] += s * h1r; a3[1] += s * h1i;
        }
      }
    }
  }

} // namespace b200
