// The Wilson / Wilson-clover stencil for ONE output site, written once and shared by every kernel
// flavour (interior, exterior, tiled, fused-pack) and by the test-only host twin.
//
// Reference behaviour being reproduced (not copied): /root/reference/include/kernels/dslash_wilson.cuh:84-197
// (applyWilson + wilson::operator()), dslash_wilson_clover.cuh:38-105, dslash_wilson_clover_preconditioned.cuh:37-117,
// dslash_helper.cuh:32-242 (isActive / isComplete / doHalo / doBulk).
#pragma once

#include "core.h"
#include "clover.h"

namespace b200
{

  enum KernelType { K_INTERIOR = 0, K_EXTERIOR_ALL = 1, K_FULL = 2 };
  // OP_TM / OP_TM_PC / OP_TM_PC_PRE: the degenerate twisted-mass epilogues on the same stencil
  // (include/kernels/dslash_twisted_mass.cuh:33-70, dslash_twisted_mass_preconditioned.cuh:48-175)
  enum OpType { OP_WILSON = 0, OP_CLOVER = 1, OP_CLOVER_PC = 2, OP_TM = 3, OP_TM_PC = 4, OP_TM_PC_PRE = 5 };

  constexpr int kMaxParity = 2;

  // Kernel parameter block (passed by value; ~0.5 KB).
  template <class P, int recon> struct DslashArgs {
    using real = typename P::real;
    Geom geom;
    SpinorView<P> out[kMaxParity], in[kMaxParity], x[kMaxParity]; // indexed by the parity the view holds
    GaugeView<P, recon> U;
    CloverView<P> A;          // clover term (OP_CLOVER) or its inverse / itself for dynamic inversion (OP_CLOVER_PC)
    GhostView<P> ghost[4][2]; // received half spinors: [dim][0 = from the backward neighbour, 1 = from the forward one]
    size_t ghost_parity_stride[4]; // elements of P::store between the parity-0 and parity-1 halves of a face buffer
    size_t ghost_norm_parity_stride[4];
    real a;                   // xpay coefficient (twisted-mass preconditioned ops: the scale of the twist rotation)
    int n_parity;             // 1: `parity` only; 2: both (blockIdx.y / loop selects)
    int parity;
    int comm_dim[4];          // dimension d is partitioned: hops across its boundary come from ghost[d]
    int threads_ext[5];       // EXTERIOR_ALL: prefix sums of 2*face_cb[d] over partitioned dims
    const unsigned *wait_flag[4][2]; // arrival flags written by the neighbours' pack kernels (nullptr: stream-ordered)
    unsigned seq;             // value the flags must have reached
    int *timeout_flag;        // set to 1 if a wait gives up
    // Twisted-mass ops have no clover term: their twist factor (sign already flipped for dagger) travels in the unused
    // clover slot A.diagonal.  Adding a field would change sizeof(DslashArgs), shift the kernel parameters behind it and
    // make ptxas re-schedule the Wilson / clover kernels that were measured on hardware (checked with cuobjdump).
    B2_HD real twist_b() const { return A.diagonal; }
  };

  // CTA -> 4-d tile of checkerboard sites, thread -> site inside the tile (x fastest so that a warp's 16-byte plane
  // loads cover contiguous 256..512-byte runs).  grid = (nt0*nt1, nt2, nt3 * n_parity); the thread index decomposes by
  // shifts (tile extents are powers of two) and the only division is a multiply-high: no runtime integer division.
  struct TileMap {
    int sh[4];          // log2 of the tile extents: [0] in checkerboard sites (x/2), [1..3] in sites
    int nt[4];          // tiles per dimension (whole lattice)
    int org[4], cnt[4]; // the launch covers the box of tiles [org, org + cnt)
    unsigned cnt0_magic; // floor(2^32 / cnt[0]) + 1 (cnt[0] >= 2); blockIdx.x / cnt[0] == umulhi(blockIdx.x, magic)
  };

  // Up to 8 boxes of boundary tiles (two per partitioned dimension) enumerated by one 1-d grid
  struct SlabTable {
    int n;
    int cta_start[9];
    int org[8][4], cnt[8][4];
  };

  B2_HD unsigned mulhi_u32(unsigned a, unsigned b)
  {
#if defined(__CUDA_ARCH__)
    return __umulhi(a, b);
#else
    return (unsigned)(((unsigned long long)a * b) >> 32);
#endif
  }

  // thread `tid` of the CTA that owns tile (b0,b1,b2,b3) -> its site; false if the (ragged) tile sticks out of the lattice
  B2_HD bool tile_thread_site(int *x, int &x_cb, const Geom &g, const TileMap &tm, int parity, int b0, int b1, int b2, int b3,
                              unsigned tid)
  {
    const int l = (int)tid;
    const int l0 = l & ((1 << tm.sh[0]) - 1);
    const int l1 = (l >> tm.sh[0]) & ((1 << tm.sh[1]) - 1);
    const int l2 = (l >> (tm.sh[0] + tm.sh[1])) & ((1 << tm.sh[2]) - 1);
    const int l3 = l >> (tm.sh[0] + tm.sh[1] + tm.sh[2]);
    const int xh = (b0 << tm.sh[0]) + l0;
    x[1] = (b1 << tm.sh[1]) + l1;
    x[2] = (b2 << tm.sh[2]) + l2;
    x[3] = (b3 << tm.sh[3]) + l3;
    if (xh >= g.Xh0 || x[1] >= g.X[1] || x[2] >= g.X[2] || x[3] >= g.X[3]) return false;
    x[0] = 2 * xh + ((x[1] + x[2] + x[3] + parity) & 1);
    x_cb = ((x[3] * g.X[2] + x[2]) * g.X[1] + x[1]) * g.Xh0 + xh;
    return true;
  }

  // box launch: grid = (cnt0*cnt1, cnt2, cnt3 * n_parity)
  B2_HD bool tile_site(int *x, int &x_cb, int &parity, const Geom &g, const TileMap &tm, int n_parity, int arg_parity,
                       unsigned bx, unsigned by, unsigned bz, unsigned tid)
  {
    const int b1 = tm.cnt[0] == 1 ? (int)bx : (int)mulhi_u32(bx, tm.cnt0_magic);
    const int b0 = (int)bx - b1 * tm.cnt[0];
    const int b2 = (int)by;
    int b3 = (int)bz;
    parity = arg_parity;
    if (n_parity == 2) {
      parity = b3 >= tm.cnt[3] ? 1 : 0;
      b3 -= parity * tm.cnt[3];
    }
    return tile_thread_site(x, x_cb, g, tm, parity, tm.org[0] + b0, tm.org[1] + b1, tm.org[2] + b2, tm.org[3] + b3, tid);
  }

  // slab launch: grid = (total CTAs of all slabs, n_parity)
  B2_HD bool slab_site(int *x, int &x_cb, const Geom &g, const TileMap &tm, const SlabTable &st, int parity, unsigned bx,
                       unsigned tid)
  {
    int s = 0;
#pragma unroll
    for (int k = 1; k < 8; k++)
      if (k < st.n && (int)bx >= st.cta_start[k]) s = k;
    int l = (int)bx - st.cta_start[s];
    const int b0 = l % st.cnt[s][0];
    l /= st.cnt[s][0];
    const int b1 = l % st.cnt[s][1];
    l /= st.cnt[s][1];
    const int b2 = l % st.cnt[s][2];
    const int b3 = l / st.cnt[s][2];
    return tile_thread_site(x, x_cb, g, tm, parity, st.org[s][0] + b0, st.org[s][1] + b1, st.org[s][2] + b2, st.org[s][3] + b3, tid);
  }

  // which spin pair the t-direction projector keeps: P(3,+1) -> upper (spins 0,1), P(3,-1) -> lower
  template <class P, bool upper, Cache c = Cache::REUSE, bool scaled = true>
  B2_HD void load_spin_pair(typename P::real *h, const SpinorView<P> &f, int x_cb)
  {
    if constexpr (P::Ns == 8) { // fixed point, 3 planes of 8: reals 0..11 live in planes 0,1 ; 12..23 in planes 1,2
      typename P::real t[16];
      f.template load_planes<upper ? 0 : 1, 2, c>(t, x_cb);
      if constexpr (scaled) {
        const float n = f.load_norm(x_cb);
#pragma unroll
        for (int i = 0; i < 12; i++) h[i] = (upper ? t[i] : t[i + 4]) * n;
      } else { // raw fixed-point values; the caller folds the norm into the accumulation
#pragma unroll
        for (int i = 0; i < 12; i++) h[i] = upper ? t[i] : t[i + 4];
      }
    } else {
      constexpr int np = 12 / P::Ns;
      f.template load_planes<upper ? 0 : np, np, c>(h, x_cb);
    }
  }

  // ---- one hop, source on this rank (periodic wrap inside the local lattice)
  // checkerboard index of the neighbour of x in direction +-d (periodic wrap)
  template <bool fwd> B2_HD int neighbor_cb(const int *x, const Geom &g, int d)
  {
    int y[4] = {x[0], x[1], x[2], x[3]};
    if (fwd)
      y[d] = (x[d] + 1 >= g.X[d]) ? 0 : x[d] + 1;
    else
      y[d] = (x[d] - 1 < 0) ? g.X[d] - 1 : x[d] - 1;
    return cb_from_coords(y, g);
  }

  // Links whose packed form is small enough (<= 48 B: fp32 recon-12/8, every half format) are fetched for all 8 hops
  // before the first hop is computed (<= 96 registers of raw vectors): one exposed DRAM round trip per site for the
  // link stream instead of one per hop.  Wider links (fp64, fp32 recon-18) would not fit the register file.
#ifndef B2_PRELOAD_LINKS
#define B2_PRELOAD_LINKS 1
#endif
  template <class P, int recon> struct PreloadLinks {
    static constexpr bool value = B2_PRELOAD_LINKS && (sizeof(typename GaugeView<P, recon>::Raw) <= 48);
  };

  // v <- s (v + b i gamma5 v).  In the UKQCD basis gamma5 exchanges the spin pairs: (i gamma5 v)_s = i v_{s +- 2}
  // (include/color_spinor.h:254-262, igamma(4)).
  template <typename real> B2_HD void twist_apply(real *v, real s, real b)
  {
#pragma unroll
    for (int sp = 0; sp < 2; sp++) {
#pragma unroll
      for (int c = 0; c < 3; c++) {
        const int u = (sp * 3 + c) * 2, l = ((sp + 2) * 3 + c) * 2;
        const real ur = v[u], ui = v[u + 1], lr = v[l], li = v[l + 1];
        v[u] = s * (ur - b * li);
        v[u + 1] = s * (ui + b * lr);
        v[l] = s * (lr - b * ui);
        v[l + 1] = s * (li + b * ur);
      }
    }
  }

  // `in` is passed explicitly so that the multi-RHS kernels can aim the same code at any source; `lc` is the cache
  // policy of the link loads; `pretwist`: the neighbour spinor is rotated by a (1 + i b gamma5) before it is projected
  // (symmetric preconditioned twisted-mass dagger, applyWilsonTM)
  template <class P, int recon, bool dagger, bool fwd, Cache lc = Cache::STREAM, bool pretwist = false>
  B2_HD void hop_from(typename P::real *r, const DslashArgs<P, recon> &arg, const SpinorView<P> &in, const int *x, int x_cb,
                      int parity, int d, const typename GaugeView<P, recon>::Raw *raw = nullptr)
  {
    using real = typename P::real;
    const Geom &g = arg.geom;
    constexpr int sign = fwd ? (dagger ? +1 : -1) : (dagger ? -1 : +1);
    real u[18], h[12];
    const int n_cb = neighbor_cb<fwd>(x, g, d);
    if (raw)
      arg.U.unpack(u, *raw, d, fwd ? x_cb : n_cb);
    else if (fwd)
      arg.U.template load<lc>(u, d, x_cb, parity);
    else
      arg.U.template load<lc>(u, d, n_cb, 1 - parity);
    if constexpr (pretwist) { // gamma5 mixes the spin pairs: the full spinor is needed in every direction
      real v[24];
      in.load(v, n_cb);
      twist_apply(v, arg.a, arg.twist_b());
      project(h, v, d, sign);
    } else if (d == 3) {
      real t[12];
      load_spin_pair<P, (sign > 0)>(t, in, n_cb);
      twice12(h, t);
    } else {
      real v[24];
      in.load(v, n_cb);
      project(h, v, d, sign);
    }
    su3_mul<!fwd>(r, u, h);
  }

  template <class P, int recon, bool dagger, bool fwd>
  B2_HD void hop_local(typename P::real *r, const DslashArgs<P, recon> &arg, const int *x, int x_cb, int parity, int d,
                       const typename GaugeView<P, recon>::Raw *raw = nullptr)
  {
    hop_from<P, recon, dagger, fwd>(r, arg, arg.in[1 - parity], x, x_cb, parity, d, raw);
  }

  // Half precision: keep the int16 values of link and neighbour spinor unscaled through projection and SU(3) multiply
  // (exact small integers in fp32) and apply link scale x block-float norm (x 2 for the t direction) in the single
  // FFMA per component that accumulates the hop.  Removes ~250 of the 2 400 instructions per site of the issue-bound
  // half kernels.  B2_HALF_DEFERRED_SCALE=0 restores the scale-on-load arithmetic.
#ifndef B2_HALF_DEFERRED_SCALE
#define B2_HALF_DEFERRED_SCALE 1
#endif
  template <class P> struct DeferredScale {
    static constexpr bool value = P::fixed && B2_HALF_DEFERRED_SCALE;
  };

  // r = (U or U^dagger) P h with everything unscaled; `scale` is the factor the result still has to be multiplied by
  template <class P, int recon, bool dagger, bool fwd, Cache lc = Cache::STREAM, bool pretwist = false>
  B2_HD void hop_from_deferred(typename P::real *r, typename P::real &scale, const DslashArgs<P, recon> &arg,
                               const SpinorView<P> &in, const int *x, int x_cb, int parity, int d,
                               const typename GaugeView<P, recon>::Raw *raw = nullptr)
  {
    using real = typename P::real;
    const Geom &g = arg.geom;
    constexpr int sign = fwd ? (dagger ? +1 : -1) : (dagger ? -1 : +1);
    real u[18], h[12], us;
    const int n_cb = neighbor_cb<fwd>(x, g, d);
    if (raw) {
      arg.U.unpack_deferred(u, us, *raw, d, fwd ? x_cb : n_cb);
    } else {
      typename GaugeView<P, recon>::Raw w;
      arg.U.template load_raw<lc>(w, d, fwd ? x_cb : n_cb, fwd ? parity : 1 - parity);
      arg.U.unpack_deferred(u, us, w, d, fwd ? x_cb : n_cb);
    }
    const real n = in.load_norm(n_cb);
    if constexpr (pretwist) { // the rotation is linear, so it commutes with the deferred scale; project() carries t's factor 2
      real v[24];
      in.template load_planes<0, 24 / P::Ns>(v, n_cb);
      twist_apply(v, arg.a, arg.twist_b());
      project(h, v, d, sign);
      scale = us * n;
    } else if (d == 3) {
      load_spin_pair<P, (sign > 0), Cache::REUSE, false>(h, in, n_cb);
      scale = (us * n) * (real)2;
    } else {
      real v[24];
      in.template load_planes<0, 24 / P::Ns>(v, n_cb);
      project(h, v, d, sign);
      scale = us * n;
    }
    su3_mul<!fwd>(r, u, h);
  }

  // acc += hop (+ optional 0/1 mask for the masked interior kernel); every local hop of every kernel goes through here
  template <class P, int recon, bool dagger, bool fwd, bool masked, Cache lc = Cache::STREAM, bool pretwist = false>
  B2_HD void hop_add(typename P::real *acc, const DslashArgs<P, recon> &arg, const SpinorView<P> &in, const int *x, int x_cb,
                     int parity, int d, const typename GaugeView<P, recon>::Raw *raw, typename P::real mask)
  {
    using real = typename P::real;
    constexpr int sign = fwd ? (dagger ? +1 : -1) : (dagger ? -1 : +1);
    real r[12];
    if constexpr (DeferredScale<P>::value) {
      real scale;
      hop_from_deferred<P, recon, dagger, fwd, lc, pretwist>(r, scale, arg, in, x, x_cb, parity, d, raw);
      if constexpr (masked) scale *= mask;
      reconstruct_add_scaled(acc, r, d, sign, scale);
    } else {
      hop_from<P, recon, dagger, fwd, lc, pretwist>(r, arg, in, x, x_cb, parity, d, raw);
      if constexpr (masked) {
#pragma unroll
        for (int i = 0; i < 12; i++) r[i] *= mask;
      }
      reconstruct_add(acc, r, d, sign);
    }
  }

  // ---- one hop across a partitioned face: pre-projected half spinor from the ghost buffer, backward link from the pad
  template <class P, int recon, bool fwd>
  B2_HD void hop_ghost(typename P::real *r, const DslashArgs<P, recon> &arg, const int *x, int x_cb, int parity, int d)
  {
    using real = typename P::real;
    const Geom &g = arg.geom;
    real u[18], h[12];
    const int fidx = face_index(x, g, d);
    if (fwd)
      arg.U.load(u, d, x_cb, parity);
    else
      arg.U.load(u, d, g.volume_cb + fidx, 1 - parity); // ghost link lives in the pad
    GhostView<P> gv = arg.ghost[d][fwd ? 1 : 0];
    gv.v += (1 - parity) * arg.ghost_parity_stride[d];
    if constexpr (P::fixed) gv.norm += (1 - parity) * arg.ghost_norm_parity_stride[d];
    gv.load(h, fidx);
    su3_mul<!fwd>(r, u, h);
  }

  // Accumulate the hops of one output site.
  //   kt == K_INTERIOR     : every hop whose source is local (periodic wrap inside non-partitioned dims).
  //                          Written WITHOUT branches: all 16 loads of the 8 hops are unconditional so that the
  //                          compiler can issue the loads of later hops while earlier ones are being multiplied
  //                          (memory-level parallelism per warp); with partitioned dims (`part`) a hop that would
  //                          cross a partitioned boundary still loads its periodic image but is masked to zero.
  //   kt == K_EXTERIOR_ALL : only hops that cross a partitioned boundary, sources read from the ghost buffers
  //   kt == K_FULL         : all 8 hops, each from the ghost buffer if it crosses a partitioned face, else local --
  //                          used for the boundary tiles once the halo has arrived (no read-modify-write pass)
  template <class P, int recon, bool dagger, KernelType kt, bool part = true, bool pretwist = false>
  B2_HD void wilson_hops(typename P::real *acc, const DslashArgs<P, recon> &arg, const int *x, int x_cb, int parity)
  {
    using real = typename P::real;
    const Geom &g = arg.geom;
    constexpr bool preload = (kt == K_INTERIOR) && PreloadLinks<P, recon>::value;
    typename GaugeView<P, recon>::Raw raw[preload ? 8 : 1];
    if constexpr (preload) {
#pragma unroll
      for (int d = 0; d < 4; d++) {
        arg.U.load_raw(raw[2 * d], d, x_cb, parity);
        arg.U.load_raw(raw[2 * d + 1], d, neighbor_cb<false>(x, g, d), 1 - parity);
      }
    }
#pragma unroll
    for (int d = 0; d < 4; d++) {
      { // forward hop: U_d(x) P(d, dagger ? + : -) in(x + d)
        constexpr int sign = dagger ? +1 : -1;
        const bool ghost = (x[d] + 1 >= g.X[d]) && arg.comm_dim[d];
        real r[12];
        if constexpr (kt == K_INTERIOR) {
          hop_add<P, recon, dagger, true, part, Cache::STREAM, pretwist>(acc, arg, arg.in[1 - parity], x, x_cb, parity, d,
                                                                         preload ? &raw[2 * d] : nullptr, ghost ? (real)0 : (real)1);
        } else if constexpr (kt == K_EXTERIOR_ALL) {
          if (ghost) {
            hop_ghost<P, recon, true>(r, arg, x, x_cb, parity, d);
            reconstruct_add(acc, r, d, sign);
          }
        } else if constexpr (DeferredScale<P>::value) {
          if (ghost) {
            hop_ghost<P, recon, true>(r, arg, x, x_cb, parity, d);
            reconstruct_add(acc, r, d, sign);
          } else {
            hop_add<P, recon, dagger, true, false>(acc, arg, arg.in[1 - parity], x, x_cb, parity, d, nullptr, (real)1);
          }
        } else {
          if (ghost)
            hop_ghost<P, recon, true>(r, arg, x, x_cb, parity, d);
          else
            hop_local<P, recon, dagger, true>(r, arg, x, x_cb, parity, d);
          reconstruct_add(acc, r, d, sign);
        }
      }
      { // backward hop: U_d(x - d)^dagger P(d, dagger ? - : +) in(x - d)
        constexpr int sign = dagger ? -1 : +1;
        const bool ghost = (x[d] - 1 < 0) && arg.comm_dim[d];
        real r[12];
        if constexpr (kt == K_INTERIOR) {
          hop_add<P, recon, dagger, false, part, Cache::STREAM, pretwist>(acc, arg, arg.in[1 - parity], x, x_cb, parity, d,
                                                                          preload ? &raw[2 * d + 1] : nullptr, ghost ? (real)0 : (real)1);
        } else if constexpr (kt == K_EXTERIOR_ALL) {
          if (ghost) {
            hop_ghost<P, recon, false>(r, arg, x, x_cb, parity, d);
            reconstruct_add(acc, r, d, sign);
          }
        } else if constexpr (DeferredScale<P>::value) {
          if (ghost) {
            hop_ghost<P, recon, false>(r, arg, x, x_cb, parity, d);
            reconstruct_add(acc, r, d, sign);
          } else {
            hop_add<P, recon, dagger, false, false>(acc, arg, arg.in[1 - parity], x, x_cb, parity, d, nullptr, (real)1);
          }
        } else {
          if (ghost)
            hop_ghost<P, recon, false>(r, arg, x, x_cb, parity, d);
          else
            hop_local<P, recon, dagger, false>(r, arg, x, x_cb, parity, d);
          reconstruct_add(acc, r, d, sign);
        }
      }
    }
  }

  // true if every hop of this site is accounted for once the current kernel has run
  // (dslash_helper.cuh:70-89 isComplete): interior kernel -> site touches no partitioned boundary.
  template <class P, int recon> B2_HD bool site_is_interior(const DslashArgs<P, recon> &arg, const int *x)
  {
    bool inner = true;
#pragma unroll
    for (int d = 0; d < 4; d++)
      if (arg.comm_dim[d] && (x[d] == 0 || x[d] == arg.geom.X[d] - 1)) inner = false;
    return inner;
  }

  // Full site update for the interior kernel.
  //   OP_WILSON    : out = D in                     | xpay: out = x + a D in
  //   OP_CLOVER    : (xpay only)                      out = A x + a D in
  //   OP_CLOVER_PC : out = A^{-1} D in              | xpay: out = x + a A^{-1} D in
  // With partitioned dims, boundary sites only store their partial sum (the exterior kernel finishes them).
  template <class P, int recon, bool dagger, bool xpay, OpType op, bool part = true>
  B2_HD void dslash_site_interior(const DslashArgs<P, recon> &arg, const int *x, int x_cb, int parity)
  {
    using real = typename P::real;
    real acc[24];
#pragma unroll
    for (int i = 0; i < 24; i++) acc[i] = 0;
    wilson_hops<P, recon, dagger, K_INTERIOR, part, op == OP_TM_PC_PRE>(acc, arg, x, x_cb, parity);

    const bool complete = part ? site_is_interior(arg, x) : true;
    if constexpr (op == OP_CLOVER_PC) {
      if (complete) clover_apply_site<P, true>(acc, arg.A, x_cb, parity);
    }
    if constexpr (op == OP_TM_PC) {
      if (complete) twist_apply(acc, arg.a, arg.twist_b()); // a (1 + i b gamma5) D in
    }
    if constexpr (xpay) {
      real xv[24];
      arg.x[parity].template load<Cache::STREAM>(xv, x_cb);
      if constexpr (op == OP_CLOVER) clover_apply_site<P, false>(xv, arg.A, x_cb, parity);
      if constexpr (op == OP_TM) twist_apply(xv, (real)1, arg.twist_b()); // (1 + i b gamma5) x + a D in
      if constexpr (op == OP_TM_PC || op == OP_TM_PC_PRE) { // `a` is the rotation's scale here: plain x + ...
        if (complete) {
#pragma unroll
          for (int i = 0; i < 24; i++) acc[i] = xv[i] + acc[i];
        }
      } else if (op != OP_CLOVER_PC || complete) {
#pragma unroll
        for (int i = 0; i < 24; i++) acc[i] = xv[i] + arg.a * acc[i];
      }
      // OP_CLOVER_PC on an incomplete site: store the bare partial sum; x and a are applied by the exterior kernel
      // after A^{-1} (dslash_wilson_clover_preconditioned.cuh:74-101)
    }
    arg.out[parity].save(acc, x_cb);
  }

  // Complete update of a boundary site once the halo is there: all hops (local or ghost), then clover / xpay exactly as
  // for an unpartitioned lattice.  Together with the interior launch over the non-boundary tiles this replaces the
  // reference's "interior partial sums + exterior read-modify-write" split (include/kernels/dslash_wilson.cuh:186-195).
  template <class P, int recon, bool dagger, bool xpay, OpType op>
  B2_HD void dslash_site_full(const DslashArgs<P, recon> &arg, const int *x, int x_cb, int parity)
  {
    using real = typename P::real;
    real acc[24];
#pragma unroll
    for (int i = 0; i < 24; i++) acc[i] = 0;
    wilson_hops<P, recon, dagger, K_FULL>(acc, arg, x, x_cb, parity);
    if constexpr (op == OP_CLOVER_PC) clover_apply_site<P, true>(acc, arg.A, x_cb, parity);
    if constexpr (op == OP_TM_PC) twist_apply(acc, arg.a, arg.twist_b());
    if constexpr (xpay) {
      real xv[24];
      arg.x[parity].template load<Cache::STREAM>(xv, x_cb);
      if constexpr (op == OP_CLOVER) clover_apply_site<P, false>(xv, arg.A, x_cb, parity);
      if constexpr (op == OP_TM) twist_apply(xv, (real)1, arg.twist_b());
#pragma unroll
      for (int i = 0; i < 24; i++) acc[i] = xv[i] + (op == OP_TM_PC ? acc[i] : arg.a * acc[i]);
    }
    arg.out[parity].save(acc, x_cb);
  }

  // ------------------------------------------------------------------ multi-RHS (batched) stencil
  // NS sources share one gauge (and clover) field: the reference batches them through cvector_ref and a source index
  // in the thread grid (include/kernels/dslash_wilson.cuh:37-40,65-69, include/dslash_helper.cuh src_idx), relying on
  // the caches to serve the repeated link loads.  Here ONE THREAD owns a site for all NS sources: each link is loaded
  // and reconstructed once into registers and multiplied into NS independent accumulators, so the link stream (2/3 of
  // the single-source traffic) is amortised exactly -- B_min per source = 8G/NS + 2S -- and every thread has NS times
  // as many independent spinor loads in flight.
  template <class P, int NS> struct MrhsFields {
    SpinorView<P> out[NS][kMaxParity], in[NS][kMaxParity], x[NS][kMaxParity]; // [source][parity the view holds]
  };

  template <class P, int recon, bool dagger, bool fwd, int NS>
  B2_HD void hop_local_mrhs(typename P::real (*acc)[24], const DslashArgs<P, recon> &arg, const MrhsFields<P, NS> &f,
                            const int *x, int x_cb, int parity, int d, const typename GaugeView<P, recon>::Raw *raw)
  {
    using real = typename P::real;
    const Geom &g = arg.geom;
    constexpr int sign = fwd ? (dagger ? +1 : -1) : (dagger ? -1 : +1);
    real u[18];
    real us = (real)1; // deferred link scale (fixed point only)
    const int n_cb = neighbor_cb<fwd>(x, g, d);
    if constexpr (DeferredScale<P>::value) {
      if (raw) {
        arg.U.unpack_deferred(u, us, *raw, d, fwd ? x_cb : n_cb);
      } else {
        typename GaugeView<P, recon>::Raw w;
        arg.U.load_raw(w, d, fwd ? x_cb : n_cb, fwd ? parity : 1 - parity);
        arg.U.unpack_deferred(u, us, w, d, fwd ? x_cb : n_cb);
      }
    } else {
      if (raw)
        arg.U.unpack(u, *raw, d, fwd ? x_cb : n_cb);
      else if (fwd)
        arg.U.load(u, d, x_cb, parity);
      else
        arg.U.load(u, d, n_cb, 1 - parity);
    }
#pragma unroll
    for (int s = 0; s < NS; s++) {
      const SpinorView<P> &in = f.in[s][1 - parity];
      real h[12], r[12];
      if constexpr (DeferredScale<P>::value) { // same arithmetic as hop_from_deferred (bit-identical per source)
        const real n = in.load_norm(n_cb);
        real scale;
        if (d == 3) {
          load_spin_pair<P, (sign > 0), Cache::REUSE, false>(h, in, n_cb);
          scale = (us * n) * (real)2;
        } else {
          real v[24];
          in.template load_planes<0, 24 / P::Ns>(v, n_cb);
          project(h, v, d, sign);
          scale = us * n;
        }
        su3_mul<!fwd>(r, u, h);
        reconstruct_add_scaled(acc[s], r, d, sign, scale);
      } else {
        if (d == 3) {
          real t[12];
          load_spin_pair<P, (sign > 0)>(t, in, n_cb);
          twice12(h, t);
        } else {
          real v[24];
          in.load(v, n_cb);
          project(h, v, d, sign);
        }
        su3_mul<!fwd>(r, u, h);
        reconstruct_add(acc[s], r, d, sign);
      }
    }
  }

  // Unpartitioned lattices only (the launcher falls back to per-source launches otherwise).  The per-source arithmetic
  // is the single-source one operation for operation, so results are bit-identical to NS separate applications.
  template <class P, int recon, bool dagger, bool xpay, OpType op, int NS>
  B2_HD void dslash_site_mrhs(const DslashArgs<P, recon> &arg, const MrhsFields<P, NS> &f, const int *x, int x_cb, int parity)
  {
    using real = typename P::real;
    const Geom &g = arg.geom;
    real acc[NS][24];
#pragma unroll
    for (int s = 0; s < NS; s++)
#pragma unroll
      for (int i = 0; i < 24; i++) acc[s][i] = 0;

    constexpr bool preload = PreloadLinks<P, recon>::value;
    typename GaugeView<P, recon>::Raw raw[preload ? 8 : 1];
    if constexpr (preload) {
#pragma unroll
      for (int d = 0; d < 4; d++) {
        arg.U.load_raw(raw[2 * d], d, x_cb, parity);
        arg.U.load_raw(raw[2 * d + 1], d, neighbor_cb<false>(x, g, d), 1 - parity);
      }
    }
#pragma unroll
    for (int d = 0; d < 4; d++) {
      hop_local_mrhs<P, recon, dagger, true, NS>(acc, arg, f, x, x_cb, parity, d, preload ? &raw[2 * d] : nullptr);
      hop_local_mrhs<P, recon, dagger, false, NS>(acc, arg, f, x, x_cb, parity, d, preload ? &raw[2 * d + 1] : nullptr);
    }
#pragma unroll
    for (int s = 0; s < NS; s++) {
      if constexpr (op == OP_CLOVER_PC) clover_apply_site<P, true>(acc[s], arg.A, x_cb, parity);
      if constexpr (xpay) {
        real xv[24];
        f.x[s][parity].template load<Cache::STREAM>(xv, x_cb);
        if constexpr (op == OP_CLOVER) clover_apply_site<P, false>(xv, arg.A, x_cb, parity);
#pragma unroll
        for (int i = 0; i < 24; i++) acc[s][i] = xv[i] + arg.a * acc[s][i];
      }
      f.out[s][parity].save(acc[s], x_cb);
    }
  }

  // Multi-RHS, CTA flavour: one thread = one (site, source) pair, the sources of a site sit in the same CTA
  // (threadIdx.y), and the links are loaded with the default caching policy so that the first warp's miss fills L1 for
  // its siblings.  Register footprint and instruction stream per thread are those of the single-source kernel; what
  // shrinks is the DRAM traffic per source.  The reference's multi-RHS kernels work this way (source index in the
  // thread grid, include/dslash_helper.cuh:664-713).
  constexpr int kMaxRhs = 16;
  template <class P> struct MrhsViews {
    SpinorView<P> out[kMaxRhs][kMaxParity], in[kMaxRhs][kMaxParity], x[kMaxRhs][kMaxParity];
  };

  template <class P, int recon, bool dagger, bool xpay, OpType op, Cache lc, bool preload_links = true>
  B2_HD void dslash_site_src(const DslashArgs<P, recon> &arg, const SpinorView<P> &in, const SpinorView<P> &out,
                             const SpinorView<P> &xf, const int *x, int x_cb, int parity)
  {
    using real = typename P::real;
    const Geom &g = arg.geom;
    real acc[24];
#pragma unroll
    for (int i = 0; i < 24; i++) acc[i] = 0;
    constexpr bool preload = preload_links && PreloadLinks<P, recon>::value;
    typename GaugeView<P, recon>::Raw raw[preload ? 8 : 1];
    if constexpr (preload) {
#pragma unroll
      for (int d = 0; d < 4; d++) {
        arg.U.template load_raw<lc>(raw[2 * d], d, x_cb, parity);
        arg.U.template load_raw<lc>(raw[2 * d + 1], d, neighbor_cb<false>(x, g, d), 1 - parity);
      }
    }
#pragma unroll
    for (int d = 0; d < 4; d++) {
      hop_add<P, recon, dagger, true, false, lc>(acc, arg, in, x, x_cb, parity, d, preload ? &raw[2 * d] : nullptr, (real)1);
      hop_add<P, recon, dagger, false, false, lc>(acc, arg, in, x, x_cb, parity, d, preload ? &raw[2 * d + 1] : nullptr, (real)1);
    }
    if constexpr (op == OP_CLOVER_PC) clover_apply_site<P, true>(acc, arg.A, x_cb, parity);
    if constexpr (xpay) {
      real xv[24];
      xf.template load<Cache::STREAM>(xv, x_cb);
      if constexpr (op == OP_CLOVER) clover_apply_site<P, false>(xv, arg.A, x_cb, parity);
#pragma unroll
      for (int i = 0; i < 24; i++) acc[i] = xv[i] + arg.a * acc[i];
    }
    out.save(acc, x_cb);
  }

  // Exterior update: out += ghost hops (read-modify-write), applying what the interior kernel had to defer.
  template <class P, int recon, bool dagger, bool xpay, OpType op>
  B2_HD void dslash_site_exterior(const DslashArgs<P, recon> &arg, const int *x, int x_cb, int parity)
  {
    using real = typename P::real;
    real acc[24];
#pragma unroll
    for (int i = 0; i < 24; i++) acc[i] = 0;
    wilson_hops<P, recon, dagger, K_EXTERIOR_ALL>(acc, arg, x, x_cb, parity);
    real partial[24];
    arg.out[parity].template load<Cache::COHERENT>(partial, x_cb); // read-modify-write of `out`: not the .nc path
    if constexpr (op == OP_CLOVER_PC || op == OP_TM_PC) {
#pragma unroll
      for (int i = 0; i < 24; i++) acc[i] += partial[i];
      if constexpr (op == OP_CLOVER_PC)
        clover_apply_site<P, true>(acc, arg.A, x_cb, parity);
      else
        twist_apply(acc, arg.a, arg.twist_b());
      if constexpr (xpay) {
        real xv[24];
        arg.x[parity].template load<Cache::STREAM>(xv, x_cb);
#pragma unroll
        for (int i = 0; i < 24; i++) acc[i] = xv[i] + (op == OP_TM_PC ? acc[i] : arg.a * acc[i]);
      }
    } else {
#pragma unroll
      for (int i = 0; i < 24; i++) acc[i] = partial[i] + (xpay ? arg.a * acc[i] : acc[i]);
    }
    arg.out[parity].save(acc, x_cb);
  }

  // Fused-exterior thread -> (dim, face, face index) decode and the corner-ownership rule: a boundary site that lies
  // on several partitioned faces is updated once, by the thread of the highest such dimension (backward face before
  // forward face when X[d] == 2 would alias; we require X[d] >= 4 for partitioned dims so faces never alias).
  // Returns false if this thread has nothing to do.  (dslash_helper.cuh:202-242 restated.)
  template <class P, int recon>
  B2_HD bool exterior_thread_site(int *x, int &x_cb, const DslashArgs<P, recon> &arg, int tid, int parity)
  {
    const Geom &g = arg.geom;
    int d = 0;
#pragma unroll
    for (int k = 0; k < 4; k++)
      if (tid >= arg.threads_ext[k + 1]) d = k + 1;
    // threads_ext[k+1]-threads_ext[k] is 0 for non-partitioned dims, so d lands on a partitioned dim
    const int local = tid - arg.threads_ext[d];
    const int face = local >= g.face_cb[d] ? 1 : 0;
    const int idx = local - face * g.face_cb[d];
    coords_from_face(x, g, d, face ? g.X[d] - 1 : 0, idx, parity);
    // ownership: skip if a higher partitioned dimension also has this site on one of its faces
#pragma unroll
    for (int e = 0; e < 4; e++)
      if (e > d && arg.comm_dim[e] && (x[e] == 0 || x[e] == g.X[e] - 1)) return false;
    x_cb = cb_from_coords(x, g);
    return true;
  }

} // namespace b200
