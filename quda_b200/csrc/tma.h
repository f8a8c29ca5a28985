// TMA-staged, time-marching interior kernel: plan, tensor-map descriptions, per-thread shared-memory offsets and the
// site arithmetic.  Everything here is `B2_HD` so that the test-only host twin can run the SAME plan / offset / site code
// against an emulated shared memory filled by emulated box loads (tests/hosttwin) -- the CUDA-only parts (mbarrier,
// cp.async.bulk.tensor) live in tma_kernel.cuh.
//
// What it replaces: the reference's interior kernel gathers the 8 neighbour spinors straight from global memory and
// leaves their reuse to L1/L2 (/root/reference/include/kernels/dslash_wilson.cuh:84-161); on B200 that pulls 404 MB
// through the L2 -> SM crossbar for 302 MB of compulsory traffic (fp32 recon-12, DESIGN.md section 6).  Here a persistent
// CTA owns an (all x) x TY x TZ tile of one parity and marches through t:
//   * the input-spinor slice t+1 (tile rows only) and the y/z halo rows of slice t arrive in shared memory by TMA box
//     loads, several slices ahead of their use; slices t-1, t, t+1 stay resident, so every input site crosses the
//     L2 -> SM path (1 + halo) times instead of ~4 times;
//   * the 8 links of a site are a pure stream (each is read exactly once).  Two ways of feeding them, selected by
//     TmaPlan::n_link_slots:
//       >0 (default) TMA stages: one direction pair (forward + backward link of dimension d) per stage through a ring in
//          shared memory.  Shared memory only holds ~2 stages in flight (48 KB), less than bandwidth x DRAM latency, so
//          the producer first pulls the link boxes into L2 two items ahead (cp.async.bulk.prefetch.tensor) and the
//          staged loads only have to cover the L2 -> SM latency;
//       0  register stream: a thread re-issues the loads of a direction pair for a later step into the registers the
//          pair just consumed.  Measured slower on B200 (profiles/r02_tma_regstream_*): under the 168-register cap of a
//          9-warp CTA ptxas sinks the prefetch loads back down to their first use;
//   * a producer warp issues the box loads, the consumer warps wait on mbarriers -- no __syncthreads in the loop.
// Work is the linearised (tile, t) sequence cut into gridDim.x equal ranges (148 SMs do not divide 2^k tiles).
#pragma once

#include "dslash_site.h"

namespace b200
{

  constexpr int kTmaMaxCenterSlots = 8; // slices t-1, t, t+1 live + look-ahead
  constexpr int kTmaMaxHaloSlots = 4;   // halo rows of slice t live + look-ahead
  constexpr int kTmaMaxLinkSlots = 4;
  constexpr int kTmaSmemBudget = 227 * 1024;
  constexpr int kTmaMaxConsumers = 256;

  // box shapes; one tensor map per (output parity, shape)
  enum TmaMapId {
    TM_SC = 0,  // spinor tile rows      (TY, TZ)
    TM_SY = 1,  // spinor y-halo rows    (1, TZ)
    TM_SZ = 2,  // spinor z-halo rows    (TY, 1)
    TM_GF = 3,  // forward links, output parity           (TY, TZ)
    TM_GB = 4,  // backward links x / t, other parity     (TY, TZ)
    TM_GYA = 5, // backward y links, row y0-1             (1, TZ)
    TM_GYB = 6, // backward y links, rows y0 .. y0+TY-2   (TY-1, TZ)
    TM_GZA = 7, // backward z links, row z0-1             (TY, 1)
    TM_GZB = 8, // backward z links, rows z0 .. z0+TZ-2   (TY, TZ-1)
    TM_COUNT = 9
  };

  // Description of one tiled tensor map over a native field: 5-d (u32 lane within an x row, plane, y, z, t).
  // The device launcher turns it into a CUtensorMap; the host twin interprets it directly.
  struct TmaDesc {
    const void *base;
    unsigned long long dim[5];    // elements (u32) / planes / sites
    unsigned long long stride[5]; // bytes; stride[0] = 4
    unsigned box[5];
    int valid;                    // 0: shape has a zero extent (TY == 1 or TZ == 1) or is not used in this mode
  };

  struct TmaPlan {
    int Xh, Y, Z, T;
    int TY, TZ, nty, ntz;
    int n_parity, parity;
    int n_items;      // n_parity * nty * ntz * T
    int n_consumers;  // Xh * TY * TZ
    int n_cwarps;     // consumer warps
    int svec, gvec;   // bytes per spinor / gauge vector
    int SP, GP;       // planes per spinor / per link
    int srow, grow;   // bytes of one (y,z) row record: SP * svec * Xh, GP * gvec * Xh
    int NC, NH;       // tile rows, halo rows
    int center_bytes, halo_bytes, link_bytes; // per slot (128-byte aligned)
    int n_center_slots, n_halo_slots, n_link_slots; // n_link_slots == 0: links are a register stream
    int l2_prefetch_items; // shared-memory link stages: items of look-ahead of the L2 prefetch of the link boxes (0: off)
    int off_center, off_halo, off_link, off_bar, smem_bytes;
  };

  B2_HD int tma_align128(int v) { return (v + 127) & ~127; }

  // mbarrier slots inside the barrier block (8 bytes each)
  B2_HD int tma_bar_full_c(int s) { return s; }
  B2_HD int tma_bar_empty_c(int s) { return kTmaMaxCenterSlots + s; }
  B2_HD int tma_bar_full_h(int s) { return 2 * kTmaMaxCenterSlots + s; }
  B2_HD int tma_bar_empty_h(int s) { return 2 * kTmaMaxCenterSlots + kTmaMaxHaloSlots + s; }
  B2_HD int tma_bar_full_l(int s) { return 2 * kTmaMaxCenterSlots + 2 * kTmaMaxHaloSlots + s; }
  B2_HD int tma_bar_empty_l(int s) { return 2 * kTmaMaxCenterSlots + 2 * kTmaMaxHaloSlots + kTmaMaxLinkSlots + s; }
  constexpr int kTmaBarriers = 2 * kTmaMaxCenterSlots + 2 * kTmaMaxHaloSlots + 2 * kTmaMaxLinkSlots;

  // position in a ring of R slots: slot index + parity of the current pass over the ring (the mbarrier phase parity)
  struct TmaPos {
    int slot;
    unsigned phase;
  };
  B2_HD TmaPos tma_pos_next(TmaPos p, int R)
  {
    if (++p.slot == R) {
      p.slot = 0;
      p.phase ^= 1u;
    }
    return p;
  }

  // tuning knobs of the plan (0 = built-in choice)
  struct TmaKnobs {
    int ty, tz;          // tile
    int link_slots;      // 0: shared-memory stages, as many as fit (default); >= 2: that many stages; -1: register stream
    int center_slots, halo_slots; // register-stream mode: cap the spinor rings
    int l2_prefetch;     // shared-memory link stages: L2 prefetch look-ahead in items (<= 0: off, the default)
  };

  // Build the plan for a lattice / precision / reconstruct.  Returns false if this shape is not served by the TMA
  // kernel (the caller falls back to the gather kernel): x rows must fit one box, the tile must divide the lattice and
  // the spinor slices (+ >= 2 link stages in the shared-memory link mode) must fit in shared memory.
  template <class P, int recon> B2_HD bool tma_make_plan(TmaPlan &p, const Geom &g, int n_parity, int parity, const TmaKnobs &k)
  {
    using GV = GaugeView<P, recon>;
    p.Xh = g.Xh0;
    p.Y = g.X[1];
    p.Z = g.X[2];
    p.T = g.X[3];
    p.n_parity = n_parity;
    p.parity = parity;
    p.svec = (int)sizeof(typename P::svec);
    p.gvec = (int)sizeof(typename GV::V);
    p.SP = 24 / P::Ns;
    p.GP = GV::M;
    if (P::fixed) return false;                                  // block-float norms would need their own maps
    if (p.svec * p.Xh / 4 > 256 || p.gvec * p.Xh / 4 > 256) return false; // box extent limit
    if ((p.svec * p.Xh) % 16 || (p.gvec * p.Xh) % 16) return false;      // inner box bytes / strides: multiples of 16
    if (p.T < 3) return false;                                   // t-1, t, t+1 must be distinct slices
    // tile: powers of two dividing Y and Z, grown alternately (y first) up to the consumer budget
    const int budget = sizeof(typename P::real) == 8 ? 128 : kTmaMaxConsumers;
    int ty = 1, tz = 1;
    if (k.ty > 0 && k.tz > 0) {
      ty = k.ty;
      tz = k.tz;
      if (p.Y % ty || p.Z % tz) return false;
    } else {
      for (;;) {
        bool grown = false;
        if (ty <= tz && p.Y % (2 * ty) == 0 && p.Xh * 2 * ty * tz <= budget) { ty *= 2; grown = true; }
        else if (p.Z % (2 * tz) == 0 && p.Xh * ty * 2 * tz <= budget) { tz *= 2; grown = true; }
        else if (p.Y % (2 * ty) == 0 && p.Xh * 2 * ty * tz <= budget) { ty *= 2; grown = true; }
        if (!grown) break;
      }
    }
    if (p.Xh * ty * tz > kTmaMaxConsumers) return false;
    p.TY = ty;
    p.TZ = tz;
    p.nty = p.Y / ty;
    p.ntz = p.Z / tz;
    p.n_items = n_parity * p.nty * p.ntz * p.T;
    p.n_consumers = p.Xh * ty * tz;
    p.n_cwarps = (p.n_consumers + 31) / 32;
    p.srow = p.SP * p.svec * p.Xh;
    p.grow = p.GP * p.gvec * p.Xh;
    p.NC = ty * tz;
    p.NH = 2 * tz + 2 * ty;
    p.center_bytes = tma_align128(p.NC * p.srow);
    // halo regions (ym, yp, zm, zp) each start 128-byte aligned
    p.halo_bytes = 2 * tma_align128(tz * p.srow) + 2 * tma_align128(ty * p.srow);
    // link stage: forward block, then the backward block (two boxes for y and z: region A, region B)
    // (region A holds max(TY,TZ) rows, region B the remaining NC - min(TY,TZ); the x / t boxes of NC rows start at A)
    {
      const int mx = ty > tz ? ty : tz, mn = ty > tz ? tz : ty;
      int bwd = tma_align128(mx * p.grow) + tma_align128((p.NC - mn) * p.grow);
      if (bwd < tma_align128(p.NC * p.grow)) bwd = tma_align128(p.NC * p.grow);
      p.link_bytes = tma_align128(p.NC * p.grow) + bwd;
    }
    const int avail = kTmaSmemBudget - 1024;
    if (k.link_slots >= 0) { // links through shared memory: minimal spinor rings, the rest to link stages
      p.n_center_slots = 4;
      p.n_halo_slots = 2;
      int nl = (avail - 4 * p.center_bytes - 2 * p.halo_bytes) / p.link_bytes;
      if (nl > kTmaMaxLinkSlots) nl = kTmaMaxLinkSlots;
      if (k.link_slots >= 2 && k.link_slots < nl) nl = k.link_slots;
      if (nl < 2) return false;
      p.n_link_slots = nl;
    } else { // register stream: shared memory holds spinors only -> deeper rings (a centre slot per halo slot first)
      p.n_link_slots = 0;
      int nc = 4, nh = 2;
      for (;;) {
        if (nc < kTmaMaxCenterSlots && nc - 2 <= nh && (nc + 1) * p.center_bytes + nh * p.halo_bytes <= avail)
          nc++;
        else if (nh < kTmaMaxHaloSlots && nc * p.center_bytes + (nh + 1) * p.halo_bytes <= avail)
          nh++;
        else
          break;
      }
      if (k.center_slots >= 4 && k.center_slots < nc) nc = k.center_slots;
      if (k.halo_slots >= 2 && k.halo_slots < nh) nh = k.halo_slots;
      if (nc * p.center_bytes + nh * p.halo_bytes > avail) return false;
      p.n_center_slots = nc;
      p.n_halo_slots = nh;
    }
    p.l2_prefetch_items = k.l2_prefetch <= 0 ? 0 : k.l2_prefetch; // (measured: the extra producer work costs more than it hides)
    p.off_center = 0;
    p.off_halo = p.off_center + p.n_center_slots * p.center_bytes;
    p.off_link = p.off_halo + p.n_halo_slots * p.halo_bytes;
    p.off_bar = p.off_link + p.n_link_slots * p.link_bytes;
    p.smem_bytes = p.off_bar + 1024;
    return p.smem_bytes <= kTmaSmemBudget;
  }

  // byte offsets of the regions inside a halo slot / a link stage
  B2_HD int tma_halo_ym(const TmaPlan &) { return 0; }
  B2_HD int tma_halo_yp(const TmaPlan &p) { return tma_align128(p.TZ * p.srow); }
  B2_HD int tma_halo_zm(const TmaPlan &p) { return 2 * tma_align128(p.TZ * p.srow); }
  B2_HD int tma_halo_zp(const TmaPlan &p) { return 2 * tma_align128(p.TZ * p.srow) + tma_align128(p.TY * p.srow); }
  B2_HD int tma_link_bwd_a(const TmaPlan &p) { return tma_align128(p.NC * p.grow); }
  B2_HD int tma_link_bwd_b(const TmaPlan &p)
  {
    return tma_align128(p.NC * p.grow) + tma_align128((p.TY > p.TZ ? p.TY : p.TZ) * p.grow);
  }

  // ---- tensor-map descriptions ------------------------------------------------------------------------------------
  // field of one parity: (u32 lane, plane, y, z, t)
  B2_HD void tma_desc_field(TmaDesc &d, const void *base, int vec_bytes, int planes, size_t plane_stride_sites, const TmaPlan &p,
                            int box_planes, int by, int bz)
  {
    d.base = base;
    d.dim[0] = (unsigned long long)(vec_bytes / 4) * p.Xh;
    d.dim[1] = planes;
    d.dim[2] = p.Y;
    d.dim[3] = p.Z;
    d.dim[4] = p.T;
    d.stride[0] = 4;
    d.stride[1] = (unsigned long long)vec_bytes * plane_stride_sites;
    d.stride[2] = (unsigned long long)vec_bytes * p.Xh;
    d.stride[3] = d.stride[2] * p.Y;
    d.stride[4] = d.stride[3] * p.Z;
    d.box[0] = (unsigned)d.dim[0];
    d.box[1] = box_planes;
    d.box[2] = by;
    d.box[3] = bz;
    d.box[4] = 1;
    d.valid = (by > 0 && bz > 0) ? 1 : 0;
  }

  // all maps for output parity `par` (input spinor and backward links have parity 1 - par)
  template <class P, int recon> B2_HD void tma_make_descs(TmaDesc *d, const DslashArgs<P, recon> &arg, const TmaPlan &p, int par)
  {
    const void *in = arg.in[1 - par].v;
    const size_t sst = arg.in[1 - par].stride;
    tma_desc_field(d[TM_SC], in, p.svec, p.SP, sst, p, p.SP, p.TY, p.TZ);
    tma_desc_field(d[TM_SY], in, p.svec, p.SP, sst, p, p.SP, 1, p.TZ);
    tma_desc_field(d[TM_SZ], in, p.svec, p.SP, sst, p, p.SP, p.TY, 1);
    const void *gf = arg.U.g[par], *gb = arg.U.g[1 - par];
    const size_t gst = arg.U.stride;
    tma_desc_field(d[TM_GF], gf, p.gvec, 4 * p.GP, gst, p, p.GP, p.TY, p.TZ);
    tma_desc_field(d[TM_GB], gb, p.gvec, 4 * p.GP, gst, p, p.GP, p.TY, p.TZ);
    tma_desc_field(d[TM_GYA], gb, p.gvec, 4 * p.GP, gst, p, p.GP, 1, p.TZ);
    tma_desc_field(d[TM_GYB], gb, p.gvec, 4 * p.GP, gst, p, p.GP, p.TY - 1, p.TZ);
    tma_desc_field(d[TM_GZA], gb, p.gvec, 4 * p.GP, gst, p, p.GP, p.TY, 1);
    tma_desc_field(d[TM_GZB], gb, p.gvec, 4 * p.GP, gst, p, p.GP, p.TY, p.TZ - 1);
    if (p.n_link_slots == 0)
      for (int k = TM_GF; k < TM_COUNT; k++) d[k].valid = 0; // register-stream links: no gauge maps
  }

  // a tensor map is only usable if the hardware constraints hold (cuTensorMapEncodeTiled): 16-byte aligned base and strides
  B2_HD bool tma_desc_ok(const TmaDesc &d)
  {
    if (!d.valid) return true;
    if (((unsigned long long)(size_t)d.base) & 15) return false;
    for (int i = 1; i < 5; i++)
      if (d.stride[i] % 16 || d.stride[i] >= (1ull << 40)) return false;
    for (int i = 0; i < 5; i++)
      if (d.box[i] == 0 || d.box[i] > 256) return false;
    return true;
  }

  // ---- work items ---------------------------------------------------------------------------------------------------
  struct TmaItem {
    int par, y0, z0, t; // output parity, tile origin, time slice
  };

  B2_HD void tma_item(TmaItem &it, const TmaPlan &p, int w)
  {
    const int tile = w / p.T;
    it.t = w - tile * p.T;
    const int per_par = p.nty * p.ntz;
    const int pi = tile / per_par;
    const int r = tile - pi * per_par;
    const int tzi = r / p.nty;
    it.par = p.n_parity == 2 ? pi : p.parity;
    it.y0 = (r - tzi * p.nty) * p.TY;
    it.z0 = tzi * p.TZ;
  }

  // item w + 1 given item w (the common case -- same tile, next slice -- without integer division)
  B2_HD void tma_item_next(TmaItem &nx, const TmaItem &it, const TmaPlan &p, int w_next)
  {
    if (it.t + 1 < p.T) {
      nx = it;
      nx.t = it.t + 1;
    } else {
      tma_item(nx, p, w_next);
    }
  }

  B2_HD void tma_work_range(int &w0, int &w1, const TmaPlan &p, int cta, int n_cta)
  {
    w0 = (int)((long long)p.n_items * cta / n_cta);
    w1 = (int)((long long)p.n_items * (cta + 1) / n_cta);
  }

  // One box load: which map, where (coordinates: lane, plane, y, z, t), destination offset inside the slot.
  struct TmaBox {
    int map, c[5], dst;
  };

  B2_HD int tma_wrap(int v, int n) { return v < 0 ? v + n : (v >= n ? v - n : v); }

  // input-spinor tile rows of slice s (already wrapped into [0, T))
  B2_HD void tma_center_box(TmaBox &b, const TmaItem &it, int s)
  {
    b.map = TM_SC;
    b.c[0] = 0, b.c[1] = 0, b.c[2] = it.y0, b.c[3] = it.z0, b.c[4] = s;
    b.dst = 0;
  }

  // the four halo boxes of slice it.t
  B2_HD void tma_halo_boxes(TmaBox *b, const TmaPlan &p, const TmaItem &it)
  {
    for (int k = 0; k < 4; k++) b[k].c[0] = 0, b[k].c[1] = 0, b[k].c[2] = it.y0, b[k].c[3] = it.z0, b[k].c[4] = it.t;
    b[0].map = TM_SY, b[0].c[2] = tma_wrap(it.y0 - 1, p.Y), b[0].dst = tma_halo_ym(p);
    b[1].map = TM_SY, b[1].c[2] = tma_wrap(it.y0 + p.TY, p.Y), b[1].dst = tma_halo_yp(p);
    b[2].map = TM_SZ, b[2].c[3] = tma_wrap(it.z0 - 1, p.Z), b[2].dst = tma_halo_zm(p);
    b[3].map = TM_SZ, b[3].c[3] = tma_wrap(it.z0 + p.TZ, p.Z), b[3].dst = tma_halo_zp(p);
  }

  // boxes of link stage (item, d): returns how many (2 or 3)
  B2_HD int tma_link_boxes(TmaBox *b, const TmaPlan &p, const TmaItem &it, int d)
  {
    for (int k = 0; k < 3; k++) b[k].c[0] = 0, b[k].c[1] = d * p.GP, b[k].c[2] = it.y0, b[k].c[3] = it.z0, b[k].c[4] = it.t;
    b[0].map = TM_GF, b[0].dst = 0;
    int n = 2;
    switch (d) {
    case 0: b[1].map = TM_GB, b[1].dst = tma_link_bwd_a(p); break;
    case 1:
      b[1].map = TM_GYA, b[1].c[2] = tma_wrap(it.y0 - 1, p.Y), b[1].dst = tma_link_bwd_a(p);
      if (p.TY > 1) b[2].map = TM_GYB, b[2].dst = tma_link_bwd_b(p), n = 3;
      break;
    case 2:
      b[1].map = TM_GZA, b[1].c[3] = tma_wrap(it.z0 - 1, p.Z), b[1].dst = tma_link_bwd_a(p);
      if (p.TZ > 1) b[2].map = TM_GZB, b[2].dst = tma_link_bwd_b(p), n = 3;
      break;
    default: b[1].map = TM_GB, b[1].c[4] = tma_wrap(it.t - 1, p.T), b[1].dst = tma_link_bwd_a(p); break;
    }
    return n;
  }

  // The producer's program: the order in which the box loads of the work range [w0, w1) are requested.  Every request
  // may block until its ring slot has been released, so the order must follow the order in which the slots become free:
  //   link stage (w, d)      -- slot of stage (w, d) - NL, released when the consumers are done with that direction pair;
  //   "early" loads of w + 1 -- the slice the item needs first that its predecessor did not already hold (t + 1, or
  //                             t - 1 at the start of a chunk) and its halo rows: with minimal rings their slots are
  //                             released at the end of item w - 1, i.e. together with link stage (w - 1, 3): requested
  //                             just before link stage (w, NL);
  //   "late" loads           -- chunk start only: slices t and t + 1, whose slots the previous chunk releases at its very
  //                             end: requested after the last link stage of item w.
  // Centre, halo and link requests each carry consecutive sequence numbers (n-th load of that ring).
  // `Issuer` provides center(n, item, slice), halo(n, item), link(ln, item, d): the CUDA kernel waits on the empty
  // barrier and issues the TMA loads, the host twin records / replays them.
  template <class Issuer> B2_HD void tma_producer_program(const TmaPlan &plan, int w0, int w1, Issuer &is)
  {
    const int NL = plan.n_link_slots;
    int cn = 0, hn = 0;
    long long ln = 0;
    TmaItem it;
    tma_item(it, plan, w0);
    // chunk start: slices t-1 (early), t and t+1 (late)
    is.center(cn, it, tma_wrap(it.t - 1, plan.T));
    is.halo(hn, it);
    is.center(cn + 1, it, it.t);
    is.center(cn + 2, it, tma_wrap(it.t + 1, plan.T));
    // Shared memory holds only ~2 link stages in flight, less than bandwidth x DRAM latency: the link boxes are therefore
    // first pulled into L2 `pf` items ahead (cp.async.bulk.prefetch.tensor, no shared memory involved), so that the
    // staged loads only have to cover the L2 -> SM latency.
    const int pf = NL > 0 ? plan.l2_prefetch_items : 0;
    for (int k = 1; k < pf && w0 + k < w1; k++) {
      TmaItem pi;
      tma_item(pi, plan, w0 + k);
      for (int d = 0; d < 4; d++) is.prefetch_link(pi, d);
    }
    for (int w = w0; w < w1; w++) {
      if (pf > 0 && w + pf < w1) {
        TmaItem pi;
        tma_item(pi, plan, w + pf);
        for (int d = 0; d < 4; d++) is.prefetch_link(pi, d);
      }
      const bool last = (w == w1 - 1) || (it.t == plan.T - 1);
      const int cn_next = cn + (last ? 3 : 1);
      TmaItem nx = it;
      const bool have_next = w + 1 < w1;
      if (have_next) tma_item_next(nx, it, plan, w + 1);
#pragma unroll 1
      for (int d = 0; d <= 4; d++) { // (not unrolled: the producer's code competes with the consumers' for the 32 KB L1.5 I-cache)
        if (have_next && (d == NL || (d == 4 && NL >= 4))) { // early loads of the next item
          if (last)
            is.center(cn_next, nx, tma_wrap(nx.t - 1, plan.T));
          else
            is.center(cn_next + 2, nx, tma_wrap(nx.t + 1, plan.T));
          is.halo(hn + 1, nx);
        }
        if (d < 4 && NL > 0) is.link(ln++, it, d);
      }
      if (have_next && last) {
        is.center(cn_next + 1, nx, nx.t);
        is.center(cn_next + 2, nx, tma_wrap(nx.t + 1, plan.T));
      }
      cn = cn_next;
      hn++;
      it = nx;
    }
  }

  B2_HD int tma_box_bytes(const TmaDesc &d) { return (int)(4u * d.box[0] * d.box[1] * d.box[2] * d.box[3] * d.box[4]); }

  // ---- per-thread shared-memory offsets -----------------------------------------------------------------------------
  struct TmaThread {
    int active;
    int xh, ly, lz;
    int o_row;                      // own tile row record (centre slots): (lz*TY + ly) * srow
    int o_yp, o_ym, o_zp, o_zm;     // neighbour row records: offset inside the centre slot or the halo slot
    int h_yp, h_ym, h_zp, h_zm;     // 1: the record lives in the halo slot
    int g_f, g_bx, g_by, g_bz, g_bt; // link row records inside a stage (without the x lane)
  };

  B2_HD void tma_thread_init(TmaThread &th, const TmaPlan &p, int tid)
  {
    th.active = tid < p.n_consumers;
    const int l = th.active ? tid : 0;
    th.xh = l % p.Xh;
    const int r = l / p.Xh;
    th.ly = r % p.TY;
    th.lz = r / p.TY;
    const int row = th.lz * p.TY + th.ly;
    th.o_row = row * p.srow;
    th.h_yp = th.ly + 1 >= p.TY;
    th.o_yp = th.h_yp ? tma_halo_yp(p) + th.lz * p.srow : (row + 1) * p.srow;
    th.h_ym = th.ly == 0;
    th.o_ym = th.h_ym ? tma_halo_ym(p) + th.lz * p.srow : (row - 1) * p.srow;
    th.h_zp = th.lz + 1 >= p.TZ;
    th.o_zp = th.h_zp ? tma_halo_zp(p) + th.ly * p.srow : (row + p.TY) * p.srow;
    th.h_zm = th.lz == 0;
    th.o_zm = th.h_zm ? tma_halo_zm(p) + th.ly * p.srow : (row - p.TY) * p.srow;
    th.g_f = row * p.grow;
    th.g_bx = tma_link_bwd_a(p) + row * p.grow;
    th.g_bt = th.g_bx;
    th.g_by = th.ly == 0 ? tma_link_bwd_a(p) + th.lz * p.grow : tma_link_bwd_b(p) + (th.lz * (p.TY - 1) + th.ly - 1) * p.grow;
    th.g_bz = th.lz == 0 ? tma_link_bwd_a(p) + th.ly * p.grow : tma_link_bwd_b(p) + ((th.lz - 1) * p.TY + th.ly) * p.grow;
  }

  // Checkerboard indices of one output site of an item: the site itself (forward links, output, x, clover), its four
  // backward neighbours (backward links; periodic wrap inside the local lattice) and rpar = (y + z + t + parity) & 1,
  // which fixes x = 2 xh + rpar and with it which x lane of the input row the +-x neighbours sit in.
  struct TmaSite {
    int x_cb, b[4], rpar, par;
  };

  B2_HD void tma_site(TmaSite &s, const TmaPlan &p, const TmaThread &th, const TmaItem &it)
  {
    const int y = it.y0 + th.ly, z = it.z0 + th.lz;
    const int row = z * p.Y + y;
    const int slice = p.Xh * p.Y * p.Z;
    const int in_slice = row * p.Xh + th.xh;
    s.par = it.par;
    s.rpar = (y + z + it.t + it.par) & 1;
    s.x_cb = it.t * slice + in_slice;
    const int xhm = s.rpar ? th.xh : (th.xh == 0 ? p.Xh - 1 : th.xh - 1);
    s.b[0] = it.t * slice + row * p.Xh + xhm;
    s.b[1] = s.x_cb + (y == 0 ? (p.Y - 1) * p.Xh : -p.Xh);
    s.b[2] = s.x_cb + (z == 0 ? (p.Z - 1) * p.Y * p.Xh : -p.Y * p.Xh);
    s.b[3] = (it.t == 0 ? p.T - 1 : it.t - 1) * slice + in_slice;
  }

  // ---- shared-memory loads --------------------------------------------------------------------------------------------
#if defined(__CUDACC__)
  using sptr = unsigned; // shared::cta window address (nvcc's host pass never executes the loads below)
#else
  using sptr = const unsigned char *; // host twin: emulated shared memory
#endif

  template <typename V> B2_HD V lds(sptr p)
  {
#if defined(__CUDA_ARCH__)
    static_assert(sizeof(V) == 16 || sizeof(V) == 8, "vector width");
    if constexpr (sizeof(V) == 16) {
      uint4 r;
      asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(p));
      return *reinterpret_cast<V *>(&r);
    } else {
      uint2 r;
      asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "r"(p));
      return *reinterpret_cast<V *>(&r);
    }
#elif defined(__CUDACC__)
    (void)p;
    return V {};
#else
    V v;
    memcpy(&v, p, sizeof(V));
    return v;
#endif
  }

  // planes [p0, p0 + np) of the spinor record at `rec` (already offset to this thread's x lane); plane stride = row_bytes
  template <class P, int p0, int np> B2_HD void lds_planes(typename P::real *out, sptr rec, int row_bytes)
  {
    using V = typename P::svec;
#pragma unroll
    for (int i = 0; i < np; i++) {
      const V t = lds<V>(rec + (p0 + i) * row_bytes);
      vec_to_real(out + i * P::Ns, t);
    }
  }

  template <class P, int recon> B2_HD void lds_link(typename GaugeView<P, recon>::Raw &raw, sptr rec, int row_bytes)
  {
    using GV = GaugeView<P, recon>;
#pragma unroll
    for (int i = 0; i < GV::M; i++) raw.w[i] = lds<typename GV::V>(rec + i * row_bytes);
  }

  // One hop with the neighbour spinor in shared memory and the link already unpacked; arithmetic identical to hop_from
  // (dslash_site.h) operation for operation.
  template <class P, bool dagger, bool fwd, int d>
  B2_HD void tma_hop(typename P::real *acc, const typename P::real *u, sptr spinor_rec, int srow_bytes)
  {
    using real = typename P::real;
    constexpr int sign = fwd ? (dagger ? +1 : -1) : (dagger ? -1 : +1);
    real h[12], r[12];
    if constexpr (d == 3) {
      constexpr int np = 12 / P::Ns;
      real t[12];
      lds_planes<P, (sign > 0) ? 0 : np, np>(t, spinor_rec, srow_bytes);
      twice12(h, t);
    } else {
      real v[24];
      lds_planes<P, 0, 24 / P::Ns>(v, spinor_rec, srow_bytes);
      project(h, v, d, sign);
    }
    su3_mul<!fwd>(r, u, h);
    reconstruct_add(acc, r, d, sign);
  }

  // Slot bases of the current item
  struct TmaBases {
    sptr cm, c0, cp, halo; // centre slots holding slices t-1, t, t+1; halo slot of slice t
  };

  // shared-memory records of the forward / backward neighbour spinor of dimension d (x lane included)
  template <int d> B2_HD void tma_neighbours(sptr &nf, sptr &nb, const TmaPlan &p, const TmaThread &th, const TmaBases &b, int rpar)
  {
    const int xs = th.xh * p.svec;
    if constexpr (d == 0) {
      const int xhp = rpar ? (th.xh + 1 == p.Xh ? 0 : th.xh + 1) : th.xh;
      const int xhm = rpar ? th.xh : (th.xh == 0 ? p.Xh - 1 : th.xh - 1);
      nf = b.c0 + th.o_row + xhp * p.svec;
      nb = b.c0 + th.o_row + xhm * p.svec;
    } else if constexpr (d == 1) {
      nf = (th.h_yp ? b.halo : b.c0) + th.o_yp + xs;
      nb = (th.h_ym ? b.halo : b.c0) + th.o_ym + xs;
    } else if constexpr (d == 2) {
      nf = (th.h_zp ? b.halo : b.c0) + th.o_zp + xs;
      nb = (th.h_zm ? b.halo : b.c0) + th.o_zm + xs;
    } else {
      nf = b.cp + th.o_row + xs;
      nb = b.cm + th.o_row + xs;
    }
  }

  // forward + backward hop of dimension d, links from the shared-memory stage `stage`
  template <class P, int recon, bool dagger, int d>
  B2_HD void tma_hop_pair(typename P::real *acc, const GaugeView<P, recon> &U, const TmaPlan &p, const TmaThread &th,
                          const TmaBases &b, sptr stage, const TmaSite &s)
  {
    using real = typename P::real;
    const int srow_b = p.svec * p.Xh, grow_b = p.gvec * p.Xh; // plane strides inside a record
    sptr nf, nb;
    tma_neighbours<d>(nf, nb, p, th, b, s.rpar);
    const int xhm = s.rpar ? th.xh : (th.xh == 0 ? p.Xh - 1 : th.xh - 1);
    const int g_b = d == 0 ? th.g_bx + xhm * p.gvec : (d == 1 ? th.g_by : (d == 2 ? th.g_bz : th.g_bt)) + th.xh * p.gvec;
    typename GaugeView<P, recon>::Raw raw;
    real u[18];
    lds_link<P, recon>(raw, stage + th.g_f + th.xh * p.gvec, grow_b);
    U.unpack(u, raw, d, s.x_cb);
    tma_hop<P, dagger, true, d>(acc, u, nf, srow_b);
    lds_link<P, recon>(raw, stage + g_b, grow_b);
    U.unpack(u, raw, d, s.b[d]);
    tma_hop<P, dagger, false, d>(acc, u, nb, srow_b);
  }

  // Register-stream links: lk[2e], lk[2e+1] hold the packed forward / backward link of dimension e.  At step d the pair
  // of dimension d is consumed (unpacked right here) and the loads of the pair that will be needed PD steps later --
  // dimension (d + PD) % 4 of this item, or of the next one (`nx`) once d + PD wraps -- are issued into its registers,
  // which have been dead since that pair was consumed.  PD = 4 gives every load a whole item (~4 us) at 96 live link
  // registers (fp32 recon-12), PD = 2 half an item at 48.
  template <class P, int recon, bool dagger, int d, int PD>
  B2_HD void tma_hop_pair_stream(typename P::real *acc, const GaugeView<P, recon> &U, typename GaugeView<P, recon>::Raw *lk,
                                 const TmaPlan &p, const TmaThread &th, const TmaBases &b, const TmaSite &s, const TmaSite &nx,
                                 bool have_next)
  {
    using real = typename P::real;
    static_assert(PD >= 1 && PD <= 4, "prefetch distance in direction pairs");
    constexpr int e = (d + PD) & 3;
    constexpr bool wraps = d + PD >= 4;
    const int srow_b = p.svec * p.Xh;
    sptr nf, nb;
    tma_neighbours<d>(nf, nb, p, th, b, s.rpar);
    real u[18];
    const bool reload = !wraps || have_next;
    const TmaSite &tg = wraps ? nx : s;
    U.unpack(u, lk[2 * d], d, s.x_cb);
    if (reload) U.template load_raw<Cache::STREAM>(lk[2 * e], e, tg.x_cb, tg.par);
    tma_hop<P, dagger, true, d>(acc, u, nf, srow_b);
    U.unpack(u, lk[2 * d + 1], d, s.b[d]);
    if (reload) U.template load_raw<Cache::STREAM>(lk[2 * e + 1], e, tg.b[e], 1 - tg.par);
    tma_hop<P, dagger, false, d>(acc, u, nb, srow_b);
  }

  // the first PD direction pairs of a site (start of a work range: nothing has been prefetched yet)
  template <class P, int recon, int PD>
  B2_HD void tma_load_links(typename GaugeView<P, recon>::Raw *lk, const GaugeView<P, recon> &U, const TmaSite &s)
  {
#pragma unroll
    for (int d = 0; d < PD; d++) {
      U.template load_raw<Cache::STREAM>(lk[2 * d], d, s.x_cb, s.par);
      U.template load_raw<Cache::STREAM>(lk[2 * d + 1], d, s.b[d], 1 - s.par);
    }
  }

  // clover / twist / xpay epilogue and store: the `complete` branch of dslash_site_interior (unpartitioned lattice)
  template <class P, int recon, bool dagger, bool xpay, OpType op>
  B2_HD void tma_epilogue(typename P::real *acc, const DslashArgs<P, recon> &arg, int x_cb, int parity)
  {
    using real = typename P::real;
    if constexpr (op == OP_CLOVER_PC) clover_apply_site<P, true>(acc, arg.A, x_cb, parity);
    if constexpr (op == OP_TM_PC) twist_apply(acc, arg.a, arg.twist_b());
    if constexpr (xpay) {
      real xv[24];
      arg.x[parity].template load<Cache::STREAM>(xv, x_cb);
      if constexpr (op == OP_CLOVER) clover_apply_site<P, false>(xv, arg.A, x_cb, parity);
      if constexpr (op == OP_TM) twist_apply(xv, (real)1, arg.twist_b());
      if constexpr (op == OP_TM_PC) {
#pragma unroll
        for (int i = 0; i < 24; i++) acc[i] = xv[i] + acc[i];
      } else {
#pragma unroll
        for (int i = 0; i < 24; i++) acc[i] = xv[i] + arg.a * acc[i];
      }
    }
    arg.out[parity].save(acc, x_cb);
  }

} // namespace b200
