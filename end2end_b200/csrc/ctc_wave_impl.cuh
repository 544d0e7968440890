// K2 "wave" kernel -- the whole fused loss path (row log-softmax, alpha/beta lattice, gradient write) for
// small alphabets, organised so that the per-frame dependent chain carries nothing but the recurrence.
//
// Replaces CTCLossEngine::compute_2d (src/losses/ctc_loss.cpp:15-118): extended targets (:25-31),
// alpha (:33-61), loss (:63-70), beta (:72-100), alpha+beta / gradient (:102-117), plus F.log_softmax
// (pytorch_end2end/modules/ctc_loss.py:40) and the exp(logits) term of the gradient (:117).
//
// Design (DESIGN.md section 4, "K2w"):
//  * One 2-CTA cluster per utterance: CTA 0 sweeps alpha forward in time, CTA 1 sweeps beta backward,
//    concurrently on two SMs.  The beta recursion is the alpha recursion of the REVERSED label sequence
//    over REVERSED time, so both CTAs run the same code: the backward CTA reverses its labels once and
//    indexes lattice cell m' = S-1-m.  Each sweep stores its first half of the frames to a global stash
//    (L2), the two meet once through a global flag, and in its second half each multiplies its own cells
//    with the other sweep's stashed row: the dependent chain is T frames, not 2T.
//  * Warp roles inside a CTA, decoupled by shared-memory rings and monotonic progress words
//    (st.release / ld.acquire at CTA scope, no block barrier anywhere in the frame loops):
//      producers : fused row log-softmax, ONE LANE PER FRAME over blocks of 32 frames (no cross-lane
//                  reductions); emissions p(t,v) land as doubles in the E ring, blocks ahead of the sweep.
//      lattice   : NW warps, K cells per lane (cells alternate blank,label).  The s-1/s-2 transitions
//                  cross lanes with one 64-bit shuffle; they cross WARPS through a 16-byte self-validating
//                  shared-memory slot per frame (value + exponent + sequence tag in one vector store), so
//                  warp w runs one 4-frame group behind warp w-1: a software wavefront.  Frames are swept
//                  in fully unrolled groups of four with the group's emissions and boundary slots fetched
//                  up front; each frame the lanes drop the top 32 bits of their cells (+ the lane's block
//                  exponent) into the `val` ring and do nothing else.
//      combiners : drain the val ring, frames round-robin.  First half: copy rows to the global stash.
//                  Second half: cp.async-prefetch the other sweep's stashed row, multiply, normalise by
//                  Z = sum_s alpha*beta, write each label cell's posterior into a row GROUPED BY SYMBOL
//                  (counting sort of the labels, built once) and sum every symbol's contiguous slice in a
//                  fixed order -- no atomics, bitwise reproducible -- into the gradient row
//                  scale * (softmax - posterior).
//  * Arithmetic: LINEAR-domain fp64 with a per-lane block exponent (value = x * 2^e).  A cell update is
//    DADD (+ DFMA for the repeat-label skip) + DMUL; the block exponents are re-centred once per 4-frame
//    group from a snapshot two frames earlier, folded into the emission multipliers; a massless lane takes
//    the exponent of the nearest lane with mass below it (ballot + indexed shuffle).
//  * The kernel image must stay small: with three roles resident on every SM the instruction cache is a
//    first-order constraint (DESIGN.md), hence runtime `BWD` outside the lattice loop and rolled loops in
//    the producer / prologue paths.  One lattice loop serves every wavefront position: a copy per position
//    (first / middle / last warp) made the loop branch-free too, but measured 137 us instead of 101 on c2.
#pragma once
#include <cstdlib>
#include <type_traits>

#include "common.cuh"

namespace e2e {
namespace {

struct WaveParams {
  const void* logits; int dtype; long long sb, st;
  void* grads; long long gsb, gst; double scale;
  const void* targets; int tgt_is64; long long ts_b;
  const void* in_len; const void* tgt_len; int len_is64;
  int B, T, V, Lmax, blank, from_logits;
  void* losses;
  int* status; int* flags; int* meet;
  uint32_t* stash;     // [B*T][32*NW*(K+1)]: K*lanes cell words, then one exponent per lane
  long long* dbg;      // E2E_CTC_WAVE_DBG=1: [cta 0/1][warp 16][8] cycle counters of utterance 0 (else NULL)
  WaveLayout L;
};

// control block (shared memory, ints)
struct WaveCtl {
  volatile int e_ready[4];       // producer pw: its 32-frame blocks pw, pw+NP, ... below this value are in the E ring
  volatile int lat_prog[8];      // lattice warp w: frames [0, value) swept and dropped into the val ring
  volatile int comb_done[8];     // combiner q: the next frame it will take (all its earlier frames are done)
  int zero;                      // no path survives / NaN input
  volatile int occ_ready;        // the label occurrence lists (CSR by symbol) are built
  int misc[2];
  double tail_x[2]; int tail_e[2]; int tail_on[2];
  double lse[4];
};

// ---- PTX wrappers -----------------------------------------------------------------------------
__device__ __forceinline__ uint32_t wv_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void wv_cp_async_cg16(void* smem_dst, const void* gmem_src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(wv_smem_u32(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void wv_cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void wv_cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ uint4 wv_ld_volatile_v4(const void* p) {
  uint4 r;
  // no "memory" clobber: the slot is self-validating (sequence tag inside the 16 bytes), nothing else is ordered by it
  asm volatile("ld.volatile.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(wv_smem_u32(p)));
  return r;
}
// the same store, predicated inside the asm so that the caller stays branch-free
__device__ __forceinline__ void wv_st_volatile_v4_if(void* p, uint4 v, int on) {
  asm volatile("{\n\t.reg .pred pp;\n\tsetp.ne.s32 pp, %5, 0;\n\t@pp st.volatile.shared.v4.u32 [%0], {%1,%2,%3,%4};\n\t}"
               ::"r"(wv_smem_u32(p)), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "r"(on));
}
__device__ __forceinline__ void wv_st_volatile_v4(void* p, uint4 v) {
  asm volatile("st.volatile.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(wv_smem_u32(p)), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w));
}
__device__ __forceinline__ int wv_ld_acquire_gpu(const int* p) {
  int r;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(r) : "l"(p) : "memory");
  return r;
}
// progress words: release stores / acquire loads at CTA scope (lighter than a fence around a volatile access)
__device__ __forceinline__ void wv_st_release(volatile int* p, int v) {
  asm volatile("st.release.cta.shared.s32 [%0], %1;" ::"r"(wv_smem_u32(const_cast<int*>(p))), "r"(v) : "memory");
}
__device__ __forceinline__ int wv_ld_acquire(const volatile int* p) {
  int r;
  asm volatile("ld.acquire.cta.shared.s32 %0, [%1];" : "=r"(r) : "r"(wv_smem_u32(const_cast<int*>(p))) : "memory");
  return r;
}
__device__ __forceinline__ double wv_hi2d(uint32_t h) { return __hiloint2double((int)h, 0); }
// A stashed row is written once and read once: after the read its L2 lines are dead.  Dropping them (no write-back)
// keeps the stash -- 33 MB per c2 launch, L2-resident between its write and its read -- out of DRAM altogether.
__device__ __forceinline__ void wv_discard_l2_128(const void* p) {
  asm volatile("discard.global.L2 [%0], 128;" ::"l"(p) : "memory");
}

// p(t, v) relative to the row's log-sum-exp, as a double: the exponent argument is formed as torch's fp32
// log_softmax does ((x - max) - logsum, fp32) for raw logits, so the emission equals exp(double(lp32)) of the
// reference up to one fp32 exp rounding.
__device__ __noinline__ double wv_emission_lp(float x, float m, float ls) {
  const double d = (double)x - ((double)m + (double)ls);
  const float hi = (float)d;
  if (!(hi > -INFINITY)) return hi != hi ? (double)hi : 0.0;   // -inf (a masked symbol) -> exact zero, NaN -> NaN
  const float lo = (float)(d - (double)hi);
  return (double)expf(hi) * (1.0 + (double)lo);
}
__device__ __forceinline__ double wv_emission(float x, float m, float ls, int from_logits) {
  if (from_logits) return (double)expf((x - m) - ls);
  return wv_emission_lp(x, m, ls);
}

struct WaveView {
  int* lab; int* occ; double* E; uint32_t* valw; int* vale; uint32_t* stage; float* post; uint4* bnd; WaveCtl* ctl;
};
__device__ __forceinline__ WaveView wv_carve(unsigned char* base, const WaveLayout& L) {
  WaveView v;
  v.lab = reinterpret_cast<int*>(base + L.off_lab);
  v.occ = reinterpret_cast<int*>(base + L.off_occ);
  v.E = reinterpret_cast<double*>(base + L.off_E);
  v.valw = reinterpret_cast<uint32_t*>(base + L.off_valw);
  v.vale = reinterpret_cast<int*>(base + L.off_vale);
  v.stage = reinterpret_cast<uint32_t*>(base + L.off_stage);
  v.post = reinterpret_cast<float*>(base + L.off_acc);
  v.bnd = reinterpret_cast<uint4*>(base + L.off_bnd);
  v.ctl = reinterpret_cast<WaveCtl*>(base + L.off_ctl);
  return v;
}

#ifdef E2E_WAVE_DBG
#define WV_DBG_ADD(slot, val) do { if (dbgp) dbgp[slot] += (val); } while (0)
#define WV_CLK() (dbgp ? clock64() : 0ll)
#else
#define WV_DBG_ADD(slot, val) do { (void)dbgp; } while (0)
#define WV_CLK() (0ll)
#endif

template <int N>
__device__ __forceinline__ int wv_min_prog(const volatile int* a, int n) {
  int m = wv_ld_acquire(a);
#pragma unroll
  for (int k = 1; k < N; k++) if (k < n) m = min(m, wv_ld_acquire(a + k));
  return m;
}

// ---- producers: fused row log-softmax -> E ring ---------------------------------------------------
// A producer warp converts a block of 32 frames at a time with ONE LANE PER FRAME: no cross-lane reductions, so
// a row costs ~25 instructions per frame instead of ~110 with warp-shuffle max / sum.  The lanes read 32
// different rows per load instruction; the rows are consecutive in memory (or at least each row is one or two
// 128-byte lines), so after the first touch the loads are L1 hits.  REG (V <= 32): the row stays in registers.
constexpr int kWavePB = 32;   // frames per producer block

__device__ __forceinline__ float wv_load_logit(const void* base, int dtype, long long idx) {
  if (dtype == E2E_F32) return __ldg(reinterpret_cast<const float*>(base) + idx);
  const unsigned short r = __ldg(reinterpret_cast<const unsigned short*>(base) + idx);
  return dtype == E2E_BF16 ? __uint_as_float((uint32_t)r << 16) : __half2float(__ushort_as_half(r));
}

template <bool REG>
__device__ __noinline__ double wave_produce_block(const WaveParams& p, const WaveView& sv, long long xbase, int Ti,
                                                  int i0, int lane, bool BWD) {
  const WaveLayout& L = p.L;
  const int i = i0 + lane;
  if (i >= Ti) return 0.0;
  const long long ro = xbase + (long long)(BWD ? (Ti - 1 - i) : i) * p.st;
  double* Ef = sv.E + (i & (L.R - 1));   // this frame's slot of the column-major ring: symbol v at Ef[v * ecs]
  const int V = p.V, ecs = L.ecs;
  float m = -INFINITY, s = 0.f;
  bool nan = false;
  if (REG) {
    float xv[32];
#pragma unroll
    for (int v = 0; v < 32; v++) xv[v] = v < V ? wv_load_logit(p.logits, p.dtype, ro + v) : -INFINITY;
#pragma unroll
    for (int v = 0; v < 32; v++) { nan |= xv[v] != xv[v]; m = fmaxf(m, xv[v]); }
#pragma unroll
    for (int v = 0; v < 32; v++) s += expf(xv[v] - m);   // exp(-inf) = 0 for the padding columns
    float ls = logf(s);
    if (nan) { m = NAN; ls = NAN; }
#pragma unroll
    for (int v = 0; v < 32; v++) if (v < V) Ef[v * ecs] = wv_emission(xv[v], m, ls, p.from_logits);
    const double mls = (double)m + (double)ls;
    Ef[V * ecs] = 0.0;                                   // the column padding cells read
    Ef[(V + 1) * ecs] = p.from_logits ? 1.0 : exp(mls);  // turns the emission back into exp(x)
    return mls;
  } else {
    for (int v = 0; v < V; v++) { const float x = wv_load_logit(p.logits, p.dtype, ro + v); nan |= x != x; m = fmaxf(m, x); }
    for (int v = 0; v < V; v++) s += expf(wv_load_logit(p.logits, p.dtype, ro + v) - m);
    float ls = logf(s);
    if (nan) { m = NAN; ls = NAN; }
    for (int v = 0; v < V; v++) Ef[v * ecs] = wv_emission(wv_load_logit(p.logits, p.dtype, ro + v), m, ls, p.from_logits);
    const double mls = (double)m + (double)ls;
    Ef[V * ecs] = 0.0;
    Ef[(V + 1) * ecs] = p.from_logits ? 1.0 : exp(mls);
    return mls;
  }
}

template <int NW>
__device__ void wave_producer(const WaveParams& p, const WaveView& sv, int b, int Ti, int pw, int lane, bool BWD, long long* dbgp) {
  const long long tstart = WV_CLK();
  constexpr int PB = kWavePB;
  const WaveLayout& L = p.L;
  const int nblocks = (Ti + PB - 1) / PB;
  const long long xbase = (long long)b * p.sb;
  double lse = 0.0;
  for (int bi = pw; bi < nblocks; bi += L.NP) {
    const int need = bi * PB + PB - L.R;   // frames below `need` must have left the ring
    if (need > 0) {
      const long long t0 = WV_CLK();
      while (wv_min_prog<8>(sv.ctl->lat_prog, NW) < need || wv_min_prog<8>(sv.ctl->comb_done, L.NC) < need) { if (L.nap) __nanosleep(L.nap); }
      WV_DBG_ADD(1, WV_CLK() - t0);
    }
    if (p.V <= 32) lse += wave_produce_block<true>(p, sv, xbase, Ti, bi * PB, lane, BWD);
    else lse += wave_produce_block<false>(p, sv, xbase, Ti, bi * PB, lane, BWD);
    __syncwarp();
    if (lane == 0) wv_st_release(&sv.ctl->e_ready[pw], bi + 1);
  }
  lse = warp_sum(lse);   // fixed order: deterministic loss for log-prob input
  if (lane == 0) sv.ctl->lse[pw] = lse;
  WV_DBG_ADD(0, WV_CLK() - tstart);
}

// ---- lattice warps ----------------------------------------------------------------------------------
// Frames are swept in groups of four (two groups per hand-off chunk) with the group fully unrolled: the
// block exponents are re-centred once per group (snapshot at the third frame, folded into the emission
// multipliers of the next group's first frame), so a frame is the recurrence, one shuffle, one boundary
// slot and two shared-memory stores.  Four frames shrink a cell by at most 2^-600 (fp32 emissions are
// >= 2^-149), well inside the fp64 range below the re-centred block maximum.
// The frames of a full group are straight-line code (no branch or reconvergence point between them, one
// divergence check per group): whether the warp takes its boundary cell from warp w-1 (HIN) or hands one to
// warp w+1 (HOUT) enters the frame body only through selects and a predicated store, and the first group (no
// boundary into frame 0, no re-centring to apply) is peeled off the loop.
template <int K, int NW, bool BWD>
__device__ void wave_lattice(const WaveParams& p, const WaveView& sv, int b, int Ti, int Li, int w, int lane, long long* dbgp) {
  const bool HIN = NW > 1 && w > 0, HOUT = NW > 1 && w + 1 < NW;
  const long long tstart = WV_CLK();
  constexpr unsigned FULL = 0xffffffffu;
  constexpr int H = K / 2, LANES = 32 * NW, CF = kWaveCF, RB = kWaveRB, G = 4, NC = wave_combiners(NW);
  const WaveLayout& L = p.L;
  const int S = 2 * Li + 1;
  const int g = w * 32 + lane;
  const int m0 = g * K;

  const double* ecol[H];   // emission-ring column of each label cell (the zero column past L_i)
  double skipd[H];         // 1.0 where the label cell may also gather from s-2 (a different, non-blank label), else 0.0
#pragma unroll
  for (int h = 0; h < H; h++) {
    const int li = g * H + h;
    const bool lv = li < Li;
    const int lab = sv.lab[li];        // padded with blank past L_i
    ecol[h] = sv.E + (size_t)(lv ? lab : p.V) * L.ecs;
    const bool sk = lv && li >= 1 && lab != p.blank && lab != sv.lab[li - 1];
    skipd[h] = sk ? 1.0 : 0.0;
  }
  const double* const bcol = sv.E + (size_t)p.blank * L.ecs;

  double x[K];
#pragma unroll
  for (int j = 0; j < K; j++) x[j] = (m0 + j == 0) ? 1.0 : 0.0;   // a virtual frame before the first: all mass on cell 0
  int e = 0;
  double fb = lane == 0 ? 0.0 : 1.0;
  int en_next = 0;
  double f_next = 1.0, fb_next = fb;
  int src_e = 0;                       // exponent of the last boundary value received from the previous warp
  const uint4* const bnd_in = sv.bnd + (size_t)(w > 0 ? w - 1 : 0) * RB;
  uint4* const bnd_out = sv.bnd + (size_t)w * RB;

  auto chunk_wait = [&](int i0) {
    // one optimistic pass with all the progress words in flight together; the slow loops only when one is behind
    const int bi = i0 / kWavePB;   // the producer block the chunk belongs to
    const volatile int* er = &sv.ctl->e_ready[bi & (L.NP - 1)];
    const int needv = i0 + CF - L.RV;        // frames below this have left the val ring
    const int needb = i0 + CF - RB + 1;      // the boundary slots this chunk overwrites have been read
    const int ev = wv_ld_acquire(er);
    const int cm = wv_min_prog<NC>(sv.ctl->comb_done, NC);
    const int lp = HOUT ? wv_ld_acquire(&sv.ctl->lat_prog[w + 1]) : 0x7fffffff;
    if (ev <= bi || cm < needv || lp < needb) {
      const long long t0 = WV_CLK();
      while (wv_ld_acquire(er) <= bi) {}
      const long long t1 = WV_CLK();
      while (wv_min_prog<NC>(sv.ctl->comb_done, NC) < needv) {}
      const long long t2 = WV_CLK();
      if (HOUT) { while (wv_ld_acquire(&sv.ctl->lat_prog[w + 1]) < needb) {} }
      WV_DBG_ADD(1, t1 - t0); WV_DBG_ADD(2, t2 - t1); WV_DBG_ADD(3, WV_CLK() - t2);
    }
  };

  // One group of G frames.  FULLG (all G frames exist): the boundary slots of the whole group are fetched up
  // front -- the warp waits for the previous warp to finish the group's third frame, so it runs one group
  // behind it -- and the body is straight-line code the compiler can schedule across frames.  Otherwise (the
  // last, partial group) every frame polls its own slot.  FIRST: the group of frame 0.
  auto group = [&](auto full_c, auto first_c, int i0) {
    constexpr bool FULLG = decltype(full_c)::value, FIRST = decltype(first_c)::value;
    // emissions of the whole group up front (rows past T_i are stale ring memory: loaded, never used); R is a
    // multiple of G, so the group's frames are adjacent in every column
    const int f0 = i0 & (L.R - 1);
    double mb[G], ml[G][H];
#pragma unroll
    for (int k = 0; k < G; k++) {
      mb[k] = bcol[f0 + k];
#pragma unroll
      for (int h = 0; h < H; h++) ml[k][h] = ecol[h][f0 + k];
    }
    // boundary slots: RB is a multiple of G, so frames i0 .. i0+G-1 sit in slots r0 .. r0+G-1 (no wrap)
    const int r0 = i0 & (RB - 1);
    uint4 qg[G];
#pragma unroll
    for (int k = 0; k < G; k++) qg[k] = make_uint4(0u, 0u, 0u, 0u);
    if (FULLG && HIN) {
      const int last = i0 + G - 2;   // frame i needs the boundary of frame i-1
      const long long t0 = WV_CLK();
      do { qg[G - 1] = wv_ld_volatile_v4(bnd_in + r0 + G - 2); } while ((int)qg[G - 1].w != last + 1);
      WV_DBG_ADD(4, WV_CLK() - t0);
      if (!FIRST) qg[0] = wv_ld_volatile_v4(bnd_in + ((i0 - 1) & (RB - 1)));
#pragma unroll
      for (int k = 1; k < G - 1; k++) qg[k] = wv_ld_volatile_v4(bnd_in + r0 + k - 1);
    }
    uint32_t* const valw0 = sv.valw + ((size_t)(i0 & (L.RV - 1)) * LANES + g) * K;
    int* const vale0 = sv.vale + (size_t)(i0 & (L.RV - 1)) * LANES + g;
#pragma unroll
    for (int k = 0; k < G; k++) {
      const int i = i0 + k;
      if (FULLG || i < Ti) {
        const bool apply = !FIRST && k == 0;            // the re-centring of the previous group
        const bool bnd_on = HIN && (!FIRST || k > 0);   // a boundary value arrives from the previous warp
        // boundary cell from the previous lane; from the previous warp through its slot
        // explicit roundings in the recurrence: with the group in straight-line code the compiler would otherwise
        // contract a product with the next frame's sum into an FMA, and the cells would change in the last bit
        double bxs = __dmul_rn(__shfl_up_sync(FULL, x[K - 1], 1), fb);
        const uint4* slot = bnd_in + ((i - 1) & (RB - 1));
        uint4 q = qg[k];
        if (!FULLG && bnd_on) q = wv_ld_volatile_v4(slot);
        if (FULLG && (!FIRST || k > 0)) {   // selects, no branch: q is all zero in the first warp
          src_e = HIN ? (int)q.z : src_e;
          const double bin = __dmul_rn(__hiloint2double((int)q.y, (int)q.x), pow2i(min(src_e - e, 600)));   // bounded: a few more lane hops (2^192 each) before the next re-centring cannot overflow
          bxs = (HIN && lane == 0) ? bin : bxs;
        }
        if (k == 2) {
          // where the lane's scale should move (applied at the next group's first frame): block maximum into [1,2)
          int mhi = 0;
#pragma unroll
          for (int j = 0; j < K; j++) mhi = max(mhi, __double2hiint(x[j]));
          // New exponent of the lane: its own block maximum, but for a lane WITH mass never more than kExpSlack
          // below the new exponent of the lane its mass comes from (so incoming cells are scaled by at most
          // 2^kExpSlack: no overflow when a large mass follows a tiny front trickle -- tight alignments under
          // very peaky emissions); a lane WITHOUT mass takes the exponent of the nearest lane with mass below
          // it exactly (below the first such lane of warps > 0: the last boundary exponent), so the front
          // always runs into a scale that is at most a few frames stale.  Both rules are one prefix maximum:
          //   en_i = max_{j <= i} (own_j + D_j) - D_i,   D_i = kExpSlack * #{lanes with mass <= i}.
          constexpr int kExpSlack = 192;
          const bool alive = mhi != 0;
          const unsigned live = __ballot_sync(FULL, alive);
          const int D = kExpSlack * __popc(live & ((2u << lane) - 1u));
          int v = alive ? e + ((mhi >> 20) - 1023) + D : 2 * kNegExp;
          v = HIN ? max(v, src_e) : v;                // the previous warp's boundary lane, as lane -1 (D = 0)
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(FULL, v, d);
            v = lane >= d ? max(v, t) : v;
          }
          const int en = v < kNegExp ? e : v - D;     // nothing with mass up to here: keep the scale
          const int nb_en = __shfl_up_sync(FULL, en, 1);
          en_next = en;
          f_next = pow2i(e - en);
          fb_next = lane == 0 ? 0.0 : pow2i(nb_en - en);
        }
        double mulb = mb[k], mull[H];
#pragma unroll
        for (int h = 0; h < H; h++) mull[h] = ml[k][h];
        if (apply) {
          mulb = __dmul_rn(mulb, f_next);
#pragma unroll
          for (int h = 0; h < H; h++) mull[h] = __dmul_rn(mull[h], f_next);
        }
        // cell j gathers j, j-1 and (label cells, when allowed) j-2 of the previous frame; in place, top down
        double so[K];
#pragma unroll
        for (int j = K - 1; j >= 2; j--) {
          double a = __dadd_rn(x[j], x[j - 1]);
          if (j & 1) a = fma(skipd[j >> 1], x[j - 2], a);
          so[j] = a;
          x[j] = __dmul_rn(a, (j & 1) ? mull[j >> 1] : mulb);
        }
        if (!FULLG && bnd_on) {
          const long long t0 = WV_CLK();
          while ((int)q.w != i) q = wv_ld_volatile_v4(slot);
          WV_DBG_ADD(4, WV_CLK() - t0);
          src_e = (int)q.z;
          const double bin = __dmul_rn(__hiloint2double((int)q.y, (int)q.x), pow2i(min(src_e - e, 600)));
          if (lane == 0) bxs = bin;
        }
        {
          so[1] = fma(skipd[0], bxs, __dadd_rn(x[1], x[0]));
          x[1] = __dmul_rn(so[1], mull[0]);
          so[0] = __dadd_rn(x[0], bxs);
          x[0] = __dmul_rn(so[0], mulb);
        }
        // drop the frame into the val ring: alpha with its emission (forward), beta before its emission (backward)
        {
          uint32_t wd[K];
#pragma unroll
          for (int j = 0; j < K; j++) wd[j] = (uint32_t)(BWD ? __double2hiint(so[j]) : __double2hiint(x[j]));
#pragma unroll
          for (int u = 0; u < K / 4; u++)
            reinterpret_cast<uint4*>(valw0 + (size_t)k * LANES * K)[u] = make_uint4(wd[4 * u], wd[4 * u + 1], wd[4 * u + 2], wd[4 * u + 3]);
          vale0[(size_t)k * LANES] = BWD ? e : (apply ? en_next : e);
        }
        if (apply) { e = en_next; fb = fb_next; }
        wv_st_volatile_v4_if(bnd_out + r0 + k,
                             make_uint4((uint32_t)__double2loint(x[K - 1]), (uint32_t)__double2hiint(x[K - 1]), (uint32_t)e, (uint32_t)(i + 1)),
                             HOUT && lane == 31);
      }
    }
  };

  // frames [0, n) swept and in the val ring (combiners and the ring owners poll this): after every group.  Once per
  // 8-frame chunk measured slower on c2 (137 -> 146 us, in the build with a lattice loop per wavefront position,
  // DESIGN.md K2w): the combiners then take frames in bursts of eight and the lattice warps wait for the val ring
  auto publish = [&](int n) {
    __syncwarp();
    if (lane == 0) wv_st_release(&sv.ctl->lat_prog[w], n);
  };
  chunk_wait(0);
  if (Ti < G) {
    group(std::false_type{}, std::true_type{}, 0);
  } else {
    group(std::true_type{}, std::true_type{}, 0);
    publish(G);
    int i0 = G;
    for (; i0 + G <= Ti; i0 += G) {
      if ((i0 & (CF - 1)) == 0) chunk_wait(i0);
      group(std::true_type{}, std::false_type{}, i0);
      publish(i0 + G);
    }
    if (i0 < Ti) {
      if ((i0 & (CF - 1)) == 0) chunk_wait(i0);
      group(std::false_type{}, std::false_type{}, i0);
    }
  }
  publish(Ti);
  WV_DBG_ADD(0, WV_CLK() - tstart);
  // exit cells S-1 and S-2 of the last frame: Z = their sum (ctc_loss.cpp:63-70)
#pragma unroll
  for (int j = 0; j < K; j++) {
    const int m = m0 + j;
    if (m == S - 1) { sv.ctl->tail_x[0] = x[j]; sv.ctl->tail_e[0] = e; sv.ctl->tail_on[0] = 1; }
    if (m == S - 2) { sv.ctl->tail_x[1] = x[j]; sv.ctl->tail_e[1] = e; sv.ctl->tail_on[1] = 1; }
  }
}

// ---- combiner warps ---------------------------------------------------------------------------------
template <int K, int NW>
__device__ void wave_combiner(const WaveParams& p, const WaveView& sv, int b, int Ti, int Li, int q, int lane, bool BWD, long long* dbgp) {
  const long long tstart = WV_CLK();
  constexpr unsigned FULL = 0xffffffffu;
  constexpr int H = K / 2, LANES = 32 * NW, CELLS = LANES * K, ROWW = LANES * (K + 1), PF = kWavePF;
  constexpr int SROW = ROWW + 4;   // staged row: the stashed row + a zero word (index ROWW) that cells past the lattice pair with
  constexpr int KLOG = K == 4 ? 2 : 3;
  const WaveLayout& L = p.L;
  const int NC = L.NC;
  const int S = 2 * Li + 1;
  const int tm = Ti / 2;
  const int nstore = BWD ? (Ti - tm) : tm;          // frames this sweep stores; the rest it combines
  const int nstore_peer = Ti - nstore;
  auto frame_t = [&](int i) { return BWD ? (Ti - 1 - i) : i; };
  uint32_t* const stash_b = p.stash + (size_t)b * p.T * ROWW;
  uint32_t* const stage = sv.stage + (size_t)q * PF * SROW;
  float* const post = sv.post + (size_t)q * (LANES * H + 4);   // this warp's label posteriors of one frame, grouped by symbol
  int* const rank = sv.occ;                                    // label index -> its slot in that grouping ...
  int* const ofs = sv.occ + LANES * H;                         // ... symbol v owns slots [ofs[v], ofs[v+1])

  auto wait_val = [&](int i) {
    const long long t0 = WV_CLK();
    while (wv_min_prog<8>(sv.ctl->lat_prog, NW) <= i) { if (L.nap) __nanosleep(L.nap); }
    WV_DBG_ADD(1, WV_CLK() - t0);
  };
  auto done = [&](int i) {
    __syncwarp();
    if (lane == 0) wv_st_release(&sv.ctl->comb_done[q], i + NC);
  };
  auto prefetch = [&](int i2, int slot) {   // the other sweep's stored row of my frame i2 -> staging slot
    if (i2 < Ti) {
      uint32_t* dst = stage + (size_t)slot * SROW;
      const uint32_t* src = stash_b + (size_t)frame_t(i2) * ROWW;
      for (int u = lane; u < ROWW / 4; u += 32) wv_cp_async_cg16(dst + 4 * u, src + 4 * u);
    }
  };

  if (q == 0) {
    // Occurrence lists of the utterance's labels by symbol (a counting sort, built once while the first frames
    // are swept): the gradient row then GATHERS the posteriors of a symbol's label cells in a fixed order --
    // no shared-memory atomics, and the sum is bitwise reproducible.
    int base = 0;
    for (int v0 = 0; v0 < p.V; v0 += 32) {
      const int v = v0 + lane;
      int c = 0;
      if (v < p.V) for (int li = 0; li < Li; li++) c += (sv.lab[li] == v);
      int inc = c;   // inclusive scan over the 32 symbols of this pass
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(FULL, inc, o); if (lane >= o) inc += t; }
      int k = base + inc - c;
      if (v < p.V) {
        ofs[v] = k;
        for (int li = 0; li < Li; li++) if (sv.lab[li] == v) rank[li] = k++;
      }
      base += __shfl_sync(FULL, inc, 31);
    }
    if (lane == 0) ofs[p.V] = base;
    __syncwarp();
    if (lane == 0) wv_st_release(&sv.ctl->occ_ready, 1);
  }

  int i = q;
  // ---- first half: val ring -> global stash ----
  for (; i < nstore; i += NC) {
    wait_val(i);
    const size_t ent0 = (size_t)(i & (L.RV - 1)) * LANES;
    uint32_t* row = stash_b + (size_t)frame_t(i) * ROWW;
#pragma unroll
    for (int u = 0; u < NW; u++) {
      const int g = lane + 32 * u;
#pragma unroll
      for (int v = 0; v < K / 4; v++)
        reinterpret_cast<uint4*>(row + (size_t)g * K)[v] = reinterpret_cast<const uint4*>(sv.valw + (ent0 + g) * K)[v];
      row[CELLS + g] = (uint32_t)sv.vale[ent0 + g];
    }
    if (i + NC >= nstore) {   // my last stored row: publish to the other CTA
      __syncwarp();
      if (lane == 0) { __threadfence(); atomicAdd(p.meet + 2 * b + (BWD ? 1 : 0), 1); }
    }
    done(i);
  }
  WV_DBG_ADD(2, WV_CLK() - tstart);
  if (i >= Ti) return;
  const long long tmeet = WV_CLK();
  // ---- meet: the other sweep's stored rows must be visible ----
  {
    const int want = min(NC, nstore_peer);
    const int* flag = p.meet + 2 * b + (BWD ? 0 : 1);
    while (wv_ld_acquire_gpu(flag) < want) __nanosleep(64);
    while (wv_ld_acquire(&sv.ctl->occ_ready) == 0) __nanosleep(64);
  }
  WV_DBG_ADD(4, WV_CLK() - tmeet);
  const long long tsecond = WV_CLK();
  for (int u = 0; u < PF; u++) { prefetch(i + u * NC, u); wv_cp_async_commit(); }

  // Per lane: the lattice lanes g = lane + 32u it multiplies.  My cell m = g*K + j is the other sweep's cell
  // mp = S-1-m: cells j <= r = (S-1) mod K of a lane sit in the other sweep's lane lA = mp0 >> KLOG, the rest in
  // lA - 1, so a lane pairs with two block exponents.  Cells past the lattice (mp < 0) pair with the zero word.
  int mp0[NW];              // other-sweep index of my cell j = 0
  int slot[NW][H];          // where the posterior of label cell j = 2h+1 goes (a spare slot past L_i)
#pragma unroll
  for (int u = 0; u < NW; u++) {
    const int g = lane + 32 * u;
    mp0[u] = S - 1 - g * K;
#pragma unroll
    for (int h = 0; h < H; h++) slot[u][h] = g * H + h < Li ? rank[g * H + h] : LANES * H;
  }
  const int r = (S - 1) & (K - 1);

  bool have_z = false;
  double cz = 0.0;   // 2^31 / Z as mantissa in [1,2); its exponent is folded into Ez
  int Ez = 0;
  const float sc = (float)p.scale;
  for (int k = 0; i < Ti; i += NC, ++k) {
    wait_val(i);
    { const long long t0 = WV_CLK(); wv_cp_async_wait<PF - 1>(); __syncwarp(); WV_DBG_ADD(5, WV_CLK() - t0); }
    const uint32_t* orow = stage + (size_t)(k % PF) * SROW;
    if ((ROWW * 4) % 128 == 0) {   // the row is staged: its global copy is dead (rows are 128-byte multiples at 256-byte aligned bases)
      const char* dead = reinterpret_cast<const char*>(stash_b + (size_t)frame_t(i) * ROWW);
      for (int u = lane; u < ROWW * 4 / 128; u += 32) wv_discard_l2_128(dead + (size_t)u * 128);
    }
    const size_t ent0 = (size_t)(i & (L.RV - 1)) * LANES;
    const uint32_t* valw_row = sv.valw + ent0 * K;
    const int* vale_row = sv.vale + ent0;
    double pr[NW][K];
    int ElA[NW], ElB[NW];
#pragma unroll
    for (int u = 0; u < NW; u++) {
      const int g = lane + 32 * u;
      uint32_t wd[K];
#pragma unroll
      for (int v = 0; v < K / 4; v++) {
        const uint4 t4 = reinterpret_cast<const uint4*>(valw_row + (size_t)g * K)[v];
        wd[4 * v] = t4.x; wd[4 * v + 1] = t4.y; wd[4 * v + 2] = t4.z; wd[4 * v + 3] = t4.w;
      }
      const int em = vale_row[g];
      const int lA = mp0[u] >> KLOG;   // arithmetic shift: negative past the lattice
      ElA[u] = em + (int)orow[CELLS + max(lA, 0)];
      ElB[u] = em + (int)orow[CELLS + max(lA - 1, 0)];
#pragma unroll
      for (int j = 0; j < K; j++) {
        const int mp = mp0[u] - j;
        pr[u][j] = wv_hi2d(wd[j]) * wv_hi2d(orow[mp >= 0 ? mp : ROWW]);
      }
    }
    if (!have_z) {
      // Z = sum_s alpha(t,s) * beta(t,s), the same for every frame: taken once per combiner warp
      int emax = 4 * kNegExp;
#pragma unroll
      for (int u = 0; u < NW; u++)
#pragma unroll
        for (int j = 0; j < K; j++) if (pr[u][j] > 0.0) emax = max(emax, j <= r ? ElA[u] : ElB[u]);
      emax = warp_max_int(emax);
      double tot = 0.0;
#pragma unroll
      for (int u = 0; u < NW; u++) {
        const double fA = pow2i(ElA[u] - emax), fB = pow2i(ElB[u] - emax);
#pragma unroll
        for (int j = 0; j < K; j++) if (pr[u][j] > 0.0) tot += pr[u][j] * (j <= r ? fA : fB);
      }
      tot = warp_sum(tot);
      // 2^31 / Z = cz * 2^kz with cz in [1,2): the power of two moves into Ez, so the per-cell scale
      // 2^(El - Ez) * cz stays finite whatever stale exponent a massless lane carries (0 * finite = 0).
      // tot == 0 or NaN: the lattice tail flags the utterance and the block is overwritten with NaN.
      const double rz = 2147483648.0 / tot;
      const int kz = ((__double2hiint(rz) >> 20) & 0x7ff) - 1023;
      cz = __hiloint2double((__double2hiint(rz) & 0x800fffff) | 0x3ff00000, __double2loint(rz));
      Ez = emax - kz;
      have_z = true;
    }
    // posteriors scaled by 2^31: blank cells are summed as fixed point (one warp-wide integer add), label
    // cells go to this warp's row by label index
    uint32_t bsum = 0u;
#pragma unroll
    for (int u = 0; u < NW; u++) {
      const double sA = pow2i(ElA[u] - Ez) * cz, sB = pow2i(ElB[u] - Ez) * cz;
#pragma unroll
      for (int j = 0; j < K; j++) {
        const double pv = pr[u][j] * (j <= r ? sA : sB);
        if (j & 1) post[slot[u][j >> 1]] = (float)pv;
        else bsum += __double2uint_rn(pv);
      }
    }
    const uint32_t qb = __reduce_add_sync(FULL, bsum);
    __syncwarp();
    // gradient row: scale * (softmax - posterior); log-prob input: exp(lp) - posterior (the engine contract).
    // A lane sums the posteriors of its symbol's label cells in list order.
    {
      const int t = frame_t(i);
      const double* Ef = sv.E + (i & (L.R - 1));
      const int ecs = L.ecs;
      const float rs = (float)Ef[(p.V + 1) * ecs];
      const long long gbase = (long long)b * p.gsb + (long long)t * p.gst;
      for (int v = lane; v < p.V; v += 32) {
        // the symbol's label cells are contiguous in the row: four independent partial sums, fixed order
        float a0 = v == p.blank ? (float)qb : 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
        const int k1 = ofs[v + 1];
        for (int kk = ofs[v]; kk < k1; kk += 4) {
          a0 += post[kk];
          a1 += kk + 1 < k1 ? post[kk + 1] : 0.f;
          a2 += kk + 2 < k1 ? post[kk + 2] : 0.f;
          a3 += kk + 3 < k1 ? post[kk + 3] : 0.f;
        }
        const float a = (a0 + a1) + (a2 + a3);
        const float gv = sc * ((float)Ef[v * ecs] * rs - a * (1.f / 2147483648.f));
        if (p.dtype == E2E_F32) reinterpret_cast<float*>(p.grads)[gbase + v] = gv;
        else if (p.dtype == E2E_BF16) reinterpret_cast<__nv_bfloat16*>(p.grads)[gbase + v] = __float2bfloat16_rn(gv);
        else reinterpret_cast<__half*>(p.grads)[gbase + v] = __float2half_rn(gv);
      }
    }
    __syncwarp();
    prefetch(i + PF * NC, k % PF);
    wv_cp_async_commit();
    done(i);
  }
  wv_cp_async_wait<0>();
  WV_DBG_ADD(3, WV_CLK() - tsecond);
  WV_DBG_ADD(0, WV_CLK() - tstart);
}

// ---- kernel -------------------------------------------------------------------------------------------
template <int K, int NW>
__device__ void wave_roles(const WaveParams& p, const WaveView& sv, int b, int Ti, int Li, int w, int lane, bool BWD) {
  const WaveLayout& L = p.L;
  long long* dbgp = (p.dbg != nullptr && b == 0 && lane == 0 && w < 16) ? p.dbg + ((BWD ? 16 : 0) + w) * 8 : nullptr;
  // Warp w runs on scheduler (SM sub-partition) w % 4, each with its own small L0 instruction cache.  With
  // `by_smsp` the roles are laid out so that every sub-partition runs ONE role's loop (lattice on 0,
  // combiners on 1 and 2, producers on 3): three interleaved loops do not fit an L0 and the sweep
  // starves on instruction fetch otherwise.
  int role, idx;   // 0 lattice, 1 combiner, 2 producer, 3 idle
  if (L.by_smsp) {
    const int sub = w & 3, r = w >> 2;
    if (sub == 0) { role = r < NW ? 0 : 3; idx = r; }
    else if (sub == 3) { role = r < L.NP ? 2 : 3; idx = r; }
    else { idx = 2 * r + (sub - 1); role = idx < L.NC ? 1 : 3; }
  } else {
    const int first_comb = L.NP, first_lat = L.NP + L.NC;
    if (w >= first_lat) { role = 0; idx = w - first_lat; }
    else if (w >= first_comb) { role = 1; idx = w - first_comb; }
    else { role = 2; idx = w; }
  }
  if (role == 0) {
    if (BWD) wave_lattice<K, NW, true>(p, sv, b, Ti, Li, idx, lane, dbgp);
    else wave_lattice<K, NW, false>(p, sv, b, Ti, Li, idx, lane, dbgp);
  } else if (role == 1) {
    wave_combiner<K, NW>(p, sv, b, Ti, Li, idx, lane, BWD, dbgp);
  } else if (role == 2) {
    w = idx;
    wave_producer<NW>(p, sv, b, Ti, w, lane, BWD, dbgp);
    // padding frames t >= T_i: exp(lp) for log-prob input (the engine contract, ctc_loss.cpp:105-117),
    // 0 for fused-logits input (what the reference's log_softmax backward leaves there)
    for (int r = Ti + (BWD ? 1 : 0) + 2 * w; r < p.T; r += 2 * L.NP) {
      const long long xo = (long long)b * p.sb + (long long)r * p.st;
      const long long go = (long long)b * p.gsb + (long long)r * p.gst;
      for (int v = lane; v < p.V; v += 32) {
        double gq = 0.0;
        if (!p.from_logits) gq = (double)expf(load_as_float(p.logits, p.dtype, xo + v));
        store_from_double(p.grads, p.dtype, go + v, p.scale * gq);
      }
    }
  }
}

template <int K, int NW>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(32 * (NW <= 4 ? 16 : 32), 1)
ctc_wave_kernel(const WaveParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr int H = K / 2, LANES = 32 * NW;
  const WaveView sv = wv_carve(smem_raw, p.L);
  __shared__ int pre[4];

  const int b = blockIdx.x >> 1;
  const bool bwd = (blockIdx.x & 1) != 0;
  const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
  const int nwarps = blockDim.x >> 5;

  const long long Ti_ll = load_index(p.in_len, p.len_is64, b);
  const long long Li_ll = load_index(p.tgt_len, p.len_is64, b);
  int bad = 0;
  if (Ti_ll < 1 || Ti_ll > p.T) bad |= kBadFrames;
  if (Li_ll < 0 || Li_ll > p.Lmax) bad |= kBadTargetLen;
  const int Ti = (int)Ti_ll, Li = bad ? 0 : (int)Li_ll;
  if (tid < 4) pre[tid] = 0;
  __syncthreads();
  int rep = 0, badlab = 0;
  // the backward CTA sweeps the reversed label sequence
  for (int i = tid; i < Li; i += blockDim.x) {
    const long long v = load_index(p.targets, p.tgt_is64, (long long)b * p.ts_b + i);
    if (v < 0 || v >= p.V) badlab = kBadLabel;
    sv.lab[bwd ? (Li - 1 - i) : i] = (int)v;
  }
  for (int i = Li + tid; i < LANES * H + 1; i += blockDim.x) sv.lab[i] = p.blank;   // cells past the lattice carry zero mass
  __syncthreads();
  for (int i = tid + 1; i < Li; i += blockDim.x) rep += (sv.lab[i] == sv.lab[i - 1]);
  if (rep) atomicAdd(&pre[1], rep);
  if (badlab) atomicOr(&pre[0], badlab);
  __syncthreads();
  bad |= pre[0];
  rep = pre[1];
  const long long gfill_base = (long long)b * p.gsb;
  if (bad || Ti < Li + rep) {
    // out-of-range lengths / labels (undefined behaviour in the reference): NaN loss + status bits;
    // no alignment exists (T < L + repeats): loss = +inf.  Either way the gradient block is all NaN
    // (-inf - (-inf) in the reference, ctc_loss.cpp:116-117), padding rows included.
    if (tid == 0 && !bwd) {
      if (bad) atomicOr(p.status, bad);
      p.flags[b] = bad ? kFlagInvalid : kFlagInfeasible;
      store_from_double(p.losses, p.dtype, b, bad ? (double)NAN : (double)INFINITY);
    }
    for (int r = 2 * w + (bwd ? 1 : 0); r < p.T; r += 2 * nwarps)
      for (int v = lane; v < p.V; v += 32) store_from_double(p.grads, p.dtype, gfill_base + (long long)r * p.gst + v, (double)NAN);
    return;
  }
  {  // control block, accumulators and boundary slots start at zero
    uint32_t* z = reinterpret_cast<uint32_t*>(smem_raw + p.L.off_acc);
    const int n = (p.L.total - p.L.off_acc) >> 2;
    for (int k = tid; k < n; k += blockDim.x) z[k] = 0u;
  }
  for (int k = tid; k < p.L.NC * kWavePF; k += blockDim.x) {   // the zero word (+ padding) after each staged row
    uint32_t* zw = sv.stage + (size_t)k * (LANES * (K + 1) + 4) + LANES * (K + 1);
    zw[0] = 0u; zw[1] = 0u; zw[2] = 0u; zw[3] = 0u;
  }
  __syncthreads();
  if (tid < p.L.NC) sv.ctl->comb_done[tid] = tid;
  __syncthreads();

  wave_roles<K, NW>(p, sv, b, Ti, Li, w, lane, bwd);
  __syncthreads();

  // loss = -log(alpha[S-1][T-1] + alpha[S-2][T-1]) (ctc_loss.cpp:63-70) from the live fp64 state of the
  // forward sweep (the backward sweep's exit cells give the same Z: it only needs the zero test).
  // Emissions were normalised per row, so for log-prob input the row normalisers are added back.
  if (tid == 0) {
    WaveCtl* c = sv.ctl;
    const double x0 = c->tail_on[0] ? c->tail_x[0] : 0.0, x1 = c->tail_on[1] ? c->tail_x[1] : 0.0;
    const int e0 = (c->tail_on[0] && x0 > 0.0) ? c->tail_e[0] : 4 * kNegExp;
    const int e1 = (c->tail_on[1] && x1 > 0.0) ? c->tail_e[1] : 4 * kNegExp;
    const int emax = max(e0, e1);
    double z = 0.0;
    if (x0 > 0.0) z += x0 * pow2i(e0 - emax);
    if (x1 > 0.0) z += x1 * pow2i(e1 - emax);
    if (x0 != x0 || x1 != x1) z = NAN;
    double loss = INFINITY;
    if (z > 0.0) {
      loss = -(log(z) + (double)emax * 0.69314718055994530942);
      if (!p.from_logits) { for (int k = 0; k < p.L.NP; k++) loss -= c->lse[k]; }
    } else {   // no path survives (exact-zero emissions): +inf; NaN input: NaN.  NaN gradient block either way
      if (z != z) loss = NAN;
      c->zero = 1;
    }
    if (!bwd) {
      p.flags[b] = z > 0.0 ? 0 : kFlagInfeasible;
      store_from_double(p.losses, p.dtype, b, loss);
    }
  }
  __syncthreads();
  if (sv.ctl->zero) {
    // each CTA overwrites the rows it wrote: its combined frames and its share of the padding rows
    const int tm = Ti / 2;
    for (int r = w; r < p.T; r += nwarps) {
      const bool mine = r < Ti ? (bwd ? r < tm : r >= tm) : (((r - Ti) & 1) == (bwd ? 1 : 0));
      if (!mine) continue;
      for (int v = lane; v < p.V; v += 32) store_from_double(p.grads, p.dtype, gfill_base + (long long)r * p.gst + v, (double)NAN);
    }
  }
}

template <int K, int NW>
int launch_wave_k(const WaveParams& wp, cudaStream_t s) {
  // the dynamic shared-memory opt-in is PER DEVICE: cached per device ordinal (it only ever grows)
  static int attr_smem[64];
  int dev = 0;
  E2E_CUDA_TRY(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64 || wp.L.total > attr_smem[dev]) {
    E2E_CUDA_TRY(cudaFuncSetAttribute(ctc_wave_kernel<K, NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, wp.L.total));
    if (dev >= 0 && dev < 64) attr_smem[dev] = wp.L.total;
  }
  const unsigned threads = 32u * (unsigned)wp.L.nwarps;
  KernelTimer timer(kKernelLattice, s);
  ctc_wave_kernel<K, NW><<<2u * (unsigned)wp.B, threads, (size_t)wp.L.total, s>>>(wp);
  E2E_CUDA_TRY(cudaGetLastError());
  return E2E_OK;
}

}  // namespace
}  // namespace e2e
