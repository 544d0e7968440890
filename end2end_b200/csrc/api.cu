// C ABI of libe2e_ctc.so (include/e2e_ctc.h): argument checking, workspace planning, kernel
// sequencing, and the host-buffer engine.  No torch / pybind11 types cross this boundary.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <mutex>
#include <new>
#include <vector>

#include "common.cuh"

namespace e2e {

static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};
static std::atomic<int> g_force_kernel{-1};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// ---- launch accounting and optional kernel timing --------------------------------------------
// With profiling on, every kernel launch is bracketed by a pair of CUDA events recorded on the
// launching stream; e2e_ctc_profile_read() resolves them.  Off (default): one relaxed atomic add.
struct EventPair { cudaEvent_t a, b; int kind; };
static std::mutex g_prof_mu;
static std::atomic<int> g_prof_on{0};
static std::vector<EventPair> g_prof_pending;
static std::vector<std::pair<cudaEvent_t, cudaEvent_t>> g_prof_free;
static thread_local EventPair t_open{nullptr, nullptr, -1};
static thread_local int t_capturing = 0;       // a CUDA-graph capture is in progress on this thread: count, do not time
static thread_local uint64_t t_captured = 0;

void launch_begin(int kind, cudaStream_t s) {
  if (t_capturing) { t_captured++; return; }       // the graph's launches are counted when the graph is launched
  g_launches.fetch_add(1, std::memory_order_relaxed);
  if (!g_prof_on.load(std::memory_order_relaxed)) return;
  std::lock_guard<std::mutex> lk(g_prof_mu);
  EventPair ev{nullptr, nullptr, kind};
  if (!g_prof_free.empty()) { ev.a = g_prof_free.back().first; ev.b = g_prof_free.back().second; g_prof_free.pop_back(); }
  else if (cudaEventCreate(&ev.a) != cudaSuccess || cudaEventCreate(&ev.b) != cudaSuccess) return;
  cudaEventRecord(ev.a, s);
  t_open = ev;
}
void launch_end(int kind, cudaStream_t s) {
  if (t_open.kind != kind || !t_open.a) return;
  cudaEventRecord(t_open.b, s);
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof_pending.push_back(t_open);
  t_open = EventPair{nullptr, nullptr, -1};
}

static inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }
static inline size_t elem_size(int dtype) {
  switch (dtype) {
    case E2E_F32: return 4;
    case E2E_BF16: case E2E_F16: return 2;
    case E2E_F64: return 8;
  }
  return 0;
}
static inline int align16i(size_t x) { return (int)((x + 15) & ~(size_t)15); }
static int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return (v && *v) ? atoi(v) : dflt;
}

constexpr int kMaxTargets = 639;      // 32 lanes x 10 blocks x 4 cells = 1280 >= 2L+1
constexpr int kMaxAlphabet = 32768;

static int check_desc(const e2e_ctc_desc* d, bool need_targets) {
  if (!d) { set_error("null descriptor"); return E2E_ERR_INVALID_ARGUMENT; }
  if (d->batch < 1 || d->max_frames < 1 || d->alphabet < 1) {
    set_error("bad shape B=%d T=%d V=%d", d->batch, d->max_frames, d->alphabet);
    return E2E_ERR_INVALID_ARGUMENT;
  }
  if (elem_size(d->dtype) == 0) { set_error("bad dtype %d", d->dtype); return E2E_ERR_INVALID_ARGUMENT; }
  if (d->blank_idx < 0 || d->blank_idx >= d->alphabet) {
    set_error("blank_idx %d outside [0,%d)", d->blank_idx, d->alphabet);
    return E2E_ERR_INVALID_ARGUMENT;
  }
  if ((d->lengths_itype != E2E_I32 && d->lengths_itype != E2E_I64) ||
      (d->targets_itype != E2E_I32 && d->targets_itype != E2E_I64)) {
    set_error("bad index type");
    return E2E_ERR_INVALID_ARGUMENT;
  }
  if (d->alphabet > kMaxAlphabet) {
    set_error("alphabet %d exceeds this build's limit %d", d->alphabet, kMaxAlphabet);
    return E2E_ERR_UNSUPPORTED;
  }
  if (need_targets) {
    if (d->max_targets < 0) { set_error("bad max_targets %d", d->max_targets); return E2E_ERR_INVALID_ARGUMENT; }
    if (d->max_targets > kMaxTargets) {
      set_error("target length %d exceeds this build's limit %d", d->max_targets, kMaxTargets);
      return E2E_ERR_UNSUPPORTED;
    }
  }
  return E2E_OK;
}

// One-warp-per-sweep kernel: variants by cells per lane; f64 inputs use a subset (compile time).
static const int kSweepK[] = {2, 4, 6, 8, 10, 12, 14, 16, 20, 24, 28, 32, 36, 40};
static const int kSweepK64[] = {2, 4, 8, 16, 24, 40};

static bool make_sweep_plan(const e2e_ctc_desc& d, bool fused, LossPlan* p) {
  const int S = 2 * d.max_targets + 1;
  const bool f64 = d.dtype == E2E_F64;
  int K = 0;
  if (f64) { for (int k : kSweepK64) if (32 * k >= S) { K = k; break; } }
  else { for (int k : kSweepK) if (32 * k >= S) { K = k; break; } }
  if (!K) return false;
  p->kind = kPlanSweep;
  p->K = K; p->NW = 1; p->cells = 32 * K;
  p->words = (K + 1 + 3) & ~3;
  p->dense = fused && d.alphabet <= kDenseMaxAlphabet;
  const int rowlen = p->dense ? d.alphabet : d.max_targets + 1;
  p->post_stride = p->cells / 2 + 4;
  p->vpad = p->dense ? ((d.alphabet + 1 + 3) & ~3) : 0;
  const int H = K / 2, PF = K >= 24 ? kSweepPFWide : kSweepPFSmall;
  const int et = f64 ? 8 : 4;
  const int esz = f64 ? 8 : (d.dtype == E2E_F32 ? 4 : 2);
  SweepLayout L;
  L.vpad = p->vpad;
  L.es = p->dense ? ((d.alphabet + 1) | 1) : (1 + 32 * H);
  if (f64) L.rawrow = rowlen * 8;
  else if (p->dense) L.rawrow = ((((d.alphabet * esz + 2 + 3) >> 2)) | 1) * 4;
  else L.rawrow = ((d.max_targets + 1) | 1) * 4;
  auto layout = [&](int cf) {
    L.cf = cf;
    size_t off = 0;
    L.off_lab = 0; off = (size_t)align16i((size_t)(32 * H + 1) * 4);
    L.off_warp = (int)off;
    size_t w = 0;
    L.w_E = (int)w; w = (size_t)align16i(w + (size_t)cf * L.es * et);
    L.w_raw = (int)w; w = (size_t)align16i(w + (size_t)cf * L.rawrow);
    L.w_stat = (int)w; w += (size_t)cf * 16;
    L.w_rs = (int)w; w = (size_t)align16i(w + (size_t)cf * 4);
    L.w_acc = (int)w; w += (size_t)2 * L.vpad * 4;
    L.w_stage = (int)w; w += (size_t)PF * 32 * p->words * 4;
    L.warp_bytes = (int)w;
    return off + 2 * w;
  };
  int cf = 32;
  // several CTAs per SM when the batch is large; otherwise whatever fits
  static const int want_kb = env_int("E2E_CTC_SWEEP_SMEM_KB", 0);   // experiments only
  // more than four CTAs per SM's worth of utterances (4 x 148): seven CTAs per SM (<= 32 KB each, 128 registers: the
  // whole batch in ONE wave) beat four with longer emission chunks -- c3 (B=1024): 267 -> 229 us; up to 592 utterances
  // four CTAs per SM already hold the batch and the 32-frame chunks win (B=512: 140 us)
  const size_t want = want_kb > 0 ? (size_t)want_kb * 1024
                                  : (d.batch > 4 * 148 && K <= 8 ? 32 * 1024 : (d.batch > 148 ? 56 * 1024 : 200 * 1024));   // wide variants are register-bound at four CTAs per SM
  while (cf > 8 && layout(cf) > want) cf >>= 1;
  const size_t smem = layout(cf);
  if (smem > 220 * 1024) return false;
  p->sw = L;
  p->smem = smem;
  const size_t rows = (size_t)d.batch * d.max_frames;
  size_t off = 0;
  p->off_status = off; off += 256;
  p->off_meet = off;
  p->off_flags = off; off += align256((size_t)d.batch * 4);
  // Wide lattices run four CTAs per SM; a batch of several waves ends with a tail of half-empty SMs unless the long
  // utterances go first (the hardware hands out CTAs in index order): c5 (B=2048) 11.7 -> see DESIGN.md
  p->off_order = 0;
  if (K >= 16 && d.batch > 4 * 148) { p->off_order = off; off += align256((size_t)d.batch * 4); }
  p->off_stats = off; off += p->dense ? 0 : align256(rows * (f64 ? 16 : 8));
  p->off_stash = off; off += align256(rows * 32 * p->words * 4);
  p->off_post = off; off += p->dense ? 0 : align256(rows * p->post_stride * 4);
  p->total = off;
  return true;
}

// Wave kernel (fused small-alphabet path): variants by (cells per lane, lattice warps per sweep).
static bool make_wave_plan(const e2e_ctc_desc& d, bool fused, LossPlan* p) {
  if (!fused || d.dtype == E2E_F64 || d.alphabet > kDenseMaxAlphabet) return false;
  // Latency shapes only -- at most two rounds of resident clusters (one 2-CTA cluster per utterance, one CTA per
  // SM: B <= 148) and two to four lattice warps per sweep; measured on c2-shaped batches the wave kernel wins up
  // to B = 148 and ties at B = 256; larger batches and short lattices are throughput-bound.
  static const int kVar[][2] = {{4, 1}, {4, 2}, {4, 4}, {4, 8}, {8, 8}};
  const int S = 2 * d.max_targets + 1;
  int K = 0, NW = 0;
  for (const auto& v : kVar)
    if (32 * v[0] * v[1] >= S && !K) { K = v[0]; NW = v[1]; }
  if (d.batch > 148 || NW > 4 || (NW == 1 && 2 * d.batch > 148)) return false;
  if (!K) return false;
  WaveLayout L;
  L.K = K; L.NW = NW;
  L.NC = wave_combiners(NW);
  L.NP = NW >= 4 ? 2 : 1;
  // experiment knobs (read once per process; a production process never sets them)
  static const int wv_np = env_int("E2E_CTC_WAVE_NP", 0), wv_nap = env_int("E2E_CTC_WAVE_NAP", -1),
                   wv_smsp = env_int("E2E_CTC_WAVE_BY_SMSP", 0), wv_r = env_int("E2E_CTC_WAVE_R", 0), wv_rv = env_int("E2E_CTC_WAVE_RV", 0);
  if (wv_np == 1 || wv_np == 2 || wv_np == 4) L.NP = wv_np;
  L.nap = wv_nap >= 0 ? wv_nap : 32;
  L.by_smsp = wv_smsp ? 1 : 0;
  if (L.by_smsp) {
    int r = NW > L.NP ? NW : L.NP;
    if ((L.NC + 1) / 2 > r) r = (L.NC + 1) / 2;
    L.nwarps = 4 * r;
  } else {
    L.nwarps = NW + L.NC + L.NP;
  }
  if (L.nwarps > (NW <= 4 ? 16 : 32)) return false;
  const int lanes = 32 * NW, roww = lanes * (K + 1);
  const int ecols = d.alphabet + 2;   // V symbols, the zero column padding cells read, the row normaliser
  L.vpad = (d.alphabet + 3) & ~3;
  L.RV = lanes * K >= 1024 ? 16 : 32;
  if (wv_rv == 8 || wv_rv == 16 || wv_rv == 32 || wv_rv == 64) L.RV = wv_rv;
  L.R = 128;   // producer blocks are 32 frames: two per producer in flight
  if (wv_r == 64 || wv_r == 128 || wv_r == 256) L.R = wv_r;
  if (L.R < 64 || (L.R & (L.R - 1))) return false;
  while (L.R > 64 && (size_t)(L.R + 1) * ecols * 8 > (size_t)(NW >= 4 ? 64 : 40) * 1024) L.R >>= 1;
  L.ecs = L.R + 1;
  if (L.RV > L.R / 2) L.RV = L.R / 2;
  if (L.RV < kWaveCF || (L.RV & (L.RV - 1))) return false;
  size_t off = 0;
  L.off_lab = 0; off = (size_t)align16i((size_t)(lanes * K / 2 + 1) * 4);
  L.off_occ = (int)off; off = (size_t)align16i(off + (size_t)(lanes * K / 2 + d.alphabet + 2) * 4);   // label indices by symbol + offsets
  L.off_E = (int)off; off = (size_t)align16i(off + (size_t)ecols * L.ecs * 8);
  L.off_valw = (int)off; off += (size_t)L.RV * lanes * K * 4;
  L.off_vale = (int)off; off += (size_t)L.RV * lanes * 4;
  L.off_stage = (int)off; off += (size_t)L.NC * kWavePF * (roww + 4) * 4;
  L.off_acc = (int)off; off += (size_t)L.NC * (lanes * K / 2 + 4) * 4;   // one row of label posteriors per combiner warp (+ a spare slot)
  L.off_bnd = (int)off; off += (size_t)NW * kWaveRB * 16;
  L.off_ctl = (int)off; off += wave_ctl_bytes();
  L.total = (int)off;
  if (off > 220 * 1024) return false;
  p->kind = kPlanWave; p->wv = L;
  p->K = K; p->NW = NW; p->cells = lanes * K; p->words = K + 1;
  p->dense = 1; p->vpad = L.vpad; p->post_stride = 0;
  p->smem = off;
  const size_t rows = (size_t)d.batch * d.max_frames;
  size_t o = 0;
  p->off_status = o; o += 256;
  p->off_meet = o; o += align256((size_t)d.batch * 8);
  p->off_flags = o; o += align256((size_t)d.batch * 4);
  p->off_stats = o;
  p->off_stash = o; o += align256(rows * roww * 4);
  p->off_post = o;
  p->total = o;
  return true;
}

// Tuning overrides for the lattice kernel's role counts and ring sizes, read ONCE per process (experiments
// run one configuration per process; a production process never sets them).
struct FzTune { int nc, np, nwarps, rv, r, pf, nap, cf, latency, dbg; };
static const FzTune& fz_tune() {
  static const FzTune t = {env_int("E2E_CTC_NC", 0), env_int("E2E_CTC_NP", 0), env_int("E2E_CTC_NWARPS", 0),
                           env_int("E2E_CTC_RV", 0), env_int("E2E_CTC_R", 0), env_int("E2E_CTC_PF", 0),
                           env_int("E2E_CTC_NAP", -1), env_int("E2E_CTC_CF", 0), env_int("E2E_CTC_LATENCY", -1), env_int("E2E_CTC_DBG", 0)};
  return t;
}

static bool make_fused_plan(const e2e_ctc_desc& d, bool fused, LossPlan* p) {
  const int Lmax = d.max_targets, V = d.alphabet;
  const int NB = Lmax <= 63 ? 1 : (Lmax <= 127 ? 2 : (Lmax <= 255 ? 4 : (Lmax <= kMaxTargets ? 10 : 0)));
  if (!NB) return false;
  const FzTune& tn = fz_tune();
  const bool dense = fused && V <= kDenseMaxAlphabet;

  // latency shapes: every CTA of the launch has an SM to itself (one 2-CTA cluster per utterance), so the
  // CTA is laid out for the shortest per-frame chain; otherwise several CTAs share an SM and the layout is
  // sized for occupancy
  bool latency = 2 * d.batch <= 148;
  // gather mode (K1 and K3 do the streaming): the kernel is a latency chain per CTA even with two CTAs on an SM --
  // the eight-warp layout (four combiners) measured 9 % faster than the occupancy layout on BASELINE config 4
  if (!dense && 2 * d.batch <= 2 * 148) latency = true;
  if (tn.latency == 0 || tn.latency == 1) latency = tn.latency == 1;
  FzLayout L;
  memset(&L, 0, sizeof(L));
  L.NB = NB;
  L.gather = dense ? 0 : 1;
  L.dbg = tn.dbg;
  const bool heavy_rows = !dense || V > 32;   // producer work per frame: a whole row of > 32 symbols, or a gather
  const int maxw = NB <= 4 ? 8 : 5;   // (six or eight combiner warps measured no better than four)
  const int nsc = NB <= 4 ? 1 : 0;              // scaler warp (exponent snapshots): every class but the large-lattice one
  if (NB == 10) { L.NP = 1; L.NC = 3; L.nwarps = 5; }
  else if (latency) { L.NP = 2; L.NC = 4; L.nwarps = 8; }
  else { L.NP = heavy_rows ? 2 : 1; L.NC = NB >= 4 ? 3 : 2; L.nwarps = 1 + nsc + L.NP + L.NC; }
  if (tn.np == 1 || tn.np == 2 || tn.np == 4) L.NP = tn.np;   // a power of two (the lattice masks with NP-1)
  if (tn.nc >= 1 && tn.nc <= 8) L.NC = tn.nc;
  if (tn.nwarps) L.nwarps = tn.nwarps;
  if (L.nwarps < 1 + nsc + L.NP + L.NC) L.nwarps = 1 + nsc + L.NP + L.NC;
  if (L.nwarps > maxw) return false;
  L.PF = (latency && NB < 10) ? 4 : 2;
  if (tn.pf == 2 || tn.pf == 4) L.PF = tn.pf;
  L.CF = NB == 10 ? 4 : 8;
  if (tn.cf == 4 || tn.cf == 8) L.CF = tn.cf;
  L.RV = NB == 10 ? 8 : 16;
  if (tn.rv >= 8 && !(tn.rv & (tn.rv - 1))) L.RV = tn.rv;
  if (L.RV < 2 * L.CF) L.RV = 2 * L.CF;
  L.nap = tn.nap >= 0 ? tn.nap : 32;
  L.es = dense ? ((V + 2) | 1) : (64 * NB + 1);   // odd: the producers' lane-per-frame stores are bank-conflict free
  L.PB = 8;            // frames per producer block (one warp per frame, four frames in flight)
  L.pb_log2 = 3;
  L.R = 2 * L.PB;                                 // at least two producer blocks in the ring, four when they fit 32 KB
  // gather mode: four blocks -- a producer's block is two dependent L2 round trips (~4k cycles), twice what the sweep
  // needs for a block, so with two blocks in the ring the lattice warp waited for emissions 45 % of its time (measured)
  if ((size_t)4 * L.PB * L.es * 8 <= (size_t)(dense ? 32 : 48) * 1024) L.R = 4 * L.PB;
  while (L.R < 128 && (size_t)2 * L.R * L.es * 8 <= (size_t)(latency ? 48 : 24) * 1024) L.R *= 2;
  if (tn.r >= 2 * L.PB && !(tn.r & (tn.r - 1))) L.R = tn.r;
  if (dense && d.dtype != E2E_F64 && V <= 32 && L.R < 64) L.R = 64;   // the lane-per-frame row producer (<= 32 symbols) works in passes of 32 frames: two in the ring
  if (L.R > 16 * L.PB) L.R = 16 * L.PB;   // at most 16 emission blocks (one mbarrier each)
  if (L.RV > 32) L.RV = 32;
  auto ilog2 = [](int v) { int k = 0; while ((1 << k) < v) k++; return k; };
  L.rv_log2 = ilog2(L.RV);
  L.neb_log2 = ilog2(L.R / L.PB);
  L.neb_mask = L.R / L.PB - 1;
  const int nbp = (NB + 3) & ~3;
  L.vframe = NB * 640 + 32 * nbp * 4;
  L.srow = 640 * NB;
  L.prow = dense ? ((V + 4) & ~3) : 0;   // dense: per-symbol fixed-point accumulators of one frame + a spare slot
  size_t off = 0;
  L.off_lab = 0; off = (size_t)align16i((size_t)(64 * NB + 1) * 4);
  L.off_occ = (int)off; off = (size_t)align16i(off + (size_t)nsc * 2 * 20 * 32 * NB);   // scale table: 2 slots x 32*NB blocks x {f, fb, en}
  L.off_E = (int)off; off = (size_t)align16i(off + (size_t)L.R * L.es * 8);
  L.off_val = (int)off; off += (size_t)L.RV * L.vframe;
  L.off_stage = (int)off; off += (size_t)L.NC * L.PF * L.srow;
  L.off_post = (int)off; off = (size_t)align16i(off + (size_t)L.NC * L.prow * 4);
  L.off_ctl = (int)off; off += fused_ctl_bytes();
  L.total = (int)off;
  if (off > 220 * 1024) return false;
  // roles: warp 0 sweeps the lattice; the helpers go to warps on the OTHER SM sub-partitions first (warp w
  // runs on scheduler w % 4), combiners before producers
  for (int w = 0; w < 16; w++) { L.role[w] = 3; L.ridx[w] = 0; }
  L.role[0] = 0;
  {
    int order[16], n = 0;
    for (int w = 1; w < L.nwarps; w++) if (w % 4 != 0) order[n++] = w;
    for (int w = 1; w < L.nwarps; w++) if (w % 4 == 0) order[n++] = w;
    int k = 0;
    for (int q = 0; q < L.NC; q++) { L.role[order[k]] = 1; L.ridx[order[k]] = (signed char)q; k++; }
    for (int q = 0; q < L.NP; q++) { L.role[order[k]] = 2; L.ridx[order[k]] = (signed char)q; k++; }
    if (nsc) L.role[order[n - 1]] = 4;   // the scaler is light: it takes the last warp (the lattice warp's sub-partition when there are 8)
  }
  p->kind = kPlanFused;
  p->fz = L;
  p->dense = dense ? 1 : 0;
  p->cells = 128 * NB;
  p->post_stride = p->cells / 2 + 4;
  p->roww = 5 * 32 * NB;
  p->smem = off;
  const size_t rows = (size_t)d.batch * d.max_frames;
  size_t o = 0;
  p->off_status = o; o += 256;
  p->off_meet = o; o += align256((size_t)d.batch * 8);
  p->off_flags = o; o += align256((size_t)d.batch * 4);
  p->off_stats = o; o += dense ? 0 : align256(rows * (d.dtype == E2E_F64 ? 16 : 8));
  p->off_stash = o; o += align256(rows * p->roww * 4);
  p->off_post = o; o += dense ? 0 : align256(rows * p->post_stride * 4);
  p->emis_stride = dense ? 0 : Lmax + 1;         // [label 0 .. label Lmax-1 | blank] doubles per frame, written by K1
  p->off_emis = o; o += dense ? 0 : align256(rows * (size_t)p->emis_stride * 8);
  p->total = o;
  return true;
}


// Which lattice kernel runs a shape (all three are parity-tested against the oracle on the shapes they take):
//  * wave kernel: latency shapes (B <= 148 utterances, small alphabet, 128..255 labels) -- four lattice warps per sweep;
//  * one-warp-per-sweep kernel: throughput shapes with small alphabets (many utterances per SM);
//  * general kernel: everything else -- large alphabets (gather mode), and a single label symbol (V == 2, where the
//    sweep kernel's lane-exponent rule loses the only feasible path of a tight alignment under very peaky
//    emissions: round 1's open parity corner; the general kernel's per-block exponents do not).
bool make_loss_plan(const e2e_ctc_desc& d, bool fused, LossPlan* p) {
  memset(p, 0, sizeof(*p));
  const int force = g_force_kernel.load(std::memory_order_relaxed);   // testing hook: 0 general, 1 wave, 2 sweep (when the shape allows)
  const bool gather = !fused || d.alphabet > kDenseMaxAlphabet;
  if (force == kPlanFused) return make_fused_plan(d, fused, p);
  if (force == kPlanWave && make_wave_plan(d, fused, p)) return true;
  if (force == kPlanSweep && make_sweep_plan(d, fused, p)) return true;
  if (d.alphabet == 2) return make_fused_plan(d, fused, p);
  if (gather && d.batch <= 256 && make_fused_plan(d, fused, p)) return true;
  // lattices of <= 256 cells (the wave kernel would run them on one or two lattice warps with its small helper set) in
  // batches that leave every cluster an SM pair's worth of room: the general kernel beats both the wave kernel (c1: 24.0
  // against 27.5 us; B=64, T=400, <= 63 / 95 / 127 labels: 94 / 115 / 113 against 138 / 152 / 151 us) and the two-warp sweep
  // CTA (a c3-shaped bucket of 128 utterances, one rank of an 8-GPU job: 103 against 131 us).  From 128 labels on the wave
  // kernel's four lattice warps win (113 against 138 us).
  if (!gather && 2 * d.max_targets + 1 <= 256 && d.batch <= 148 && make_fused_plan(d, fused, p)) return true;
  memset(p, 0, sizeof(*p));
  if (make_wave_plan(d, fused, p)) return true;
  memset(p, 0, sizeof(*p));
  if (make_sweep_plan(d, fused, p)) return true;
  memset(p, 0, sizeof(*p));
  return make_fused_plan(d, fused, p);
}

static int check_ws(const void* ws, size_t have, size_t need) {
  if (!ws || (reinterpret_cast<uintptr_t>(ws) & 255)) { set_error("workspace null or not 256-byte aligned"); return E2E_ERR_WORKSPACE; }
  if (have < need) { set_error("workspace too small: %zu < %zu bytes", have, need); return E2E_ERR_WORKSPACE; }
  return E2E_OK;
}

// split path: K1 row statistics + lattice (gather mode; posteriors left in the workspace for K3)
static int loss_forward(const e2e_ctc_desc& d, const LossPlan& p, const void* logits, const void* targets,
                        const void* in_len, const void* tgt_len, void* losses, char* ws, cudaStream_t s) {
  E2E_CUDA_TRY(cudaMemsetAsync(ws + p.off_status, 0, p.off_flags, s));   // status word + the meet flags
  const bool emis = p.kind == kPlanFused && p.emis_stride > 0;
  int rc = launch_row_stats(d, logits, ws + p.off_stats, emis ? reinterpret_cast<double*>(ws + p.off_emis) : nullptr,
                            p.emis_stride, targets, in_len, tgt_len, s);
  if (rc != E2E_OK) return rc;
  if (p.kind == kPlanSweep) return launch_sweep(d, p, logits, targets, in_len, tgt_len, losses, nullptr, 1.0, ws, s);
  return launch_fused(d, p, logits, targets, in_len, tgt_len, losses, nullptr, 1.0, ws, s);
}

// loss + gradient (scale folded in) in as few launches as the shape allows:
// dense shapes: ONE kernel; otherwise K1 + lattice + K3
static int loss_fwd_bwd(const e2e_ctc_desc& d, const LossPlan& p, const void* logits, const void* targets,
                        const void* in_len, const void* tgt_len, void* losses, void* grads, double scale,
                        char* ws, cudaStream_t s) {
  if (p.dense) {
    E2E_CUDA_TRY(cudaMemsetAsync(ws + p.off_status, 0, p.off_flags, s));   // status word + the meet flags
    if (p.kind == kPlanWave) return launch_wave(d, p, logits, targets, in_len, tgt_len, losses, grads, scale, ws, s);
    if (p.kind == kPlanSweep) return launch_sweep(d, p, logits, targets, in_len, tgt_len, losses, grads, scale, ws, s);
    return launch_fused(d, p, logits, targets, in_len, tgt_len, losses, grads, scale, ws, s);
  }
  int rc = loss_forward(d, p, logits, targets, in_len, tgt_len, losses, ws, s);
  if (rc != E2E_OK) return rc;
  return launch_grad(d, p, logits, targets, in_len, tgt_len, nullptr, 0, scale, grads, ws, s);
}

// ---- host-buffer engine -------------------------------------------------------------------------
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int ensure(size_t n) {
    if (n <= cap) return E2E_OK;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    const size_t want = align256(n + n / 8);
    E2E_CUDA_TRY(cudaMalloc(&p, want));
    cap = want;
    return E2E_OK;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

}  // namespace e2e

struct e2e_ctc_engine {
  int device = 0;
  cudaStream_t stream = nullptr;
  e2e::DevBuf logits, grads, targets, in_len, tgt_len, losses, ws, decoded, decoded_len;
  uint64_t h2d = 0, d2h = 0, zero_copy_bytes = 0;
  // chunked host pipeline: copy-in stream, compute streams, copy-out stream, one event pair per chunk
  static constexpr int kMaxChunks = 8, kComputeStreams = 8;   // one compute stream per chunk: chunks never queue behind each other
  cudaStream_t s_in = nullptr, s_out = nullptr, s_comp[kComputeStreams] = {};
  cudaEvent_t ev_in[kMaxChunks] = {}, ev_comp[kMaxChunks] = {}, ev_free = nullptr;
  bool pipe_ready = false;
};

using namespace e2e;

extern "C" {

const char* e2e_ctc_version(void) { return "e2e_ctc 0.1.0 (sm_100a, abi 1)"; }
const char* e2e_last_error_string(void) { return g_err; }
uint64_t e2e_ctc_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int e2e_ctc_profile_enable(int32_t on) {
  g_prof_on.store(on ? 1 : 0, std::memory_order_relaxed);
  return E2E_OK;
}

int e2e_ctc_profile_read(double* ms, uint64_t* launches, int32_t n_kinds) {
  if (!ms || !launches || n_kinds < kMinProfileKinds) { set_error("profile_read needs %d slots", (int)kMinProfileKinds); return E2E_ERR_INVALID_ARGUMENT; }
  for (int i = 0; i < n_kinds; i++) { ms[i] = 0.0; launches[i] = 0; }
  std::lock_guard<std::mutex> lk(g_prof_mu);
  for (EventPair& ev : g_prof_pending) {
    E2E_CUDA_TRY(cudaEventSynchronize(ev.b));
    float t = 0.f;
    E2E_CUDA_TRY(cudaEventElapsedTime(&t, ev.a, ev.b));
    if (ev.kind < n_kinds) {
      ms[ev.kind] += (double)t;
      launches[ev.kind] += 1;
    }
    g_prof_free.emplace_back(ev.a, ev.b);
  }
  g_prof_pending.clear();
  return E2E_OK;
}

/* testing hook (not part of the public header): force a lattice kernel where the shape allows it.
 * -1 automatic, 0 general kernel, 1 wave kernel, 2 one-warp-per-sweep kernel */
int e2e_ctc_debug_force_kernel(int32_t kind) { g_force_kernel.store(kind, std::memory_order_relaxed); return E2E_OK; }

int e2e_ctc_get_limits(e2e_ctc_limits* out) {
  if (!out) { set_error("null limits"); return E2E_ERR_INVALID_ARGUMENT; }
  out->max_alphabet = kMaxAlphabet;
  out->max_targets = kMaxTargets;
  out->abi_version = E2E_CTC_ABI_VERSION;
  out->sm_arch = 100;
  return E2E_OK;
}

size_t e2e_ctc_loss_workspace_bytes(const e2e_ctc_desc* desc) {
  if (check_desc(desc, true) != E2E_OK) return 0;
  LossPlan p;
  LossPlan q;
  if (!make_loss_plan(*desc, false, &p) || !make_loss_plan(*desc, true, &q)) { set_error("no lattice configuration for max_targets=%d", desc->max_targets); return 0; }
  return p.total > q.total ? p.total : q.total;
}

int e2e_ctc_loss_forward_device(const e2e_ctc_desc* desc, const void* logits, const void* targets,
                                const void* logits_lengths, const void* targets_lengths, void* losses,
                                void* workspace, size_t workspace_bytes, void* cuda_stream) {
  int rc = check_desc(desc, true);
  if (rc != E2E_OK) return rc;
  if (!logits || !logits_lengths || !targets_lengths || !losses || (!targets && desc->max_targets > 0)) {
    set_error("null pointer argument");
    return E2E_ERR_INVALID_ARGUMENT;
  }
  LossPlan p;
  if (!make_loss_plan(*desc, false, &p)) { set_error("no lattice configuration for max_targets=%d", desc->max_targets); return E2E_ERR_UNSUPPORTED; }
  rc = check_ws(workspace, workspace_bytes, p.total);
  if (rc != E2E_OK) return rc;
  return loss_forward(*desc, p, logits, targets, logits_lengths, targets_lengths, losses,
                      reinterpret_cast<char*>(workspace), reinterpret_cast<cudaStream_t>(cuda_stream));
}

int e2e_ctc_loss_backward_device(const e2e_ctc_desc* desc, const void* logits, const void* targets,
                                 const void* logits_lengths, const void* targets_lengths,
                                 const void* grad_out, int32_t grad_out_count, double host_scale,
                                 void* grads, void* workspace, size_t workspace_bytes, void* cuda_stream) {
  int rc = check_desc(desc, true);
  if (rc != E2E_OK) return rc;
  if (!logits || !logits_lengths || !targets_lengths || !grads || (!targets && desc->max_targets > 0)) {
    set_error("null pointer argument");
    return E2E_ERR_INVALID_ARGUMENT;
  }
  if (grad_out && grad_out_count != 1 && grad_out_count != desc->batch) {
    set_error("grad_out_count must be 1 or B");
    return E2E_ERR_INVALID_ARGUMENT;
  }
  LossPlan p;
  if (!make_loss_plan(*desc, false, &p)) { set_error("no lattice configuration"); return E2E_ERR_UNSUPPORTED; }
  rc = check_ws(workspace, workspace_bytes, p.total);
  if (rc != E2E_OK) return rc;
  return launch_grad(*desc, p, logits, targets, logits_lengths, targets_lengths, grad_out, grad_out_count,
                     host_scale, grads, reinterpret_cast<const char*>(workspace),
                     reinterpret_cast<cudaStream_t>(cuda_stream));
}

static int step_impl(const e2e_ctc_desc* desc, const void* logits, const void* targets, const void* logits_lengths,
                     const void* targets_lengths, void* losses, void* grads, double grad_scale, void* reduced,
                     double* reduced_f64, double reduce_scale, void* workspace, size_t workspace_bytes, cudaStream_t s) {
  int rc = check_desc(desc, true);
  if (rc != E2E_OK) return rc;
  if (!logits || !logits_lengths || !targets_lengths || !losses || !grads || (!targets && desc->max_targets > 0)) {
    set_error("null pointer argument");
    return E2E_ERR_INVALID_ARGUMENT;
  }
  LossPlan p;
  if (!make_loss_plan(*desc, true, &p)) { set_error("no lattice configuration for max_targets=%d", desc->max_targets); return E2E_ERR_UNSUPPORTED; }
  rc = check_ws(workspace, workspace_bytes, p.total);
  if (rc != E2E_OK) return rc;
  rc = loss_fwd_bwd(*desc, p, logits, targets, logits_lengths, targets_lengths, losses, grads, grad_scale,
                    reinterpret_cast<char*>(workspace), s);
  if (rc != E2E_OK) return rc;
  if (reduced || reduced_f64) return launch_reduce(losses, desc->dtype, desc->batch, reduce_scale, reduced, reduced_f64, s);
  return E2E_OK;
}

int e2e_ctc_loss_fwd_bwd_device(const e2e_ctc_desc* desc, const void* logits, const void* targets,
                                const void* logits_lengths, const void* targets_lengths, void* losses,
                                void* grads, void* workspace, size_t workspace_bytes, void* cuda_stream) {
  return step_impl(desc, logits, targets, logits_lengths, targets_lengths, losses, grads, 1.0, nullptr, nullptr, 1.0,
                   workspace, workspace_bytes, reinterpret_cast<cudaStream_t>(cuda_stream));
}

int e2e_ctc_loss_step_device(const e2e_ctc_desc* desc, const void* logits, const void* targets,
                             const void* logits_lengths, const void* targets_lengths, void* losses,
                             void* grads, double grad_scale, void* reduced, double* reduced_f64,
                             double reduce_scale, void* workspace, size_t workspace_bytes, void* cuda_stream) {
  return step_impl(desc, logits, targets, logits_lengths, targets_lengths, losses, grads, grad_scale, reduced,
                   reduced_f64, reduce_scale, workspace, workspace_bytes, reinterpret_cast<cudaStream_t>(cuda_stream));
}

int e2e_ctc_scale_rows_device(const e2e_ctc_desc* desc, void* grads, const void* grad_out, int32_t grad_out_count,
                              void* cuda_stream) {
  int rc = check_desc(desc, false);
  if (rc != E2E_OK) return rc;
  if (!grads || !grad_out || (grad_out_count != 1 && grad_out_count != desc->batch)) {
    set_error("scale_rows: grads / grad_out required, grad_out_count must be 1 or B");
    return E2E_ERR_INVALID_ARGUMENT;
  }
  return launch_scale_rows(*desc, grads, grad_out, grad_out_count, reinterpret_cast<cudaStream_t>(cuda_stream));
}

int e2e_ctc_loss_reduce_device(const void* losses, int32_t dtype, int32_t batch, double scale, void* out,
                               double* out_f64, void* cuda_stream) {
  if (!losses || batch < 1 || elem_size(dtype) == 0 || (!out && !out_f64)) {
    set_error("bad reduce arguments");
    return E2E_ERR_INVALID_ARGUMENT;
  }
  return launch_reduce(losses, dtype, batch, scale, out, out_f64, reinterpret_cast<cudaStream_t>(cuda_stream));
}

int e2e_ctc_loss_check_device(const void* workspace, int32_t* status_host, void* cuda_stream) {
  if (!workspace || !status_host) { set_error("null pointer argument"); return E2E_ERR_INVALID_ARGUMENT; }
  cudaStream_t s = reinterpret_cast<cudaStream_t>(cuda_stream);
  E2E_CUDA_TRY(cudaMemcpyAsync(status_host, workspace, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  E2E_CUDA_TRY(cudaStreamSynchronize(s));
  return E2E_OK;
}

size_t e2e_ctc_greedy_workspace_bytes(const e2e_ctc_desc* desc) {
  if (check_desc(desc, false) != E2E_OK) return 0;
  return align256((size_t)desc->batch * desc->max_frames * sizeof(int));
}

int e2e_ctc_greedy_decode_device(const e2e_ctc_desc* desc, const void* logits, const void* logits_lengths,
                                 int64_t* decoded, int64_t* decoded_lengths, void* workspace,
                                 size_t workspace_bytes, void* cuda_stream) {
  int rc = check_desc(desc, false);
  if (rc != E2E_OK) return rc;
  if (!logits || !decoded || !decoded_lengths) { set_error("null pointer argument"); return E2E_ERR_INVALID_ARGUMENT; }
  rc = check_ws(workspace, workspace_bytes, e2e_ctc_greedy_workspace_bytes(desc));
  if (rc != E2E_OK) return rc;
  return launch_greedy(*desc, logits, logits_lengths, decoded, decoded_lengths,
                       reinterpret_cast<char*>(workspace), reinterpret_cast<cudaStream_t>(cuda_stream));
}

// ---- LM-free prefix beam search (SURVEY 8(f3)) -----------------------------------------------------------
static int check_beam(const e2e_ctc_desc* desc, int32_t beam_width, int32_t n_best, int32_t space_idx, double wip) {
  int rc = check_desc(desc, false);
  if (rc != E2E_OK) return rc;
  if (beam_width < 1) { set_error("beam_width %d < 1", beam_width); return E2E_ERR_INVALID_ARGUMENT; }
  if (n_best < 1 || n_best > beam_width) {
    set_error("n_best %d outside [1, beam_width = %d]", n_best, beam_width);
    return E2E_ERR_INVALID_ARGUMENT;
  }
  if (space_idx < -1 || space_idx >= desc->alphabet) { set_error("space_idx %d outside [-1,%d)", space_idx, desc->alphabet); return E2E_ERR_INVALID_ARGUMENT; }
  if (!(wip == wip) || wip == INFINITY || wip == -INFINITY) { set_error("wip must be finite"); return E2E_ERR_INVALID_ARGUMENT; }
  if (!beam_supported(*desc, beam_width)) {
    set_error("beam search: beam_width %d with alphabet %d exceeds this build's limits (beam_width <= 256, beam and bitmap state <= 200 KB of shared memory)",
              beam_width, desc->alphabet);
    return E2E_ERR_UNSUPPORTED;
  }
  return E2E_OK;
}

size_t e2e_ctc_beam_nbest_workspace_bytes(const e2e_ctc_desc* desc, int32_t beam_width, int32_t n_best) {
  if (check_beam(desc, beam_width, n_best, -1, 0.0) != E2E_OK) return 0;
  return align256(beam_workspace_bytes(*desc, beam_width));   // the trie; the n_best backtraces need nothing more
}

size_t e2e_ctc_beam_workspace_bytes(const e2e_ctc_desc* desc, int32_t beam_width) {
  return e2e_ctc_beam_nbest_workspace_bytes(desc, beam_width, 1);
}

int e2e_ctc_beam_nbest_device(const e2e_ctc_desc* desc, int32_t beam_width, int32_t n_best, int32_t space_idx, double wip,
                              const void* logits, const void* logits_lengths, int64_t* decoded, int64_t* decoded_lengths,
                              double* scores, double* log_probs, int64_t* ties, void* workspace, size_t workspace_bytes,
                              void* cuda_stream) {
  int rc = check_beam(desc, beam_width, n_best, space_idx, wip);
  if (rc != E2E_OK) return rc;
  if (!logits || !decoded || !decoded_lengths || !scores) { set_error("null pointer argument"); return E2E_ERR_INVALID_ARGUMENT; }
  rc = check_ws(workspace, workspace_bytes, e2e_ctc_beam_nbest_workspace_bytes(desc, beam_width, n_best));
  if (rc != E2E_OK) return rc;
  return launch_beam(*desc, beam_width, n_best, space_idx, wip, logits, logits_lengths, decoded, decoded_lengths, scores,
                     log_probs, ties, reinterpret_cast<char*>(workspace), reinterpret_cast<cudaStream_t>(cuda_stream));
}

int e2e_ctc_beam_decode_device(const e2e_ctc_desc* desc, int32_t beam_width, int32_t space_idx, double wip,
                               const void* logits, const void* logits_lengths, int64_t* decoded, int64_t* decoded_lengths,
                               int64_t* ties, void* workspace, size_t workspace_bytes, void* cuda_stream) {
  int rc = check_beam(desc, beam_width, 1, space_idx, wip);
  if (rc != E2E_OK) return rc;
  if (!logits || !decoded || !decoded_lengths) { set_error("null pointer argument"); return E2E_ERR_INVALID_ARGUMENT; }
  rc = check_ws(workspace, workspace_bytes, e2e_ctc_beam_workspace_bytes(desc, beam_width));
  if (rc != E2E_OK) return rc;
  return launch_beam(*desc, beam_width, 1, space_idx, wip, logits, logits_lengths, decoded, decoded_lengths, nullptr, nullptr,
                     ties, reinterpret_cast<char*>(workspace), reinterpret_cast<cudaStream_t>(cuda_stream));
}

// ---- CTC log-likelihood of N hypotheses per utterance (K9) -------------------------------------------
static int check_score(const e2e_ctc_desc* desc, int32_t n_hyp) {
  int rc = check_desc(desc, true);
  if (rc != E2E_OK) return rc;
  if (n_hyp < 1) { set_error("n_hyp %d < 1", n_hyp); return E2E_ERR_INVALID_ARGUMENT; }
  if (desc->max_targets > 0 && desc->targets_stride_b < desc->max_targets) {
    set_error("hypothesis row stride %lld < max_targets %d", (long long)desc->targets_stride_b, desc->max_targets);
    return E2E_ERR_INVALID_ARGUMENT;
  }
  if (desc->logits_stride_b < 0 || desc->logits_stride_t < 0) { set_error("negative logits stride"); return E2E_ERR_INVALID_ARGUMENT; }
  if ((long long)desc->batch * n_hyp > 0x7fffffffLL) {
    set_error("batch %d x n_hyp %d hypotheses exceed this build's limit", desc->batch, n_hyp);
    return E2E_ERR_UNSUPPORTED;
  }
  if (!score_supported(*desc)) {
    set_error("score: max_targets %d with alphabet %d does not fit shared memory", desc->max_targets, desc->alphabet);
    return E2E_ERR_UNSUPPORTED;
  }
  return E2E_OK;
}

size_t e2e_ctc_score_workspace_bytes(const e2e_ctc_desc* desc, int32_t n_hyp) {
  if (check_score(desc, n_hyp) != E2E_OK) return 0;
  return 256;   // nothing is stashed; 0 stays the "unsupported" answer
}

int e2e_ctc_score_device(const e2e_ctc_desc* desc, int32_t n_hyp, const void* logits, const void* hyps,
                         const void* logits_lengths, const void* hyp_lengths, double* scores, void* workspace,
                         size_t workspace_bytes, void* cuda_stream) {
  int rc = check_score(desc, n_hyp);
  if (rc != E2E_OK) return rc;
  if (!logits || !hyp_lengths || !scores || (!hyps && desc->max_targets > 0)) {
    set_error("null pointer argument");
    return E2E_ERR_INVALID_ARGUMENT;
  }
  rc = check_ws(workspace, workspace_bytes, e2e_ctc_score_workspace_bytes(desc, n_hyp));
  if (rc != E2E_OK) return rc;
  return launch_score(*desc, n_hyp, logits, hyps, logits_lengths, hyp_lengths, scores,
                      reinterpret_cast<cudaStream_t>(cuda_stream));
}

// ---- the scorer's backward (K10 + row kernel) ------------------------------------------------------------
static int check_score_backward(const e2e_ctc_desc* desc, int32_t n_hyp) {
  int rc = check_score(desc, n_hyp);
  if (rc != E2E_OK) return rc;
  if (desc->grads_stride_b < 0 || desc->grads_stride_t < 0) { set_error("negative gradient stride"); return E2E_ERR_INVALID_ARGUMENT; }
  if (!score_backward_supported(*desc)) {
    set_error("score backward: max_targets %d with alphabet %d does not fit shared memory", desc->max_targets, desc->alphabet);
    return E2E_ERR_UNSUPPORTED;
  }
  return E2E_OK;
}

size_t e2e_ctc_score_backward_workspace_bytes(const e2e_ctc_desc* desc, int32_t n_hyp) {
  if (check_score_backward(desc, n_hyp) != E2E_OK) return 0;
  return score_backward_workspace_bytes(*desc, n_hyp);   // 0 (message set) on overflow
}

int e2e_ctc_score_backward_device(const e2e_ctc_desc* desc, int32_t n_hyp, const void* logits, const void* hyps,
                                  const void* logits_lengths, const void* hyp_lengths, const double* grad_scores,
                                  void* grads, void* workspace, size_t workspace_bytes, void* cuda_stream) {
  int rc = check_score_backward(desc, n_hyp);
  if (rc != E2E_OK) return rc;
  if (!logits || !hyp_lengths || !grad_scores || !grads || (!hyps && desc->max_targets > 0)) {
    set_error("null pointer argument");
    return E2E_ERR_INVALID_ARGUMENT;
  }
  const size_t need = e2e_ctc_score_backward_workspace_bytes(desc, n_hyp);
  if (need == 0) return E2E_ERR_UNSUPPORTED;
  rc = check_ws(workspace, workspace_bytes, need);
  if (rc != E2E_OK) return rc;
  return launch_score_backward(*desc, n_hyp, logits, hyps, logits_lengths, hyp_lengths, grad_scores, grads,
                               reinterpret_cast<char*>(workspace), reinterpret_cast<cudaStream_t>(cuda_stream));
}

// ---- word / token errors of N hypotheses per utterance (K11) -----------------------------------------------------
static int check_edit(const e2e_ctc_edit_desc* d) {
  if (!d) { set_error("null descriptor"); return E2E_ERR_INVALID_ARGUMENT; }
  if (d->batch < 1 || d->n_hyp < 1 || d->hyp_width < 0 || d->ref_width < 0) {
    set_error("bad shape batch=%d n_hyp=%d hyp_width=%d ref_width=%d", d->batch, d->n_hyp, d->hyp_width, d->ref_width);
    return E2E_ERR_INVALID_ARGUMENT;
  }
  if ((d->tokens_itype != E2E_I32 && d->tokens_itype != E2E_I64) || (d->lengths_itype != E2E_I32 && d->lengths_itype != E2E_I64)) {
    set_error("bad index type");
    return E2E_ERR_INVALID_ARGUMENT;
  }
  if (d->separator < -1) { set_error("separator %d: -1 (token level) or a token id >= 0 (word level)", d->separator); return E2E_ERR_INVALID_ARGUMENT; }
  if ((d->hyp_width > 0 && d->hyp_stride_b < d->hyp_width) || (d->ref_width > 0 && d->ref_stride_b < d->ref_width)) {
    set_error("row stride below the width: hyps %lld < %d or refs %lld < %d", (long long)d->hyp_stride_b, d->hyp_width,
              (long long)d->ref_stride_b, d->ref_width);
    return E2E_ERR_INVALID_ARGUMENT;
  }
  if (d->ref_width > 4095 || d->hyp_width > 65535) {
    set_error("edit distance: reference width %d (limit 4095) or hypothesis width %d (limit 65535) exceeds this build's limits",
              d->ref_width, d->hyp_width);
    return E2E_ERR_UNSUPPORTED;
  }
  if ((long long)d->batch * ((d->n_hyp + 7) / 8) > 0x7fffffffLL) {
    set_error("batch %d x n_hyp %d hypotheses exceed the grid (2^31 - 1 CTAs)", d->batch, d->n_hyp);
    return E2E_ERR_UNSUPPORTED;
  }
  return E2E_OK;
}

size_t e2e_ctc_edit_distance_workspace_bytes(const e2e_ctc_edit_desc* desc) {
  if (check_edit(desc) != E2E_OK) return 0;
  return 256;   // nothing is stashed; 0 stays the "unsupported" answer
}

int e2e_ctc_edit_distance_device(const e2e_ctc_edit_desc* desc, const void* hyps, const void* hyp_lengths,
                                 const void* refs, const void* ref_lengths, int64_t* errors, int64_t* substitutions,
                                 int64_t* insertions, int64_t* deletions, int64_t* reference_units,
                                 void* workspace, size_t workspace_bytes, void* cuda_stream) {
  int rc = check_edit(desc);
  if (rc != E2E_OK) return rc;
  if (!hyp_lengths || !ref_lengths || !errors || !substitutions || !insertions || !deletions || !reference_units ||
      (!hyps && desc->hyp_width > 0) || (!refs && desc->ref_width > 0)) {
    set_error("null pointer argument");
    return E2E_ERR_INVALID_ARGUMENT;
  }
  rc = check_ws(workspace, workspace_bytes, e2e_ctc_edit_distance_workspace_bytes(desc));
  if (rc != E2E_OK) return rc;
  return launch_edit_distance(*desc, hyps, hyp_lengths, refs, ref_lengths, errors, substitutions, insertions, deletions,
                              reference_units, reinterpret_cast<cudaStream_t>(cuda_stream));
}

// ---- pinned host memory for result buffers -------------------------------------------------------
// The host-buffer entry points write their results straight into PINNED caller buffers (see e2e_ctc_engine_loss_host);
// a binding that has no pinned allocator of its own takes its result buffers from here.
int e2e_ctc_host_alloc(size_t bytes, void** out) {
  if (!out || bytes == 0) { set_error("host_alloc: bad arguments"); return E2E_ERR_INVALID_ARGUMENT; }
  *out = nullptr;
  E2E_CUDA_TRY(cudaHostAlloc(out, bytes, cudaHostAllocPortable));
  return E2E_OK;
}

int e2e_ctc_host_free(void* p) {
  if (!p) return E2E_OK;
  E2E_CUDA_TRY(cudaFreeHost(p));
  return E2E_OK;
}

// ---- Viterbi forced alignment (SURVEY 8(f2)) -------------------------------------------------------
// The alignment has its own width limit (viterbi_supported), not the loss kernels' kMaxTargets.
static int check_viterbi(const e2e_ctc_desc* desc, int32_t is_ctc) {
  int rc = check_desc(desc, false);
  if (rc != E2E_OK) return rc;
  if (desc->max_targets < 0) { set_error("bad max_targets %d", desc->max_targets); return E2E_ERR_INVALID_ARGUMENT; }
  return viterbi_supported(*desc, is_ctc ? 1 : 0) ? E2E_OK : E2E_ERR_UNSUPPORTED;
}

size_t e2e_ctc_viterbi_workspace_bytes(const e2e_ctc_desc* desc, int32_t is_ctc) {
  if (check_viterbi(desc, is_ctc) != E2E_OK) return 0;
  return align256(viterbi_workspace_bytes(*desc, is_ctc ? 1 : 0, 1, 0));
}

int e2e_ctc_viterbi_align_device(const e2e_ctc_desc* desc, int32_t is_ctc, const void* log_probs, const void* targets,
                                 const void* logits_lengths, const void* targets_lengths, int64_t* aligned,
                                 void* workspace, size_t workspace_bytes, void* cuda_stream) {
  int rc = check_viterbi(desc, is_ctc);
  if (rc != E2E_OK) return rc;
  if (!log_probs || !logits_lengths || !targets_lengths || !aligned || (!targets && desc->max_targets > 0)) {
    set_error("null pointer argument");
    return E2E_ERR_INVALID_ARGUMENT;
  }
  rc = check_ws(workspace, workspace_bytes, e2e_ctc_viterbi_workspace_bytes(desc, is_ctc));
  if (rc != E2E_OK) return rc;
  return launch_viterbi(*desc, is_ctc ? 1 : 0, 1, 0, log_probs, targets, logits_lengths, targets_lengths, aligned, nullptr,
                        nullptr, nullptr, reinterpret_cast<char*>(workspace), reinterpret_cast<cudaStream_t>(cuda_stream));
}

// ---- Viterbi alignment of N hypotheses per utterance (K1 + K6) ---------------------------------------------------------
static int check_align_nbest(const e2e_ctc_desc* desc, int32_t n_hyp) {
  int rc = check_viterbi(desc, 1);
  if (rc != E2E_OK) return rc;
  if (n_hyp < 1) { set_error("n_hyp %d < 1", n_hyp); return E2E_ERR_INVALID_ARGUMENT; }
  if (desc->max_targets > 0 && desc->targets_stride_b < desc->max_targets) {
    set_error("hypothesis row stride %lld < max_targets %d", (long long)desc->targets_stride_b, desc->max_targets);
    return E2E_ERR_INVALID_ARGUMENT;
  }
  if (desc->logits_stride_b < 0 || desc->logits_stride_t < 0) { set_error("negative logits stride"); return E2E_ERR_INVALID_ARGUMENT; }
  if ((long long)desc->batch * n_hyp > 0x7fffffffLL) {
    set_error("batch %d x n_hyp %d lattices exceed the grid (2^31 - 1 CTAs)", desc->batch, n_hyp);
    return E2E_ERR_UNSUPPORTED;
  }
  return E2E_OK;
}

size_t e2e_ctc_align_nbest_workspace_bytes(const e2e_ctc_desc* desc, int32_t n_hyp) {
  if (check_align_nbest(desc, n_hyp) != E2E_OK) return 0;
  return align256(viterbi_workspace_bytes(*desc, 1, n_hyp, desc->from_logits ? 1 : 0));   // 0 (message set) on overflow
}

int e2e_ctc_align_nbest_device(const e2e_ctc_desc* desc, int32_t n_hyp, const void* logits, const void* hyps,
                               const void* logits_lengths, const void* hyp_lengths, int64_t* aligned, int64_t* token_starts,
                               int64_t* token_ends, double* path_scores, void* workspace, size_t workspace_bytes,
                               void* cuda_stream) {
  int rc = check_align_nbest(desc, n_hyp);
  if (rc != E2E_OK) return rc;
  if (!logits || !hyp_lengths || !aligned || !path_scores || (desc->max_targets > 0 && (!hyps || !token_starts || !token_ends))) {
    set_error("null pointer argument");
    return E2E_ERR_INVALID_ARGUMENT;
  }
  const size_t need = e2e_ctc_align_nbest_workspace_bytes(desc, n_hyp);
  if (need == 0) return E2E_ERR_UNSUPPORTED;
  rc = check_ws(workspace, workspace_bytes, need);
  if (rc != E2E_OK) return rc;
  return launch_viterbi(*desc, 1, n_hyp, desc->from_logits ? 1 : 0, logits, hyps, logits_lengths, hyp_lengths, aligned,
                        desc->max_targets > 0 ? token_starts : nullptr, desc->max_targets > 0 ? token_ends : nullptr,
                        path_scores, reinterpret_cast<char*>(workspace), reinterpret_cast<cudaStream_t>(cuda_stream));
}

// ---- CTC without blank (SURVEY 8(f4)) ---------------------------------------------------------------
size_t e2e_ctc_noblank_workspace_bytes(const e2e_ctc_desc* desc) {
  if (!desc || desc->batch < 1 || desc->max_frames < 1 || desc->alphabet < 1 || desc->max_targets < 0 || elem_size(desc->dtype) == 0) {
    set_error("bad descriptor");
    return 0;
  }
  if (!noblank_supported(*desc)) return 0;
  return align256(noblank_workspace_bytes(*desc));
}

int e2e_ctc_noblank_fwd_bwd_device(const e2e_ctc_desc* desc, int32_t space_idx, const void* log_probs, const void* targets,
                                   const void* logits_lengths, const void* targets_lengths, void* losses, void* grads,
                                   void* workspace, size_t workspace_bytes, void* cuda_stream) {
  const size_t need = e2e_ctc_noblank_workspace_bytes(desc);
  if (!need) return desc && desc->max_targets >= 0 && !noblank_supported(*desc) ? E2E_ERR_UNSUPPORTED : E2E_ERR_INVALID_ARGUMENT;
  if (!log_probs || !logits_lengths || !targets_lengths || !losses || !grads || (!targets && desc->max_targets > 0)) {
    set_error("null pointer argument");
    return E2E_ERR_INVALID_ARGUMENT;
  }
  if (space_idx < -1 || space_idx >= desc->alphabet) { set_error("space_idx %d outside [-1,%d)", space_idx, desc->alphabet); return E2E_ERR_INVALID_ARGUMENT; }
  if ((desc->lengths_itype != E2E_I32 && desc->lengths_itype != E2E_I64) || (desc->targets_itype != E2E_I32 && desc->targets_itype != E2E_I64)) {
    set_error("bad index type");
    return E2E_ERR_INVALID_ARGUMENT;
  }
  int rc = check_ws(workspace, workspace_bytes, need);
  if (rc != E2E_OK) return rc;
  return launch_noblank(*desc, space_idx, log_probs, targets, logits_lengths, targets_lengths, losses, grads,
                        reinterpret_cast<char*>(workspace), reinterpret_cast<cudaStream_t>(cuda_stream));
}

// ---- CUDA-graph step ------------------------------------------------------------------------------
// SURVEY 8(f1): the whole training step of the loss -- status/meet memset, lattice kernel(s), loss reduction and
// (multi-GPU) the scalar all-reduce -- captured ONCE for a fixed set of buffers and replayed with one
// cudaGraphLaunch: the step costs the host ~one driver call instead of 3-5 launches plus their argument marshalling.
}  // extern "C"

struct e2e_ctc_graph {
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  uint64_t kernels = 0;       // kernels of this library inside the graph (launch accounting)
  int device = 0;
};

extern "C" {

int e2e_ctc_graph_create(const e2e_ctc_desc* desc, const void* logits, const void* targets, const void* logits_lengths,
                         const void* targets_lengths, void* losses, void* grads, double grad_scale, void* reduced,
                         double* reduced_f64, double reduce_scale, void* workspace, size_t workspace_bytes,
                         e2e_ctc_comm* comm, e2e_ctc_graph** out) {
  if (!out) { set_error("null out pointer"); return E2E_ERR_INVALID_ARGUMENT; }
  *out = nullptr;
  if (comm && !reduced) { set_error("graph: the all-reduce needs the reduced-loss buffer"); return E2E_ERR_INVALID_ARGUMENT; }
  e2e_ctc_graph* g = new (std::nothrow) e2e_ctc_graph();
  if (!g) { set_error("out of host memory"); return E2E_ERR_CUDA; }
  cudaStream_t cs = nullptr;
  cudaError_t ce = cudaGetDevice(&g->device);
  if (ce == cudaSuccess) ce = cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking);
  if (ce != cudaSuccess) { set_error("graph: %s", cudaGetErrorString(ce)); delete g; return E2E_ERR_CUDA; }
  // a first plain run on the capture stream: one-time attribute opt-ins and lazy module loading must not
  // happen inside the capture (and argument errors surface here, outside it)
  int rc = step_impl(desc, logits, targets, logits_lengths, targets_lengths, losses, grads, grad_scale, reduced,
                     reduced_f64, reduce_scale, workspace, workspace_bytes, cs);
  if (rc == E2E_OK && cudaStreamSynchronize(cs) != cudaSuccess) { set_error("graph: warm-up run failed"); rc = E2E_ERR_CUDA; }
  if (rc != E2E_OK) { cudaStreamDestroy(cs); delete g; return rc; }
  ce = cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal);
  if (ce != cudaSuccess) { set_error("cudaStreamBeginCapture: %s", cudaGetErrorString(ce)); cudaStreamDestroy(cs); delete g; return E2E_ERR_CUDA; }
  t_capturing = 1; t_captured = 0;
  rc = step_impl(desc, logits, targets, logits_lengths, targets_lengths, losses, grads, grad_scale, reduced,
                 reduced_f64, reduce_scale, workspace, workspace_bytes, cs);
  if (rc == E2E_OK && comm) rc = e2e_ctc_comm_allreduce_sum(comm, reduced, 1, desc->dtype, cs);
  t_capturing = 0;
  g->kernels = t_captured;
  ce = cudaStreamEndCapture(cs, &g->graph);
  if (rc == E2E_OK && ce != cudaSuccess) { set_error("cudaStreamEndCapture: %s", cudaGetErrorString(ce)); rc = E2E_ERR_CUDA; }
  if (rc == E2E_OK) {
    ce = cudaGraphInstantiate(&g->exec, g->graph, 0);
    if (ce != cudaSuccess) { set_error("cudaGraphInstantiate: %s", cudaGetErrorString(ce)); rc = E2E_ERR_CUDA; }
  }
  cudaStreamDestroy(cs);
  if (rc != E2E_OK) {
    if (g->graph) cudaGraphDestroy(g->graph);
    delete g;
    return rc;
  }
  *out = g;
  return E2E_OK;
}

int e2e_ctc_graph_launch(e2e_ctc_graph* g, void* cuda_stream) {
  if (!g || !g->exec) { set_error("null graph"); return E2E_ERR_INVALID_ARGUMENT; }
  E2E_CUDA_TRY(cudaGraphLaunch(g->exec, reinterpret_cast<cudaStream_t>(cuda_stream)));
  g_launches.fetch_add(g->kernels, std::memory_order_relaxed);
  return E2E_OK;
}

void e2e_ctc_graph_destroy(e2e_ctc_graph* g) {
  if (!g) return;
  if (g->exec) cudaGraphExecDestroy(g->exec);
  if (g->graph) cudaGraphDestroy(g->graph);
  delete g;
}

// ---- engine ---------------------------------------------------------------------------------------
int e2e_ctc_engine_create(int32_t device, e2e_ctc_engine** out) {
  if (!out) { set_error("null out pointer"); return E2E_ERR_INVALID_ARGUMENT; }
  *out = nullptr;
  int n = 0;
  E2E_CUDA_TRY(cudaGetDeviceCount(&n));
  if (device < 0 || device >= n) {
    set_error("CUDA device %d not present (%d devices); this engine has no CPU fallback", device, n);
    return E2E_ERR_CUDA;
  }
  E2E_CUDA_TRY(cudaSetDevice(device));
  e2e_ctc_engine* e = new (std::nothrow) e2e_ctc_engine();
  if (!e) { set_error("out of host memory"); return E2E_ERR_CUDA; }
  e->device = device;
  cudaError_t ce = cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking);
  if (ce != cudaSuccess) { set_error("cudaStreamCreate: %s", cudaGetErrorString(ce)); delete e; return E2E_ERR_CUDA; }
  *out = e;
  return E2E_OK;
}

void e2e_ctc_engine_destroy(e2e_ctc_engine* e) {
  if (!e) return;
  cudaSetDevice(e->device);
  if (e->stream) { cudaStreamSynchronize(e->stream); cudaStreamDestroy(e->stream); }
  if (e->pipe_ready) {
    cudaStreamSynchronize(e->s_out);
    cudaStreamDestroy(e->s_in); cudaStreamDestroy(e->s_out);
    for (cudaStream_t c : e->s_comp) cudaStreamDestroy(c);
    for (int k = 0; k < e2e_ctc_engine::kMaxChunks; k++) { cudaEventDestroy(e->ev_in[k]); cudaEventDestroy(e->ev_comp[k]); }
    cudaEventDestroy(e->ev_free);
  }
  DevBuf* bufs[] = {&e->logits, &e->grads, &e->targets, &e->in_len, &e->tgt_len, &e->losses, &e->ws, &e->decoded, &e->decoded_len};
  for (DevBuf* b : bufs) b->release();
  delete e;
}

// A host buffer the GPU can address directly (pinned, mapped: cudaHostAlloc / cudaHostRegister under unified
// addressing)?  Then kernels may write their results straight into it -- the stores travel over PCIe while the
// kernel runs, instead of a device->host copy after it.
static bool host_device_ptr(const void* host, void** dev) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, host) != cudaSuccess) { cudaGetLastError(); return false; }
  if (a.type != cudaMemoryTypeHost || !a.devicePointer) return false;
  *dev = a.devicePointer;
  return true;
}

// dense [B,T,V] block in either batch-major or time-major order?
static bool dense_block(const e2e_ctc_desc& d, int64_t sb, int64_t st) {
  const int64_t B = d.batch, T = d.max_frames, V = d.alphabet;
  return (sb == T * V && st == V) || (sb == V && st == B * V) || (B == 1 && st == V) || (T == 1 && sb == V);
}

int e2e_ctc_engine_loss_host(e2e_ctc_engine* e, const e2e_ctc_desc* desc, const void* logits,
                             const void* targets, const void* logits_lengths, const void* targets_lengths,
                             void* losses, void* grads) {
  if (!e) { set_error("null engine"); return E2E_ERR_INVALID_ARGUMENT; }
  int rc = check_desc(desc, true);
  if (rc != E2E_OK) return rc;
  if (!logits || !logits_lengths || !targets_lengths || !losses || !grads || (!targets && desc->max_targets > 0)) {
    set_error("null pointer argument");
    return E2E_ERR_INVALID_ARGUMENT;
  }
  const e2e_ctc_desc& d = *desc;
  if (!dense_block(d, d.logits_stride_b, d.logits_stride_t) || !dense_block(d, d.grads_stride_b, d.grads_stride_t) ||
      (d.max_targets > 0 && d.targets_stride_b != d.max_targets)) {
    set_error("host tensors must be dense (batch-major or time-major contiguous)");
    return E2E_ERR_INVALID_ARGUMENT;
  }
  // The buffers are on the host: lengths and labels outside their legal range (undefined behaviour in the
  // reference, forward_backward.cpp:38-52 indexes with them) are rejected here, before anything is enqueued.
  {
    auto idx = [](const void* q, int is64, size_t i) -> long long {
      return is64 ? reinterpret_cast<const long long*>(q)[i] : (long long)reinterpret_cast<const int*>(q)[i];
    };
    const int l64 = d.lengths_itype == E2E_I64, t64 = d.targets_itype == E2E_I64;
    for (int b = 0; b < d.batch; b++) {
      const long long Ti = idx(logits_lengths, l64, (size_t)b), Li = idx(targets_lengths, l64, (size_t)b);
      if (Ti < 1 || Ti > d.max_frames) { set_error("logits_lengths must be in [1, %d] (utterance %d: %lld)", d.max_frames, b, Ti); return E2E_ERR_LENGTHS; }
      if (Li < 0 || Li > d.max_targets) { set_error("targets_lengths must be in [0, %d] (utterance %d: %lld)", d.max_targets, b, Li); return E2E_ERR_LENGTHS; }
      for (long long i = 0; i < Li; i++) {
        const long long v = idx(targets, t64, (size_t)b * d.max_targets + (size_t)i);
        if (v < 0 || v >= d.alphabet) { set_error("target labels must be in [0, %d) (utterance %d, position %lld: %lld)", d.alphabet, b, i, v); return E2E_ERR_LENGTHS; }
      }
    }
  }
  LossPlan p;
  if (!make_loss_plan(d, true, &p)) { set_error("no lattice configuration for max_targets=%d", d.max_targets); return E2E_ERR_UNSUPPORTED; }
  E2E_CUDA_TRY(cudaSetDevice(e->device));
  const size_t es = elem_size(d.dtype);
  const size_t n_log = (size_t)d.batch * d.max_frames * d.alphabet * es;
  const size_t n_tgt = (size_t)d.batch * d.max_targets * (d.targets_itype == E2E_I64 ? 8 : 4);
  const size_t n_len = (size_t)d.batch * (d.lengths_itype == E2E_I64 ? 8 : 4);
  const size_t n_loss = (size_t)d.batch * es;
  e->h2d = n_log + n_tgt + 2 * n_len;
  e->d2h = n_loss + n_log;

  // Utterances are independent, so a batch-major batch is cut into chunks of utterances that flow through
  // three stages on separate streams -- copy in, kernels, copy out -- and the PCIe transfers of one chunk
  // overlap the kernels of another (both copy directions run at once).  Time-major host tensors (a chunk
  // of utterances is not contiguous there) and small batches take the single-stream path.
  const bool batch_major = d.logits_stride_b == (int64_t)d.max_frames * d.alphabet && d.logits_stride_t == d.alphabet &&
                           d.grads_stride_b == d.logits_stride_b && d.grads_stride_t == d.logits_stride_t;
  // Results go STRAIGHT into the caller's buffers when those are pinned host memory (what torch's pin_memory /
  // cudaHostAlloc give): the kernels' gradient and loss stores cross PCIe while the lattice is still being swept,
  // and the device->host copy stage disappears (c2: 258 -> 212 us per call, measured).  Reading the logits the same way is
  // NOT a win (uncoalesced 4-byte loads over PCIe: 428 us), so inputs are still staged by the copy engine; the
  // small index tensors are read in place when pinned (a few hundred bytes per utterance, once).
  const int zc_env = env_int("E2E_CTC_HOST_ZERO_COPY", -1);
  void *zc_grads = nullptr, *zc_losses = nullptr;
  const bool zc = zc_env != 0 && host_device_ptr(grads, &zc_grads) && host_device_ptr(losses, &zc_losses);
  void *zc_tgt = nullptr, *zc_il = nullptr, *zc_tl = nullptr;
  const bool zc_idx = zc && (n_tgt == 0 || host_device_ptr(targets, &zc_tgt)) && host_device_ptr(logits_lengths, &zc_il) &&
                      host_device_ptr(targets_lengths, &zc_tl);
  e->zero_copy_bytes = zc ? n_loss + n_log : 0;   // (h2d / d2h keep counting every byte that crosses PCIe, whoever moves it)
  int nch = env_int("E2E_CTC_HOST_CHUNKS", -1);
  if (nch < 0) {
    nch = (int)(n_log / (768 * 1024));          // aim at chunks of >= 0.75 MB of logits
    // a latency-bound fused kernel takes as long for a third of the batch as for all of it: with no copy-out stage
    // left to overlap, cutting a small batch only delays the last chunk's kernel behind more, slower, copies
    if (zc && p.dense && n_log <= ((size_t)6 << 20)) nch = 1;
  }
  if (nch > e2e_ctc_engine::kMaxChunks) nch = e2e_ctc_engine::kMaxChunks;
  if (nch > d.batch) nch = d.batch;
  if (!batch_major || nch < 2) {
    if ((rc = e->logits.ensure(n_log)) || (rc = e->grads.ensure(n_log)) || (rc = e->targets.ensure(n_tgt + 8)) ||
        (rc = e->in_len.ensure(n_len)) || (rc = e->tgt_len.ensure(n_len)) || (rc = e->losses.ensure(n_loss)) ||
        (rc = e->ws.ensure(p.total)))
      return rc;
    cudaStream_t s = e->stream;
    E2E_CUDA_TRY(cudaMemcpyAsync(e->logits.p, logits, n_log, cudaMemcpyHostToDevice, s));
    if (!zc_idx) {
      if (n_tgt) E2E_CUDA_TRY(cudaMemcpyAsync(e->targets.p, targets, n_tgt, cudaMemcpyHostToDevice, s));
      E2E_CUDA_TRY(cudaMemcpyAsync(e->in_len.p, logits_lengths, n_len, cudaMemcpyHostToDevice, s));
      E2E_CUDA_TRY(cudaMemcpyAsync(e->tgt_len.p, targets_lengths, n_len, cudaMemcpyHostToDevice, s));
    }
    rc = loss_fwd_bwd(d, p, e->logits.p, zc_idx ? zc_tgt : e->targets.p, zc_idx ? zc_il : e->in_len.p, zc_idx ? zc_tl : e->tgt_len.p,
                      zc ? zc_losses : e->losses.p, zc ? zc_grads : e->grads.p, 1.0, reinterpret_cast<char*>(e->ws.p), s);
    if (rc != E2E_OK) return rc;
    if (!zc) {
      E2E_CUDA_TRY(cudaMemcpyAsync(losses, e->losses.p, n_loss, cudaMemcpyDeviceToHost, s));
      E2E_CUDA_TRY(cudaMemcpyAsync(grads, e->grads.p, n_log, cudaMemcpyDeviceToHost, s));
    }
    E2E_CUDA_TRY(cudaStreamSynchronize(s));
    return E2E_OK;
  }

  if (!e->pipe_ready) {
    E2E_CUDA_TRY(cudaStreamCreateWithFlags(&e->s_in, cudaStreamNonBlocking));
    E2E_CUDA_TRY(cudaStreamCreateWithFlags(&e->s_out, cudaStreamNonBlocking));
    for (cudaStream_t& c : e->s_comp) E2E_CUDA_TRY(cudaStreamCreateWithFlags(&c, cudaStreamNonBlocking));
    for (int k = 0; k < e2e_ctc_engine::kMaxChunks; k++) {
      E2E_CUDA_TRY(cudaEventCreateWithFlags(&e->ev_in[k], cudaEventDisableTiming));
      E2E_CUDA_TRY(cudaEventCreateWithFlags(&e->ev_comp[k], cudaEventDisableTiming));
    }
    E2E_CUDA_TRY(cudaEventCreateWithFlags(&e->ev_free, cudaEventDisableTiming));
    e->pipe_ready = true;
  }
  // chunk plans (a chunk may pick a different kernel than the whole batch would) and workspace offsets
  const int per = (d.batch + nch - 1) / nch;
  nch = (d.batch + per - 1) / per;
  LossPlan cp[e2e_ctc_engine::kMaxChunks];
  e2e_ctc_desc cd[e2e_ctc_engine::kMaxChunks];
  size_t ws_off[e2e_ctc_engine::kMaxChunks + 1];
  ws_off[0] = 0;
  for (int k = 0; k < nch; k++) {
    cd[k] = d;
    cd[k].batch = (k + 1) * per <= d.batch ? per : d.batch - k * per;
    if (!make_loss_plan(cd[k], true, &cp[k])) { set_error("no lattice configuration for a chunk of the batch"); return E2E_ERR_UNSUPPORTED; }
    ws_off[k + 1] = ws_off[k] + align256(cp[k].total);
  }
  if ((rc = e->logits.ensure(n_log)) || (rc = e->grads.ensure(n_log)) || (rc = e->targets.ensure(n_tgt + 8)) ||
      (rc = e->in_len.ensure(n_len)) || (rc = e->tgt_len.ensure(n_len)) || (rc = e->losses.ensure(n_loss)) ||
      (rc = e->ws.ensure(ws_off[nch])))
    return rc;
  const size_t row_b = (size_t)d.max_frames * d.alphabet * es;            // bytes of one utterance's logits
  const size_t tg_b = (size_t)d.max_targets * (d.targets_itype == E2E_I64 ? 8 : 4);
  const size_t len_b = d.lengths_itype == E2E_I64 ? 8 : 4;
  // E2E_CTC_HOST_TRACE=1: device timeline of this call (timing events on the three stages) + host issue times, to stderr
  static const int trace = env_int("E2E_CTC_HOST_TRACE", 0);
  cudaEvent_t tr[4 * e2e_ctc_engine::kMaxChunks + 2] = {};
  double host_us[e2e_ctc_engine::kMaxChunks + 2] = {};
  auto now_us = []() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e6 + ts.tv_nsec * 1e-3; };
  const double host_t0 = now_us();
  if (trace) {
    for (cudaEvent_t& ev : tr) cudaEventCreate(&ev);
    cudaEventRecord(tr[4 * nch], e->s_in);
  }
  if (!zc_idx) {
    if (n_tgt) E2E_CUDA_TRY(cudaMemcpyAsync(e->targets.p, targets, n_tgt, cudaMemcpyHostToDevice, e->s_in));
    E2E_CUDA_TRY(cudaMemcpyAsync(e->in_len.p, logits_lengths, n_len, cudaMemcpyHostToDevice, e->s_in));
    E2E_CUDA_TRY(cudaMemcpyAsync(e->tgt_len.p, targets_lengths, n_len, cudaMemcpyHostToDevice, e->s_in));
  }
  char* const d_tgt = reinterpret_cast<char*>(zc_idx ? zc_tgt : e->targets.p);
  char* const d_il = reinterpret_cast<char*>(zc_idx ? zc_il : e->in_len.p);
  char* const d_tl = reinterpret_cast<char*>(zc_idx ? zc_tl : e->tgt_len.p);
  for (int k = 0; k < nch; k++) {
    const size_t b0 = (size_t)k * per, nb = (size_t)cd[k].batch;
    char* dl = reinterpret_cast<char*>(e->logits.p) + b0 * row_b;
    char* dg = reinterpret_cast<char*>(zc ? zc_grads : e->grads.p) + b0 * row_b;
    char* dls = reinterpret_cast<char*>(zc ? zc_losses : e->losses.p) + b0 * es;
    E2E_CUDA_TRY(cudaMemcpyAsync(dl, reinterpret_cast<const char*>(logits) + b0 * row_b, nb * row_b, cudaMemcpyHostToDevice, e->s_in));
    E2E_CUDA_TRY(cudaEventRecord(e->ev_in[k], e->s_in));
    cudaStream_t sc = e->s_comp[k % e2e_ctc_engine::kComputeStreams];
    E2E_CUDA_TRY(cudaStreamWaitEvent(sc, e->ev_in[k], 0));
    if (trace) { cudaEventRecord(tr[4 * k], e->s_in); cudaEventRecord(tr[4 * k + 1], sc); }
    rc = loss_fwd_bwd(cd[k], cp[k], dl, d_tgt + b0 * tg_b, d_il + b0 * len_b, d_tl + b0 * len_b, dls, dg, 1.0,
                      reinterpret_cast<char*>(e->ws.p) + ws_off[k], sc);
    if (rc != E2E_OK) { cudaDeviceSynchronize(); return rc; }
    E2E_CUDA_TRY(cudaEventRecord(e->ev_comp[k], sc));
    E2E_CUDA_TRY(cudaStreamWaitEvent(e->s_out, e->ev_comp[k], 0));      // s_out joins every chunk: one synchronize at the end
    if (trace) cudaEventRecord(tr[4 * k + 2], sc);
    if (!zc) {
      E2E_CUDA_TRY(cudaMemcpyAsync(reinterpret_cast<char*>(grads) + b0 * row_b, dg, nb * row_b, cudaMemcpyDeviceToHost, e->s_out));
      E2E_CUDA_TRY(cudaMemcpyAsync(reinterpret_cast<char*>(losses) + b0 * es, dls, nb * es, cudaMemcpyDeviceToHost, e->s_out));
    }
    if (trace) { cudaEventRecord(tr[4 * k + 3], e->s_out); host_us[k] = now_us() - host_t0; }
  }
  E2E_CUDA_TRY(cudaStreamSynchronize(e->s_out));
  if (trace) {
    const double host_done = now_us() - host_t0;
    fprintf(stderr, "[e2e host trace] %d chunks; host: ", nch);
    for (int k = 0; k < nch; k++) fprintf(stderr, "issued[%d] %.0f us  ", k, host_us[k]);
    fprintf(stderr, "synced %.0f us\n", host_done);
    for (int k = 0; k < nch; k++) {
      float a = 0, b = 0, c = 0, dd = 0;
      cudaEventElapsedTime(&a, tr[4 * nch], tr[4 * k]); cudaEventElapsedTime(&b, tr[4 * nch], tr[4 * k + 1]);
      cudaEventElapsedTime(&c, tr[4 * nch], tr[4 * k + 2]); cudaEventElapsedTime(&dd, tr[4 * nch], tr[4 * k + 3]);
      fprintf(stderr, "  chunk %d (%d utt): copy-in done %.0f us, kernels %.0f -> %.0f us, copy-out done %.0f us\n", k, cd[k].batch,
              a * 1e3, b * 1e3, c * 1e3, dd * 1e3);
    }
    for (cudaEvent_t& ev : tr) cudaEventDestroy(ev);
  }
  return E2E_OK;
}

int e2e_ctc_engine_greedy_host(e2e_ctc_engine* e, const e2e_ctc_desc* desc, const void* logits,
                               const void* logits_lengths, int64_t* decoded, int64_t* decoded_lengths) {
  if (!e) { set_error("null engine"); return E2E_ERR_INVALID_ARGUMENT; }
  int rc = check_desc(desc, false);
  if (rc != E2E_OK) return rc;
  if (!logits || !decoded || !decoded_lengths) { set_error("null pointer argument"); return E2E_ERR_INVALID_ARGUMENT; }
  const e2e_ctc_desc& d = *desc;
  if (!dense_block(d, d.logits_stride_b, d.logits_stride_t)) {
    set_error("host logits must be dense (batch-major or time-major contiguous)");
    return E2E_ERR_INVALID_ARGUMENT;
  }
  E2E_CUDA_TRY(cudaSetDevice(e->device));
  const size_t n_log = (size_t)d.batch * d.max_frames * d.alphabet * elem_size(d.dtype);
  const size_t n_len = (size_t)d.batch * (d.lengths_itype == E2E_I64 ? 8 : 4);
  const size_t n_dec = (size_t)d.batch * d.max_frames * 8, n_dl = (size_t)d.batch * 8;
  const size_t n_ws = e2e_ctc_greedy_workspace_bytes(desc);
  if ((rc = e->logits.ensure(n_log)) || (rc = e->in_len.ensure(n_len)) || (rc = e->decoded.ensure(n_dec)) ||
      (rc = e->decoded_len.ensure(n_dl)) || (rc = e->ws.ensure(n_ws)))
    return rc;
  cudaStream_t s = e->stream;
  E2E_CUDA_TRY(cudaMemcpyAsync(e->logits.p, logits, n_log, cudaMemcpyHostToDevice, s));
  if (logits_lengths) E2E_CUDA_TRY(cudaMemcpyAsync(e->in_len.p, logits_lengths, n_len, cudaMemcpyHostToDevice, s));
  rc = launch_greedy(d, e->logits.p, logits_lengths ? e->in_len.p : nullptr, reinterpret_cast<int64_t*>(e->decoded.p),
                     reinterpret_cast<int64_t*>(e->decoded_len.p), reinterpret_cast<char*>(e->ws.p), s);
  if (rc != E2E_OK) return rc;
  E2E_CUDA_TRY(cudaMemcpyAsync(decoded, e->decoded.p, n_dec, cudaMemcpyDeviceToHost, s));
  E2E_CUDA_TRY(cudaMemcpyAsync(decoded_lengths, e->decoded_len.p, n_dl, cudaMemcpyDeviceToHost, s));
  E2E_CUDA_TRY(cudaStreamSynchronize(s));
  e->h2d = n_log + (logits_lengths ? n_len : 0);
  e->d2h = n_dec + n_dl;
  return E2E_OK;
}

// decode (n_best == 1, scores == NULL) and the N-best list share one path; results land in the engine's decoded /
// decoded_len buffers (decoded_len: lengths [B,N], ties [B], scores [B,N], log_probs [B,N])
static int engine_beam_host(e2e_ctc_engine* e, const e2e_ctc_desc* desc, int32_t beam_width, int32_t n_best, int32_t space_idx,
                            double wip, const void* logits, const void* logits_lengths, int64_t* decoded,
                            int64_t* decoded_lengths, double* scores, double* log_probs, int64_t* ties) {
  if (!e) { set_error("null engine"); return E2E_ERR_INVALID_ARGUMENT; }
  int rc = check_beam(desc, beam_width, n_best, space_idx, wip);
  if (rc != E2E_OK) return rc;
  if (!logits || !decoded || !decoded_lengths) { set_error("null pointer argument"); return E2E_ERR_INVALID_ARGUMENT; }
  const e2e_ctc_desc& d = *desc;
  if (!dense_block(d, d.logits_stride_b, d.logits_stride_t)) {
    set_error("host logits must be dense (batch-major or time-major contiguous)");
    return E2E_ERR_INVALID_ARGUMENT;
  }
  E2E_CUDA_TRY(cudaSetDevice(e->device));
  const size_t n_log = (size_t)d.batch * d.max_frames * d.alphabet * elem_size(d.dtype);
  const size_t n_len = (size_t)d.batch * (d.lengths_itype == E2E_I64 ? 8 : 4);
  const size_t n_hyp = (size_t)d.batch * n_best;
  const size_t n_dec = n_hyp * d.max_frames * 8, n_dl = n_hyp * 8, n_ties = (size_t)d.batch * 8;
  const size_t n_ws = e2e_ctc_beam_nbest_workspace_bytes(desc, beam_width, n_best);
  if ((rc = e->logits.ensure(n_log)) || (rc = e->in_len.ensure(n_len)) || (rc = e->decoded.ensure(n_dec)) ||
      (rc = e->decoded_len.ensure(n_dl + n_ties + (scores ? 2 * n_dl : 0))) || (rc = e->ws.ensure(n_ws)))
    return rc;
  cudaStream_t s = e->stream;
  E2E_CUDA_TRY(cudaMemcpyAsync(e->logits.p, logits, n_log, cudaMemcpyHostToDevice, s));
  if (logits_lengths) E2E_CUDA_TRY(cudaMemcpyAsync(e->in_len.p, logits_lengths, n_len, cudaMemcpyHostToDevice, s));
  int64_t* d_len = reinterpret_cast<int64_t*>(e->decoded_len.p);
  int64_t* d_ties = d_len + n_hyp;
  double* d_scores = scores ? reinterpret_cast<double*>(d_ties + d.batch) : nullptr;
  double* d_lp = scores && log_probs ? d_scores + n_hyp : nullptr;
  rc = launch_beam(d, beam_width, n_best, space_idx, wip, e->logits.p, logits_lengths ? e->in_len.p : nullptr,
                   reinterpret_cast<int64_t*>(e->decoded.p), d_len, d_scores, d_lp, d_ties, reinterpret_cast<char*>(e->ws.p), s);
  if (rc != E2E_OK) return rc;
  E2E_CUDA_TRY(cudaMemcpyAsync(decoded, e->decoded.p, n_dec, cudaMemcpyDeviceToHost, s));
  E2E_CUDA_TRY(cudaMemcpyAsync(decoded_lengths, d_len, n_dl, cudaMemcpyDeviceToHost, s));
  if (ties) E2E_CUDA_TRY(cudaMemcpyAsync(ties, d_ties, n_ties, cudaMemcpyDeviceToHost, s));
  if (d_scores) E2E_CUDA_TRY(cudaMemcpyAsync(scores, d_scores, n_dl, cudaMemcpyDeviceToHost, s));
  if (d_lp) E2E_CUDA_TRY(cudaMemcpyAsync(log_probs, d_lp, n_dl, cudaMemcpyDeviceToHost, s));
  E2E_CUDA_TRY(cudaStreamSynchronize(s));
  e->h2d = n_log + (logits_lengths ? n_len : 0);
  e->d2h = n_dec + n_dl + (ties ? n_ties : 0) + (d_scores ? n_dl : 0) + (d_lp ? n_dl : 0);
  return E2E_OK;
}

int e2e_ctc_engine_beam_host(e2e_ctc_engine* e, const e2e_ctc_desc* desc, int32_t beam_width, int32_t space_idx, double wip,
                             const void* logits, const void* logits_lengths, int64_t* decoded, int64_t* decoded_lengths,
                             int64_t* ties) {
  return engine_beam_host(e, desc, beam_width, 1, space_idx, wip, logits, logits_lengths, decoded, decoded_lengths, nullptr,
                          nullptr, ties);
}

int e2e_ctc_engine_beam_nbest_host(e2e_ctc_engine* e, const e2e_ctc_desc* desc, int32_t beam_width, int32_t n_best,
                                   int32_t space_idx, double wip, const void* logits, const void* logits_lengths,
                                   int64_t* decoded, int64_t* decoded_lengths, double* scores, double* log_probs,
                                   int64_t* ties) {
  if (!scores) { set_error("null pointer argument"); return E2E_ERR_INVALID_ARGUMENT; }
  return engine_beam_host(e, desc, beam_width, n_best, space_idx, wip, logits, logits_lengths, decoded, decoded_lengths,
                          scores, log_probs, ties);
}

int e2e_ctc_engine_last_traffic(const e2e_ctc_engine* e, uint64_t* h2d_bytes, uint64_t* d2h_bytes) {
  if (!e) { set_error("null engine"); return E2E_ERR_INVALID_ARGUMENT; }
  if (h2d_bytes) *h2d_bytes = e->h2d;
  if (d2h_bytes) *d2h_bytes = e->d2h;
  return E2E_OK;
}

}  // extern "C"
