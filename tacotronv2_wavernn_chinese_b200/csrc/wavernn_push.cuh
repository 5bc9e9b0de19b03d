// WaveRNN per-sample recurrence, "push" kernel: the small-batch (B <= 32 rows per GPU) form of the weight-stationary grid.
//
// Same decomposition as wavernn_grid.cuh -- 128 co-resident CTAs (cooperative launch), CTA c keeps the rows of every layer
// that produce hidden units / fc rows [4c, 4c+4) and classes [8c, 8c+8) in shared memory for the whole launch -- but the
// five exchanges of a sample step (reference loop wavernn/models/fatchord_version.py:201-237) no longer go through a
// grid barrier followed by a load of the activations.  At B <= 32 a step is pure latency (FMA floor 4 us at 32 rows), and
// the barrier round (bar.sync + red.release + spin on ld.acquire + bar.sync = 1.27 us measured) plus the L2 pull after it
// was ~75 % of the 17.7 us (B <= 4) / 29.4 us (B = 32) step of the round-1 kernel.  Here:
//
//   * FLAG-IN-DATA exchange.  Every exchanged activation vector lives in L2 as [producer CTA][row][4 units] fp32, two
//     parity copies, pre-filled with a sentinel bit pattern (0xFFFFFFFF, a NaN no arithmetic here can produce).  A
//     producer simply stores its 4 x G values; a consumer thread loads the float4 it needs straight into registers with
//     ld.relaxed.gpu and re-polls until none of the four words is the sentinel -- the data IS the flag, one L2 round trip
//     instead of fence + flag + poll + load.  A producer re-arms the OTHER parity copy of its own entries (sentinel stores +
//     __threadfence) right after it has seen every CTA's winner of the previous step, i.e. when every consumer of that
//     copy is provably done and long before anybody can poll it again (proof at `rearm` below).
//   * The sampled label travels the same way: every CTA publishes its local Gumbel-max winner per row as one 64-bit word
//     (ordered key | inverted class | 22-bit step tag -- 8-byte stores are single-copy atomic) and every CTA reduces the
//     128 winners itself; no atomics, no barrier.
//   * No shared-memory staging: thread (row lane, k queue) loads exactly the float4s it multiplies (G/4 per vector), all
//     rows of the phase are accumulated in registers, k queues are reduced by shuffles + one 16-warp pass through shared
//     memory.
//   * CONDITIONING HOISTED (SURVEY 7.1-5): the 112 conditioning columns of the I layer / GRU-1 and the 32 aux columns of
//     GRU-2, fc1, fc2 never enter the serial path.  push_cond_table_kernel computes, once per utterance and FRAME,
//     W.mel[f] (FIR linearity: W.(sum_j fir[ph][j] mel[f_j]) = sum_j fir[ph][j] (W.mel[f_j])) and W.aux[f] + bias for
//     the 52 conditioned rows of every CTA; the kernel combines <= 6 table rows per output row for step t+1 while it
//     waits for fc2's exchange of step t.  This also removes the [S][80][B] sample-rate mel buffer of the round-1 path.
//   * The two recurrent projections W_hh1.h1(t), W_hh2.h2(t) (42 % of the MACs) do not depend on the sample drawn at
//     step t: they run in the shadow of the NEXT exchange (after GRU-2 / fc1 have published) and are consumed one step later.
//
// Per step and CTA:  P01 winners(t-1) -> x, GRU-1 gate math (all matrix work precomputed) -> publish h1, x1
//                    P2  x1 -> W_ih2 (12 x 512) -> gate math -> publish h2, x2      | shadow: W_hh1.h1(t)
//                    P3  x2 -> fc1 (4 x 512)  -> publish f1                          | shadow: W_hh2.h2(t)
//                    P4  f1 -> fc2 (4 x 512)  -> publish f2                          | shadow: conditioning of step t+1
//                    P5  f2 -> fc3 (8 x 512)  -> Gumbel-max over the CTA's 8 classes -> publish winner
#pragma once
#include "common.cuh"
#include "wavernn_upsample.cuh"
#include "wavernn_grid.cuh"

namespace b200tts {

constexpr int kPushThreads = 512;
constexpr int kPushWarps = kPushThreads / 32;
constexpr uint32_t kPushSentinel = 0xFFFFFFFFu;
constexpr int kPushCondRows = 52;   // per CTA and frame: 16 mel projections | 16 + 12 + 4 + 4 aux projections (+ bias)
constexpr int kPushVecs = 6;        // h1, x1, h2, x2, f1, f2
enum { PV_H1 = 0, PV_X1, PV_H2, PV_X2, PV_F1, PV_F2 };

struct PushModel {          // layout of one CTA's weight blob (offsets in floats, 16-byte aligned)
  int ncta, R, F, NC;
  int ohh1, oih2, ohh2;     // [12][R]  row = gate*4 + unit ; W_ih2 without its aux columns
  int ofc1, ofc2, ofc3;     // [4][R], [4][F], [8][F]
  int oAx;                  // [16]: coefficient of the fed-back sample x in the 4 I rows and the 12 folded GRU-1 rows
  int obhh1, obhh2, obfc3;  // [12], [12], [8]
  int blob;
  int ok;
};

struct PushArgs {
  const float* wblob;            // [ncta][blob]
  float* vec;                    // [6][2][ncta][G][4]   exchanged activations (sentinel pre-filled)
  unsigned long long* best;      // [ncta][G]            winners, tagged with the step
  int* error;                    // set non-zero when a poll timed out
  const float* tab;              // [n_src][T+1][ncta][52] conditioning tables (push_cond_table_kernel)
  const float* fir;              // [hop][NT] composite polyphase FIR of the upsampling network
  int NT;
  int B, S, T, hop, steps;
  int ng;                        // multi-group kernel (wavernn_pushmg.cuh): groups of 32 rows; vec is [ng][6][2][ncta][32][4], best [ng][ncta][32]
  int row_stride;                // 0: row u is utterance u.  > 0 (fold-with-overlap): row u = samples [u*row_stride, ...) of utterance 0
  int S_src;                     // samples of the source utterance (conditioning is ZERO beyond, fatchord_version.py:315-317)
  int rng_mode;
  unsigned long long seed, utt_offset;
  const unsigned long long* utt_ids;   // optional [B]: global utterance index of every row (overrides utt_offset + row)
  const float* q;                // [S][B][NC]
  const int16_t* teacher;        // [B][S]
  float* logits_out;             // [S][B][NC]
  int16_t* labels;               // [B][S]
  long long* prof;               // optional [ncta][16] cycle counters of thread 0
  // PACKED rows (ragged sets, pipeline.py): row u runs a QUEUE of utterances back to back -- segment k of row u is utterance
  // pack_utt[u*pack_segs + k] from step pack_start[u*(pack_segs+1) + k] (next entry = its end; utt < 0 = no more work) -- and
  // restarts from the zero state at every segment start, so every utterance gets exactly the arithmetic of a stand-alone run.
  // B then counts UTTERANCES (labels [B][S], tables [B][T+1]...), the kernel runs G rows for `steps` lock-steps.
  const int* pack_utt;           // [pack_rows][pack_segs]
  const int* pack_start;         // [pack_rows][pack_segs + 1]
  int pack_segs, pack_rows;      // kernel rows >= pack_rows are idle
  // STREAMING (wavernn_push_kernel<G, true>, b200tts_wavernn_generate_stream; plain batches only): while it runs, CTA 0 writes
  // the final fp64 wave sample of every row -- the value finish_wave_kernel writes for the same label and position -- to
  // caller-owned pinned host memory and publishes how many lock-steps are there.  Appended last: the offsets of the fields
  // above, and with them the code of every other kernel that takes PushArgs, stay as they are.
  double* h_wave;                // device alias of pinned host memory [B][(T-1)*hop]
  long long* h_progress;         // device alias of a pinned int64: lock-steps whose samples are in h_wave (< 0: the kernel gave up)
  int chunk_steps;               // publish every chunk_steps lock-steps (and once after the last)
  const int* d_utt_frames;       // optional [B]: own frame count of each row (truncation / fade as finish_wave_kernel)
  int fade_len, mu_law;
};

struct PushRowState {            // per-row bookkeeping in shared memory (normal mode: row u == utterance u from step 0, forever)
  int utt[32], t0[32], end[32], k[32];     // current segment: utterance (-1 idle), first step, first step of the NEXT segment, index
  int putt[32], pn[32];                    // (utterance, local step) the row was at in the PREVIOUS step (whose winner P01 collects)
  int rst[32];                             // the current step is the first of a segment: x = 0, h1 = h2 = 0
};
// (utterance, local step) of row u at step t+1, seen from step t
__device__ __forceinline__ void push_row_next(const PushArgs& A, const PushRowState& R, int u, int t1, int& utt, int& n) {
  if (t1 < R.end[u]) { utt = R.utt[u]; n = t1 - R.t0[u]; return; }
  const int k1 = R.k[u] + 1;
  utt = (A.pack_utt && u < A.pack_rows && k1 < A.pack_segs) ? A.pack_utt[u * A.pack_segs + k1] : -1;
  n = t1 - R.end[u];
}

// ---- L2-coherent accessors ---------------------------------------------------------------------------------------
__device__ __forceinline__ float4 ld_relaxed_f4(const float* p) {
  float4 v;
  asm volatile("ld.relaxed.gpu.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed_f32(float* p, float v) {
  asm volatile("st.relaxed.gpu.global.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_u32(float* p, uint32_t v) {
  asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_relaxed_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ bool f4_ready(const float4& v) {
  return __float_as_uint(v.x) != kPushSentinel && __float_as_uint(v.y) != kPushSentinel &&
         __float_as_uint(v.z) != kPushSentinel && __float_as_uint(v.w) != kPushSentinel;
}

// A poll gives up after ~2 s (a peer CTA is gone) or as soon as any CTA has raised the global error flag.
struct PollGuard {
  int* error;
  long long t0;
  unsigned spins;
  bool aborted;
  __device__ __forceinline__ void begin() { spins = 0; }
  __device__ __forceinline__ bool expired() {
    if ((++spins & 1023u) != 0u) return false;
    if (spins == 1024u) t0 = clock64();
    if (*reinterpret_cast<volatile int*>(error) != 0 || clock64() - t0 > 4000000000LL) {
      atomicExch(error, 1);
      aborted = true;
      return true;
    }
    return false;
  }
};

// ---- exchange protocol ------------------------------------------------------------------------------------------
// Measured in isolation (tools/exchange_bench.cu -> profiles/r02_exchange_bench.txt, cycles per all-to-all exchange of
// a [128][G][4] vector by 128 CTAs, G = 4 / 8 / 32):  counter barrier + loads 3511 / 3600 / 4106;  every thread
// spinning on its own entries 1558 / 2033 / 4140;  one canary warp (on the data or on replicated hint words) releasing
// the block through a barrier 2928-3761 / 3780-4545 / 6754-7465.  The direct spin wins: detection and delivery are the
// same L2 round trip.  Every thread issues ALL its loads first and re-polls only what still carries a sentinel.
template <int NL>
__device__ __forceinline__ void poll_entries(const float* base, const int (&off)[NL], float4 (&a)[NL], PollGuard& g) {
#pragma unroll
  for (int i = 0; i < NL; ++i) a[i] = ld_relaxed_f4(base + off[i]);
  unsigned pending = 0;
#pragma unroll
  for (int i = 0; i < NL; ++i) pending |= f4_ready(a[i]) ? 0u : (1u << i);
  if (pending) {
    g.begin();
    while (pending && !g.aborted) {
#pragma unroll
      for (int i = 0; i < NL; ++i)
        if (pending & (1u << i)) {
          a[i] = ld_relaxed_f4(base + off[i]);
          if (f4_ready(a[i])) pending &= ~(1u << i);
        }
      if (pending && g.expired()) break;
    }
  }
}

// winner word: ordered-float key (32) | 1023 - class (10) | step tag (22)
__device__ __forceinline__ unsigned long long push_pack(float key, uint32_t cls, uint32_t tag) {
  uint32_t u = __float_as_uint(key);
  u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return ((unsigned long long)u << 32) | ((unsigned long long)(1023u - cls) << 22) | (unsigned long long)(tag & 0x3FFFFFu);
}
__device__ __forceinline__ uint32_t push_cls(unsigned long long p) { return 1023u - (uint32_t)((p >> 22) & 1023u); }

template <int G> struct PushTraits {
  static constexpr int UT = (G >= 16) ? 2 : 1;             // rows per thread in the GEMMs
  static constexpr int NU = G / UT;                        // row lanes
  static constexpr int NKQ = kPushThreads / NU;            // k queues
  static constexpr int NKB = 128 / NKQ;                    // producer blocks (float4 columns) per thread and row
  static constexpr int NL = NKB * UT;                      // float4 loads per thread and vector = G/4
  static constexpr int kPartFloats = kPushWarps * 16 * G;        // up to 16 rows per pass (W_ih2 12 + fc1 4 on x1)
  static_assert(NU >= 4 && NU <= 32 && NKQ * NKB == 128 && NL * 4 == G && (32 / NU) * NKB == 8 && (NKB == 1 || NKB == 2 || NKB == 4), "mapping");
  // shared memory after the weight blob (floats)
  static constexpr int oPartX = 0;
  static constexpr int oPartY = oPartX + kPartFloats;
  static constexpr int oCond = oPartY + kPartFloats;       // [2][36][G]
  static constexpr int oGh1 = oCond + 2 * 36 * G;          // [12][G]
  static constexpr int oGh2 = oGh1 + 12 * G;               // [12][G]
  static constexpr int oSmax = oGh2 + 12 * G;              // u64 [16][G]
  static constexpr int oKeys = oSmax + 2 * kPushWarps * G; // u64 [8][G]
  static constexpr int oXs = oKeys + 2 * 8 * G;            // [G] fed-back sample
  static constexpr int oFir = oXs + ((G + 3) & ~3);        // [hop*NT]
  static constexpr int scratch_floats(int hop, int NT) { return oFir + ((hop * NT + 3) & ~3); }
};

// ---- one GEMM pass over this thread's NKB producer blocks x UT rows.  The 128 four-term dot products of an output (one
//      per producer block kb) are combined in ONE fixed order for every G: pairwise by bit 0, 1, 2 of kb (inside the thread
//      while it owns the pair, by warp shuffle otherwise; 8 consecutive kb per warp for every G), then the 16 warps in
//      sequence (push_part_sum).  A row's result is therefore bit-identical whatever batch it is generated in (G = 4 ... 32),
//      which is what lets N ranks reproduce the single-rank labels exactly.  Partials to part[(warp*ROWS + r)*G + u]. -------
template <int G>
__device__ __forceinline__ void push_load(const float* vecbase, float4 (&a)[PushTraits<G>::NL], int ul, int kq, PollGuard& pg) {
  using PT = PushTraits<G>;
  constexpr int UT = PT::UT, NU = PT::NU, NKB = PT::NKB, NL = PT::NL;
  int off[NL];
#pragma unroll
  for (int i = 0; i < NKB; ++i)
#pragma unroll
    for (int j = 0; j < UT; ++j) off[i * UT + j] = ((kq * NKB + i) * G + ul + NU * j) * 4;
  poll_entries<NL>(vecbase, off, a, pg);
}
// (settling and multiplying block by block, so that the FMAs of block i overlap the loads of block i+1, was measured SLOWER:
//  19.4 vs 14.4 us per step at 16 rows, 24.9 vs 21.7 at 32 -- the per-block leaves no longer fit the register file)
template <int G, int ROWS>
__device__ __forceinline__ void push_mma(const float* __restrict__ W /*[ROWS][512] smem*/, const float4 (&a)[PushTraits<G>::NL], float* part,
                                         int ul, int kq, int warp, int lane) {
  using PT = PushTraits<G>;
  constexpr int UT = PT::UT, NU = PT::NU, NKB = PT::NKB;
  float acc[ROWS][UT];
  const float4* W4 = reinterpret_cast<const float4*>(W);
#pragma unroll
  for (int r = 0; r < ROWS; ++r) {
    float leaf[NKB][UT];
#pragma unroll
    for (int i = 0; i < NKB; ++i) {
      const float4 w = W4[r * 128 + kq * NKB + i];
      if constexpr (UT == 2) {
        // packed fp32: both rows of this thread against one broadcast weight (bit-identical to two scalar FMA chains)
        const float4 v0 = a[i * 2], v1 = a[i * 2 + 1];
        float2 s2 = __ffma2_rn(make_float2(v0.x, v1.x), make_float2(w.x, w.x), make_float2(0.f, 0.f));
        s2 = __ffma2_rn(make_float2(v0.y, v1.y), make_float2(w.y, w.y), s2);
        s2 = __ffma2_rn(make_float2(v0.z, v1.z), make_float2(w.z, w.z), s2);
        s2 = __ffma2_rn(make_float2(v0.w, v1.w), make_float2(w.w, w.w), s2);
        leaf[i][0] = s2.x; leaf[i][1] = s2.y;
      } else {
        const float4 v = a[i];
        float s1 = fmaf(w.x, v.x, 0.f);
        s1 = fmaf(w.y, v.y, s1); s1 = fmaf(w.z, v.z, s1); s1 = fmaf(w.w, v.w, s1);
        leaf[i][0] = s1;
      }
    }
#pragma unroll
    for (int j = 0; j < UT; ++j) {
      if constexpr (NKB == 4) acc[r][j] = (leaf[0][j] + leaf[1][j]) + (leaf[2][j] + leaf[3][j]);
      else if constexpr (NKB == 2) acc[r][j] = leaf[0][j] + leaf[1][j];
      else acc[r][j] = leaf[0][j];
    }
  }
  // the remaining levels of the 8-block tree: k queues that share the warp sit at lanes ul + NU*m
#pragma unroll
  for (int o = NU; o < 32; o <<= 1)
#pragma unroll
    for (int r = 0; r < ROWS; ++r)
#pragma unroll
      for (int j = 0; j < UT; ++j) acc[r][j] += __shfl_xor_sync(0xffffffffu, acc[r][j], o);
  if (lane < NU) {
#pragma unroll
    for (int r = 0; r < ROWS; ++r)
#pragma unroll
      for (int j = 0; j < UT; ++j) part[(warp * ROWS + r) * G + ul + NU * j] = acc[r][j];
  }
}
template <int G, int ROWS>
__device__ __forceinline__ void push_gemm(const float* __restrict__ W /*[ROWS][512] smem*/, const float* vecbase, float* part,
                                          int ul, int kq, int warp, int lane, PollGuard& pg) {
  float4 a[PushTraits<G>::NL];
  push_load<G>(vecbase, a, ul, kq, pg);
  push_mma<G, ROWS>(W, a, part, ul, kq, warp, lane);
}

template <int G, int ROWS>
__device__ __forceinline__ float push_part_sum(const float* part, int r, int u) {
  float v = 0.f;
#pragma unroll
  for (int w = 0; w < kPushWarps; ++w) v += part[(w * ROWS + r) * G + u];
  return v;
}

// Conditioning of step `t`.  Rows 0-15 (I rows 0-3 and the folded GRU-1 rows: FIR-combined mel projections + aux projection
// + bias) change every sample -> push_cond16, one (row, cond row) item per thread at 32 rows, all (<= 1 + kMaxTaps) table
// loads of an item in flight at once.  Rows 16-35 (GRU-2 12, fc1 4, fc2 4: aux projection + bias) are constant within a
// frame -> push_cond20, refreshed only when the next step starts a new frame (every step in fold mode, where rows sit at
// different phases).
template <int G>
__device__ __forceinline__ void push_cond16(const PushArgs& A, const PushRowState& R, const float* fir_s, float* cdst, int c, int ncta, int t,
                                            int tid) {
  const size_t fstride = (size_t)ncta * kPushCondRows;
  const int fr0 = t / A.hop, ph0 = t - fr0 * A.hop;                   // plain batch: every row is at the same frame / phase
  // items start at thread 4G: the gate threads (0 ... 4G-1) are busy with the fc2 gate, the re-arm and its fence at this point
  for (int it = (tid + kPushThreads - 4 * G) % kPushThreads; it < 16 * G; it += kPushThreads) {
    const int u = it >> 4, r = it & 15;
    int src = u, fr = fr0, ph = ph0;
    bool beyond = false;
    if (A.row_stride) {
      const long long n = (long long)u * A.row_stride + t;
      src = 0;
      beyond = n >= A.S_src;                                           // past the source utterance: zero mel and aux -> bias only
      fr = beyond ? A.T : (int)(n / A.hop);
      ph = beyond ? 0 : (int)(n - (long long)fr * A.hop);
    } else if (A.pack_utt) {
      int n;
      push_row_next(A, R, u, t, src, n);
      if (src < 0) { cdst[r * G + u] = 0.f; continue; }                // idle row
      fr = n / A.hop;
      ph = n - fr * A.hop;
    }
    const float* row = A.tab + (((size_t)src * (A.T + 1) + fr) * ncta + c) * kPushCondRows;
    float v = __ldg(row + 16 + r);
    float pm[kMaxTaps];
#pragma unroll
    for (int j = 0; j < kMaxTaps; ++j) {
      const int f = fr + j - A.NT / 2;
      pm[j] = (!beyond && j < A.NT && f >= 0 && f < A.T) ? __ldg(row + ((ptrdiff_t)(f - fr)) * (ptrdiff_t)fstride + r) : 0.f;
    }
#pragma unroll
    for (int j = 0; j < kMaxTaps; ++j)
      if (j < A.NT) v = fmaf(fir_s[ph * A.NT + j], pm[j], v);          // an absent frame contributes fir * 0 = 0 exactly
    cdst[r * G + u] = v;
  }
}
template <int G>
__device__ __forceinline__ void push_cond20(const PushArgs& A, const PushRowState& R, float* cdst, int c, int ncta, int t, int tid) {
  const int fr0 = t / A.hop;
  for (int it = tid; it < 20 * G; it += kPushThreads) {
    const int u = it / 20, r = it - u * 20;
    int src = u, fr = fr0;
    if (A.row_stride) {
      const long long n = (long long)u * A.row_stride + t;
      src = 0;
      fr = n >= A.S_src ? A.T : (int)(n / A.hop);
    } else if (A.pack_utt) {
      int n;
      push_row_next(A, R, u, t, src, n);
      if (src < 0) { cdst[r * G + u] = 0.f; continue; }
      fr = n / A.hop;
    }
    cdst[r * G + u] = __ldg(A.tab + (((size_t)src * (A.T + 1) + fr) * ncta + c) * kPushCondRows + 32 + r);
  }
}

// ---- streaming (STREAM = true) ----------------------------------------------------------------------------------------
// The samples are written and published by the LAST G threads of CTA 0 -- never gate threads (tid < 4G <= 128), which run the
// gpu-scope fence of the re-arm every step and would otherwise wait there for host-bound stores -- in the shadow of the fc2
// exchange.  Sample n of a row is final once the winner of step n is known (P01 of step n+1); it is stored in step n+1's P4
// shadow, so after the P4 barrier of step t the samples of steps < t-1 are in h_wave: t-1 is what step t may publish.
struct PushStreamSmem {
  double dec[1024];              // wave_decode of every label (the fp64 pow of decode_mu_law leaves the per-step path)
  double step;                   // wave_fade_step(fade_len)
  int wlen[32];                  // own wave length of every row
  int lab[32];                   // label of the step collected in this step's P01 (written by the gate threads)
};
__device__ __forceinline__ PushStreamSmem& push_stream_smem() {
  __shared__ PushStreamSmem s;   // allocated only in the kernels that call this: the streaming instantiations
  return s;
}
__device__ __forceinline__ void push_stream_publish(const PushArgs& A, long long steps_done) {
  // the block barrier before this call orders CTA 0's earlier sample stores; the fence makes them visible system-wide
  // before the count that announces them (the host reads it with an acquire load)
  asm volatile("fence.acq_rel.sys;" ::: "memory");
  asm volatile("st.release.sys.global.s64 [%0], %1;" ::"l"(A.h_progress), "l"(steps_done) : "memory");
}
template <int G>
__device__ __forceinline__ void push_stream_sample(const PushArgs& A, const PushStreamSmem& ss, int tid, int n) {
  const int u = tid - (kPushThreads - G);
  const int wave_len_max = (A.T - 1) * A.hop;
  if (u < 0 || u >= A.B || n >= wave_len_max) return;      // (the last hop of steps is not part of the wave, :184)
  const int wl = ss.wlen[u];
  A.h_wave[(size_t)u * wave_len_max + n] = n < wl ? wave_fade(ss.dec[ss.lab[u]], n, wl, A.fade_len, ss.step) : 0.0;
}

template <int G, bool STREAM>
__global__ void __launch_bounds__(kPushThreads, 1) wavernn_push_kernel(PushModel M, PushArgs A) {
  using PT = PushTraits<G>;
  constexpr int NU = PT::NU;
  extern __shared__ __align__(16) float smem[];
  float* Wb = smem;
  float* sc = smem + M.blob;
  float* partX = sc + PT::oPartX;
  float* partY = sc + PT::oPartY;
  float* cond = sc + PT::oCond;
  float* gh1 = sc + PT::oGh1;
  float* gh2 = sc + PT::oGh2;
  unsigned long long* smax = reinterpret_cast<unsigned long long*>(sc + PT::oSmax);
  unsigned long long* skeys = reinterpret_cast<unsigned long long*>(sc + PT::oKeys);
  float* xs = sc + PT::oXs;
  float* fir_s = sc + PT::oFir;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c = blockIdx.x, ncta = gridDim.x;
  const int ul = tid % NU, kq = tid / NU;                 // GEMM mapping
  const int gu = tid % G, gj = tid / G;                   // gate mapping: row gu, unit gj (threads < 4G)
  const bool gate = tid < 4 * G;
  const float ncls_m1 = (float)(M.NC - 1);
  const size_t vstride = (size_t)ncta * G * 4;            // floats per parity copy of one vector
  auto vecp = [&](int which, int parity) { return A.vec + ((size_t)which * 2 + parity) * vstride; };

  {   // one-time load of this CTA's weight blob: TMA bulk copies signalled through an mbarrier
    __shared__ __align__(8) unsigned long long wbar;
    const char* src = reinterpret_cast<const char*>(A.wblob + (size_t)c * M.blob);
    const unsigned total = (unsigned)M.blob * 4u;
    if (tid == 0) mbar_init(&wbar, 1);
    __syncthreads();
    if (tid == 0) {
      mbar_expect_tx(&wbar, total);
      for (unsigned off = 0; off < total; off += 32768u)
        tma_bulk_g2s(reinterpret_cast<char*>(Wb) + off, src + off, min(32768u, total - off), &wbar);
    }
    mbar_wait(&wbar, 0);
  }
  for (int i = tid; i < A.hop * A.NT; i += kPushThreads) fir_s[i] = A.fir[i];
  for (int i = tid; i < 12 * G; i += kPushThreads) { gh1[i] = 0.f; gh2[i] = 0.f; }     // W_hh . 0  (h1 = h2 = 0, :194-195)
  __shared__ PushRowState R;
  if (tid < G) {
    // state "before step 0": an empty segment ending at step 0, so that push_row_next(..., t = 0) finds segment 0
    R.k[tid] = -1; R.utt[tid] = -1; R.t0[tid] = 0; R.end[tid] = 0; R.putt[tid] = -1; R.pn[tid] = 0; R.rst[tid] = 1;
    if (!A.pack_utt) {                                     // plain batch / folds: row u is utterance u from step 0 to the end
      R.k[tid] = 0; R.utt[tid] = tid < A.B ? tid : -1; R.end[tid] = 0x7fffffff;
    }
  }
  __syncthreads();
  float* cond16 = cond;                       // [2][16][G]  rows 0-15 of step t (parity buffers, written one step ahead)
  float* cond20 = cond + 2 * 16 * G;          // [20][G]     rows 16-35 of the current frame
  push_cond16<G>(A, R, fir_s, cond16, c, ncta, 0, tid);
  push_cond20<G>(A, R, cond20, c, ncta, 0, tid);
  __syncthreads();
  if (A.pack_utt && tid < G) {                             // enter segment 0 (kernel rows beyond the schedule stay idle)
    const bool live = tid < A.pack_rows && A.pack_segs > 0;
    R.k[tid] = 0;
    R.utt[tid] = live ? A.pack_utt[tid * A.pack_segs] : -1;
    R.t0[tid] = 0;
    R.end[tid] = live ? A.pack_start[tid * (A.pack_segs + 1) + 1] : 0x7fffffff;
  }
  if constexpr (STREAM) {
    if (c == 0) {
      PushStreamSmem& ss = push_stream_smem();
      for (int l = tid; l < M.NC; l += kPushThreads) ss.dec[l] = wave_decode(l, (double)(M.NC - 1), A.mu_law);
      if (tid < A.B && tid < G) ss.wlen[tid] = wave_row_len(A.d_utt_frames, tid, (A.T - 1) * A.hop, A.hop);
      if (tid == 0) ss.step = wave_fade_step(A.fade_len);
    }
  }
  __syncthreads();

  PollGuard pg{A.error, 0, 0, false};
  float h1own = 0.f, h2own = 0.f;                          // gate threads: state of unit 4c+gj, row gu
  __shared__ long long s_pf[12];                           // optional per-phase cycle counters of thread 0 (debug)
  __shared__ long long s_tmark;
  if (tid == 0) {
    for (int i = 0; i < 12; ++i) s_pf[i] = 0;
    s_tmark = clock64();
  }
#define PUSH_MARK(slot)                          \
  do {                                           \
    if (A.prof && tid == 0) {                    \
      const long long now_ = clock64();          \
      s_pf[slot] += now_ - s_tmark;              \
      s_tmark = now_;                            \
    }                                            \
  } while (0)
  // a poll gave up (~2 s without a peer): the whole block leaves; a streaming CTA 0 first tells the host waiters
#define PUSH_GIVE_UP()                                                                 \
  do {                                                                                 \
    if constexpr (STREAM) {                                                            \
      if (c == 0 && tid == kPushThreads - 1) push_stream_publish(A, -1);               \
    }                                                                                  \
    return;                                                                            \
  } while (0)

  constexpr int NCQ = kPushThreads / G, NREC = 128 / NCQ;   // winner records per thread = G/4
  const int cq = tid / G;
  for (int t = 0; t <= A.steps; ++t) {
    const int par = t & 1;
    // ================= P01: winners of step t-1 -> label -> GRU 1 =================
    float x = 0.f;
    if (t > 0) {
      const unsigned long long want = (unsigned long long)((uint32_t)t & 0x3FFFFFu);
      unsigned long long rec[NREC];
#pragma unroll
      for (int i = 0; i < NREC; ++i) rec[i] = ld_relaxed_u64(A.best + (size_t)(cq + NCQ * i) * G + gu);
      unsigned long long bestp = 0ull;
#pragma unroll
      for (int i = 0; i < NREC; ++i) {
        unsigned long long v = rec[i];
        if ((v & 0x3FFFFFull) != want) {
          const unsigned long long* p = A.best + (size_t)(cq + NCQ * i) * G + gu;
          pg.begin();
          while (true) {
            v = ld_relaxed_u64(p);
            if ((v & 0x3FFFFFull) == want || pg.expired()) break;
          }
        }
        bestp = v > bestp ? v : bestp;
      }
      PUSH_MARK(0);
#pragma unroll
      for (int o = G; o < 32; o <<= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, bestp, o);
        bestp = other > bestp ? other : bestp;
      }
      if (lane < G) smax[warp * G + lane] = bestp;
      if (__syncthreads_or(pg.aborted ? 1 : 0)) PUSH_GIVE_UP();
      if (gate) {                                           // every warp covered different producers: reduce the 16 warps
        unsigned long long b = 0ull;
#pragma unroll
        for (int w = 0; w < kPushWarps; ++w) { const unsigned long long v = smax[w * G + gu]; b = v > b ? v : b; }
        const int label = (int)push_cls(b);
        const int putt = R.putt[gu], pn = R.pn[gu];         // where this row was at step t-1
        if (putt >= 0) {
          if (c == 0 && gj == 0) {
            A.labels[(size_t)putt * A.S + pn] = (int16_t)label;
            if constexpr (STREAM) push_stream_smem().lab[gu] = label;
          }
          const int fb = A.teacher ? (int)A.teacher[(size_t)putt * A.S + pn] : label;
          x = label_to_float(fb, ncls_m1);
        }
      }
    }
    if (t == A.steps) break;                                // the extra trip only collects the last winner
    const bool restart = gate && R.rst[gu] != 0;            // first step of an utterance: x = 0, h1 = h2 = 0 (:194-196)
    if (gate) {
      if (restart) { x = 0.f; h1own = 0.f; }
      const float* cd = cond16 + par * 16 * G;
      const float* wAx = Wb + M.oAx;
      const float* bhh = Wb + M.obhh1;
      const float iout = fmaf(wAx[gj], x, cd[gj * G + gu]);
      const float gir = fmaf(wAx[4 + gj], x, cd[(4 + gj) * G + gu]);
      const float giz = fmaf(wAx[8 + gj], x, cd[(8 + gj) * G + gu]);
      const float gin = fmaf(wAx[12 + gj], x, cd[(12 + gj) * G + gu]);
      const float g1r = restart ? 0.f : gh1[gj * G + gu], g1z = restart ? 0.f : gh1[(4 + gj) * G + gu],
                  g1n = restart ? 0.f : gh1[(8 + gj) * G + gu];            // W_hh1 . 0
      const float h = gru_update(gir, giz, gin, g1r + bhh[gj], g1z + bhh[4 + gj], g1n + bhh[8 + gj], h1own);
      h1own = h;
      const size_t e = ((size_t)c * G + gu) * 4 + gj;
      st_relaxed_f32(vecp(PV_H1, par) + e, h);
      st_relaxed_f32(vecp(PV_X1, par) + e, iout + h);
    }
    __syncwarp();      // (4G < 32: lanes that skip the gate block must not run ahead into a spin loop and steal its issue slots)
    PUSH_MARK(1);

    // ================= P2: W_ih2 (12 rows) AND fc1 (4 rows) on x1(t) =================
    // x2 = x1 + h2 is never exchanged: fc1 . x2 = fc1 . x1 + fc1 . h2, the first half is taken here while x1 is in registers,
    // the second in P3 from the h2 registers W_hh2 needs anyway -- one vector less through L2 per step.
    float f1x = 0.f;                                          // gate threads: (fc1 . x1)[4c + gj] of row gu
    // h1(t) was published together with x1(t): up to 16 rows (<= 4 float4 per vector and thread) its loads are issued with
    // the x1 loads, so the W_hh1 pass below starts from registers instead of paying another L2 round trip
    constexpr bool kPrefetchH1 = PT::NL <= 4;
    float4 ah1[kPrefetchH1 ? PT::NL : 1];
    {
      float4 a[PT::NL];
      push_load<G>(vecp(PV_X1, par), a, ul, kq, pg);
      if constexpr (kPrefetchH1) push_load<G>(vecp(PV_H1, par), ah1, ul, kq, pg);
      push_mma<G, 16>(Wb + M.oih2, a, partX, ul, kq, warp, lane);
    }
    PUSH_MARK(2);
    if (__syncthreads_or(pg.aborted ? 1 : 0)) PUSH_GIVE_UP();
    if (gate) {
      const float* cd = cond20;
      const float* bhh = Wb + M.obhh2;
      if (restart) h2own = 0.f;
      const float g2r = restart ? 0.f : gh2[gj * G + gu], g2z = restart ? 0.f : gh2[(4 + gj) * G + gu],
                  g2n = restart ? 0.f : gh2[(8 + gj) * G + gu];            // W_hh2 . 0
      const float h = gru_update(push_part_sum<G, 16>(partX, gj, gu) + cd[gj * G + gu],
                                 push_part_sum<G, 16>(partX, 4 + gj, gu) + cd[(4 + gj) * G + gu],
                                 push_part_sum<G, 16>(partX, 8 + gj, gu) + cd[(8 + gj) * G + gu], g2r + bhh[gj], g2z + bhh[4 + gj],
                                 g2n + bhh[8 + gj], h2own);
      h2own = h;
      f1x = push_part_sum<G, 16>(partX, 12 + gj, gu);
      st_relaxed_f32(vecp(PV_H2, par) + ((size_t)c * G + gu) * 4 + gj, h);
    }
    __syncwarp();
    PUSH_MARK(3);
    // shadow: W_hh1 . h1(t) for step t+1
    if constexpr (kPrefetchH1) push_mma<G, 12>(Wb + M.ohh1, reinterpret_cast<const float4 (&)[PT::NL]>(ah1), partY, ul, kq, warp, lane);
    else push_gemm<G, 12>(Wb + M.ohh1, vecp(PV_H1, par), partY, ul, kq, warp, lane, pg);
    if (__syncthreads_or(pg.aborted ? 1 : 0)) PUSH_GIVE_UP();
    for (int i = tid; i < 12 * G; i += kPushThreads) gh1[i] = push_part_sum<G, 12>(partY, i / G, i % G);
    PUSH_MARK(4);

    // ================= P3: h2(t) once: fc1 (critical), then W_hh2 . h2(t) for step t+1 from the same registers =================
    {
      float4 a[PT::NL];
      push_load<G>(vecp(PV_H2, par), a, ul, kq, pg);
      push_mma<G, 4>(Wb + M.ofc1, a, partX, ul, kq, warp, lane);
      PUSH_MARK(5);
      if (__syncthreads_or(pg.aborted ? 1 : 0)) PUSH_GIVE_UP();
      if (gate) {
        const float v = (f1x + push_part_sum<G, 4>(partX, gj, gu)) + cond20[(12 + gj) * G + gu];
        st_relaxed_f32(vecp(PV_F1, par) + ((size_t)c * G + gu) * 4 + gj, fmaxf(v, 0.f));
      }
      __syncwarp();
      push_mma<G, 12>(Wb + M.ohh2, a, partY, ul, kq, warp, lane);
    }
    if (__syncthreads_or(pg.aborted ? 1 : 0)) PUSH_GIVE_UP();
    for (int i = tid; i < 12 * G; i += kPushThreads) gh2[i] = push_part_sum<G, 12>(partY, i / G, i % G);
    PUSH_MARK(6);

    // ================= P4: fc2 + relu on f1(t) =================
    push_gemm<G, 4>(Wb + M.ofc2, vecp(PV_F1, par), partX, ul, kq, warp, lane, pg);
    // the fc2 conditioning value is taken BEFORE the barrier: after it the other threads may refresh cond20 for the next frame
    const float cv4 = gate ? cond20[(16 + gj) * G + gu] : 0.f;
    PUSH_MARK(7);
    if (__syncthreads_or(pg.aborted ? 1 : 0)) PUSH_GIVE_UP();
    if (gate) {
      const float v = push_part_sum<G, 4>(partX, gj, gu) + cv4;
      const size_t e = ((size_t)c * G + gu) * 4 + gj;
      st_relaxed_f32(vecp(PV_F2, par) + e, fmaxf(v, 0.f));
      // REARM (shadow of the f2 exchange).  Every CTA's winner of step t-1 was seen at the top of this step, and a CTA
      // publishes its winner LAST in a step: all reads of the step t-1 vectors, which live in the other parity copy, are
      // over everywhere -- this thread's entries of that copy can take the sentinel again.  Nobody polls that copy for
      // step t+1 before it has seen THIS CTA's winner of step t, which is stored below after two block barriers that
      // follow this fence: the sentinels are performed gpu-wide by then.
#pragma unroll
      for (int v6 = 0; v6 < kPushVecs; ++v6)
        if (v6 != PV_X2) st_relaxed_u32(vecp(v6, par ^ 1) + e, kPushSentinel);      // (x2 is not exchanged by this kernel)
      asm volatile("fence.acq_rel.gpu;" ::: "memory");
    }
    __syncwarp();
    if constexpr (STREAM) {      // shadow: sample of step t-1 to the host; every chunk_steps steps announce the samples of steps < t-1
      if (c == 0 && t > 0) {
        push_stream_sample<G>(A, push_stream_smem(), tid, t - 1);
        if (tid == kPushThreads - 1 && t > 1 && (t - 1) % A.chunk_steps == 0) push_stream_publish(A, t - 1);
      }
    }
    // shadow: conditioning of step t+1 (rows 0-15 into the other parity buffer; rows 16-35 only when a new frame starts)
    if (t + 1 < A.steps) {
      push_cond16<G>(A, R, fir_s, cond16 + (par ^ 1) * 16 * G, c, ncta, t + 1, tid);
      if (A.row_stride || A.pack_utt || (t + 1) % A.hop == 0) push_cond20<G>(A, R, cond20, c, ncta, t + 1, tid);
    }
    PUSH_MARK(8);

    // ================= P5: fc3 on f2(t) + Gumbel-max over this CTA's 8 classes =================
    push_gemm<G, 8>(Wb + M.ofc3, vecp(PV_F2, par), partY, ul, kq, warp, lane, pg);
    PUSH_MARK(9);
    if (__syncthreads_or(pg.aborted ? 1 : 0)) PUSH_GIVE_UP();
    if (tid < 8 * G) {
      const int r = tid / G, u = tid % G;
      const int cls = c * kCPC + r;
      const float l = push_part_sum<G, 8>(partY, r, u) + Wb[M.obfc3 + r];
      float qv = 1.0f;
      const int utt = R.utt[u], n = t - R.t0[u];               // plain batch: utt == u, n == t
      if (utt >= 0) {
        if (A.rng_mode == 0) {
          float q4[4];
          philox_exp4(A.seed, A.utt_ids ? A.utt_ids[utt] : A.utt_offset + (unsigned long long)utt, (uint32_t)n, (uint32_t)(cls >> 2), q4);
          qv = q4[cls & 3];
        } else {
          qv = __ldg(A.q + ((size_t)n * A.B + utt) * M.NC + cls);
        }
        if (A.logits_out) A.logits_out[((size_t)n * A.B + utt) * M.NC + cls] = l;
      }
      skeys[r * G + u] = push_pack(l - logf(qv), (uint32_t)cls, (uint32_t)(t + 1));
    }
    __syncthreads();
    if (tid < G) {
      unsigned long long b = skeys[tid];
#pragma unroll
      for (int r = 1; r < 8; ++r) { const unsigned long long v = skeys[r * G + tid]; b = v > b ? v : b; }
      st_relaxed_u64(A.best + (size_t)c * G + tid, b);
      // row bookkeeping for step t+1 (read by the gate threads after the barrier of the next winner poll)
      R.putt[tid] = R.utt[tid];
      R.pn[tid] = t - R.t0[tid];
      int rst = 0;
      if (t + 1 >= R.end[tid]) {                               // the row's utterance ends with this step: enter its next segment
        const int k1 = R.k[tid] + 1, e0 = R.end[tid];
        R.k[tid] = k1;
        const bool more = A.pack_utt && tid < A.pack_rows && k1 < A.pack_segs;
        R.utt[tid] = more ? A.pack_utt[tid * A.pack_segs + k1] : -1;
        R.t0[tid] = e0;
        R.end[tid] = more ? A.pack_start[tid * (A.pack_segs + 1) + k1 + 1] : 0x7fffffff;
        rst = 1;
      }
      R.rst[tid] = rst;
    }
    __syncwarp();
    PUSH_MARK(10);
  }
  if constexpr (STREAM) {        // the last trip collected the winner of step steps-1 and left before its P4: store, then announce all
    if (c == 0) {
      __syncthreads();
      if (A.steps > 0) push_stream_sample<G>(A, push_stream_smem(), tid, A.steps - 1);
      __syncthreads();
      if (tid == kPushThreads - 1) push_stream_publish(A, A.steps);
    }
  }
  if (A.prof && tid == 0)
    for (int i = 0; i < 12; ++i) A.prof[(size_t)c * 12 + i] = s_pf[i];
#undef PUSH_GIVE_UP
#undef PUSH_MARK
}

// ---- conditioning tables: tab[u][f][c][52] for f in [0, T]; frame T carries the bias only (zero conditioning) ------------
// cw: per CTA [16][feat] mel rows | [36][aux] aux rows | [36] bias   (floats; see pack in b200tts_api.cu)
struct PushCondW {
  const float* wm;      // [ncta][16][feat]
  const float* wa;      // [ncta][36][aux]
  const float* bias;    // [ncta][36]
  int ncta, feat, aux;
};
template <int FT>
__global__ void push_cond_table_kernel(PushCondW W, const float* __restrict__ mel /*[B][feat][T]*/,
                                       const float* __restrict__ aux_frames /*[B][T][4*aux]*/, int B, int T,
                                       float* __restrict__ tab /*[Brows][T+1][ncta][52]*/) {
  extern __shared__ float sm[];
  float* sm_mel = sm;                          // [feat][FT]
  float* sm_aux = sm + W.feat * FT;            // [4*aux][FT]
  const int u = blockIdx.y, f0 = blockIdx.x * FT;
  const int O = 4 * W.aux;
  const bool real = u < B;
  for (int i = threadIdx.x; i < W.feat * FT; i += blockDim.x) {
    const int k = i / FT, ff = f0 + i % FT;
    sm_mel[i] = (real && ff < T) ? mel[((size_t)u * W.feat + k) * T + ff] : 0.f;
  }
  for (int i = threadIdx.x; i < O * FT; i += blockDim.x) {
    const int k = i / FT, ff = f0 + i % FT;
    sm_aux[i] = (real && ff < T) ? aux_frames[((size_t)u * T + ff) * O + k] : 0.f;
  }
  __syncthreads();
  const int nout = W.ncta * kPushCondRows;
  for (int o = threadIdx.x; o < nout; o += blockDim.x) {
    const int c = o / kPushCondRows, row = o % kPushCondRows;
    float acc[FT];
    if (row < 16) {
#pragma unroll
      for (int i = 0; i < FT; ++i) acc[i] = 0.f;
      const float* w = W.wm + ((size_t)c * 16 + row) * W.feat;
      for (int k = 0; k < W.feat; ++k) {
        const float wk = __ldg(w + k);
#pragma unroll
        for (int i = 0; i < FT; ++i) acc[i] = fmaf(wk, sm_mel[k * FT + i], acc[i]);
      }
    } else {
      const int pr = row - 16;                                      // 0-15 a1 | 16-27 a2 | 28-31 a3 | 32-35 a4
      const int seg = pr < 16 ? 0 : (pr < 28 ? 1 : (pr < 32 ? 2 : 3));
      const float* w = W.wa + ((size_t)c * 36 + pr) * W.aux;
      const float b = __ldg(W.bias + (size_t)c * 36 + pr);
#pragma unroll
      for (int i = 0; i < FT; ++i) acc[i] = 0.f;
      for (int k = 0; k < W.aux; ++k) {
        const float wk = __ldg(w + k);
#pragma unroll
        for (int i = 0; i < FT; ++i) acc[i] = fmaf(wk, sm_aux[(seg * W.aux + k) * FT + i], acc[i]);
      }
#pragma unroll
      for (int i = 0; i < FT; ++i) acc[i] += b;
      if (!real) {
#pragma unroll
        for (int i = 0; i < FT; ++i) acc[i] = 0.f;
      }
      // frame T (and padding frames of the last tile): zero conditioning -> bias only
#pragma unroll
      for (int i = 0; i < FT; ++i)
        if (f0 + i >= T) acc[i] = real ? b : 0.f;
    }
#pragma unroll
    for (int i = 0; i < FT; ++i) {
      const int ff = f0 + i;
      if (ff <= T) tab[(((size_t)u * (T + 1) + ff) * W.ncta + c) * kPushCondRows + row] = (row < 16 && ff >= T) ? 0.f : acc[i];
    }
  }
}

// fills the exchange buffers with the sentinel pattern and clears the winner slots / error flag
__global__ void push_init_kernel(uint32_t* __restrict__ vec, size_t nvec, unsigned long long* __restrict__ best, size_t nbest,
                                 int* __restrict__ error) {
  const size_t i0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x, st = (size_t)gridDim.x * blockDim.x;
  for (size_t i = i0; i < nvec; i += st) vec[i] = kPushSentinel;
  for (size_t i = i0; i < nbest; i += st) best[i] = 0ull;
  if (i0 == 0) *error = 0;
}

}  // namespace b200tts
