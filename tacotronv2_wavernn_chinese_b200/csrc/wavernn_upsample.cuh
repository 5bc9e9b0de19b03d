// WaveRNN conditioning network on the GPU.
//
// Replaces UpsampleNetwork.forward (reference wavernn/models/fatchord_version.py:82-89):
//   * MelResNet (:31-48, ResBlock :13-28) evaluated at FRAME rate -- the reference stretches its output x hop
//     afterwards (:84), so aux is constant within a hop and is never materialised at sample rate here.
//   * the three Stretch2d + Conv2d stages (:73-80, :86-87) collapsed into one polyphase FIR of `hop` phases x NT
//     taps over the zero-padded frame sequence.  The composite taps are derived on the host (double precision)
//     by pushing an impulse through the stages; the stages' own zero padding only disturbs samples inside the
//     `indent` that :88 trims away (reach 341 samples < indent 550 for factors (5,5,11)).
#pragma once
#include "common.cuh"

namespace b200tts {

constexpr int kMaxTaps = 7;

struct ResnetParams {
  // all weights are transposed to [in][out] so that thread `c` (output channel) reads coalesced
  const float* conv_in_t;   // [feat*k][C]   (index (i*k + j)*C + c)
  const float* bn_scale;    // [(1 + 2*blocks)][C]   gamma / sqrt(var + eps)
  const float* bn_shift;    // [(1 + 2*blocks)][C]   beta - mean * scale
  const float* res_w_t;     // [blocks][2][C][C]     (in-major)
  const float* conv_out_t;  // [C][O]
  const float* conv_out_b;  // [O]
  int feat, k, C, O, blocks, pad;
};

// One CTA = FT frames of one utterance; thread c owns channel c for all FT frames.
template <int FT>
__global__ void melresnet_kernel(ResnetParams P, const float* __restrict__ mel /*[B][feat][T]*/,
                                                        int T, float* __restrict__ aux_frames /*[B][T][O]*/) {
  extern __shared__ float sm[];
  const int C = P.C;
  float* xin = sm;                              // [feat*k][FT]
  float* act = xin + P.feat * P.k * FT;         // [C][FT]
  float* tmp = act + C * FT;                    // [C][FT]
  const int b = blockIdx.y, f0 = blockIdx.x * FT, c = threadIdx.x;
  const float* melb = mel + (size_t)b * P.feat * T;
  // gather the k-frame windows; frame index into the padded sequence is f + j, i.e. unpadded f + j - pad
  for (int e = threadIdx.x; e < P.feat * P.k * FT; e += blockDim.x) {
    int ft = e % FT, ij = e / FT, j = ij % P.k, i = ij / P.k;
    int fr = f0 + ft + j - P.pad;
    xin[e] = (fr >= 0 && fr < T && f0 + ft < T) ? melb[(size_t)i * T + fr] : 0.f;
  }
  __syncthreads();
  float acc[FT];
  if (c < C) {
#pragma unroll
    for (int t = 0; t < FT; ++t) acc[t] = 0.f;
    for (int e = 0; e < P.feat * P.k; ++e) {
      float w = P.conv_in_t[(size_t)e * C + c];
#pragma unroll
      for (int t = 0; t < FT; ++t) acc[t] = fmaf(w, xin[e * FT + t], acc[t]);
    }
    float s = P.bn_scale[c], h = P.bn_shift[c];
#pragma unroll
    for (int t = 0; t < FT; ++t) act[c * FT + t] = fmaxf(fmaf(acc[t], s, h), 0.f);
  }
  __syncthreads();
  for (int blk = 0; blk < P.blocks; ++blk) {
    const float* w1 = P.res_w_t + (size_t)(blk * 2) * C * C;
    const float* w2 = w1 + (size_t)C * C;
    if (c < C) {
#pragma unroll
      for (int t = 0; t < FT; ++t) acc[t] = 0.f;
      for (int i = 0; i < C; ++i) {
        float w = w1[(size_t)i * C + c];
#pragma unroll
        for (int t = 0; t < FT; ++t) acc[t] = fmaf(w, act[i * FT + t], acc[t]);
      }
      float s = P.bn_scale[(1 + 2 * blk) * C + c], h = P.bn_shift[(1 + 2 * blk) * C + c];
#pragma unroll
      for (int t = 0; t < FT; ++t) tmp[c * FT + t] = fmaxf(fmaf(acc[t], s, h), 0.f);
    }
    __syncthreads();
    if (c < C) {
#pragma unroll
      for (int t = 0; t < FT; ++t) acc[t] = 0.f;
      for (int i = 0; i < C; ++i) {
        float w = w2[(size_t)i * C + c];
#pragma unroll
        for (int t = 0; t < FT; ++t) acc[t] = fmaf(w, tmp[i * FT + t], acc[t]);
      }
      float s = P.bn_scale[(2 + 2 * blk) * C + c], h = P.bn_shift[(2 + 2 * blk) * C + c];
      // act[c][*] is only re-read by its own thread here (residual); everybody else reads tmp -> no hazard
#pragma unroll
      for (int t = 0; t < FT; ++t) act[c * FT + t] = fmaf(acc[t], s, h) + act[c * FT + t];
    }
    __syncthreads();
  }
  for (int o = threadIdx.x; o < P.O; o += blockDim.x) {
#pragma unroll
    for (int t = 0; t < FT; ++t) acc[t] = 0.f;
    for (int i = 0; i < C; ++i) {
      float w = P.conv_out_t[(size_t)i * P.O + o];
#pragma unroll
      for (int t = 0; t < FT; ++t) acc[t] = fmaf(w, act[i * FT + t], acc[t]);
    }
    float bias = P.conv_out_b[o];
#pragma unroll
    for (int t = 0; t < FT; ++t)
      if (f0 + t < T) aux_frames[((size_t)b * T + f0 + t) * P.O + o] = acc[t] + bias;
  }
}

// mels_up[b][n][c] = sum_j fir[ph][j] * melpad[b][c][fr + j - NT/2],  n' = n + pad*hop, fr = n'/hop, ph = n'%hop
__global__ void mel_fir_kernel(const float* __restrict__ mel /*[B][feat][T]*/, const float* __restrict__ fir /*[hop][NT]*/,
                               int T, int feat, int hop, int pad, int NT, float* __restrict__ mels_up /*[B][T*hop][feat]*/) {
  const int b = blockIdx.y;
  const size_t S = (size_t)T * hop;
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < S * feat; e += (size_t)gridDim.x * blockDim.x) {
    int c = (int)(e % feat);
    size_t n = e / feat;
    size_t np = n + (size_t)pad * hop;
    int fr = (int)(np / hop), ph = (int)(np % hop);
    float acc = 0.f;
    for (int j = 0; j < NT; ++j) {
      int f = fr + j - NT / 2 - pad;   // unpadded frame index
      if (f >= 0 && f < T) acc = fmaf(fir[ph * NT + j], mel[((size_t)b * feat + c) * T + f], acc);
    }
    mels_up[((size_t)b * S + n) * feat + c] = acc;
  }
}

__global__ void aux_repeat_kernel(const float* __restrict__ aux_frames, int T, int hop, int O, float* __restrict__ aux_full) {
  const int b = blockIdx.y;
  const size_t S = (size_t)T * hop;
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < S * O; e += (size_t)gridDim.x * blockDim.x) {
    int o = (int)(e % O);
    size_t n = e / O;
    aux_full[((size_t)b * S + n) * O + o] = aux_frames[((size_t)b * T + n / hop) * O + o];
  }
}

// ---- fold_with_overlap (fatchord_version.py:293-340): ONE utterance's conditioning -> per-fold rows ----------------
// Fold u covers samples [u*(target+overlap), u*(target+overlap) + target + 2*overlap); positions beyond S read as 0
// (the reference zero-pads BOTH mels and aux after the end, :326-330).  aux is emitted per SAMPLE here (hop = 1 for the
// generation kernels) because fold boundaries need not be hop aligned.
// K-major layout for the grid kernel: mels_T[t][c][u], aux_T[t][o][u]
__global__ void fold_cond_T_kernel(const float* __restrict__ mels_up /*[S][feat]*/, const float* __restrict__ aux_frames /*[T][O]*/,
                                   int S, int hop, int feat, int O, int L, int stride, int nfold, int Bp,
                                   float* __restrict__ mels_T /*[L][feat][Bp]*/, float* __restrict__ aux_T /*[L][O][Bp]*/) {
  const size_t total = (size_t)L * (feat + O) * Bp;
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
    const int u = (int)(e % Bp);
    const size_t r = e / Bp;
    const int c = (int)(r % (feat + O));
    const int t = (int)(r / (feat + O));
    const long long pos = (long long)u * stride + t;
    const bool in = u < nfold && pos < S;
    if (c < feat) mels_T[((size_t)t * feat + c) * Bp + u] = in ? mels_up[(size_t)pos * feat + c] : 0.f;
    else aux_T[((size_t)t * O + (c - feat)) * Bp + u] = in ? aux_frames[(size_t)(pos / hop) * O + (c - feat)] : 0.f;
  }
}
// row-major layout for the utterance kernel: mels_f[u][t][c], aux_f[u][t][o]
__global__ void fold_cond_kernel(const float* __restrict__ mels_up, const float* __restrict__ aux_frames, int S, int hop, int feat,
                                 int O, int L, int stride, int nfold, float* __restrict__ mels_f, float* __restrict__ aux_f) {
  const size_t total = (size_t)nfold * L * (feat + O);
  for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(e % (feat + O));
    const size_t r = e / (feat + O);
    const int t = (int)(r % L);
    const int u = (int)(r / L);
    const long long pos = (long long)u * stride + t;
    const bool in = pos < S;
    if (c < feat) mels_f[((size_t)u * L + t) * feat + c] = in ? mels_up[(size_t)pos * feat + c] : 0.f;
    else aux_f[((size_t)u * L + t) * O + (c - feat)] = in ? aux_frames[(size_t)(pos / hop) * O + (c - feat)] : 0.f;
  }
}

// np.linspace(-1, 1, flen)[k]: -1 + k * 2/(flen-1), exactly +1 at the last point; a ONE point linspace is [-1]
__device__ __forceinline__ double xfade_t(int k, int flen) {
  if (flen <= 1) return -1.0;
  return (k == flen - 1) ? 1.0 : (-1.0 + k * (2.0 / (flen - 1)));
}

// xfade_and_unfold (fatchord_version.py:342-405) + the generate() epilogue (:247-258), fp64:
// decode every fold's labels, apply the equal-power fade-in/out over `overlap` (first half of the fade-in is silence),
// overlap-add at stride target+overlap, truncate to wave_len, 20-hop linear fade-out.
__global__ void xfade_unfold_kernel(const int16_t* __restrict__ labels /*[nfold][L]*/, int nfold, int L, int target, int overlap,
                                    int wave_len, int fade_len, int ncls, int mu_law, const int* __restrict__ gen_error,
                                    double* __restrict__ wave /*[wave_len]*/) {
  const double mu = (double)(ncls - 1);
  const bool poisoned = gen_error && *gen_error;    // the generation kernel timed out: never hand back plausible-looking audio
  const int stride = target + overlap;
  const int silence = overlap / 2, flen = overlap - silence;
  const double lin_step = -1.0 / (double)(fade_len - 1);
  for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < wave_len; n += gridDim.x * blockDim.x) {
    double acc = 0.0;
    int u_hi = n / stride;                          // last fold that can start at or before n
    if (u_hi >= nfold) u_hi = nfold - 1;
    for (int u = u_hi; u >= 0 && u >= u_hi - 1; --u) {
      const int t = n - u * stride;
      if (t < 0 || t >= L) continue;
      float yf = label_to_float((int)labels[(size_t)u * L + t], (float)(ncls - 1));
      double y = (double)yf;
      if (mu_law) {
        const double a = fabs(y), sgn = (y > 0.0) - (y < 0.0);
        y = sgn / mu * (pow(1.0 + mu, a) - 1.0);
      }
      // np.linspace(-1, 1, flen)[k] = -1 + k * 2/(flen-1)
      if (t < overlap) {
        double g = 0.0;
        if (t >= silence) { const int k = t - silence; const double tt = xfade_t(k, flen); g = sqrt(0.5 * (1.0 + tt)); }
        y *= g;
      }
      if (t >= L - overlap) {
        const int k2 = t - (L - overlap);
        double g = 1.0;
        if (k2 >= silence) { const int k = k2 - silence; const double tt = xfade_t(k, flen); g = sqrt(0.5 * (1.0 - tt)); }
        y *= g;
      }
      acc += y;
    }
    const int k = n - (wave_len - fade_len);
    if (k >= 0) acc *= (k == fade_len - 1) ? 0.0 : (1.0 + (double)k * lin_step);
    wave[n] = poisoned ? nan("") : acc;
  }
}

// The two halves of the generate() epilogue for ONE sample, shared by finish_wave_kernel and the streaming push kernel (which
// decodes through a table built with wave_decode and fades in the loop), so that both produce the same bits:
//   wave_decode: label -> float64, decode_mu_law (dsp.py:98-103) when mu_law is set
//   wave_fade:   20-hop linear fade-out of sample i of a row truncated at wave_len (fatchord_version.py:256-258);
//                step = wave_fade_step(fade_len) = np.linspace(1, 0, fade_len)[1]
__device__ __forceinline__ double wave_decode(int label, double mu, int mu_law) {
  float yf = label_to_float(label, (float)mu);
  double y = (double)yf;
  if (mu_law) {
    double a = fabs(y);
    double sgn = (y > 0.0) - (y < 0.0);
    y = sgn / mu * (pow(1.0 + mu, a) - 1.0);
  }
  return y;
}
__device__ __forceinline__ double wave_fade_step(int fade_len) { return -1.0 / (double)(fade_len - 1); }
__device__ __forceinline__ double wave_fade(double y, int i, int wave_len, int fade_len, double step) {
  int k = i - (wave_len - fade_len);
  if (k >= 0) y *= (k == fade_len - 1) ? 0.0 : (1.0 + (double)k * step);
  return y;
}
// length of row b of a ragged batch: its own (T_b - 1) * hop, capped at the launch's
__device__ __forceinline__ int wave_row_len(const int* utt_frames, int b, int wave_len_max, int hop) {
  return utt_frames ? min(wave_len_max, max(0, (utt_frames[b] - 1) * hop)) : wave_len_max;
}

// generate() epilogue (fatchord_version.py:243-258): float64, decode_mu_law (dsp.py:98-103), truncate, 20-hop fade.
// `utt_frames` (optional, [B]): true frame count of each row of a zero-padded ragged batch -> that row is truncated / faded at
// ITS OWN (T_b - 1) * hop like a batch-1 run of the reference, and zero beyond.
__global__ void finish_wave_kernel(const int16_t* __restrict__ labels /*[B][S]*/, int S, int wave_len_max, int fade_len,
                                   int ncls, int mu_law, const int* __restrict__ utt_frames, int hop,
                                   const int* __restrict__ gen_error, double* __restrict__ wave /*[B][wave_len_max]*/) {
  const int b = blockIdx.y;
  const bool poisoned = gen_error && *gen_error;    // the generation kernel timed out: never hand back plausible-looking audio
  const double mu = (double)(ncls - 1);
  const double step = wave_fade_step(fade_len);
  const int wave_len = wave_row_len(utt_frames, b, wave_len_max, hop);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < wave_len_max; i += gridDim.x * blockDim.x) {
    if (i >= wave_len) { wave[(size_t)b * wave_len_max + i] = 0.0; continue; }
    const double y = wave_fade(wave_decode((int)labels[(size_t)b * S + i], mu, mu_law), i, wave_len, fade_len, step);
    wave[(size_t)b * wave_len_max + i] = poisoned ? nan("") : y;
  }
}

}  // namespace b200tts
