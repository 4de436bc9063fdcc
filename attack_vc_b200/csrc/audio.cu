// audio.cu -- mel front-end and Griffin-Lim back-end (SURVEY.md §8f rank 4; reference data_utils.py:16-31, 65-197) on B200.
//
// What runs here is the arithmetic between a trimmed waveform and the normalised log-mel the attacks consume, and back:
//   wav2mel  (file2mel :99-114)  pre-emphasis -> STFT -> |.| -> mel basis -> 20 log10 -> clip to [1e-8, 1]
//   mel2wav  (mel2wav :149-164)  inverse scaling -> inv_mel_matrix -> Griffin-Lim (n_iter x [ISTFT, STFT, unit phase]) -> de-emphasis
// librosa.load / effects.trim stay host I/O.  Griffin-Lim is where the time goes once the attack is fast (SURVEY §8f):
// 2 n_iter + 1 transforms per utterance.  Both transforms are dense GEMMs against precomputed DFT matrices on the tensor
// cores -- conv2d_tc_kernel as a plain GEMM: TMA-fed operands, 3xTF32, chunked fp32 accumulation -- because a frame count of
// a few hundred rows x n_fft = 2048 is exactly the shape that kernel is built for, and an FFT would be a new kernel family
// used nowhere else on the path.  Everything between the GEMMs is one small elementwise / gather kernel each.
//   frames [F, n_fft] (reflect-centred, Hann-windowed, written directly as hi / lo planes)
//     x W_fwd^T [n_fft -> re(0..n_fft/2) | im(0..n_fft/2)]            -> spectrum [F, NP]
//   spectrum x W_inv^T [NP -> n_fft] (numpy irfft semantics)          -> time frames [F, n_fft] -> windowed overlap-add / window sum-square
// Oracle: oracle/audio_oracle.py (numpy; pinned against scipy.signal and transformers.audio_utils -- librosa itself is not
// installed, so parity with the reference's third-party arithmetic is unpinned, see DESIGN.md).
#include <cuda_runtime.h>

#include <cmath>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../../include/avc_b200.h"
#include "common.cuh"
#include "host_util.h"
#include "conv2d_tc.cuh"

using namespace avc;

namespace {

thread_local std::string g_audio_create_error;

__device__ __forceinline__ int au_reflect(long long i, long long n) {      // np.pad(mode="reflect"): edge not repeated
  if (i < 0) i = -i;
  if (i >= n) i = 2 * (n - 1) - i;
  return (int)i;
}

// y[0] = x[0]; y[i] = x[i] - a x[i-1]                                   (data_utils.py:99)
// (x, y hold B utterances of n samples each, end to end)
__global__ void au_preemph_kernel(const float* __restrict__ x, float* __restrict__ y, long long n, int B, float a) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n * B; i += (long long)gridDim.x * blockDim.x)
    y[i] = (i % n) ? x[i] - a * x[i - 1] : x[i];
}

// frame f, sample j = wav[reflect(f hop + j - n_fft/2)] * window[j], split into 3xTF32 planes      (librosa.stft, center=True)
// (wav: one utterance of n samples)
__device__ __forceinline__ void au_frame_elem(const float* __restrict__ wav, long long n, const float* __restrict__ window, float* __restrict__ hi,
                                              float* __restrict__ lo, long long i, int f, int j, int n_fft, int hop) {
  const float w = window[j];
  const float v = w != 0.f ? wav[au_reflect((long long)f * hop + j - n_fft / 2, n)] * w : 0.f;
  const float h = tf32_hi(v);
  hi[i] = h; lo[i] = v - h;
}

// n_frames per utterance; rows of the frame matrix are (utterance, frame)
__global__ void au_frame_kernel(const float* __restrict__ wav, long long n, const float* __restrict__ window, float* __restrict__ hi,
                                float* __restrict__ lo, int n_frames, int B, int n_fft, int hop) {
  const long long tot = (long long)B * n_frames * n_fft;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < tot; i += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(i % n_fft);
    const long long r = i / n_fft;
    const int f = (int)(r % n_frames), b = (int)(r / n_frames);
    au_frame_elem(wav + (long long)b * n, n, window, hi, lo, i, f, j, n_fft, hop);
  }
}

// Ragged batches (avc_audio_*_varlen): utterance u owns samples [s_off[u], s_off[u+1]) and frame rows [f_off[u], f_off[u+1]);
// fu[r] is the utterance of frame row r.  Utterances are never empty, so the offsets are strictly increasing.
// largest u in [0, B) with off[u] <= i
__device__ __forceinline__ int au_find(const long long* __restrict__ off, int B, long long i) {
  int lo = 0, hi = B - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (off[mid] <= i) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// the pre-emphasis of au_preemph_kernel over utterances of their own lengths
__global__ void au_preemph_varlen_kernel(const float* __restrict__ x, float* __restrict__ y, const long long* __restrict__ s_off, int B, float a) {
  const long long tot = s_off[B];
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < tot; i += (long long)gridDim.x * blockDim.x)
    y[i] = (i - s_off[au_find(s_off, B, i)]) ? x[i] - a * x[i - 1] : x[i];
}

__global__ void au_frame_varlen_kernel(const float* __restrict__ wav, const long long* __restrict__ s_off, const int* __restrict__ f_off,
                                       const int* __restrict__ fu, const float* __restrict__ window, float* __restrict__ hi,
                                       float* __restrict__ lo, long long R, int n_fft, int hop) {
  const long long tot = R * n_fft;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < tot; i += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(i % n_fft);
    const long long r = i / n_fft;
    const int u = fu[r];
    const long long s0 = s_off[u];
    au_frame_elem(wav + s0, s_off[u + 1] - s0, window, hi, lo, i, (int)(r - f_off[u]), j, n_fft, hop);
  }
}

// |re + i im| of a spectrum row [re(0..nbin) | im(0..nbin) | pad]
__global__ void au_mag_kernel(const float* __restrict__ spec, float* __restrict__ mag, int n_frames, int nbin, int NP) {
  const long long tot = (long long)n_frames * nbin;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < tot; i += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(i % nbin), f = (int)(i / nbin);
    const float re = spec[(long long)f * NP + k], im = spec[(long long)f * NP + nbin + k];
    mag[i] = sqrtf(re * re + im * im);
  }
}

// mel[f][m] = clip((20 log10(max(1e-5, sum_k basis[m][k] mag[f][k])) - ref_db + max_db) / max_db, 1e-8, 1)      (:108-114)
// one warp per output; lanes stride over the bins (fixed-order tree)
// mean / std non-null: the speaker normalisation of data_utils.py:35-40 follows, (mel - mean[m]) / std[m], correctly rounded and
// unfused like the numpy code
__global__ void au_mel_kernel(const float* __restrict__ mag, const float* __restrict__ basis, float* __restrict__ mel, int n_frames, int nbin,
                              int n_mels, float ref_db, float max_db, const float* __restrict__ mean, const float* __restrict__ std) {
  const long long o = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (o >= (long long)n_frames * n_mels) return;
  const int m = (int)(o % n_mels), f = (int)(o / n_mels);
  float s = 0.f;
  for (int k = threadIdx.x & 31; k < nbin; k += 32) s = fmaf(basis[(long long)m * nbin + k], mag[(long long)f * nbin + k], s);
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
  if ((threadIdx.x & 31) == 0) {
    const float db = 20.f * log10f(fmaxf(1e-5f, s));
    const float v = fminf(fmaxf((db - ref_db + max_db) / max_db, 1e-8f), 1.f);
    mel[o] = mean ? __fdiv_rn(__fsub_rn(v, mean[m]), std[m]) : v;
  }
}

// mag[f][k] = sum_m inv[k][m] * 10^(0.05 ((clip(mel[f][m], 0, 1) * max_db) - max_db + ref_db))                 (:151-156)
// mean / std non-null: the input is first denormalised, x * std[m] + mean[m] (data_utils.py:43-47), correctly rounded and unfused
__global__ void au_invmel_kernel(const float* __restrict__ mel, const float* __restrict__ inv, float* __restrict__ mag, int n_frames, int nbin,
                                 int n_mels, float ref_db, float max_db, const float* __restrict__ mean, const float* __restrict__ std) {
  extern __shared__ float au_lin[];      // [n_mels] linear-scale mel of this frame
  const int f = blockIdx.x;
  for (int m = threadIdx.x; m < n_mels; m += blockDim.x) {
    float x = mel[(long long)f * n_mels + m];
    if (mean) x = __fadd_rn(__fmul_rn(x, std[m]), mean[m]);
    const float v = fminf(fmaxf(x, 0.f), 1.f) * max_db - max_db + ref_db;
    au_lin[m] = powf(10.f, v * 0.05f);
  }
  __syncthreads();
  for (int k = threadIdx.x; k < nbin; k += blockDim.x) {
    float s = 0.f;
    for (int m = 0; m < n_mels; ++m) s = fmaf(inv[(long long)k * n_mels + m], au_lin[m], s);
    mag[(long long)f * nbin + k] = s;
  }
}

// Griffin-Lim state X = spect * phase as 3xTF32 planes of [re | im | pad].  est == nullptr: zero phase (X_best = spect, :182)
__global__ void au_phase_kernel(const float* __restrict__ mag, const float* __restrict__ est, float* __restrict__ hi, float* __restrict__ lo,
                                int n_frames, int nbin, int NP) {
  const long long tot = (long long)n_frames * NP;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < tot; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % NP), f = (int)(i / NP);
    float v = 0.f;
    if (c < 2 * nbin) {
      const int k = c < nbin ? c : c - nbin;
      const float m = mag[(long long)f * nbin + k];
      if (!est) v = c < nbin ? m : 0.f;
      else {
        const float re = est[(long long)f * NP + k], im = est[(long long)f * NP + nbin + k];
        const float den = fmaxf(1e-8f, sqrtf(re * re + im * im));            // phase = est / max(1e-8, |est|)      (:186)
        v = m * ((c < nbin ? re : im) / den);
      }
    }
    const float h = tf32_hi(v);
    hi[i] = h; lo[i] = v - h;
  }
}

// librosa.istft after the inverse transform: y[p] = sum_f tf[f][p - f hop] w[p - f hop] / sum_f w[p - f hop]^2 (where > tiny), the
// n_fft/2 centre padding removed.  Gather form: every output sample walks the <= ceil(n_fft / hop) frames that cover it, in order.
// output sample s of one utterance whose n_frames time frames start at tf
__device__ __forceinline__ float au_ola_sample(const float* __restrict__ tf, const float* __restrict__ window, long long s, int n_frames,
                                               int n_fft, int hop) {
  const long long p = s + n_fft / 2;
  long long f_hi = p / hop;
  if (f_hi > n_frames - 1) f_hi = n_frames - 1;
  long long f_lo = (p - n_fft + hop) / hop;       // smallest f with p - f hop < n_fft  (ceil((p - n_fft + 1) / hop))
  if (p - n_fft + 1 <= 0) f_lo = 0;
  else f_lo = (p - n_fft + 1 + hop - 1) / hop;
  float acc = 0.f, wss = 0.f;
  for (long long f = f_lo; f <= f_hi; ++f) {
    const int j = (int)(p - f * hop);
    const float w = window[j];
    acc = fmaf(tf[f * n_fft + j], w, acc);
    wss = fmaf(w, w, wss);
  }
  return wss > 1.17549435e-38f ? acc / wss : acc;
}

__global__ void au_ola_kernel(const float* __restrict__ tf_all, const float* __restrict__ window, float* __restrict__ wav, long long n_out, int n_frames,
                              int B, int n_fft, int hop) {
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < n_out * B; q += (long long)gridDim.x * blockDim.x)
    wav[q] = au_ola_sample(tf_all + (q / n_out) * (long long)n_frames * n_fft, window, q % n_out, n_frames, n_fft, hop);
}

// ragged: utterance u writes samples [o_off[u], o_off[u+1]) from its frame rows [f_off[u], f_off[u+1])
__global__ void au_ola_varlen_kernel(const float* __restrict__ tf_all, const float* __restrict__ window, float* __restrict__ wav,
                                     const long long* __restrict__ o_off, const int* __restrict__ f_off, int B, int n_fft, int hop) {
  const long long tot = o_off[B];
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < tot; q += (long long)gridDim.x * blockDim.x) {
    const int u = au_find(o_off, B, q);
    wav[q] = au_ola_sample(tf_all + (long long)f_off[u] * n_fft, window, q - o_off[u], f_off[u + 1] - f_off[u], n_fft, hop);
  }
}

// scipy.signal.lfilter([1], [1, -a], x): y[n] = x[n] + a y[n-1], in place.  A 77 k-sample recurrence is 0.2 ms on one thread.
// (one thread per utterance)
__global__ void au_deemph_kernel(float* x_all, long long n, int B, float a) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  float* x = x_all + (long long)b * n;
  float acc = 0.f;
  for (long long i = 0; i < n; ++i) { acc = fmaf(a, acc, x[i]); x[i] = acc; }
}

__global__ void au_deemph_varlen_kernel(float* x_all, const long long* __restrict__ o_off, int B, float a) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  float* x = x_all + o_off[b];
  const long long n = o_off[b + 1] - o_off[b];
  float acc = 0.f;
  for (long long i = 0; i < n; ++i) { acc = fmaf(a, acc, x[i]); x[i] = acc; }
}

// ---- host: Slaney mel basis (librosa.filters.mel defaults) ------------------------------------------------------------
double au_hz_to_mel(double f) { return f >= 1000.0 ? 15.0 + std::log(f / 1000.0) / (std::log(6.4) / 27.0) : f / (200.0 / 3); }
double au_mel_to_hz(double m) { return m >= 15.0 ? 1000.0 * std::exp((std::log(6.4) / 27.0) * (m - 15.0)) : (200.0 / 3) * m; }

std::vector<float> au_mel_basis(int sr, int n_fft, int n_mels) {
  const int nbin = 1 + n_fft / 2;
  std::vector<double> mel_f(n_mels + 2);
  const double lo = au_hz_to_mel(0.0), hi = au_hz_to_mel(sr / 2.0);
  for (int i = 0; i < n_mels + 2; ++i) mel_f[i] = au_mel_to_hz(lo + (hi - lo) * i / (n_mels + 1));
  std::vector<float> w((size_t)n_mels * nbin);
  for (int i = 0; i < n_mels; ++i) {
    const double enorm = 2.0 / (mel_f[i + 2] - mel_f[i]);
    for (int k = 0; k < nbin; ++k) {
      const double f = (sr / 2.0) * k / (nbin - 1);
      const double lower = (f - mel_f[i]) / (mel_f[i + 1] - mel_f[i]), upper = (mel_f[i + 2] - f) / (mel_f[i + 2] - mel_f[i + 1]);
      w[(size_t)i * nbin + k] = (float)(std::max(0.0, std::min(lower, upper)) * enorm);
    }
  }
  return w;
}

}  // namespace

struct avc_audio_handle {
  int device = 0, sm_count = 148;
  avc_audio_desc d{};
  int nbin = 0, NP = 0;
  Arena wmem;
  SlabPool pool;
  float *window = nullptr, *basis = nullptr, *inv = nullptr;
  float *wf_h = nullptr, *wf_l = nullptr;      // forward DFT  [NP rows][n_fft]   (K-major weight operand: rows = output column)
  float *wi_h = nullptr, *wi_l = nullptr;      // inverse DFT  [n_fft rows][NP]
  float* part = nullptr; size_t part_floats = 0;
  std::string err;
  long long launches = 0;
};

namespace {

template <class Fn>
int au_guarded(avc_audio_handle* h, Fn&& fn) {
  try {
    DeviceGuard dg(h ? h->device : -1);
    fn();
    return AVC_OK;
  } catch (const Fail& f) {
    if (h) h->err = f.msg; else g_audio_create_error = f.msg;
    return f.code;
  } catch (const std::exception& e) {
    if (h) h->err = e.what(); else g_audio_create_error = e.what();
    return AVC_ERR_INVALID;
  }
}

unsigned au_grid(long long n, int sm) { return (unsigned)std::max<long long>(1, std::min<long long>((n + 255) / 256, (long long)sm * 8)); }

// Y[M, N] = X[M, K] (hi / lo planes) x W^T, W given as K-major planes [N rows][K]
void au_gemm(avc_audio_handle* h, const float* xh, const float* xl, int M, int K, const float* wh, const float* wl, int N, float* y, cudaStream_t st) {
  C2Args c{};
  c.B = 1; c.Hb = 1; c.Wb = M; c.a_wmul = c.a_hmul = 1; c.n_taps = 1;
  c.Ci = K; c.Cop = N; c.y = y; c.Ho = 1; c.Wo = M; c.Co = N; c.oh_mul = c.ow_mul = 1; c.ksplit = 1;
  c2_pick_boxes(c);
  const int tiles = c2_tiles(c);
  if (2 * tiles <= h->sm_count) c.ksplit = std::max(1, std::min({8, h->sm_count / std::max(1, tiles), c2_stages(c)}));
  if (c.ksplit > 1) {
    const size_t n = (size_t)M * N;
    if (h->part_floats < n * c.ksplit) {
      h->part = h->wmem.f(n * c.ksplit); h->part_floats = n * c.ksplit;
      CK(cudaDeviceSynchronize());
    }
    c.part = h->part; c.part_stride = (long long)n;
  }
  const WtOperand X{xh, xl, K, M, 1, 1, 1, 1};
  launch_conv2d_tc(X, wh, wl, K, N, c, h->sm_count, st, 1);
  if (c.ksplit > 1) launch_c2_finish(c, h->sm_count, st);
  h->launches += c.ksplit > 1 ? 2 : 1;
}

// B utterances of n samples -> spectrum [B*F][NP]
void au_stft(avc_audio_handle* h, Arena& mem, const float* wav, long long n, int F, int B, float* spec, cudaStream_t st) {
  const int n_fft = h->d.n_fft;
  float* fh = mem.f((size_t)B * F * n_fft); float* fl = mem.f((size_t)B * F * n_fft);
  au_frame_kernel<<<au_grid((long long)B * F * n_fft, h->sm_count), 256, 0, st>>>(wav, n, h->window, fh, fl, F, B, n_fft, h->d.hop_length);
  CK(cudaGetLastError());
  h->launches++;
  au_gemm(h, fh, fl, B * F, n_fft, h->wf_h, h->wf_l, h->NP, spec, st);
}

// spectrum planes [F][NP] -> waveform [hop (F - 1)]
void au_istft(avc_audio_handle* h, Arena& mem, const float* xh, const float* xl, int F, int B, float* tf, float* wav, cudaStream_t st) {
  const int n_fft = h->d.n_fft;
  (void)mem;
  au_gemm(h, xh, xl, B * F, h->NP, h->wi_h, h->wi_l, n_fft, tf, st);
  const long long n_out = (long long)h->d.hop_length * (F - 1);
  au_ola_kernel<<<au_grid(n_out * B, h->sm_count), 256, 0, st>>>(tf, h->window, wav, n_out, F, B, n_fft, h->d.hop_length);
  CK(cudaGetLastError());
  h->launches++;
}

}  // namespace

extern "C" {

int avc_audio_create(avc_audio_handle** out, const avc_audio_desc* d, int device) {
  if (!out) { g_audio_create_error = "null argument"; return AVC_ERR_INVALID; }
  *out = nullptr;
  return au_guarded(nullptr, [&] {
    if (!d) fail(AVC_ERR_INVALID, "null descriptor");
    if (d->n_fft < 64 || d->n_fft % 32 || d->n_fft > 8192 || d->win_length < 2 || d->win_length > d->n_fft || d->hop_length < 1 ||
        d->hop_length > d->n_fft || d->n_mels < 1 || d->n_mels > 1024 || d->sample_rate < 1 || !(d->max_db > 0.f))
      fail(AVC_ERR_INVALID, "unsupported audio parameters (n_fft a multiple of 32 in [64, 8192], win_length <= n_fft, hop_length <= n_fft)");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) fail(AVC_ERR_CUDA, "no CUDA device available (%s); libavc_b200 has no CPU fallback", cudaGetErrorString(e));
    if (device < 0 || device >= n) fail(AVC_ERR_INVALID, "device %d out of range (%d devices)", device, n);
    DeviceGuard dg(device);
    cudaDeviceProp p{};
    CK(cudaGetDeviceProperties(&p, device));
    if (p.major < 10) fail(AVC_ERR_CUDA, "device %d is sm_%d%d; libavc_b200 is built for sm_100a only", device, p.major, p.minor);
    auto h = std::make_unique<avc_audio_handle>();
    h->device = device; h->sm_count = p.multiProcessorCount; h->d = *d;
    const int N = d->n_fft, nbin = 1 + N / 2, NP = (2 * nbin + 3) / 4 * 4;
    h->nbin = nbin; h->NP = NP;
    c2_init_attributes();
    // periodic Hann of win_length, centred in n_fft (scipy get_window(fftbins=True) + librosa pad_center)
    std::vector<float> win(N, 0.f);
    const int lpad = (N - d->win_length) / 2;
    for (int i = 0; i < d->win_length; ++i) win[lpad + i] = (float)(0.5 - 0.5 * std::cos(2.0 * M_PI * i / d->win_length));
    h->window = h->wmem.upload(win);
    const std::vector<float> basis = au_mel_basis(d->sample_rate, N, d->n_mels);
    h->basis = h->wmem.upload(basis);
    {   // inv_mel_matrix (data_utils.py:16-31): m^T diag(1 / colsum(m m^T)), entries <= 1e-8 kept as they are
      std::vector<double> colsum(d->n_mels, 0.0);
      for (int i = 0; i < d->n_mels; ++i)
        for (int j = 0; j < d->n_mels; ++j) {
          double s = 0.0;
          for (int k = 0; k < nbin; ++k) s += (double)basis[(size_t)i * nbin + k] * basis[(size_t)j * nbin + k];
          colsum[j] += s;
        }
      std::vector<float> inv((size_t)nbin * d->n_mels);
      for (int k = 0; k < nbin; ++k)
        for (int m = 0; m < d->n_mels; ++m) {
          const double dm = std::fabs(colsum[m]) > 1e-8 ? 1.0 / colsum[m] : colsum[m];
          inv[(size_t)k * d->n_mels + m] = (float)(basis[(size_t)m * nbin + k] * dm);
        }
      h->inv = h->wmem.upload(inv);
    }
    // DFT matrices in fp64 with the angle reduced exactly ((k n) mod N), split into 3xTF32 planes
    auto split_upload = [&](const std::vector<float>& w, float*& hi, float*& lo) {
      std::vector<float> a(w.size()), b(w.size());
      for (size_t i = 0; i < w.size(); ++i) {
        uint32_t u;
        memcpy(&u, &w[i], 4);
        u = (u + 0x1000u) & 0xffffe000u;
        memcpy(&a[i], &u, 4);
        b[i] = w[i] - a[i];
      }
      hi = h->wmem.upload(a); lo = h->wmem.upload(b);
    };
    std::vector<float> wf((size_t)NP * N, 0.f), wi((size_t)N * NP, 0.f);
    for (int k = 0; k < nbin; ++k)
      for (int t = 0; t < N; ++t) {
        const double ang = 2.0 * M_PI * (double)(((long long)k * t) % N) / N;
        const double c = std::cos(ang), s = std::sin(ang);
        wf[(size_t)k * N + t] = (float)c;                       // re X_k =  sum x cos
        wf[(size_t)(nbin + k) * N + t] = (float)(-s);           // im X_k = -sum x sin
        const bool edge = k == 0 || k == N / 2;                 // numpy irfft: the imaginary parts of DC and Nyquist are ignored
        wi[(size_t)t * NP + k] = (float)((edge ? c : 2.0 * c) / N);
        wi[(size_t)t * NP + nbin + k] = (float)(edge ? 0.0 : -2.0 * s / N);
      }
    split_upload(wf, h->wf_h, h->wf_l);
    split_upload(wi, h->wi_h, h->wi_l);
    CK(cudaDeviceSynchronize());
    *out = h.release();
  });
}

void avc_audio_destroy(avc_audio_handle* h) {
  if (!h) return;
  DeviceGuard dg(h->device);
  cudaDeviceSynchronize();
  delete h;
}

const char* avc_audio_last_error(const avc_audio_handle* h) { return h ? h->err.c_str() : g_audio_create_error.c_str(); }
int64_t avc_audio_kernel_launches(const avc_audio_handle* h) { return h ? h->launches : -1; }
int32_t avc_audio_frames(const avc_audio_handle* h, int64_t n_samples) { return (h && n_samples > 0) ? (int32_t)(1 + n_samples / h->d.hop_length) : -1; }
int64_t avc_audio_samples(const avc_audio_handle* h, int32_t n_frames) { return (h && n_frames > 0) ? (int64_t)h->d.hop_length * (n_frames - 1) : -1; }

int avc_audio_wav2mel_batch(avc_audio_handle* h, const float* wav, int32_t B, int64_t n, float* mel, void* stream) {
  if (!h) return AVC_ERR_INVALID;
  return au_guarded(h, [&] {
    if (!wav || !mel || B < 1) fail(AVC_ERR_INVALID, "null tensor argument / bad batch");
    if (n <= h->d.n_fft / 2) fail(AVC_ERR_INVALID, "waveform of %lld samples is too short for reflect padding by n_fft / 2 = %d", (long long)n, h->d.n_fft / 2);
    cudaStream_t st = (cudaStream_t)stream;
    Arena mem(&h->pool, st);
    const int F = 1 + (int)(n / h->d.hop_length), R = B * F;
    float* pre = mem.f((size_t)n * B);
    au_preemph_kernel<<<au_grid(n * B, h->sm_count), 256, 0, st>>>(wav, pre, n, B, h->d.preemph);
    CK(cudaGetLastError());
    float* spec = mem.f((size_t)R * h->NP);
    au_stft(h, mem, pre, n, F, B, spec, st);
    float* mag = mem.f((size_t)R * h->nbin);
    au_mag_kernel<<<au_grid((long long)R * h->nbin, h->sm_count), 256, 0, st>>>(spec, mag, R, h->nbin, h->NP);
    CK(cudaGetLastError());
    const long long outs = (long long)R * h->d.n_mels;
    au_mel_kernel<<<(unsigned)((outs * 32 + 255) / 256), 256, 0, st>>>(mag, h->basis, mel, R, h->nbin, h->d.n_mels, h->d.ref_db, h->d.max_db,
                                                                      nullptr, nullptr);
    CK(cudaGetLastError());
    h->launches += 3;
    CK(cudaStreamSynchronize(st));
  });
}

int avc_audio_mel2wav_batch(avc_audio_handle* h, const float* mel, int32_t B, int32_t n_frames, int32_t n_iter, float* wav, void* stream) {
  if (!h) return AVC_ERR_INVALID;
  return au_guarded(h, [&] {
    if (!mel || !wav || B < 1) fail(AVC_ERR_INVALID, "null tensor argument / bad batch");
    if (n_frames < 2 || n_iter < 0) fail(AVC_ERR_INVALID, "bad n_frames / n_iter");
    const int F = n_frames, N = h->d.n_fft, R = B * F;
    const long long n_out = (long long)h->d.hop_length * (F - 1);
    if (n_out <= N / 2) fail(AVC_ERR_INVALID, "%d frames give %lld samples: too short for the STFT inside Griffin-Lim", F, n_out);
    cudaStream_t st = (cudaStream_t)stream;
    Arena mem(&h->pool, st);
    float* mag = mem.f((size_t)R * h->nbin);
    au_invmel_kernel<<<R, 256, h->d.n_mels * sizeof(float), st>>>(mel, h->inv, mag, R, h->nbin, h->d.n_mels, h->d.ref_db, h->d.max_db,
                                                                nullptr, nullptr);
    CK(cudaGetLastError());
    float* xh = mem.f((size_t)R * h->NP); float* xl = mem.f((size_t)R * h->NP);
    float* tf = mem.f((size_t)R * N);
    float* est = mem.f((size_t)R * h->NP);
    float* fh = mem.f((size_t)R * N); float* fl = mem.f((size_t)R * N);
    const unsigned gp = au_grid((long long)R * h->NP, h->sm_count);
    au_phase_kernel<<<gp, 256, 0, st>>>(mag, nullptr, xh, xl, R, h->nbin, h->NP);          // X_best = spect
    CK(cudaGetLastError());
    h->launches += 2;
    for (int it = 0; it < n_iter; ++it) {                                                   // data_utils.py:183-187
      au_istft(h, mem, xh, xl, F, B, tf, wav, st);
      au_frame_kernel<<<au_grid((long long)R * N, h->sm_count), 256, 0, st>>>(wav, n_out, h->window, fh, fl, F, B, N, h->d.hop_length);
      CK(cudaGetLastError());
      au_gemm(h, fh, fl, R, N, h->wf_h, h->wf_l, h->NP, est, st);
      au_phase_kernel<<<gp, 256, 0, st>>>(mag, est, xh, xl, R, h->nbin, h->NP);
      CK(cudaGetLastError());
      h->launches += 2;
    }
    au_istft(h, mem, xh, xl, F, B, tf, wav, st);                                            // :188-189
    au_deemph_kernel<<<(B + 31) / 32, 32, 0, st>>>(wav, n_out, B, h->d.preemph);            // :162
    CK(cudaGetLastError());
    h->launches++;
    CK(cudaStreamSynchronize(st));
  });
}

}  // extern "C"

namespace {

template <class T>
T* au_upload(Arena& mem, const std::vector<T>& v, cudaStream_t st) {
  T* p = mem.raw<T>(v.size());
  CK(cudaMemcpyAsync(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, st));
  return p;
}

// Offset table of a ragged batch on the device: sample offsets (B + 1), frame offsets (B + 1) and the utterance of every frame row
struct AuTable {
  long long* s_off = nullptr;
  int* f_off = nullptr;
  int* fu = nullptr;
};

AuTable au_table(Arena& mem, const std::vector<long long>& s_off, const std::vector<int>& f_off, cudaStream_t st) {
  const int B = (int)s_off.size() - 1;
  std::vector<int> fi(f_off);                      // [f_off (B + 1) | fu (R)]: one upload
  fi.reserve(fi.size() + f_off[B]);
  for (int u = 0; u < B; ++u) fi.insert(fi.end(), (size_t)(f_off[u + 1] - f_off[u]), u);
  AuTable t;
  t.s_off = au_upload(mem, s_off, st);
  t.f_off = au_upload(mem, fi, st);
  t.fu = t.f_off + B + 1;
  return t;
}

void au_check_norm(const float* mean, const float* std) {
  if ((mean == nullptr) != (std == nullptr)) fail(AVC_ERR_INVALID, "mean and std must both be given or both be NULL");
}

}  // namespace

extern "C" {

int avc_audio_wav2mel_varlen(avc_audio_handle* h, const float* wav, const int64_t* n_host, int32_t B, const float* mean, const float* std,
                             float* mel, void* stream) {
  if (!h) return AVC_ERR_INVALID;
  return au_guarded(h, [&] {
    if (!wav || !mel || !n_host || B < 1) fail(AVC_ERR_INVALID, "null tensor argument / bad batch");
    au_check_norm(mean, std);
    const int hop = h->d.hop_length;
    std::vector<long long> s_off(B + 1, 0);
    std::vector<int> f_off(B + 1, 0);
    for (int u = 0; u < B; ++u) {
      const long long n = n_host[u];
      if (n <= h->d.n_fft / 2)
        fail(AVC_ERR_INVALID, "utterance %d: waveform of %lld samples is too short for reflect padding by n_fft / 2 = %d", u, n, h->d.n_fft / 2);
      if ((long long)f_off[u] + 1 + n / hop > (1ll << 30)) fail(AVC_ERR_INVALID, "too many frames in one call");
      s_off[u + 1] = s_off[u] + n;
      f_off[u + 1] = f_off[u] + 1 + (int)(n / hop);
    }
    cudaStream_t st = (cudaStream_t)stream;
    Arena mem(&h->pool, st);
    const AuTable t = au_table(mem, s_off, f_off, st);
    const long long S = s_off[B];
    const int R = f_off[B], n_fft = h->d.n_fft;
    float* pre = mem.f((size_t)S);
    au_preemph_varlen_kernel<<<au_grid(S, h->sm_count), 256, 0, st>>>(wav, pre, t.s_off, B, h->d.preemph);
    CK(cudaGetLastError());
    float* fh = mem.f((size_t)R * n_fft); float* fl = mem.f((size_t)R * n_fft);
    au_frame_varlen_kernel<<<au_grid((long long)R * n_fft, h->sm_count), 256, 0, st>>>(pre, t.s_off, t.f_off, t.fu, h->window, fh, fl, R, n_fft, hop);
    CK(cudaGetLastError());
    float* spec = mem.f((size_t)R * h->NP);
    au_gemm(h, fh, fl, R, n_fft, h->wf_h, h->wf_l, h->NP, spec, st);
    float* mag = mem.f((size_t)R * h->nbin);
    au_mag_kernel<<<au_grid((long long)R * h->nbin, h->sm_count), 256, 0, st>>>(spec, mag, R, h->nbin, h->NP);
    CK(cudaGetLastError());
    const long long outs = (long long)R * h->d.n_mels;
    au_mel_kernel<<<(unsigned)((outs * 32 + 255) / 256), 256, 0, st>>>(mag, h->basis, mel, R, h->nbin, h->d.n_mels, h->d.ref_db, h->d.max_db,
                                                                      mean, std);
    CK(cudaGetLastError());
    h->launches += 4;
    CK(cudaStreamSynchronize(st));
  });
}

int avc_audio_mel2wav_varlen(avc_audio_handle* h, const float* mel, const int32_t* frames_host, int32_t B, int32_t n_iter, const float* mean,
                             const float* std, float* wav, void* stream) {
  if (!h) return AVC_ERR_INVALID;
  return au_guarded(h, [&] {
    if (!mel || !wav || !frames_host || B < 1) fail(AVC_ERR_INVALID, "null tensor argument / bad batch");
    if (n_iter < 0) fail(AVC_ERR_INVALID, "bad n_iter");
    au_check_norm(mean, std);
    const int N = h->d.n_fft, hop = h->d.hop_length;
    std::vector<long long> o_off(B + 1, 0);
    std::vector<int> f_off(B + 1, 0);
    for (int u = 0; u < B; ++u) {
      const int F = frames_host[u];
      if (F < 2) fail(AVC_ERR_INVALID, "utterance %d: bad n_frames %d", u, F);
      const long long n_out = (long long)hop * (F - 1);
      if (n_out <= N / 2) fail(AVC_ERR_INVALID, "utterance %d: %d frames give %lld samples: too short for the STFT inside Griffin-Lim", u, F, n_out);
      if ((long long)f_off[u] + F > (1ll << 30)) fail(AVC_ERR_INVALID, "too many frames in one call");
      o_off[u + 1] = o_off[u] + n_out;
      f_off[u + 1] = f_off[u] + F;
    }
    cudaStream_t st = (cudaStream_t)stream;
    Arena mem(&h->pool, st);
    const AuTable t = au_table(mem, o_off, f_off, st);
    const int R = f_off[B];
    float* mag = mem.f((size_t)R * h->nbin);
    au_invmel_kernel<<<R, 256, h->d.n_mels * sizeof(float), st>>>(mel, h->inv, mag, R, h->nbin, h->d.n_mels, h->d.ref_db, h->d.max_db, mean, std);
    CK(cudaGetLastError());
    float* xh = mem.f((size_t)R * h->NP); float* xl = mem.f((size_t)R * h->NP);
    float* tf = mem.f((size_t)R * N);
    float* est = mem.f((size_t)R * h->NP);
    float* fh = mem.f((size_t)R * N); float* fl = mem.f((size_t)R * N);
    const unsigned gp = au_grid((long long)R * h->NP, h->sm_count);
    const unsigned go = au_grid(o_off[B], h->sm_count), gf = au_grid((long long)R * N, h->sm_count);
    au_phase_kernel<<<gp, 256, 0, st>>>(mag, nullptr, xh, xl, R, h->nbin, h->NP);          // X_best = spect
    CK(cudaGetLastError());
    h->launches += 2;
    auto istft = [&] {
      au_gemm(h, xh, xl, R, h->NP, h->wi_h, h->wi_l, N, tf, st);
      au_ola_varlen_kernel<<<go, 256, 0, st>>>(tf, h->window, wav, t.s_off, t.f_off, B, N, hop);
      CK(cudaGetLastError());
      h->launches++;
    };
    for (int it = 0; it < n_iter; ++it) {                                                   // data_utils.py:183-187
      istft();
      au_frame_varlen_kernel<<<gf, 256, 0, st>>>(wav, t.s_off, t.f_off, t.fu, h->window, fh, fl, R, N, hop);
      CK(cudaGetLastError());
      au_gemm(h, fh, fl, R, N, h->wf_h, h->wf_l, h->NP, est, st);
      au_phase_kernel<<<gp, 256, 0, st>>>(mag, est, xh, xl, R, h->nbin, h->NP);
      CK(cudaGetLastError());
      h->launches += 2;
    }
    istft();                                                                                // :188-189
    au_deemph_varlen_kernel<<<(B + 31) / 32, 32, 0, st>>>(wav, t.s_off, B, h->d.preemph);   // :162
    CK(cudaGetLastError());
    h->launches++;
    CK(cudaStreamSynchronize(st));
  });
}

int avc_audio_wav2mel(avc_audio_handle* h, const float* wav, int64_t n, float* mel, void* stream) {
  return avc_audio_wav2mel_batch(h, wav, 1, n, mel, stream);
}
int avc_audio_mel2wav(avc_audio_handle* h, const float* mel, int32_t n_frames, int32_t n_iter, float* wav, void* stream) {
  return avc_audio_mel2wav_batch(h, mel, 1, n_frames, n_iter, wav, stream);
}

}  // extern "C"
