// wave.cu — RIFF/RIFX 16-bit PCM container parsing: the host-side I/O step in front of the path (WaveInfo::Read /
// WaveData::Read, feat/wave-reader.cc:119-310).  Pure byte handling on an in-memory file image, no device work: the
// samples stay int16 (the reference widens them to float without rescaling, wave-reader.cc:302-309; the MFCC kernel does
// that widening on the device).  The second half of the file is DownsampleWaveForm (feat/resample.cc:368-376) on the device.
// The parser accepts what the reference accepts: PCM (format 1) and WAVE_FORMAT_EXTENSIBLE with the
// PCM sub-format, 16 bits per sample, any number of channels, chunks between "fmt " and "data" skipped, "stream mode"
// sizes (0, 0xFFFFFFFF, SoX's 0x7FFFF000) meaning "data runs to the end of the image", a truncated data chunk.
#include "common.h"

namespace {

struct Cursor {
  const uint8_t *p;
  size_t n, pos;
  bool swap, ok;
  void tag(char *t) {
    if (pos + 4 > n) {
      ok = false;
      t[0] = 0;
      return;
    }
    std::memcpy(t, p + pos, 4);
    t[4] = 0;
    pos += 4;
  }
  uint32_t u32() {
    if (pos + 4 > n) {
      ok = false;
      return 0;
    }
    const uint8_t *b = p + pos;
    pos += 4;
    return swap ? ((uint32_t)b[0] << 24 | (uint32_t)b[1] << 16 | (uint32_t)b[2] << 8 | b[3])
                : ((uint32_t)b[3] << 24 | (uint32_t)b[2] << 16 | (uint32_t)b[1] << 8 | b[0]);
  }
  uint16_t u16() {
    if (pos + 2 > n) {
      ok = false;
      return 0;
    }
    const uint8_t *b = p + pos;
    pos += 2;
    return swap ? (uint16_t)(b[0] << 8 | b[1]) : (uint16_t)(b[1] << 8 | b[0]);
  }
};

}  // namespace

using vb::fail;

extern "C" {

int vbgpu_wave_parse(const void *bytes, size_t n_bytes, vbgpu_wave_info *info) {
  VB_CHECK(bytes && info, "null argument");
  std::memset(info, 0, sizeof(*info));
  Cursor c{static_cast<const uint8_t *>(bytes), n_bytes, 0, false, true};
  char t[5];
  c.tag(t);
  if (std::strcmp(t, "RIFF") == 0) c.swap = false;
  else if (std::strcmp(t, "RIFX") == 0) c.swap = true;
  else return fail(VBGPU_ERR_INVALID, "WaveData: expected RIFF or RIFX, got %s", t);
  const uint32_t riff_size = c.u32();
  c.tag(t);
  VB_CHECK(c.ok && std::strcmp(t, "WAVE") == 0, "WaveData: expected WAVE, got %s", t);
  c.tag(t);
  VB_CHECK(c.ok && std::strcmp(t, "fmt ") == 0, "WaveData: expected fmt chunk, got %s", t);
  const uint32_t fmt_size = c.u32();
  const uint16_t format = c.u16(), channels = c.u16();
  const uint32_t rate = c.u32(), byte_rate = c.u32();
  const uint16_t block_align = c.u16(), bits = c.u16();
  VB_CHECK(c.ok, "WaveData: unexpected end of file or read error");
  uint32_t fmt_read = 16;
  if (format == 1) {
    VB_CHECK(fmt_size >= 16, "WaveData: expect PCM format data to have fmt chunk of at least size 16.");
  } else if (format == 0xFFFE) {  // WAVE_FORMAT_EXTENSIBLE, PCM sub-format only (wave-reader.cc:150-172)
    const uint16_t extra = c.u16();
    VB_CHECK(c.ok && fmt_size >= 40 && extra >= 22, "WaveData: malformed WAVE_FORMAT_EXTENSIBLE format data.");
    c.u16();
    c.u32();
    const uint32_t g1 = c.u32(), g2 = c.u32(), g3 = c.u32(), g4 = c.u32();
    fmt_read = 40;
    VB_CHECK(c.ok && g1 == 0x00000001u && g2 == 0x00100000u && g3 == 0xAA000080u && g4 == 0x719B3800u,
             "WaveData: unsupported WAVE_FORMAT_EXTENSIBLE format.");
  } else {
    return fail(VBGPU_ERR_INVALID, "WaveData: can read only PCM data, format id in file is: %d", (int)format);
  }
  VB_CHECK(fmt_size >= fmt_read && c.pos + (fmt_size - fmt_read) <= c.n, "WaveData: unexpected end of file or read error");
  c.pos += fmt_size - fmt_read;
  VB_CHECK(channels != 0, "WaveData: no channels present");
  VB_CHECK(bits == 16, "WaveData: unsupported bits_per_sample = %d", (int)bits);
  VB_CHECK(byte_rate == rate * 2u * channels, "Unexpected byte rate %u vs. %u * 2 * %d", byte_rate, rate, (int)channels);
  VB_CHECK(block_align == channels * 2, "Unexpected block_align: %d vs. %d * 2", (int)block_align, (int)channels);
  c.tag(t);
  while (c.ok && std::strcmp(t, "data") != 0) {  // "fact", "LIST", ... are skipped (wave-reader.cc:196-210)
    const uint32_t sz = c.u32();
    VB_CHECK(c.ok && c.pos + sz <= c.n, "WaveData: unexpected end of file or read error");
    c.pos += sz;
    c.tag(t);
  }
  VB_CHECK(c.ok, "WaveData: unexpected end of file or read error");
  const uint32_t data_size = c.u32();
  VB_CHECK(c.ok, "WaveData: unexpected end of file or read error");
  const bool stream = riff_size == 0 || riff_size == 0xFFFFFFFFu || data_size == 0 || data_size == 0xFFFFFFFFu ||
                      data_size == 0x7FFFF000u;
  size_t avail = c.n - c.pos;
  if (!stream && data_size < avail) avail = data_size;  // a shorter image is a truncated file: keep what is there
  VB_CHECK(avail > 0, "WaveData: empty file (no data)");
  info->samp_freq = static_cast<float>(rate);
  info->num_channels = channels;
  info->num_samples = static_cast<int64_t>(avail / block_align);
  info->data_offset = static_cast<int64_t>(c.pos);
  info->reverse_bytes = c.swap ? 1 : 0;
  return 0;
}

int vbgpu_wave_channel_i16(const void *bytes, size_t n_bytes, const vbgpu_wave_info *info, int32_t channel, int16_t *out) {
  VB_CHECK(bytes && info && out, "null argument");
  if (channel < 0) channel = 0;  // compute-mfcc-feats --channel=-1: the first channel (compute-mfcc-feats.cpp:120-135)
  VB_CHECK(channel < info->num_channels, "File has %d channels; channel %d requested", info->num_channels, channel);
  VB_CHECK(info->data_offset >= 0 && (size_t)info->data_offset + (size_t)info->num_samples * info->num_channels * 2 <= n_bytes,
           "wave info does not match the image");
  const uint8_t *d = static_cast<const uint8_t *>(bytes) + info->data_offset + 2 * channel;
  const size_t step = 2 * (size_t)info->num_channels;
  for (int64_t i = 0; i < info->num_samples; i++, d += step)
    out[i] = info->reverse_bytes ? (int16_t)(uint16_t)(d[0] << 8 | d[1]) : (int16_t)(uint16_t)(d[1] << 8 | d[0]);
  return 0;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------------
// DownsampleWaveForm (feat/resample.cc:368-376): one flushed LinearResample::Resample call (resample.cc:34-160) with
// cutoff = 0.99 * new_freq / 2 and 6 zeros.  OfflineFeatureTpl::ComputeFeatures runs it when the wave's rate is above
// the options' and allow_downsample is set (feat/feature-common-inl.h:29-55).
// ---------------------------------------------------------------------------------------------------------------
struct vbgpu_resample_s {
  int device = 0;
  int32_t in_hz = 0, out_hz = 0, in_unit = 0, out_unit = 0, max_w = 0;
  vb::DevBuf d_first, d_nw, d_w, d_in, d_out;
  vb::Stream stream;
};

namespace {

int64_t gcd64(int64_t a, int64_t b) {
  while (b) {
    const int64_t t = a % b;
    a = b;
    b = t;
  }
  return a;
}

// LinearResample::FilterFunc (resample.cc:213-226): Hanning-windowed sinc
float filter_func(float t, float cutoff, int32_t num_zeros) {
  const double two_pi = 6.283185307179586476925286766559005, pi = 3.14159265358979323846;
  float window, filter;
  if (std::fabs(t) < num_zeros / (2.0 * cutoff)) window = (float)(0.5 * (1 + std::cos(two_pi * cutoff / num_zeros * t)));
  else window = 0.0f;
  if (t != 0) filter = (float)(std::sin(two_pi * cutoff * t) / (pi * t));
  else filter = (float)(2 * cutoff);
  return filter * window;
}

// out[i] = sum_k w[phase(i)][k] * in[first(i) + k] over the input indexes that exist (the flushed call assumes zeros past
// the end, resample.cc:141-157)
__global__ void __launch_bounds__(256) downsample_kernel(const float *__restrict__ in, int64_t n_in, float *__restrict__ out,
                                                         int64_t n_out, const int32_t *__restrict__ first,
                                                         const int32_t *__restrict__ nw, const float *__restrict__ w,
                                                         int32_t in_unit, int32_t out_unit, int32_t max_w) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_out; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t unit = i / out_unit;
    const int32_t ph = (int32_t)(i - unit * out_unit);
    const int64_t f = first[ph] + unit * in_unit;
    const int32_t n = nw[ph];
    const float *wp = w + (size_t)ph * max_w;
    float acc = 0.0f;
    for (int32_t k = 0; k < n; k++) {
      const int64_t idx = f + k;
      if (idx >= 0 && idx < n_in) acc = fmaf(__ldg(wp + k), __ldg(in + idx), acc);
    }
    out[i] = acc;
  }
}

}  // namespace

extern "C" {

int vbgpu_downsample_create(float orig_freq, float new_freq, int32_t device, vbgpu_resample_t *out) {
  VB_CHECK(out, "null argument");
  // the reference asserts new_freq < orig_freq (resample.cc:370); LinearResample takes the rates as int32
  VB_CHECK(new_freq < orig_freq && (int32_t)new_freq >= 1, "downsampling needs 1 <= new_freq (%g) < orig_freq (%g)", new_freq, orig_freq);
  VB_TRY(vb::check_device(device));
  vb::DeviceGuard g(device);
  std::unique_ptr<vbgpu_resample_s, decltype(&vbgpu_downsample_destroy)> h(new (std::nothrow) vbgpu_resample_s,
                                                                             vbgpu_downsample_destroy);
  if (!h) return fail(VBGPU_ERR_NOMEM, "out of host memory");
  h->device = device;
  h->in_hz = (int32_t)orig_freq;
  h->out_hz = (int32_t)new_freq;
  const float cutoff = (float)(0.99 * 0.5 * new_freq);
  const int32_t num_zeros = 6;
  const int32_t base = (int32_t)gcd64(h->in_hz, h->out_hz);
  h->in_unit = h->in_hz / base;
  h->out_unit = h->out_hz / base;
  const double window_width = num_zeros / (2.0 * cutoff);  // resample.cc:82-106
  std::vector<int32_t> first(h->out_unit), nw(h->out_unit);
  for (int32_t i = 0; i < h->out_unit; i++) {
    const double output_t = i / (double)h->out_hz, min_t = output_t - window_width, max_t = output_t + window_width;
    const int32_t lo = (int32_t)std::ceil(min_t * h->in_hz), hi = (int32_t)std::floor(max_t * h->in_hz);
    first[i] = lo;
    nw[i] = hi - lo + 1;
    h->max_w = std::max(h->max_w, nw[i]);
  }
  std::vector<float> w((size_t)h->out_unit * h->max_w, 0.0f);
  for (int32_t i = 0; i < h->out_unit; i++) {
    const double output_t = i / (double)h->out_hz;
    for (int32_t j = 0; j < nw[i]; j++) {
      const double input_t = (first[i] + j) / (double)h->in_hz, delta_t = input_t - output_t;
      w[(size_t)i * h->max_w + j] = filter_func((float)delta_t, cutoff, num_zeros) / h->in_hz;
    }
  }
  VB_TRY(h->d_first.upload(first.data(), first.size() * 4));
  VB_TRY(h->d_nw.upload(nw.data(), nw.size() * 4));
  VB_TRY(h->d_w.upload(w.data(), w.size() * 4));
  VB_TRY(h->stream.create());
  *out = h.release();
  return 0;
}

void vbgpu_downsample_destroy(vbgpu_resample_t h) {
  if (!h) return;
  vb::DeviceGuard g(h->device);
  cudaDeviceSynchronize();
  delete h;
}

// LinearResample::GetNumOutputSamples(n_in, flush = true) (resample.cc:57-80)
int64_t vbgpu_downsample_num_out(vbgpu_resample_t h, int64_t n_in) {
  if (!h || n_in < 0) return fail(VBGPU_ERR_INVALID, "bad argument");
  const int64_t tick_freq = (int64_t)h->in_hz / gcd64(h->in_hz, h->out_hz) * h->out_hz;
  const int64_t len = n_in * (tick_freq / h->in_hz);
  if (len <= 0) return 0;
  const int64_t ticks_per_out = tick_freq / h->out_hz;
  int64_t last = len / ticks_per_out;
  if (last * ticks_per_out == len) last--;
  return last + 1;
}

int vbgpu_downsample_dev(vbgpu_resample_t h, const float *d_wave, int64_t n_in, float *d_out, void *stream) {
  VB_CHECK(h && n_in >= 0, "bad argument");
  const int64_t n_out = vbgpu_downsample_num_out(h, n_in);
  if (n_out <= 0) return (int)n_out;
  VB_CHECK(d_wave && d_out, "null buffer");
  vb::DeviceGuard g(h->device);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const unsigned blocks = (unsigned)std::min<int64_t>((n_out + 255) / 256, 8LL * vb::num_sms(h->device));
  downsample_kernel<<<blocks, 256, 0, s>>>(d_wave, n_in, d_out, n_out, h->d_first.as<int32_t>(), h->d_nw.as<int32_t>(),
                                           h->d_w.as<float>(), h->in_unit, h->out_unit, h->max_w);
  VB_CUDA(cudaGetLastError());
  return 0;
}

int vbgpu_downsample_f32(vbgpu_resample_t h, const float *wave, int64_t n_in, float *out) {
  VB_CHECK(h && n_in >= 0, "bad argument");
  const int64_t n_out = vbgpu_downsample_num_out(h, n_in);
  if (n_out <= 0) return (int)n_out;
  VB_CHECK(wave && out, "null buffer");
  vb::DeviceGuard g(h->device);
  VB_TRY(h->d_in.reserve((size_t)n_in * 4));
  VB_TRY(h->d_out.reserve((size_t)n_out * 4));
  VB_CUDA(cudaMemcpyAsync(h->d_in.p, wave, (size_t)n_in * 4, cudaMemcpyHostToDevice, h->stream));
  VB_TRY(vbgpu_downsample_dev(h, h->d_in.as<float>(), n_in, h->d_out.as<float>(), h->stream));
  VB_CUDA(cudaMemcpyAsync(out, h->d_out.p, (size_t)n_out * 4, cudaMemcpyDeviceToHost, h->stream));
  VB_CUDA(cudaStreamSynchronize(h->stream));
  return 0;
}

}  // extern "C"

