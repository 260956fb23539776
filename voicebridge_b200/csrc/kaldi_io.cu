// kaldi_io.cu — the wire / disk formats on either side of the hot path (SURVEY.md §8f n2), on memory buffers, so that the
// C ABI reads and writes exactly what the recipe scripts exchange through their temp files:
//   * matrices  "FM " / "DM " (matrix/kaldi-matrix.cc:1375-1460) and CompressedMatrix "CM " / "CM2 " / "CM3 "
//     (matrix/compressed-matrix.cc:371-377,490-500,531-612,617-670), vectors "FV " / "DV ", int32 vectors
//     (util/kaldi-holder-inl.h:230-243: alignments), archive entries "key \0B<object>" (util/kaldi-holder-inl.h, kaldi-table-inl.h);
//   * model files: TransitionModel (hmm/transition-model.cc:144-177,383-409, hmm/hmm-topology.cc:128-158) -> tid2pdf,
//     AmDiagGmm / DiagGmm blocks (gmm/am-diag-gmm.cc:147-176, gmm/diag-gmm.cc:705-756; gconsts recomputed as
//     DiagGmm::ComputeGconsts does, :114-152);
//   * statistics files as gmm-acc-stats-ali writes them: transition accs "DV " + AccumAmDiagGmm::Write
//     (gmm/mle-am-diag-gmm.cc:153-166, gmm/mle-diag-gmm.cc:77-103: doubles narrowed to float on write).
// A compressed feature matrix goes to the device as it is on disk (1 byte per element over PCIe) and is expanded by a
// kernel straight into the HBM feature buffer (vbgpu_io_matrix_to_device).
#include <algorithm>
#include <cmath>
#include <new>
#include <stdexcept>
#include <string>

#include "common.h"

namespace {

struct Reader {
  const uint8_t *p;
  int64_t n, pos = 0;
  bool ok = true;
  Reader(const void *buf, int64_t len) : p(static_cast<const uint8_t *>(buf)), n(len) {}
  bool need(int64_t k) {
    if (!ok || k < 0 || pos + k > n) ok = false;
    return ok;
  }
  int peek() { return (ok && pos < n) ? p[pos] : -1; }
  void skip_binary_marker() {  // "\0B" written by WriteKaldiObject / the table holders
    if (pos + 1 < n && p[pos] == 0 && p[pos + 1] == 'B') pos += 2;
  }
  std::string token() {  // ReadToken: characters up to (and consuming) one space
    std::string t;
    while (ok && pos < n && p[pos] != ' ' && p[pos] != '\n' && t.size() < 64) t.push_back((char)p[pos++]);
    if (pos >= n || (p[pos] != ' ' && p[pos] != '\n')) ok = false;
    else pos++;
    return t;
  }
  bool expect(const char *want) { return token() == want && ok ? true : (ok = false); }
  template <typename T>
  T basic() {  // ReadBasicType, binary: one size byte then the value
    T v = T();
    if (!need(1 + (int64_t)sizeof(T)) || p[pos] != sizeof(T)) return ok = false, v;
    std::memcpy(&v, p + pos + 1, sizeof(T));
    pos += 1 + sizeof(T);
    return v;
  }
  const uint8_t *raw(int64_t bytes) {
    if (!need(bytes)) return nullptr;
    const uint8_t *r = p + pos;
    pos += bytes;
    return r;
  }
};

struct Writer {  // counts past the capacity, so that a first call with cap = 0 sizes the buffer
  uint8_t *buf;
  int64_t cap, pos = 0;
  Writer(void *b, int64_t c) : buf(static_cast<uint8_t *>(b)), cap(b ? c : 0) {}
  void raw(const void *src, int64_t bytes) {
    if (pos + bytes <= cap) std::memcpy(buf + pos, src, (size_t)bytes);
    pos += bytes;
  }
  void token(const char *t) {
    raw(t, (int64_t)strlen(t));
    raw(" ", 1);
  }
  template <typename T>
  void basic(T v) {
    const char sz = (char)sizeof(T);
    raw(&sz, 1);
    raw(&v, sizeof(T));
  }
  void float_vector(const double *v, int32_t n) {  // Vector<BaseFloat>::Write of a narrowed copy
    token("FV");
    basic<int32_t>(n);
    for (int32_t i = 0; i < n; i++) {
      const float f = (float)v[i];
      raw(&f, 4);
    }
  }
  void float_matrix(const double *m, int32_t rows, int32_t cols) {
    token("FM");
    basic<int32_t>(rows);
    basic<int32_t>(cols);
    for (int64_t i = 0; i < (int64_t)rows * cols; i++) {
      const float f = (float)m[i];
      raw(&f, 4);
    }
  }
};

enum { kFM = 1, kDM = 2, kCM = 3, kCM2 = 4, kCM3 = 5, kFV = 6, kDV = 7, kIV = 8 };

// Parses the header of the object at the reader's position; leaves the reader at the payload.
bool object_header(Reader &r, vbgpu_io_info *info) {
  const int64_t start = r.pos;
  r.skip_binary_marker();
  std::memset(info, 0, sizeof(*info));
  const int c = r.peek();
  if (c == 4) {  // BasicVectorHolder<int32>::Write (kaldi-holder-inl.h:230-243): WriteBasicType(count), then one
                 // WriteBasicType per element, i.e. a size byte in front of every int32
    const int32_t cnt = r.basic<int32_t>();
    if (!r.ok || cnt < 0) return r.ok = false;
    info->kind = kIV, info->rows = 1, info->cols = cnt;
    info->header_bytes = r.pos - start;
    info->total_bytes = info->header_bytes + 5LL * cnt;
    return r.need(5LL * cnt);
  }
  const std::string t = r.token();
  if (!r.ok) return false;
  int64_t payload = 0;
  if (t == "FM" || t == "DM") {
    const int32_t rows = r.basic<int32_t>(), cols = r.basic<int32_t>();
    if (!r.ok || rows < 0 || cols < 0) return r.ok = false;
    info->kind = t == "FM" ? kFM : kDM, info->rows = rows, info->cols = cols;
    // sizes come from an untrusted header: rows * cols * elem must fit what is left of the buffer (checked by division, the
    // product of two int32 can wrap int64 once multiplied by the element size)
    if (cols > 0 && rows > (r.n - r.pos) / (t == "FM" ? 4 : 8) / cols) return r.ok = false;
    payload = (int64_t)rows * cols * (t == "FM" ? 4 : 8);
  } else if (t == "FV" || t == "DV") {
    const int32_t dim = r.basic<int32_t>();
    if (!r.ok || dim < 0) return r.ok = false;
    info->kind = t == "FV" ? kFV : kDV, info->rows = 1, info->cols = dim;
    payload = (int64_t)dim * (t == "FV" ? 4 : 8);
  } else if (t == "CM" || t == "CM2" || t == "CM3") {
    // GlobalHeader without its format word: min_value, range, num_rows, num_cols (compressed-matrix.cc:579-590)
    const uint8_t *h = r.raw(16);
    if (!h) return false;
    int32_t rows, cols;
    std::memcpy(&info->min_value, h, 4);
    std::memcpy(&info->range, h + 4, 4);
    std::memcpy(&rows, h + 8, 4);
    std::memcpy(&cols, h + 12, 4);
    if (rows < 0 || cols < 0) return r.ok = false;
    info->kind = t == "CM" ? kCM : (t == "CM2" ? kCM2 : kCM3), info->rows = rows, info->cols = cols;
    if (cols == 0) info->rows = rows = 0;  // "empty matrix": nothing follows the header
    if (cols > 0 && (int64_t)rows > (r.n - r.pos) / cols) return r.ok = false;  // (as above: no overflow on a corrupt header)
    payload = t == "CM" ? (int64_t)cols * (8 + rows) : (int64_t)rows * cols * (t == "CM2" ? 2 : 1);
  } else {
    return r.ok = false;
  }
  info->header_bytes = r.pos - start;
  info->total_bytes = info->header_bytes + payload;
  return r.need(payload);
}

// CompressedMatrix::Uint16ToFloat / CharToFloat / the linear formats: the reference's exact expressions (float products,
// double constants), with every rounding pinned on the device (no FMA contraction) so that host and device agree bit
// for bit with CompressedMatrix::CopyToMat.
__host__ __device__ inline float mul_add_f(float a, float b, float c) {  // (a * b) + c, two roundings
#ifdef __CUDA_ARCH__
  return __fadd_rn(__fmul_rn(a, b), c);
#else
  return a * b + c;
#endif
}
__host__ __device__ inline float u16_to_float(float min_value, float range, uint16_t v) {
  // min_value + range * 1.52590218966964e-05F * value   (compressed-matrix.cc:371-377)
#ifdef __CUDA_ARCH__
  return mul_add_f(__fmul_rn(range, 1.52590218966964e-05F), (float)v, min_value);
#else
  return mul_add_f(range * 1.52590218966964e-05F, (float)v, min_value);
#endif
}
__host__ __device__ inline float char_to_float(float p0, float p25, float p75, float p100, uint8_t v) {
  // p + (q - p) * k * (1/c.0): the float product (q - p) * k widened and scaled in double, added to p in double
  float base, diff, k;
  double scale;
  if (v <= 64) base = p0, diff = p25 - p0, k = (float)v, scale = 1 / 64.0;
  else if (v <= 192) base = p25, diff = p75 - p25, k = (float)(v - 64), scale = 1 / 128.0;
  else base = p75, diff = p100 - p75, k = (float)(v - 192), scale = 1 / 63.0;
#ifdef __CUDA_ARCH__
  return (float)__dadd_rn((double)base, __dmul_rn((double)__fmul_rn(diff, k), scale));
#else
  return (float)((double)base + (double)(diff * k) * scale);
#endif
}

void expand_host(const vbgpu_io_info &info, const uint8_t *payload, float *out, int32_t stride) {
  const int32_t R = info.rows, C = info.cols;
  switch (info.kind) {
    case kFM:
      for (int32_t i = 0; i < R; i++) std::memcpy(out + (size_t)i * stride, payload + (size_t)i * C * 4, (size_t)C * 4);
      break;
    case kDM:
      for (int32_t i = 0; i < R; i++)
        for (int32_t j = 0; j < C; j++) {
          double d;
          std::memcpy(&d, payload + ((size_t)i * C + j) * 8, 8);
          out[(size_t)i * stride + j] = (float)d;
        }
      break;
    case kCM: {
      const uint8_t *bytes = payload + (size_t)C * 8;
      for (int32_t j = 0; j < C; j++) {
        uint16_t q[4];
        std::memcpy(q, payload + (size_t)j * 8, 8);
        const float p0 = u16_to_float(info.min_value, info.range, q[0]), p25 = u16_to_float(info.min_value, info.range, q[1]),
                    p75 = u16_to_float(info.min_value, info.range, q[2]), p100 = u16_to_float(info.min_value, info.range, q[3]);
        for (int32_t i = 0; i < R; i++) out[(size_t)i * stride + j] = char_to_float(p0, p25, p75, p100, bytes[(size_t)j * R + i]);
      }
      break;
    }
    case kCM2: {
      const float inc = info.range * (1.0 / 65535.0);
      for (int32_t i = 0; i < R; i++)
        for (int32_t j = 0; j < C; j++) {
          uint16_t v;
          std::memcpy(&v, payload + ((size_t)i * C + j) * 2, 2);
          out[(size_t)i * stride + j] = mul_add_f((float)v, inc, info.min_value);
        }
      break;
    }
    case kCM3: {
      const float inc = info.range * (1.0 / 255.0);
      for (int32_t i = 0; i < R; i++)
        for (int32_t j = 0; j < C; j++) out[(size_t)i * stride + j] = mul_add_f((float)payload[(size_t)i * C + j], inc, info.min_value);
      break;
    }
    default: break;
  }
}

// ---- device-side expansion ------------------------------------------------------------------------------------------
// kCM: bytes are column-major [col][row]; a 32 x 32 tile is read along rows of the byte matrix (coalesced), transposed
// through shared memory and written along feature rows (coalesced).
__global__ void expand_cm_kernel(const uint8_t *__restrict__ payload, int32_t R, int32_t C, float min_value, float range,
                                 float *__restrict__ out, int32_t stride) {
  __shared__ float tile[32][33];
  const uint16_t *hdr = reinterpret_cast<const uint16_t *>(payload);
  const uint8_t *bytes = payload + (size_t)C * 8;
  const int r0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int k = threadIdx.y; k < 32; k += blockDim.y) {
    const int c = c0 + k, r = r0 + threadIdx.x;
    if (c < C && r < R) {
      const float p0 = u16_to_float(min_value, range, hdr[4 * c]), p25 = u16_to_float(min_value, range, hdr[4 * c + 1]),
                  p75 = u16_to_float(min_value, range, hdr[4 * c + 2]), p100 = u16_to_float(min_value, range, hdr[4 * c + 3]);
      tile[k][threadIdx.x] = char_to_float(p0, p25, p75, p100, bytes[(size_t)c * R + r]);
    }
  }
  __syncthreads();
  for (int k = threadIdx.y; k < 32; k += blockDim.y) {
    const int r = r0 + k, c = c0 + threadIdx.x;
    if (r < R && c < C) out[(size_t)r * stride + c] = tile[threadIdx.x][k];
  }
}
template <typename T>
__global__ void expand_linear_kernel(const T *__restrict__ v, int32_t R, int32_t C, float min_value, float inc,
                                     float *__restrict__ out, int32_t stride) {
  const int64_t total = (int64_t)R * C;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / C;
    out[r * stride + (i - r * C)] = mul_add_f((float)v[i], inc, min_value);
  }
}
__global__ void narrow_kernel(const double *__restrict__ v, int32_t R, int32_t C, float *__restrict__ out, int32_t stride) {
  const int64_t total = (int64_t)R * C;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / C;
    out[r * stride + (i - r * C)] = (float)v[i];
  }
}

// ---- model files -----------------------------------------------------------------------------------------------------
struct Topo {
  std::vector<int32_t> phone2idx;
  std::vector<std::vector<std::vector<int32_t>>> entries;  // [entry][state] -> destination states of its transitions
  std::vector<std::vector<std::pair<int32_t, int32_t>>> pdf_classes;  // [entry][state] -> (forward, self-loop) pdf class
};
bool read_int_vector(Reader &r, std::vector<int32_t> *v) {
  if (!r.need(5) || r.p[r.pos] != 4) return r.ok = false;
  int32_t cnt;
  std::memcpy(&cnt, r.p + r.pos + 1, 4);
  r.pos += 5;
  if (cnt < 0 || !r.need(4LL * cnt)) return r.ok = false;
  v->resize(cnt);
  if (cnt) std::memcpy(v->data(), r.p + r.pos, 4 * (size_t)cnt);
  r.pos += 4LL * cnt;
  return true;
}
bool read_topology(Reader &r, Topo *t) {  // binary branch of HmmTopology::Read
  if (!r.expect("<Topology>")) return false;
  std::vector<int32_t> phones;
  if (!read_int_vector(r, &phones) || !read_int_vector(r, &t->phone2idx)) return false;
  int32_t sz = r.basic<int32_t>();
  bool is_hmm = true;
  if (sz == -1) is_hmm = false, sz = r.basic<int32_t>();
  if (!r.ok || sz < 0 || sz > 100000) return r.ok = false;
  t->entries.resize(sz);
  t->pdf_classes.resize(sz);
  for (int32_t i = 0; i < sz && r.ok; i++) {
    const int32_t ns = r.basic<int32_t>();
    if (!r.ok || ns < 0 || ns > 100000) return r.ok = false;
    t->entries[i].resize(ns);
    t->pdf_classes[i].resize(ns);
    for (int32_t j = 0; j < ns && r.ok; j++) {
      const int32_t fwd = r.basic<int32_t>();
      t->pdf_classes[i][j] = {fwd, is_hmm ? fwd : r.basic<int32_t>()};
      const int32_t nt = r.basic<int32_t>();
      if (!r.ok || nt < 0 || nt > 100000) return r.ok = false;
      for (int32_t k = 0; k < nt && r.ok; k++) {
        t->entries[i][j].push_back(r.basic<int32_t>());
        r.basic<float>();
      }
    }
  }
  return r.expect("</Topology>");
}
// TransitionModel::Read + ComputeDerived: tid2pdf[0] = -1 (transition-ids are 1-based), log_probs as stored; the topology
// and the (phone, hmm-state) of every transition state (tuples[ts - 1]) for callers that want them.
bool read_transition_model(Reader &r, std::vector<int32_t> *tid2pdf, std::vector<float> *log_probs, Topo &topo,
                           std::vector<std::pair<int32_t, int32_t>> *tuples) {
  if (!r.expect("<TransitionModel>") || !read_topology(r, &topo)) return false;
  const std::string tok = r.token();
  if (!r.ok || (tok != "<Triples>" && tok != "<Tuples>")) return r.ok = false;
  const int32_t n = r.basic<int32_t>();
  if (!r.ok || n < 0) return r.ok = false;
  tid2pdf->assign(1, -1);
  for (int32_t i = 0; i < n && r.ok; i++) {
    const int32_t phone = r.basic<int32_t>(), state = r.basic<int32_t>(), fwd = r.basic<int32_t>();
    const int32_t self = tok == "<Tuples>" ? r.basic<int32_t>() : fwd;
    if (!r.ok || phone < 0 || phone >= (int32_t)topo.phone2idx.size()) return r.ok = false;
    const int32_t e = topo.phone2idx[phone];
    if (e < 0 || e >= (int32_t)topo.entries.size() || state < 0 || state >= (int32_t)topo.entries[e].size())
      return r.ok = false;
    for (int32_t dst : topo.entries[e][state]) tid2pdf->push_back(dst == state ? self : fwd);  // IsSelfLoop
    tuples->emplace_back(phone, state);
  }
  const std::string end = r.token();
  if (!r.ok || (end != "</Triples>" && end != "</Tuples>")) return r.ok = false;
  if (!r.expect("<LogProbs>") || !r.expect("FV")) return false;
  const int32_t dim = r.basic<int32_t>();
  if (!r.ok || dim != (int32_t)tid2pdf->size()) return r.ok = false;
  const uint8_t *lp = r.raw(4LL * dim);
  if (!lp) return false;
  log_probs->resize(dim);
  std::memcpy(log_probs->data(), lp, 4 * (size_t)dim);
  return r.expect("</LogProbs>") && r.expect("</TransitionModel>");
}
bool read_float_vector(Reader &r, std::vector<float> *v) {
  const std::string t = r.token();
  if (!r.ok || (t != "FV" && t != "DV")) return r.ok = false;
  const int32_t dim = r.basic<int32_t>();
  if (!r.ok || dim < 0) return r.ok = false;
  const int es = t == "FV" ? 4 : 8;
  const uint8_t *d = r.raw((int64_t)dim * es);
  if (!d) return false;
  v->resize(dim);
  for (int32_t i = 0; i < dim; i++) {
    if (es == 4) std::memcpy(&(*v)[i], d + 4 * (size_t)i, 4);
    else {
      double x;
      std::memcpy(&x, d + 8 * (size_t)i, 8);
      (*v)[i] = (float)x;
    }
  }
  return true;
}
bool read_float_matrix(Reader &r, std::vector<float> *m, int32_t *rows, int32_t *cols) {
  vbgpu_io_info info;
  const int64_t at = r.pos;
  if (!object_header(r, &info) || (info.kind != kFM && info.kind != kDM)) return r.ok = false;
  *rows = info.rows, *cols = info.cols;
  m->resize((size_t)info.rows * info.cols);
  expand_host(info, r.p + at + info.header_bytes, m->data(), info.cols);
  r.pos = at + info.total_bytes;
  return true;
}
struct Mdl {
  int32_t D = 0, P = 0;
  std::vector<int32_t> pdf_offsets, tid2pdf;
  std::vector<float> weights, miv, iv, log_probs;
};
bool read_mdl(Reader &r, Mdl *m) {
  r.skip_binary_marker();
  if (r.peek() == '<') {  // a model file starts with the TransitionModel; a bare AmDiagGmm starts with <DIMENSION>
    const int64_t at = r.pos;
    const std::string t = r.token();
    r.pos = at;
    Topo topo;
    std::vector<std::pair<int32_t, int32_t>> tuples;
    if (t == "<TransitionModel>" && !read_transition_model(r, &m->tid2pdf, &m->log_probs, topo, &tuples)) return false;
  }
  if (!r.expect("<DIMENSION>")) return false;
  m->D = r.basic<int32_t>();
  if (!r.expect("<NUMPDFS>")) return false;
  m->P = r.basic<int32_t>();
  if (!r.ok || m->D <= 0 || m->P <= 0) return r.ok = false;
  m->pdf_offsets.assign(1, 0);
  for (int32_t p = 0; p < m->P && r.ok; p++) {
    std::string t = r.token();
    if (t != "<DiagGMM>" && t != "<DiagGMMBegin>") return r.ok = false;
    t = r.token();
    std::vector<float> w, tmp;
    if (t == "<GCONSTS>") {  // optional, and not trusted: DiagGmm::Read recomputes them
      if (!read_float_vector(r, &tmp) || !r.expect("<WEIGHTS>")) return false;
    } else if (t != "<WEIGHTS>") {
      return r.ok = false;
    }
    if (!read_float_vector(r, &w)) return false;
    int32_t r1, c1, r2, c2;
    std::vector<float> a, b;
    if (!r.expect("<MEANS_INVVARS>") || !read_float_matrix(r, &a, &r1, &c1)) return false;
    if (!r.expect("<INV_VARS>") || !read_float_matrix(r, &b, &r2, &c2)) return false;
    t = r.token();
    if (t != "</DiagGMM>" && t != "<DiagGMMEnd>") return r.ok = false;
    if (r1 != (int32_t)w.size() || r2 != r1 || c1 != m->D || c2 != m->D || r1 <= 0) return r.ok = false;
    m->weights.insert(m->weights.end(), w.begin(), w.end());
    m->miv.insert(m->miv.end(), a.begin(), a.end());
    m->iv.insert(m->iv.end(), b.begin(), b.end());
    m->pdf_offsets.push_back(m->pdf_offsets.back() + r1);
  }
  return r.ok;
}

}  // namespace

using vb::fail;

extern "C" {

int vbgpu_io_object_info(const void *buf, int64_t n, vbgpu_io_info *info) {
  VB_CHECK(buf && info && n >= 0, "bad argument");
  Reader r(buf, n);
  if (!object_header(r, info)) return fail(VBGPU_ERR_INVALID, "not a Kaldi binary matrix / vector object (or truncated)");
  return 0;
}

int vbgpu_io_read_matrix(const void *buf, int64_t n, float *out, int32_t out_stride) {
  VB_CHECK(buf && n >= 0, "bad argument");
  Reader r(buf, n);
  vbgpu_io_info info;
  if (!object_header(r, &info)) return fail(VBGPU_ERR_INVALID, "not a Kaldi binary matrix object (or truncated)");
  VB_CHECK(info.kind >= kFM && info.kind <= kCM3, "object is not a matrix");
  VB_CHECK(out_stride >= info.cols, "out_stride %d < cols %d", out_stride, info.cols);
  if (info.rows == 0 || info.cols == 0) return 0;
  VB_CHECK(out, "null output");
  expand_host(info, static_cast<const uint8_t *>(buf) + info.header_bytes, out, out_stride);
  return 0;
}

int vbgpu_io_read_vector(const void *buf, int64_t n, double *out) {
  VB_CHECK(buf && n >= 0, "bad argument");
  Reader r(buf, n);
  vbgpu_io_info info;
  if (!object_header(r, &info) || (info.kind != kFV && info.kind != kDV)) return fail(VBGPU_ERR_INVALID, "not a Kaldi binary vector");
  VB_CHECK(out || info.cols == 0, "null output");
  const uint8_t *d = static_cast<const uint8_t *>(buf) + info.header_bytes;
  for (int32_t i = 0; i < info.cols; i++) {
    if (info.kind == kFV) {
      float f;
      std::memcpy(&f, d + 4 * (size_t)i, 4);
      out[i] = f;
    } else {
      std::memcpy(&out[i], d + 8 * (size_t)i, 8);
    }
  }
  return 0;
}

int vbgpu_io_read_int32_vector(const void *buf, int64_t n, int32_t *out, int32_t cap) {
  VB_CHECK(buf && n >= 0, "bad argument");
  Reader r(buf, n);
  vbgpu_io_info info;
  if (!object_header(r, &info) || info.kind != kIV) return fail(VBGPU_ERR_INVALID, "not a Kaldi binary int32 vector");
  VB_CHECK(cap >= info.cols, "capacity %d < %d elements", cap, info.cols);
  const uint8_t *d = static_cast<const uint8_t *>(buf) + info.header_bytes;
  for (int32_t i = 0; i < info.cols; i++) {
    if (d[5 * (size_t)i] != 4) return fail(VBGPU_ERR_INVALID, "element %d of the int32 vector has size byte %d", i, d[5 * (size_t)i]);
    std::memcpy(&out[i], d + 5 * (size_t)i + 1, 4);
  }
  return info.cols;
}

int64_t vbgpu_io_write_matrix(const float *data, int32_t rows, int32_t cols, int32_t stride, void *buf, int64_t cap) {
  if (rows < 0 || cols < 0 || stride < cols || (!data && rows * cols > 0)) return fail(VBGPU_ERR_INVALID, "bad argument");
  Writer w(buf, cap);
  w.raw("\0B", 2);
  w.token("FM");
  w.basic<int32_t>(rows);
  w.basic<int32_t>(cols);
  for (int32_t i = 0; i < rows; i++) w.raw(data + (size_t)i * stride, 4LL * cols);
  return w.pos;
}

int64_t vbgpu_io_write_int32_vector(const int32_t *data, int32_t count, void *buf, int64_t cap) {
  if (count < 0 || (!data && count > 0)) return fail(VBGPU_ERR_INVALID, "bad argument");
  Writer w(buf, cap);
  w.raw("\0B", 2);
  w.basic<int32_t>(count);
  for (int32_t i = 0; i < count; i++) w.basic<int32_t>(data[i]);
  return w.pos;
}

int vbgpu_io_ark_next(const void *buf, int64_t n, int64_t pos, char *key, int32_t key_cap, int64_t *obj_pos,
                      int64_t *next_pos, vbgpu_io_info *info) {
  VB_CHECK(buf && key && key_cap > 0 && obj_pos && next_pos && info && pos >= 0, "bad argument");
  const uint8_t *p = static_cast<const uint8_t *>(buf);
  if (pos >= n) return 1;  // end of archive
  int64_t e = pos;
  while (e < n && p[e] != ' ') e++;
  if (e >= n || e == pos) return fail(VBGPU_ERR_INVALID, "archive entry at byte %lld has no key", (long long)pos);
  VB_CHECK(e - pos < key_cap, "key longer than %d bytes", key_cap - 1);
  std::memcpy(key, p + pos, (size_t)(e - pos));
  key[e - pos] = 0;
  Reader r(p + e + 1, n - e - 1);
  if (!(r.n >= 2 && p[e + 1] == 0 && p[e + 2] == 'B'))
    return fail(VBGPU_ERR_INVALID, "archive entry '%s' is not binary (no \\0B marker)", key);
  if (!object_header(r, info)) return fail(VBGPU_ERR_INVALID, "archive entry '%s': unknown or truncated object", key);
  *obj_pos = e + 1;
  *next_pos = e + 1 + info->total_bytes;
  return 0;
}

int vbgpu_io_mdl_info(const void *buf, int64_t n, int32_t *dim, int32_t *num_pdfs, int32_t *num_gauss, int32_t *num_tids) {
  VB_CHECK(buf && n >= 0, "bad argument");
  Reader r(buf, n);
  Mdl m;
  try {  // no exception crosses the C ABI: a corrupt file that asks for absurd sizes ends as an error code
    if (!read_mdl(r, &m)) return fail(VBGPU_ERR_INVALID, "not a binary Kaldi GMM model (TransitionModel + AmDiagGmm, or AmDiagGmm)");
  } catch (const std::bad_alloc &) {
    return fail(VBGPU_ERR_NOMEM, "out of memory while parsing the model");
  } catch (const std::exception &e) {
    return fail(VBGPU_ERR_INVALID, "model parse failed: %s", e.what());
  }
  if (dim) *dim = m.D;
  if (num_pdfs) *num_pdfs = m.P;
  if (num_gauss) *num_gauss = m.pdf_offsets.back();
  if (num_tids) *num_tids = m.tid2pdf.empty() ? 0 : (int32_t)m.tid2pdf.size() - 1;
  return 0;
}

int vbgpu_io_mdl_transitions(const void *buf, int64_t n, int32_t *phone, int32_t *hmm_state, int32_t *pdf_class,
                             int32_t *trans_state, int32_t *flags) {
  VB_CHECK(buf && n >= 0, "bad argument");
  Reader r(buf, n);
  Topo topo;
  std::vector<std::pair<int32_t, int32_t>> tuples;
  std::vector<int32_t> tid2pdf;
  std::vector<float> log_probs;
  try {
    r.skip_binary_marker();
    if (!read_transition_model(r, &tid2pdf, &log_probs, topo, &tuples))
      return fail(VBGPU_ERR_INVALID, "not a binary Kaldi model file starting with a TransitionModel");
  } catch (const std::bad_alloc &) {
    return fail(VBGPU_ERR_NOMEM, "out of memory while parsing the model");
  } catch (const std::exception &e) {
    return fail(VBGPU_ERR_INVALID, "model parse failed: %s", e.what());
  }
  // TransitionModel::TransitionIdToPdfClass / IsSelfLoop / IsFinal, and the check SplitToPhones makes on a phone's first
  // frame (state 0 of its topology entry emitting)
  int32_t tid = 0;
  auto put = [](int32_t *a, int32_t i, int32_t v) {
    if (a) a[i] = v;
  };
  put(phone, 0, 0), put(hmm_state, 0, 0), put(pdf_class, 0, 0), put(trans_state, 0, 0), put(flags, 0, 0);
  for (size_t ts = 0; ts < tuples.size(); ts++) {
    const int32_t ph = tuples[ts].first, st = tuples[ts].second, e = topo.phone2idx[ph];
    const auto &entry = topo.entries[e];
    const auto &pc = topo.pdf_classes[e][st];
    const int32_t emit0 = topo.pdf_classes[e][0].first != -1 ? VBGPU_TID_STATE0_EMITTING : 0;
    for (int32_t dst : entry[st]) {
      tid++;
      const bool self = dst == st;
      put(phone, tid, ph), put(hmm_state, tid, st), put(pdf_class, tid, self ? pc.second : pc.first);
      put(trans_state, tid, (int32_t)ts + 1);
      put(flags, tid, (self ? VBGPU_TID_SELF_LOOP : 0) | (dst + 1 == (int32_t)entry.size() ? VBGPU_TID_FINAL : 0) | emit0);
    }
  }
  return tid;
}

int vbgpu_io_mdl_read(const void *buf, int64_t n, int32_t *pdf_offsets, float *gconsts, float *weights, float *means_invvars,
                      float *inv_vars, int32_t *tid2pdf, float *trans_log_probs) {
  VB_CHECK(buf && n >= 0, "bad argument");
  Reader r(buf, n);
  Mdl m;
  try {
    if (!read_mdl(r, &m)) return fail(VBGPU_ERR_INVALID, "not a binary Kaldi GMM model");
  } catch (const std::bad_alloc &) {
    return fail(VBGPU_ERR_NOMEM, "out of memory while parsing the model");
  } catch (const std::exception &e) {
    return fail(VBGPU_ERR_INVALID, "model parse failed: %s", e.what());
  }
  const int32_t N = m.pdf_offsets.back(), D = m.D;
  if (pdf_offsets) std::memcpy(pdf_offsets, m.pdf_offsets.data(), 4 * (size_t)(m.P + 1));
  if (weights) std::memcpy(weights, m.weights.data(), 4 * (size_t)N);
  if (means_invvars) std::memcpy(means_invvars, m.miv.data(), 4 * (size_t)N * D);
  if (inv_vars) std::memcpy(inv_vars, m.iv.data(), 4 * (size_t)N * D);
  if (tid2pdf && !m.tid2pdf.empty()) std::memcpy(tid2pdf, m.tid2pdf.data(), 4 * m.tid2pdf.size());
  if (trans_log_probs && !m.log_probs.empty()) std::memcpy(trans_log_probs, m.log_probs.data(), 4 * m.log_probs.size());
  int bad = 0;
  if (gconsts) {  // DiagGmm::ComputeGconsts (diag-gmm.cc:114-152): the right-hand side in double, += rounds to float
    const float offset = (float)(-0.5 * 1.8378770664093454835606594728112 * D);
    for (int32_t g = 0; g < N; g++) {
      if (m.weights[g] < 0.0f) return fail(VBGPU_ERR_INVALID, "negative weight at Gaussian %d", g);
      float gc = logf(m.weights[g]) + offset;
      for (int32_t d = 0; d < D; d++) {
        const float a = m.iv[(size_t)g * D + d], b = m.miv[(size_t)g * D + d];
        gc = (float)(gc + (0.5 * logf(a) - 0.5 * b * b / a));
      }
      if (std::isnan(gc)) return fail(VBGPU_ERR_NUMERIC, "at component %d, not a number in gconst computation", g);
      if (std::isinf(gc)) {
        bad++;
        if (gc > 0) gc = -gc;
      }
      gconsts[g] = gc;
    }
  }
  return bad;
}

int64_t vbgpu_io_write_acc(int32_t num_pdfs, int32_t dim, const int32_t *pdf_offsets, const double *trans_accs,
                           int32_t n_trans, const double *occ, const double *mean_acc, const double *var_acc,
                           double tot_like, double tot_frames, void *buf, int64_t cap) {
  if (num_pdfs <= 0 || dim <= 0 || !pdf_offsets || !occ || !mean_acc || !var_acc || n_trans < 0 || (n_trans && !trans_accs))
    return fail(VBGPU_ERR_INVALID, "bad argument");
  Writer w(buf, cap);
  w.raw("\0B", 2);
  if (n_trans) {  // transition_accs.Write (Vector<double>), gmm-acc-stats-ali.cpp:124-126
    w.token("DV");
    w.basic<int32_t>(n_trans);
    w.raw(trans_accs, 8LL * n_trans);
  }
  w.token("<NUMPDFS>");
  w.basic<int32_t>(num_pdfs);
  for (int32_t p = 0; p < num_pdfs; p++) {
    const int32_t g0 = pdf_offsets[p], M = pdf_offsets[p + 1] - g0;
    w.token("<GMMACCS>");
    w.token("<VECSIZE>");
    w.basic<int32_t>(dim);
    w.token("<NUMCOMPONENTS>");
    w.basic<int32_t>(M);
    w.token("<FLAGS>");
    {  // GmmFlagsType is uint16: WriteBasicType marks unsigned integers with a NEGATIVE size byte (io-funcs-inl.h:38-40)
      const char sz = -2;
      const uint16_t flags = 0x00F;  // kGmmAll
      w.raw(&sz, 1);
      w.raw(&flags, 2);
    }
    w.token("<OCCUPANCY>");
    w.float_vector(occ + g0, M);
    w.token("<MEANACCS>");
    w.float_matrix(mean_acc + (size_t)g0 * dim, M, dim);
    w.token("<DIAGVARACCS>");
    w.float_matrix(var_acc + (size_t)g0 * dim, M, dim);
    w.token("</GMMACCS>");
  }
  w.token("<total_like>");
  w.basic<double>(tot_like);
  w.token("<total_frames>");
  w.basic<double>(tot_frames);
  return w.pos;
}

int vbgpu_io_matrix_to_device(const void *buf, int64_t n, float *d_out, int32_t out_stride, void *d_scratch,
                              int64_t scratch_bytes, void *stream) {
  VB_CHECK(buf && n >= 0, "bad argument");
  Reader r(buf, n);
  vbgpu_io_info info;
  if (!object_header(r, &info)) return fail(VBGPU_ERR_INVALID, "not a Kaldi binary matrix object (or truncated)");
  VB_CHECK(info.kind >= kFM && info.kind <= kCM3, "object is not a matrix");
  VB_CHECK(out_stride >= info.cols, "out_stride %d < cols %d", out_stride, info.cols);
  if (info.rows == 0 || info.cols == 0) return 0;
  VB_CHECK(d_out, "null output");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const uint8_t *payload = static_cast<const uint8_t *>(buf) + info.header_bytes;
  const int64_t pay_bytes = info.total_bytes - info.header_bytes;
  if (info.kind == kFM) {  // plain rows: one strided copy
    VB_CUDA(cudaMemcpy2DAsync(d_out, (size_t)out_stride * 4, payload, (size_t)info.cols * 4, (size_t)info.cols * 4,
                              (size_t)info.rows, cudaMemcpyHostToDevice, s));
    return 0;
  }
  VB_CHECK(d_scratch && scratch_bytes >= pay_bytes, "scratch of %lld bytes needed for the packed payload", (long long)pay_bytes);
  VB_CUDA(cudaMemcpyAsync(d_scratch, payload, (size_t)pay_bytes, cudaMemcpyHostToDevice, s));
  const int64_t total = (int64_t)info.rows * info.cols;
  const int grid = (int)std::min<int64_t>((total + 255) / 256, 148 * 8);
  switch (info.kind) {
    case kCM: {
      dim3 g((info.rows + 31) / 32, (info.cols + 31) / 32);
      expand_cm_kernel<<<g, dim3(32, 8), 0, s>>>(static_cast<const uint8_t *>(d_scratch), info.rows, info.cols, info.min_value,
                                                 info.range, d_out, out_stride);
      break;
    }
    case kCM2:
      expand_linear_kernel<uint16_t><<<grid, 256, 0, s>>>(static_cast<const uint16_t *>(d_scratch), info.rows, info.cols,
                                                          info.min_value, info.range * (1.0 / 65535.0), d_out, out_stride);
      break;
    case kCM3:
      expand_linear_kernel<uint8_t><<<grid, 256, 0, s>>>(static_cast<const uint8_t *>(d_scratch), info.rows, info.cols,
                                                         info.min_value, info.range * (1.0 / 255.0), d_out, out_stride);
      break;
    default:
      narrow_kernel<<<grid, 256, 0, s>>>(static_cast<const double *>(d_scratch), info.rows, info.cols, d_out, out_stride);
  }
  VB_CUDA(cudaGetLastError());
  return 0;
}

}  // extern "C"
