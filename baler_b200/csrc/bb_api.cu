// C-ABI entry points (include/baler_b200.h): context, model packing, encode / decode dispatch and
// the host-buffer compress / decompress pipelines.
#include <algorithm>
#include <cstring>
#include <new>
#include <thread>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <pthread.h>
#if defined(__linux__)
#include <sched.h>
#endif
#if defined(__x86_64__) && defined(__GNUC__)
#include <immintrin.h>
#endif

#include <cstdlib>

#include "bb_common.cuh"

extern "C" {

int bb_version(void) { return BB_VERSION; }

const char* bb_strerror(int code) {
  switch (code) {
    case BB_OK: return "ok";
    case BB_ERR_INVALID: return "baler_b200: invalid argument";
    case BB_ERR_UNSUPPORTED: return "baler_b200: shape or mode not supported by the CUDA kernels";
    case BB_ERR_NOMEM: return "baler_b200: out of memory";
    case BB_ERR_NODEVICE: return "baler_b200: no CUDA device (there is no CPU fallback)";
    case BB_ERR_OVERFLOW: return "baler_b200: fp16 split range guard tripped; use BB_PREC_FP32";
    default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "baler_b200: unknown error";
  }
}

int bb_ctx_create(int device, bb_ctx** out) {
  if (!out) return BB_ERR_INVALID;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) return BB_ERR_NODEVICE;
  if (device < 0 || device >= n) return BB_ERR_INVALID;
  BB_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  BB_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return BB_ERR_UNSUPPORTED;  // sm_100a SASS only
  bb_ctx* c = new (std::nothrow) bb_ctx();
  if (!c) return BB_ERR_NOMEM;
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  c->smem_optin = prop.sharedMemPerBlockOptin;
  *out = c;
  return BB_OK;
}

int bb_ctx_destroy(bb_ctx* ctx) {
  if (!ctx) return BB_OK;
  if (ctx->minmax_scratch) cudaFree(ctx->minmax_scratch);
  if (ctx->err_scratch) cudaFree(ctx->err_scratch);
  delete ctx;
  return BB_OK;
}

int bb_ctx_sm_count(const bb_ctx* ctx) { return ctx ? ctx->sm_count : 0; }

}  // extern "C"

namespace {

int fill_chain(Chain* c, int n_layers, const int* dims, const int* acts, const double* const* w,
               const double* const* b) {
  if (n_layers < 1 || n_layers > BB_MAX_LAYERS || !dims || !acts || !w || !b) return BB_ERR_INVALID;
  ChainDesc& d = c->desc;
  memset(&d, 0, sizeof(d));
  d.n_layers = n_layers;
  d.in_dim = dims[0];
  d.out_dim = dims[n_layers];
  for (int l = 0; l < n_layers; ++l) {
    if (dims[l] < 1 || dims[l + 1] < 1 || acts[l] < BB_ACT_NONE || acts[l] > BB_ACT_RELU || !w[l] || !b[l])
      return BB_ERR_INVALID;
    d.layer[l].K = dims[l];
    d.layer[l].N = dims[l + 1];
    d.layer[l].act = acts[l];
    c->w_host[l].assign(w[l], w[l] + (size_t)dims[l] * dims[l + 1]);
    c->b_host[l].assign(b[l], b[l] + dims[l + 1]);
  }
  return BB_OK;
}

void free_chain(Chain* c) {
  // (pointers are cleared: bb_model_destroy also runs model_trim, which releases the scratch of a live model)
  auto release = [](auto*& p) {
    if (p) cudaFree(p);
    p = nullptr;
  };
  release(c->blob_dev);
  release(c->tc_blob_dev);
  release(c->lay_blob_dev);
  release(c->lay_scratch);
  c->lay_scratch_bytes = 0;
  release(c->lay_tc_blob_dev);
  release(c->g5_blob_dev);
  release(c->g5_bias_dev);
  bb_tc_release(c);
  bb_chain_f64_release(c);
}

// the chain has a tensor-core form: one of the fused tcgen05 kernels, or the layered mma.sync GEMMs for shapes too
// large for any fused kernel
bool chain_has_tc(const Chain* c) { return c->tc_ok || (!c->f32_ok && c->lay_tc_ok); }

int resolve_precision(const bb_model* m, const Chain* c, int precision) {
  if (precision == BB_PREC_AUTO) return chain_has_tc(c) ? BB_PREC_SPLIT16 : BB_PREC_FP32;
  return precision;
}

// features (pre_* / post_*) are float32, or float64 (feat_dtype BB_F64) on the float64 path only
int run_chain(bb_model* m, const Chain* c, const void* in, int in_dtype, int64_t n_rows,
              const void* pre_min_v, const void* pre_range_v, const void* post_min_v,
              const void* post_range_v, int feat_dtype, void* out, int out_dtype, int precision, cudaStream_t stream) {
  if (!m || (!in && n_rows) || (!out && n_rows) || n_rows < 0) return BB_ERR_INVALID;
  if ((pre_min_v == nullptr) != (pre_range_v == nullptr) || (post_min_v == nullptr) != (post_range_v == nullptr))
    return BB_ERR_INVALID;
  if (precision == BB_PREC_FP64)
    return bb_chain_f64_launch(m->ctx, c, in, in_dtype, n_rows, pre_min_v, pre_range_v, post_min_v, post_range_v, feat_dtype,
                               out, out_dtype, stream);
  if ((in_dtype != BB_F32 && in_dtype != BB_F16) || (out_dtype != BB_F32 && out_dtype != BB_F16) || feat_dtype != BB_F32)
    return BB_ERR_INVALID;
  const float* pre_min = (const float*)pre_min_v;
  const float* pre_range = (const float*)pre_range_v;
  const float* post_min = (const float*)post_min_v;
  const float* post_range = (const float*)post_range_v;
  const int p = resolve_precision(m, c, precision);
  if (p == BB_PREC_FP32) {
    if (!c->f32_ok)  // weights do not fit shared memory: one GEMM launch per layer
      return bb_chain_layered_launch(m->ctx, c, in, in_dtype, n_rows, pre_min, pre_range, post_min, post_range, out,
                                     out_dtype, 0, nullptr, stream);
    return bb_chain_f32_launch(m->ctx, c, in, in_dtype, n_rows, pre_min, pre_range, post_min, post_range,
                               out, out_dtype, stream);
  }
  if (p == BB_PREC_SPLIT16 && !c->tc_ok && chain_has_tc(c))
    return bb_chain_layered_launch(m->ctx, c, in, in_dtype, n_rows, pre_min, pre_range, post_min, post_range, out, out_dtype, 1,
                                   m->flag_dev, stream);
  if (p == BB_PREC_SPLIT16 || p == BB_PREC_FAST16) {
    if (!c->tc_ok) return BB_ERR_UNSUPPORTED;
    return bb_tc_launch(m->ctx, c, in, in_dtype, n_rows, pre_min, pre_range, post_min, post_range, out,
                        out_dtype, p == BB_PREC_FAST16, m->flag_dev, stream);
  }
  return BB_ERR_INVALID;
}

size_t dtype_size(int dt) { return dt == BB_F64 ? 8 : (dt == BB_F16 ? 2 : 4); }

// host threads this process may use for the scan: the CPUs it is allowed on (a launcher may have bound the rank to its
// GPU's NUMA node), shared with the other ranks of the node (LOCAL_WORLD_SIZE, set by torchrun), at most 16
unsigned host_scan_threads() {
  unsigned hw = std::max(1u, std::thread::hardware_concurrency());
#if defined(__linux__)
  cpu_set_t set;
  if (sched_getaffinity(0, sizeof(set), &set) == 0 && CPU_COUNT(&set) > 0) hw = std::min<unsigned>(hw, (unsigned)CPU_COUNT(&set));
#endif
  unsigned ranks = 1;
  if (const char* e = getenv("LOCAL_WORLD_SIZE")) ranks = (unsigned)std::max(1, atoi(e));
  return std::max(1u, std::min(16u, hw / ranks));
}

// fp32 <-> fp64 conversion of a chunk on host threads (the reference stores float64 latents and reconstructions:
// helper.py:565).  AVX2 with non-temporal stores where the destination allows it: the output is written once and not
// read here, so the cache lines need not be fetched first (a plain store of a 3.8 GB reconstruction reads 3.8 GB too).
#if defined(__x86_64__) && defined(__GNUC__)
__attribute__((target("avx2"))) void widen_range_avx2(const float* src, double* dst, size_t lo, size_t hi) {
  size_t i = lo;
  for (; i < hi && (reinterpret_cast<uintptr_t>(dst + i) & 31u); ++i) dst[i] = (double)src[i];
  for (; i + 8 <= hi; i += 8) {
    const __m256 v = _mm256_loadu_ps(src + i);
    _mm256_stream_pd(dst + i, _mm256_cvtps_pd(_mm256_castps256_ps128(v)));
    _mm256_stream_pd(dst + i + 4, _mm256_cvtps_pd(_mm256_extractf128_ps(v, 1)));
  }
  for (; i < hi; ++i) dst[i] = (double)src[i];
  _mm_sfence();
}
__attribute__((target("avx2"))) void narrow_range_avx2(const double* src, float* dst, size_t lo, size_t hi) {
  size_t i = lo;
  for (; i < hi && (reinterpret_cast<uintptr_t>(dst + i) & 31u); ++i) dst[i] = (float)src[i];
  for (; i + 8 <= hi; i += 8) {
    const __m128 a = _mm256_cvtpd_ps(_mm256_loadu_pd(src + i)), b = _mm256_cvtpd_ps(_mm256_loadu_pd(src + i + 4));
    _mm256_stream_ps(dst + i, _mm256_set_m128(b, a));
  }
  for (; i < hi; ++i) dst[i] = (float)src[i];
  _mm_sfence();
}
#endif

// Persistent worker threads for the per-chunk conversions.  Spawning and joining 16 std::threads costs ~0.45 ms, and a
// float64 round trip converts three arrays per chunk (48 dispatches for 16 chunks: a sixth of its wall time); the pool
// hands a job to sleeping workers in a few microseconds.  One job at a time (callers queue on run_mu); the caller works
// too.  Never destroyed (no join against a library being unloaded at exit); a forked child starts a pool of its own,
// because the parent's workers do not exist there and its mutexes may be held.
class HostPool {
 public:
  static HostPool& get(unsigned want) {
    std::lock_guard<std::mutex> lk(singleton_mu());
    static std::once_flag fork_once;
    std::call_once(fork_once, [] { pthread_atfork(nullptr, nullptr, [] { slot() = nullptr; new (&singleton_mu()) std::mutex(); }); });
    HostPool*& p = slot();
    if (p == nullptr) p = new HostPool();
    p->grow(want);
    return *p;
  }
  // fn(t) for t in [0, n_tasks): tasks are claimed one by one by the workers and by the calling thread
  void run(unsigned n_tasks, const std::function<void(unsigned)>& fn) {
    if (n_tasks == 0) return;
    std::lock_guard<std::mutex> one_job(run_mu_);
    {
      std::lock_guard<std::mutex> lk(mu_);
      job_ = &fn; n_tasks_ = n_tasks; next_ = 0; left_ = n_tasks;
      ++generation_;
    }
    cv_work_.notify_all();
    work_on_current_job();
    std::unique_lock<std::mutex> lk(mu_);
    cv_done_.wait(lk, [&] { return left_ == 0; });
    job_ = nullptr;
  }

 private:
  static HostPool*& slot() { static HostPool* p = nullptr; return p; }
  static std::mutex& singleton_mu() { static std::mutex* m = new std::mutex(); return *m; }
  void grow(unsigned want) {  // (under singleton_mu) workers = want - 1: the caller is the last one
    while (workers_ + 1 < want) {
      std::thread([this] { worker(); }).detach();
      ++workers_;
    }
  }
  void work_on_current_job() {
    for (;;) {
      unsigned t;
      {
        std::lock_guard<std::mutex> lk(mu_);
        if (job_ == nullptr || next_ >= n_tasks_) return;
        t = next_++;
      }
      (*job_)(t);
      std::lock_guard<std::mutex> lk(mu_);
      if (--left_ == 0) cv_done_.notify_all();
    }
  }
  void worker() {
    uint64_t seen = 0;
    for (;;) {
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_work_.wait(lk, [&] { return generation_ != seen; });
        seen = generation_;
      }
      work_on_current_job();
    }
  }
  std::mutex mu_, run_mu_;
  std::condition_variable cv_work_, cv_done_;
  const std::function<void(unsigned)>* job_ = nullptr;
  unsigned n_tasks_ = 0, next_ = 0, left_ = 0, workers_ = 0;
  uint64_t generation_ = 0;
};

template <typename Fn>
void host_parallel_ranges(size_t n, Fn fn) {
  const unsigned hw = host_scan_threads();
  const size_t per = ((n + hw - 1) / hw + 7) & ~(size_t)7;
  if (n < (1u << 16) || hw == 1) {
    fn((size_t)0, n);
    return;
  }
  const unsigned n_tasks = (unsigned)((n + per - 1) / per);
  const std::function<void(unsigned)> task = [&](unsigned t) {
    const size_t lo = (size_t)t * per, hi = std::min(n, lo + per);
    if (lo < hi) fn(lo, hi);
  };
  HostPool::get(hw).run(n_tasks, task);
}

void widen_f32_f64(const float* src, double* dst, size_t n) {
  host_parallel_ranges(n, [=](size_t lo, size_t hi) {
#if defined(__x86_64__) && defined(__GNUC__)
    if (__builtin_cpu_supports("avx2")) { widen_range_avx2(src, dst, lo, hi); return; }
#endif
    for (size_t i = lo; i < hi; ++i) dst[i] = (double)src[i];
  });
}

void narrow_f64_f32(const double* src, float* dst, size_t n) {
  host_parallel_ranges(n, [=](size_t lo, size_t hi) {
#if defined(__x86_64__) && defined(__GNUC__)
    if (__builtin_cpu_supports("avx2")) { narrow_range_avx2(src, dst, lo, hi); return; }
#endif
    for (size_t i = lo; i < hi; ++i) dst[i] = (float)src[i];
  });
}

constexpr int64_t PIPE_CHUNK_ROWS = 1 << 21;  // rows per pipeline chunk (2 Mi rows: 192 MiB in, 120 MiB out for 24 -> 15)
constexpr int64_t PIPE_MIN_CHUNK_ROWS = 1 << 18;

// Chunking of a host table: at least ~16 chunks so that filling and draining the H2D / kernel / D2H pipeline stays a small
// part of the call (a 12.5M-row shard cut into 2Mi-row chunks spends a third of its time in fill and drain), but never
// below 256 Ki rows (per-chunk launch and event overhead) nor above 2 Mi rows (staging memory)
inline int64_t pipe_chunk_rows(int64_t n_rows) {
  int64_t c = (n_rows + 15) / 16;
  c = std::max<int64_t>(c, PIPE_MIN_CHUNK_ROWS);
  c = std::min<int64_t>(c, PIPE_CHUNK_ROWS);
  c = (c + 127) & ~(int64_t)127;  // whole 128-row tiles: chunk boundaries stay 16-byte aligned for any row width
  return std::max<int64_t>(1, std::min<int64_t>(n_rows, c));
}

int pipe_init(bb_model* m, size_t in_bytes, size_t out_bytes) {
  if (!m->s_compute) {
    BB_CUDA(cudaStreamCreateWithFlags(&m->s_copy_in, cudaStreamNonBlocking));
    BB_CUDA(cudaStreamCreateWithFlags(&m->s_compute, cudaStreamNonBlocking));
    BB_CUDA(cudaStreamCreateWithFlags(&m->s_copy_out, cudaStreamNonBlocking));
    for (int s = 0; s < 2; ++s) {
      BB_CUDA(cudaEventCreateWithFlags(&m->ev_in[s], cudaEventDisableTiming));
      BB_CUDA(cudaEventCreateWithFlags(&m->ev_done[s], cudaEventDisableTiming));
      BB_CUDA(cudaEventCreateWithFlags(&m->ev_out[s], cudaEventDisableTiming));
    }
    BB_CUDA(cudaMalloc(&m->feat_dev, 3 * sizeof(float) * std::max(m->enc.desc.in_dim, m->dec.desc.out_dim)));
  }
  const size_t need[2] = {in_bytes, out_bytes};
  for (int io = 0; io < 2; ++io) {
    if (m->stage_bytes[io] < need[io]) {
      for (int s = 0; s < 2; ++s) {
        if (m->stage_dev[io][s]) cudaFree(m->stage_dev[io][s]);
        m->stage_dev[io][s] = nullptr;
        BB_CUDA(cudaMalloc(&m->stage_dev[io][s], need[io]));
      }
      m->stage_bytes[io] = need[io];
    }
  }
  return BB_OK;
}

// pinned bounce buffers (two slots, float32 or float64 chunks) of the float64 host paths, grown on demand and kept
int pinned_init(bb_model* m, int io, size_t bytes) {
  if (m->pinned_bytes[io] >= bytes) return BB_OK;
  for (int s = 0; s < 2; ++s) {
    if (m->pinned_f32[io][s]) cudaFreeHost(m->pinned_f32[io][s]);
    m->pinned_f32[io][s] = nullptr;
  }
  m->pinned_bytes[io] = 0;
  for (int s = 0; s < 2; ++s)
    if (cudaMallocHost(&m->pinned_f32[io][s], bytes) != cudaSuccess) { cudaGetLastError(); return BB_ERR_NOMEM; }
  m->pinned_bytes[io] = bytes;
  return BB_OK;
}

// Column min / max of a host table on host threads (data_processing.find_minmax, data_processing.py:113-130), for the
// resident path of bb_compress_host: the scan reads host memory at several times the PCIe rate, so the features are known
// long before the upload of the table ends and the latent download overlaps the rest of the upload (full duplex) instead
// of following it.  Same results as colminmax_kernel: order-preserving integer keys (-0 < +0), NaN propagates per column.
// key(u) = u ^ ((u >> 31) & 0x7fffffff) as a SIGNED int is monotonic in the float value.
inline int32_t mm_key(uint32_t u) { return (int32_t)(u ^ ((uint32_t)((int32_t)u >> 31) & 0x7fffffffu)); }
inline float mm_unkey(int32_t k) {
  const uint32_t u = k >= 0 ? (uint32_t)k : ((uint32_t)k ^ 0x7fffffffu);
  float f;
  memcpy(&f, &u, 4);
  return f;
}

// scalar scan of elements [e0, e1) of the flat table; column = element index % F
void mm_scan_scalar(const uint32_t* p, int64_t e0, int64_t e1, int F, int32_t* mn, int32_t* mx, uint32_t* nan) {
  int c = (int)(e0 % F);
  for (int64_t e = e0; e < e1; ++e) {
    const uint32_t u = p[e];
    if ((u & 0x7fffffffu) > 0x7f800000u) {
      nan[c] = 1u;
    } else {
      const int32_t k = mm_key(u);
      mn[c] = k < mn[c] ? k : mn[c];
      mx[c] = k > mx[c] ? k : mx[c];
    }
    if (++c == F) c = 0;
  }
}

#if defined(__x86_64__) && defined(__GNUC__)
// AVX2: the column pattern of 8 consecutive elements repeats every L = lcm(F, 8) elements, so L / 8 vector accumulators
// cover a period; lane j of accumulator v belongs to column (8 v + j) % F
// (accumulators as plain int arrays of 8 L8 entries; kept in registers for the scan when L8 <= 4: the CMS table has L8 = 3)
__attribute__((target("avx2"))) void mm_scan_avx2(const uint32_t* p, int64_t n_periods, int L8, int32_t* mn, int32_t* mx, int32_t* nanv) {
  const __m256i mag = _mm256_set1_epi32(0x7fffffff), inf = _mm256_set1_epi32(0x7f800000);
  const __m256i imax = _mm256_set1_epi32(0x7fffffff), imin = _mm256_set1_epi32((int)0x80000000u);
#define BB_MM_STEP(U, MN, MX, NV)                                                              \
  do {                                                                                         \
    const __m256i key_ = _mm256_xor_si256(U, _mm256_and_si256(_mm256_srai_epi32(U, 31), mag)); \
    const __m256i isnan_ = _mm256_cmpgt_epi32(_mm256_and_si256(U, mag), inf);                  \
    NV = _mm256_or_si256(NV, isnan_);                                                          \
    MN = _mm256_min_epi32(MN, _mm256_blendv_epi8(key_, imax, isnan_));                         \
    MX = _mm256_max_epi32(MX, _mm256_blendv_epi8(key_, imin, isnan_));                         \
  } while (0)
  if (L8 <= 4) {
    __m256i rmn[4], rmx[4], rnv[4];
    for (int v = 0; v < L8; ++v) {
      rmn[v] = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(mn + 8 * v));
      rmx[v] = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(mx + 8 * v));
      rnv[v] = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(nanv + 8 * v));
    }
    for (int64_t q = 0; q < n_periods; ++q, p += (size_t)L8 * 8)
      for (int v = 0; v < L8; ++v) {
        const __m256i u = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(p + 8 * v));
        BB_MM_STEP(u, rmn[v], rmx[v], rnv[v]);
      }
    for (int v = 0; v < L8; ++v) {
      _mm256_storeu_si256(reinterpret_cast<__m256i*>(mn + 8 * v), rmn[v]);
      _mm256_storeu_si256(reinterpret_cast<__m256i*>(mx + 8 * v), rmx[v]);
      _mm256_storeu_si256(reinterpret_cast<__m256i*>(nanv + 8 * v), rnv[v]);
    }
    return;
  }
  for (int64_t q = 0; q < n_periods; ++q, p += (size_t)L8 * 8)
    for (int v = 0; v < L8; ++v) {
      const __m256i u = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(p + 8 * v));
      __m256i a = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(mn + 8 * v));
      __m256i b = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(mx + 8 * v));
      __m256i c = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(nanv + 8 * v));
      BB_MM_STEP(u, a, b, c);
      _mm256_storeu_si256(reinterpret_cast<__m256i*>(mn + 8 * v), a);
      _mm256_storeu_si256(reinterpret_cast<__m256i*>(mx + 8 * v), b);
      _mm256_storeu_si256(reinterpret_cast<__m256i*>(nanv + 8 * v), c);
    }
#undef BB_MM_STEP
}
#endif

void host_colminmax(const float* x, int64_t n_rows, int F, float* mn_out, float* mx_out) {
  const unsigned hw = host_scan_threads();
  int g = F, b = 8;
  while (b) { const int r = g % b; g = b; b = r; }
  const int period_rows = 8 / g, L8 = F / g;  // rows / 8-lane vectors of one period
  bool avx2 = false;
#if defined(__x86_64__) && defined(__GNUC__)
  avx2 = __builtin_cpu_supports("avx2") && L8 <= 1024;
#endif
  const int64_t periods = n_rows / period_rows;
  const int64_t per = (periods + hw - 1) / hw;
  std::vector<std::vector<int32_t>> pmn(hw, std::vector<int32_t>((size_t)F, 0x7fffffff)), pmx(hw, std::vector<int32_t>((size_t)F, (int32_t)0x80000000u));
  std::vector<std::vector<uint32_t>> pnan(hw, std::vector<uint32_t>((size_t)F, 0u));
  const uint32_t* p = reinterpret_cast<const uint32_t*>(x);
  auto work = [&](unsigned t) {
    const int64_t q0 = std::min<int64_t>(periods, (int64_t)t * per), q1 = std::min<int64_t>(periods, q0 + per);
    int32_t* mn = pmn[t].data();
    int32_t* mx = pmx[t].data();
    uint32_t* nan = pnan[t].data();
    int64_t e0 = q0 * period_rows * F;
    const int64_t e1 = (t + 1 == hw ? n_rows : q1 * period_rows) * (int64_t)F;  // the last thread also takes the ragged tail
#if defined(__x86_64__) && defined(__GNUC__)
    if (avx2 && q1 > q0) {
      std::vector<int32_t> acc(3 * (size_t)L8 * 8);
      int32_t* vmn = acc.data();
      int32_t* vmx = vmn + (size_t)L8 * 8;
      int32_t* vnan = vmx + (size_t)L8 * 8;
      for (int i = 0; i < L8 * 8; ++i) { vmn[i] = 0x7fffffff; vmx[i] = (int32_t)0x80000000u; vnan[i] = 0; }
      mm_scan_avx2(p + e0, q1 - q0, L8, vmn, vmx, vnan);
      for (int i = 0; i < L8 * 8; ++i) {
        const int c = i % F;
        mn[c] = vmn[i] < mn[c] ? vmn[i] : mn[c];
        mx[c] = vmx[i] > mx[c] ? vmx[i] : mx[c];
        nan[c] |= vnan[i] ? 1u : 0u;
      }
      e0 = q1 * period_rows * F;
    }
#endif
    mm_scan_scalar(p, e0, e1, F, mn, mx, nan);
  };
  std::vector<std::thread> th;
  for (unsigned t = 1; t < hw; ++t) th.emplace_back(work, t);
  work(0);
  for (auto& h : th) h.join();
  for (int c = 0; c < F; ++c) {
    int32_t mn = 0x7fffffff, mx = (int32_t)0x80000000u;
    uint32_t nan = 0u;
    for (unsigned t = 0; t < hw; ++t) {
      mn = std::min(mn, pmn[t][c]); mx = std::max(mx, pmx[t][c]); nan |= pnan[t][c];
    }
    const uint32_t qnan = 0x7fc00000u;
    float fn;
    memcpy(&fn, &qnan, 4);
    mn_out[c] = nan ? fn : mm_unkey(mn);
    mx_out[c] = nan ? fn : mm_unkey(mx);
  }
}

// page-locked host memory (cudaMallocHost / cudaHostRegister): copies to and from it run asynchronously at the PCIe rate
bool host_pinned(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost;
}

// memcpy of n bytes on the library's worker threads (float64 chunks between a pageable caller buffer and a pinned slot)
void copy_parallel(void* dst, const void* src, size_t n) {
  host_parallel_ranges(n, [=](size_t lo, size_t hi) { memcpy((char*)dst + lo, (const char*)src + lo, hi - lo); });
}

// device copy of the whole table between the two passes of bb_compress_host, when it fits in half of the free memory
float* resident_get(bb_model* m, size_t bytes) {
  if (getenv("BALER_B200_NO_RESIDENT")) return nullptr;  // test hook: take the two-pass streaming path of tables that do not fit
  if (m->resident_bytes >= bytes) return m->resident_dev;
  if (m->resident_dev) { cudaFree(m->resident_dev); m->resident_dev = nullptr; m->resident_bytes = 0; }
  size_t free_b = 0, total_b = 0;
  if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess || bytes >= free_b / 2) return nullptr;
  if (cudaMalloc(&m->resident_dev, bytes) != cudaSuccess) { cudaGetLastError(); m->resident_dev = nullptr; return nullptr; }
  m->resident_bytes = bytes;
  return m->resident_dev;
}

void model_trim(bb_model* m) {
  if (m->resident_dev) cudaFree(m->resident_dev);
  m->resident_dev = nullptr; m->resident_bytes = 0;
  for (int io = 0; io < 2; ++io) {
    for (int s = 0; s < 2; ++s) {
      if (m->pinned_f32[io][s]) cudaFreeHost(m->pinned_f32[io][s]);
      m->pinned_f32[io][s] = nullptr;
    }
    m->pinned_bytes[io] = 0;
  }
  // the activation scratch of the layered GEMM path (up to 2 x 1.24 GB per direction for 2000-wide layers; cudaFree waits
  // for the device, so work still using it on any stream has finished)
  for (Chain* c : {&m->enc, &m->dec}) {
    if (c->lay_scratch) cudaFree(c->lay_scratch);
    c->lay_scratch = nullptr; c->lay_scratch_bytes = 0;
    bb_chain_f64_release(c);  // the float64 weight image: packed again by the next BB_PREC_FP64 call
  }
  if (m->feat64_dev) cudaFree(m->feat64_dev);
  m->feat64_dev = nullptr;
}

// range = max - min on device (one subtraction in the table's dtype, like numpy)
template <typename T>
__global__ void range_kernel(const T* mn, const T* mx, T* rg, int c) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < c) rg[i] = mx[i] - mn[i];
}

void launch_range(const void* mn, const void* mx, void* rg, int c, int dtype, cudaStream_t s) {
  if (dtype == BB_F64) range_kernel<double><<<(c + 127) / 128, 128, 0, s>>>((const double*)mn, (const double*)mx, (double*)rg, c);
  else range_kernel<float><<<(c + 127) / 128, 128, 0, s>>>((const float*)mn, (const float*)mx, (float*)rg, c);
}

// [min | range | max] of the table's dtype on the device: float32 features in feat_dev, float64 ones in feat64_dev
int features_dev(bb_model* m, int dtype, char** out) {
  if (dtype == BB_F64 && !m->feat64_dev)
    BB_CUDA(cudaMalloc(&m->feat64_dev, 3 * sizeof(double) * std::max(m->enc.desc.in_dim, m->dec.desc.out_dim)));
  *out = dtype == BB_F64 ? (char*)m->feat64_dev : (char*)m->feat_dev;
  return BB_OK;
}

}  // namespace

extern "C" {

int bb_model_range_flag(bb_model* m, int reset, int* out);

int bb_model_create_dense(bb_ctx* ctx, int n_enc_layers, const int* enc_dims, const int* enc_acts,
                          const double* const* enc_w, const double* const* enc_b, int n_dec_layers,
                          const int* dec_dims, const int* dec_acts, const double* const* dec_w,
                          const double* const* dec_b, bb_model** out) {
  if (!ctx || !out) return BB_ERR_INVALID;
  BB_CUDA(cudaSetDevice(ctx->device));
  bb_model* m = new (std::nothrow) bb_model();
  if (!m) return BB_ERR_NOMEM;
  m->ctx = ctx;
  int rc = fill_chain(&m->enc, n_enc_layers, enc_dims, enc_acts, enc_w, enc_b);
  if (rc == BB_OK) rc = fill_chain(&m->dec, n_dec_layers, dec_dims, dec_acts, dec_w, dec_b);
  if (rc == BB_OK && m->enc.desc.out_dim != m->dec.desc.in_dim) rc = BB_ERR_INVALID;
  for (Chain* c : {&m->enc, &m->dec}) {
    if (rc != BB_OK) break;
    rc = bb_chain_f32_prepare(ctx, c);
    c->f32_ok = rc == BB_OK;
    if (rc == BB_ERR_UNSUPPORTED) rc = bb_chain_layered_prepare(ctx, c);  // too big for the fused kernels
  }
  if (rc == BB_OK) rc = (int)cudaMalloc(&m->flag_dev, sizeof(int));
  if (rc == BB_OK) rc = (int)cudaMemset(m->flag_dev, 0, sizeof(int));
  if (rc == BB_OK) {
    // the tensor-core path is optional per shape; failure to prepare it is not an error
    int t = bb_tc_prepare(ctx, &m->enc);
    if (t != BB_OK && t != BB_ERR_UNSUPPORTED) rc = t;
    t = bb_tc_prepare(ctx, &m->dec);
    if (t != BB_OK && t != BB_ERR_UNSUPPORTED) rc = t;
  }
  if (rc != BB_OK) {
    bb_model_destroy(m);
    return rc;
  }
  *out = m;
  return BB_OK;
}

int bb_model_trim(bb_model* m) {
  if (!m) return BB_ERR_INVALID;
  cudaSetDevice(m->ctx->device);
  if (m->s_compute) { cudaStreamSynchronize(m->s_copy_in); cudaStreamSynchronize(m->s_compute); cudaStreamSynchronize(m->s_copy_out); }
  model_trim(m);
  return BB_OK;
}

int bb_model_destroy(bb_model* m) {
  if (!m) return BB_OK;
  free_chain(&m->enc);
  free_chain(&m->dec);
  if (m->flag_dev) cudaFree(m->flag_dev);
  if (m->feat_dev) cudaFree(m->feat_dev);
  model_trim(m);
  for (int io = 0; io < 2; ++io)
    for (int s = 0; s < 2; ++s)
      if (m->stage_dev[io][s]) cudaFree(m->stage_dev[io][s]);
  for (int s = 0; s < 2; ++s) {
    if (m->ev_in[s]) cudaEventDestroy(m->ev_in[s]);
    if (m->ev_done[s]) cudaEventDestroy(m->ev_done[s]);
    if (m->ev_out[s]) cudaEventDestroy(m->ev_out[s]);
  }
  if (m->s_copy_in) cudaStreamDestroy(m->s_copy_in);
  if (m->s_compute) cudaStreamDestroy(m->s_compute);
  if (m->s_copy_out) cudaStreamDestroy(m->s_copy_out);
  delete m;
  return BB_OK;
}

// Test hook (not part of the public header): run one direction on the tcgen05 path and dump the scaled
// accumulator of program step `dbg_step` (before activation) to dbg_out_dev [n_rows x step width].
int bb_debug_tc_chain(bb_model* m, int decode, const void* in_dev, int64_t n_rows, void* out_dev, int fast,
                      int dbg_step, float* dbg_out_dev, int force_groups, bb_stream_t stream) {
  if (!m) return BB_ERR_INVALID;
  const Chain* c = decode ? &m->dec : &m->enc;
  return bb_tc_launch_dbg(m->ctx, c, in_dev, BB_F32, n_rows, nullptr, nullptr, nullptr, nullptr, out_dev, BB_F32, fast,
                          m->flag_dev, dbg_step, dbg_out_dev, force_groups, (cudaStream_t)stream);
}

// Test hook (not part of the public header): the kernel (a BbRoute) and tile rows of the last launch of one direction
// (0 encoder, 1 decoder), so that tests can show which kernel a shape, precision, dtype and alignment were dispatched to.
int bb_debug_last_route(bb_model* m, int direction, int* kernel, int* tile_rows) {
  if (!m || direction < 0 || direction > 1 || !kernel || !tile_rows) return BB_ERR_INVALID;
  const Chain* c = direction == 0 ? &m->enc : &m->dec;
  *kernel = c->last_route;
  *tile_rows = c->last_tile_rows;
  return BB_OK;
}

int bb_model_range_flag(bb_model* m, int reset, int* out) {
  if (!m || !out) return BB_ERR_INVALID;
  BB_CUDA(cudaMemcpy(out, m->flag_dev, sizeof(int), cudaMemcpyDeviceToHost));
  if (reset && *out) BB_CUDA(cudaMemset(m->flag_dev, 0, sizeof(int)));
  return BB_OK;
}

int bb_model_n_features(const bb_model* m) { return m ? m->enc.desc.in_dim : 0; }
int bb_model_z_dim(const bb_model* m) { return m ? m->enc.desc.out_dim : 0; }
int bb_model_chain_precision(const bb_model* m, int direction) {
  if (!m || direction < 0 || direction > 1) return BB_ERR_INVALID;
  return chain_has_tc(direction == 0 ? &m->enc : &m->dec) ? BB_PREC_SPLIT16 : BB_PREC_FP32;
}

int bb_model_auto_precision(const bb_model* m) {
  return (m && chain_has_tc(&m->enc) && chain_has_tc(&m->dec)) ? BB_PREC_SPLIT16 : BB_PREC_FP32;
}

int bb_colminmax_f32(bb_ctx* ctx, const float* x_dev, int64_t n_rows, int n_cols, float* min_dev,
                     float* max_dev, bb_stream_t stream) {
  if (!ctx || (!x_dev && n_rows) || !min_dev || !max_dev) return BB_ERR_INVALID;
  return bb_colminmax_launch(ctx, x_dev, BB_F32, n_rows, n_cols, min_dev, max_dev, 1, (cudaStream_t)stream);
}

int bb_colminmax_f64(bb_ctx* ctx, const double* x_dev, int64_t n_rows, int n_cols, double* min_dev,
                     double* max_dev, bb_stream_t stream) {
  if (!ctx || (!x_dev && n_rows) || !min_dev || !max_dev) return BB_ERR_INVALID;
  return bb_colminmax_launch(ctx, x_dev, BB_F64, n_rows, n_cols, min_dev, max_dev, 1, (cudaStream_t)stream);
}

int bb_encode_f32(bb_model* m, const float* x_dev, int64_t n_rows, const float* min_dev,
                  const float* range_dev, void* z_dev, int z_dtype, int precision, bb_stream_t stream) {
  if (!m) return BB_ERR_INVALID;
  return run_chain(m, &m->enc, x_dev, BB_F32, n_rows, min_dev, range_dev, nullptr, nullptr, BB_F32, z_dev, z_dtype,
                   precision, (cudaStream_t)stream);
}

int bb_decode_f32(bb_model* m, const void* z_dev, int z_dtype, int64_t n_rows, const float* min_dev,
                  const float* range_dev, float* y_dev, int precision, bb_stream_t stream) {
  if (!m) return BB_ERR_INVALID;
  return run_chain(m, &m->dec, z_dev, z_dtype, n_rows, nullptr, nullptr, min_dev, range_dev, BB_F32, y_dev, BB_F32,
                   precision, (cudaStream_t)stream);
}

int bb_encode_f64(bb_model* m, const double* x_dev, int64_t n_rows, const double* min_dev, const double* range_dev,
                  double* z_dev, bb_stream_t stream) {
  if (!m) return BB_ERR_INVALID;
  return run_chain(m, &m->enc, x_dev, BB_F64, n_rows, min_dev, range_dev, nullptr, nullptr, BB_F64, z_dev, BB_F64,
                   BB_PREC_FP64, (cudaStream_t)stream);
}

int bb_decode_f64(bb_model* m, const double* z_dev, int64_t n_rows, const double* min_dev, const double* range_dev,
                  double* y_dev, bb_stream_t stream) {
  if (!m) return BB_ERR_INVALID;
  return run_chain(m, &m->dec, z_dev, BB_F64, n_rows, nullptr, nullptr, min_dev, range_dev, BB_F64, y_dev, BB_F64,
                   BB_PREC_FP64, (cudaStream_t)stream);
}

int bb_host_convert(const void* src, int src_dtype, void* dst, int dst_dtype, int64_t n) {
  if (n < 0 || ((!src || !dst) && n)) return BB_ERR_INVALID;
  if (src_dtype == BB_F32 && dst_dtype == BB_F64) widen_f32_f64((const float*)src, (double*)dst, (size_t)n);
  else if (src_dtype == BB_F64 && dst_dtype == BB_F32) narrow_f64_f32((const double*)src, (float*)dst, (size_t)n);
  else return BB_ERR_INVALID;
  return BB_OK;
}

int bb_host_colminmax_f32(const float* x_host, int64_t n_rows, int n_cols, float* min_out, float* max_out) {
  if (!x_host || !min_out || !max_out || n_rows < 1 || n_cols < 1) return BB_ERR_INVALID;
  host_colminmax(x_host, n_rows, n_cols, min_out, max_out);
  return BB_OK;
}

}  // extern "C"

namespace {

// The quantised latent of bb_compress_host_packed / bb_decompress_host_packed in host memory: codes [n_rows, row_bytes]
// (row_bytes = ceil(Z * bits / 8)), lo / step [ceil(n_rows / 128), Z]
struct QHost {
  int bits;
  uint8_t* codes;
  float* lo;
  float* step;
  size_t row_bytes(int Z) const { return ((size_t)Z * bits + 7) / 8; }
};

// A chunk's quantised latent in a device staging slot, behind its float32 latent: [float32 latent | codes | lo | step],
// each part 256-byte aligned.  Chunks start on block boundaries (pipe_chunk_rows gives whole 128-row tiles), so a chunk's
// blocks are the file's.
struct QSlot {
  size_t codes_off, lo_off, step_off, bytes;
  QSlot(int64_t rows, int Z, size_t row_bytes) {
    auto up = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t nb = (size_t)((rows + BB_Q8_BLOCK_ROWS - 1) / BB_Q8_BLOCK_ROWS);
    codes_off = up((size_t)rows * Z * sizeof(float));
    lo_off = codes_off + up((size_t)rows * row_bytes);
    step_off = lo_off + up(nb * Z * sizeof(float));
    bytes = step_off + up(nb * Z * sizeof(float));
  }
};

// The host-buffer compress pipeline of bb_compress_host (x_dtype BB_F32: float32 table and features),
// bb_compress_host_f64 (x_dtype BB_F64: float64 table and features, precision BB_PREC_FP64) and bb_compress_host_packed
// (q: the float32 latent of each chunk is quantised on the device and its codes and parameters are copied out instead).
int compress_host(bb_model* m, const void* x_host, int x_dtype, int64_t n_rows, void* features_host,
                  int recompute_minmax, void* z_host, int z_dtype, int precision, const QHost* q = nullptr) {
  if (!m || (!x_host && n_rows) || (!z_host && !q && n_rows) || n_rows < 0) return BB_ERR_INVALID;
  if (q && (q->bits < BB_LATENT_MIN_BITS || q->bits > BB_LATENT_MAX_BITS)) return BB_ERR_INVALID;
  if (q && n_rows && (!q->codes || !q->lo || !q->step)) return BB_ERR_INVALID;
  if (q && (precision == BB_PREC_FP64 || x_dtype != BB_F32)) return BB_ERR_UNSUPPORTED;
  if (z_dtype != BB_F32 && z_dtype != BB_F16 && z_dtype != BB_F64) return BB_ERR_INVALID;
  if (recompute_minmax && !features_host) return BB_ERR_INVALID;
  if (x_dtype == BB_F64 && precision != BB_PREC_FP64) return BB_ERR_INVALID;
  BB_CUDA(cudaSetDevice(m->ctx->device));
  const int F = m->enc.desc.in_dim, Z = m->enc.desc.out_dim;
  const size_t xs = dtype_size(x_dtype);  // bytes per element of the table and of its features
  // device output dtype: the float32 / fp16 kernels write float32 for a float64 latent (widened on the host below); the
  // float64 kernel writes whatever is asked
  const int dev_dtype = q ? BB_F32 : (z_dtype == BB_F64 && precision != BB_PREC_FP64) ? BB_F32 : z_dtype;
  const int64_t chunk = pipe_chunk_rows(n_rows);
  const int64_t n_chunks = n_rows ? (n_rows + chunk - 1) / chunk : 0;
  const QSlot qs(chunk, Z, q ? q->row_bytes(Z) : 0);
  const size_t in_b = (size_t)chunk * F * xs, out_b = q ? qs.bytes : (size_t)chunk * Z * dtype_size(dev_dtype);
  int rc = pipe_init(m, in_b, out_b);
  if (rc != BB_OK) return rc;
  char* feat = nullptr;
  rc = features_dev(m, x_dtype, &feat);
  if (rc != BB_OK) return rc;
  char* fmin = feat;
  char* frange = feat + F * xs;
  char* fmax = feat + 2 * F * xs;
  const bool norm = features_host != nullptr;
  const char* xh = (const char*)x_host;

  // Column statistics of THIS table (helper.py:500-502): either a first streaming pass that keeps
  // the table resident when it fits, or the features handed in.
  char* resident = nullptr;
  std::vector<cudaEvent_t> ev_up;  // resident path: upload of chunk k complete
  if (norm && recompute_minmax && n_rows) {
    resident = (char*)resident_get(m, (size_t)n_rows * F * xs);
    // the host scan pays when 16 host threads are free for it (measured on a 32-CPU node: 2 ranks 483 M rows/s against 414
    // with the device pass, 4 ranks of 8 threads each 385 against 557: the scans then compete with four uploads for the host's
    // memory bandwidth; the device pass below costs nothing on the host).  (float32 tables: the host scan has no float64 form)
    if (resident && x_dtype == BB_F32 && host_scan_threads() >= 16 && !getenv("BALER_B200_DEVICE_MINMAX")) {
      // the table fits: queue the whole upload now, find the column min / max on host threads meanwhile, and let the
      // encode + latent download of the chunks that have landed run against the rest of the upload
      // (the scan starts first, on its own threads: queuing copies from pageable memory blocks the calling thread)
      std::vector<float> mm(2 * (size_t)F);
      std::thread scan(host_colminmax, (const float*)x_host, n_rows, F, mm.data(), mm.data() + F);
      ev_up.resize((size_t)n_chunks, nullptr);
      cudaError_t up_rc = cudaSuccess;
      for (int64_t k = 0; k < n_chunks && up_rc == cudaSuccess; ++k) {
        const int64_t r0 = k * chunk, rows = std::min(chunk, n_rows - r0);
        up_rc = cudaMemcpyAsync(resident + (size_t)r0 * F * xs, xh + (size_t)r0 * F * xs, (size_t)rows * F * xs, cudaMemcpyHostToDevice, m->s_copy_in);
        if (up_rc == cudaSuccess) up_rc = cudaEventCreateWithFlags(&ev_up[(size_t)k], cudaEventDisableTiming);
        if (up_rc == cudaSuccess) up_rc = cudaEventRecord(ev_up[(size_t)k], m->s_copy_in);
      }
      scan.join();
      if (up_rc != cudaSuccess) {
        for (cudaEvent_t e : ev_up) if (e) cudaEventDestroy(e);
        return (int)up_rc;
      }
      BB_CUDA(cudaMemcpyAsync(fmin, mm.data(), F * sizeof(float), cudaMemcpyHostToDevice, m->s_compute));
      BB_CUDA(cudaMemcpyAsync(fmax, mm.data() + F, F * sizeof(float), cudaMemcpyHostToDevice, m->s_compute));
      launch_range(fmin, fmax, frange, F, x_dtype, m->s_compute);
      BB_CUDA(cudaMemcpyAsync(features_host, fmin, 2 * F * xs, cudaMemcpyDeviceToHost, m->s_compute));
      BB_CUDA(cudaStreamSynchronize(m->s_compute));  // (mm goes out of scope; features_host is final)
    } else {
      // a first streaming pass for the statistics on the device (column min / max kernel per chunk as it lands), which
      // keeps the table resident when it fits; otherwise the second pass below uploads it again
      for (int64_t k = 0; k < n_chunks; ++k) {
        const int64_t r0 = k * chunk, rows = std::min(chunk, n_rows - r0);
        const int s = (int)(k & 1);
        char* dst = resident ? resident + (size_t)r0 * F * xs : (char*)m->stage_dev[0][s];
        if (!resident && k >= 2) BB_CUDA(cudaStreamWaitEvent(m->s_copy_in, m->ev_done[s], 0));
        BB_CUDA(cudaMemcpyAsync(dst, xh + (size_t)r0 * F * xs, (size_t)rows * F * xs, cudaMemcpyHostToDevice, m->s_copy_in));
        BB_CUDA(cudaEventRecord(m->ev_in[s], m->s_copy_in));
        BB_CUDA(cudaStreamWaitEvent(m->s_compute, m->ev_in[s], 0));
        rc = bb_colminmax_launch(m->ctx, dst, x_dtype, rows, F, fmin, fmax, k == 0, m->s_compute);
        if (rc != BB_OK) return rc;
        BB_CUDA(cudaEventRecord(m->ev_done[s], m->s_compute));
      }
      launch_range(fmin, fmax, frange, F, x_dtype, m->s_compute);
      BB_CUDA(cudaMemcpyAsync(features_host, fmin, 2 * F * xs, cudaMemcpyDeviceToHost, m->s_compute));
      BB_CUDA(cudaStreamSynchronize(m->s_compute));
    }
  } else if (norm) {
    BB_CUDA(cudaMemcpyAsync(fmin, features_host, 2 * F * xs, cudaMemcpyHostToDevice, m->s_compute));
  }
  struct EvGuard {  // the per-chunk upload events live for this call only
    std::vector<cudaEvent_t>& v;
    ~EvGuard() { for (cudaEvent_t e : v) if (e) cudaEventDestroy(e); }
  } ev_guard{ev_up};

  const bool widen = !q && z_dtype == BB_F64 && dev_dtype != BB_F64;  // float32 on the device, float64 in the caller's buffer
  // a float64 latent from the float64 chain lands in a pinned slot and is copied out on host threads when the caller's
  // buffer is pageable (a device-to-pageable copy runs at a fraction of the PCIe rate)
  const bool bounce = dev_dtype == BB_F64 && n_rows && !host_pinned(z_host);
  void* pinned_out[2] = {nullptr, nullptr};
  if ((widen || bounce) && n_rows) {
    if (pinned_init(m, 1, (size_t)chunk * Z * dtype_size(dev_dtype)) != BB_OK) return BB_ERR_NOMEM;
    pinned_out[0] = m->pinned_f32[1][0]; pinned_out[1] = m->pinned_f32[1][1];
  }
  auto finish_chunk = [&](int64_t k) -> int {  // host side of chunk k: wait for its D2H, widen / copy out if needed
    const int s = (int)(k & 1);
    BB_CUDA(cudaEventSynchronize(m->ev_out[s]));
    const int64_t r0 = k * chunk, rows = std::min(chunk, n_rows - r0);
    if (widen) widen_f32_f64((const float*)pinned_out[s], (double*)z_host + (size_t)r0 * Z, (size_t)rows * Z);
    else if (bounce) copy_parallel((double*)z_host + (size_t)r0 * Z, pinned_out[s], (size_t)rows * Z * sizeof(double));
    return BB_OK;
  };
  rc = BB_OK;
  for (int64_t k = 0; k < n_chunks && rc == BB_OK; ++k) {
    const int64_t r0 = k * chunk, rows = std::min(chunk, n_rows - r0);
    const int s = (int)(k & 1);
    const char* src;
    if (resident) {
      src = resident + (size_t)r0 * F * xs;
      if (!ev_up.empty()) BB_CUDA(cudaStreamWaitEvent(m->s_compute, ev_up[(size_t)k], 0));
    } else {
      if (k >= 2) BB_CUDA(cudaStreamWaitEvent(m->s_copy_in, m->ev_done[s], 0));  // slot's previous kernel finished
      BB_CUDA(cudaMemcpyAsync(m->stage_dev[0][s], xh + (size_t)r0 * F * xs, (size_t)rows * F * xs, cudaMemcpyHostToDevice, m->s_copy_in));
      BB_CUDA(cudaEventRecord(m->ev_in[s], m->s_copy_in));
      BB_CUDA(cudaStreamWaitEvent(m->s_compute, m->ev_in[s], 0));
      src = (const char*)m->stage_dev[0][s];
    }
    if (k >= 2) {
      rc = finish_chunk(k - 2);  // frees output slot s on the host side (and its pinned buffer)
      if (rc != BB_OK) break;
      BB_CUDA(cudaStreamWaitEvent(m->s_compute, m->ev_out[s], 0));
    }
    rc = run_chain(m, &m->enc, src, x_dtype, rows, norm ? fmin : nullptr, norm ? frange : nullptr, nullptr, nullptr, x_dtype,
                   m->stage_dev[1][s], dev_dtype, precision, m->s_compute);
    if (rc != BB_OK) break;
    char* out = (char*)m->stage_dev[1][s];
    if (q) {
      rc = bb_latent_quantize_launch(m->ctx, (const float*)out, rows, Z, q->bits, (uint8_t*)(out + qs.codes_off),
                                     (float*)(out + qs.lo_off), (float*)(out + qs.step_off), m->s_compute);
      if (rc != BB_OK) break;
    }
    BB_CUDA(cudaEventRecord(m->ev_done[s], m->s_compute));
    BB_CUDA(cudaStreamWaitEvent(m->s_copy_out, m->ev_done[s], 0));
    if (q) {
      const int64_t b0 = r0 / BB_Q8_BLOCK_ROWS, nb = (rows + BB_Q8_BLOCK_ROWS - 1) / BB_Q8_BLOCK_ROWS;
      BB_CUDA(cudaMemcpyAsync(q->codes + (size_t)r0 * q->row_bytes(Z), out + qs.codes_off, (size_t)rows * q->row_bytes(Z), cudaMemcpyDeviceToHost, m->s_copy_out));
      BB_CUDA(cudaMemcpyAsync(q->lo + (size_t)b0 * Z, out + qs.lo_off, (size_t)nb * Z * sizeof(float), cudaMemcpyDeviceToHost, m->s_copy_out));
      BB_CUDA(cudaMemcpyAsync(q->step + (size_t)b0 * Z, out + qs.step_off, (size_t)nb * Z * sizeof(float), cudaMemcpyDeviceToHost, m->s_copy_out));
    } else {
      void* dst = (widen || bounce) ? pinned_out[s] : (void*)((char*)z_host + (size_t)r0 * Z * dtype_size(z_dtype));
      BB_CUDA(cudaMemcpyAsync(dst, out, (size_t)rows * Z * dtype_size(dev_dtype), cudaMemcpyDeviceToHost, m->s_copy_out));
    }
    BB_CUDA(cudaEventRecord(m->ev_out[s], m->s_copy_out));
  }
  for (int64_t k = std::max<int64_t>(0, n_chunks - 2); k < n_chunks && rc == BB_OK; ++k) rc = finish_chunk(k);
  cudaStreamSynchronize(m->s_compute);
  cudaStreamSynchronize(m->s_copy_out);
  if (rc == BB_OK && precision == BB_PREC_AUTO && chain_has_tc(&m->enc)) {
    int tripped = 0;  // fp16 range guard of the split path: redo on the fp32 kernel (features are already known)
    rc = bb_model_range_flag(m, 1, &tripped);
    if (rc == BB_OK && tripped)
      return compress_host(m, x_host, x_dtype, n_rows, features_host, 0, z_host, z_dtype, BB_PREC_FP32, q);
  }
  return rc;
}

// The host-buffer decompress pipeline of bb_decompress_host (float32 features), bb_decompress_host_f64 (feat_dtype
// BB_F64: float64 features, latent and reconstruction, precision BB_PREC_FP64) and bb_decompress_host_packed (q: codes
// and parameters are copied in and dequantised to a float32 latent on the device; z_host and z_dtype are unused).
int decompress_host(bb_model* m, const void* z_host, int z_dtype, int64_t n_rows, const void* features_host,
                    int feat_dtype, void* y_host, int y_dtype, int precision, const QHost* q = nullptr) {
  if (!m || (!z_host && !q && n_rows) || (!y_host && n_rows) || n_rows < 0) return BB_ERR_INVALID;
  if (q && (q->bits < BB_LATENT_MIN_BITS || q->bits > BB_LATENT_MAX_BITS)) return BB_ERR_INVALID;
  if (q && n_rows && (!q->codes || !q->lo || !q->step)) return BB_ERR_INVALID;
  if (q && (precision == BB_PREC_FP64 || feat_dtype != BB_F32)) return BB_ERR_UNSUPPORTED;
  if (q) z_dtype = BB_F32;  // (the device latent)
  if (z_dtype != BB_F32 && z_dtype != BB_F16 && z_dtype != BB_F64) return BB_ERR_INVALID;
  if (y_dtype != BB_F32 && y_dtype != BB_F64) return BB_ERR_INVALID;
  if (feat_dtype == BB_F64 && precision != BB_PREC_FP64) return BB_ERR_INVALID;
  BB_CUDA(cudaSetDevice(m->ctx->device));
  const int F = m->dec.desc.out_dim, Z = m->dec.desc.in_dim;
  const bool f64 = precision == BB_PREC_FP64;
  // device dtypes: the float32 / fp16 kernels read a float64 latent narrowed on the host and write float32; the float64
  // kernel reads and writes the caller's dtypes
  const int dev_in = (z_dtype == BB_F64 && !f64) ? BB_F32 : z_dtype;
  const int dev_out = f64 ? y_dtype : BB_F32;
  const bool narrow = dev_in != z_dtype, widen = dev_out != y_dtype;
  // float64 chunks of the float64 chain go through the pinned slots when the caller's buffer is pageable
  const bool bounce_in = dev_in == BB_F64 && n_rows && !host_pinned(z_host);
  const bool bounce_out = dev_out == BB_F64 && n_rows && !host_pinned(y_host);
  const int64_t chunk = pipe_chunk_rows(n_rows);
  const int64_t n_chunks = n_rows ? (n_rows + chunk - 1) / chunk : 0;
  const QSlot qs(chunk, Z, q ? q->row_bytes(Z) : 0);
  const size_t in_b = q ? qs.bytes : (size_t)chunk * Z * dtype_size(dev_in), out_b = (size_t)chunk * F * dtype_size(dev_out);
  int rc = pipe_init(m, in_b, out_b);
  if (rc != BB_OK) return rc;
  char* feat = nullptr;
  rc = features_dev(m, feat_dtype, &feat);
  if (rc != BB_OK) return rc;
  char* fmin = feat;
  char* frange = feat + F * dtype_size(feat_dtype);
  const bool norm = features_host != nullptr;
  if (norm) BB_CUDA(cudaMemcpyAsync(fmin, features_host, 2 * F * dtype_size(feat_dtype), cudaMemcpyHostToDevice, m->s_compute));

  void* pin_in[2] = {nullptr, nullptr};
  void* pin_out[2] = {nullptr, nullptr};
  if (n_rows) {  // (the bounce buffers belong to the model)
    if (narrow || bounce_in) {
      if (pinned_init(m, 0, (size_t)chunk * Z * dtype_size(dev_in)) != BB_OK) return BB_ERR_NOMEM;
      pin_in[0] = m->pinned_f32[0][0]; pin_in[1] = m->pinned_f32[0][1];
    }
    if (widen || bounce_out) {
      if (pinned_init(m, 1, (size_t)chunk * F * dtype_size(dev_out)) != BB_OK) return BB_ERR_NOMEM;
      pin_out[0] = m->pinned_f32[1][0]; pin_out[1] = m->pinned_f32[1][1];
    }
  }
  auto finish_chunk = [&](int64_t k) -> int {
    const int s = (int)(k & 1);
    BB_CUDA(cudaEventSynchronize(m->ev_out[s]));
    const int64_t r0 = k * chunk, rows = std::min(chunk, n_rows - r0);
    if (widen) widen_f32_f64((const float*)pin_out[s], (double*)y_host + (size_t)r0 * F, (size_t)rows * F);
    else if (bounce_out) copy_parallel((double*)y_host + (size_t)r0 * F, pin_out[s], (size_t)rows * F * sizeof(double));
    return BB_OK;
  };
  rc = BB_OK;
  for (int64_t k = 0; k < n_chunks && rc == BB_OK; ++k) {
    const int64_t r0 = k * chunk, rows = std::min(chunk, n_rows - r0);
    const int s = (int)(k & 1);
    if (k >= 2) {
      BB_CUDA(cudaEventSynchronize(m->ev_in[s]));  // pinned input slot consumed by its H2D copy
      BB_CUDA(cudaStreamWaitEvent(m->s_copy_in, m->ev_done[s], 0));
    }
    char* in = (char*)m->stage_dev[0][s];
    if (q) {
      const int64_t b0 = r0 / BB_Q8_BLOCK_ROWS, nb = (rows + BB_Q8_BLOCK_ROWS - 1) / BB_Q8_BLOCK_ROWS;
      BB_CUDA(cudaMemcpyAsync(in + qs.codes_off, q->codes + (size_t)r0 * q->row_bytes(Z), (size_t)rows * q->row_bytes(Z), cudaMemcpyHostToDevice, m->s_copy_in));
      BB_CUDA(cudaMemcpyAsync(in + qs.lo_off, q->lo + (size_t)b0 * Z, (size_t)nb * Z * sizeof(float), cudaMemcpyHostToDevice, m->s_copy_in));
      BB_CUDA(cudaMemcpyAsync(in + qs.step_off, q->step + (size_t)b0 * Z, (size_t)nb * Z * sizeof(float), cudaMemcpyHostToDevice, m->s_copy_in));
    } else {
      const void* src = (const char*)z_host + (size_t)r0 * Z * dtype_size(z_dtype);
      if (narrow) {
        narrow_f64_f32((const double*)src, (float*)pin_in[s], (size_t)rows * Z);
        src = pin_in[s];
      } else if (bounce_in) {
        copy_parallel(pin_in[s], src, (size_t)rows * Z * sizeof(double));
        src = pin_in[s];
      }
      BB_CUDA(cudaMemcpyAsync(in, src, (size_t)rows * Z * dtype_size(dev_in), cudaMemcpyHostToDevice, m->s_copy_in));
    }
    BB_CUDA(cudaEventRecord(m->ev_in[s], m->s_copy_in));
    BB_CUDA(cudaStreamWaitEvent(m->s_compute, m->ev_in[s], 0));
    if (k >= 2) {
      rc = finish_chunk(k - 2);
      if (rc != BB_OK) break;
      BB_CUDA(cudaStreamWaitEvent(m->s_compute, m->ev_out[s], 0));
    }
    if (q) {
      rc = bb_latent_dequantize_launch(m->ctx, q->bits, (const uint8_t*)(in + qs.codes_off), (const float*)(in + qs.lo_off),
                                       (const float*)(in + qs.step_off), rows, Z, (float*)in, m->s_compute);
      if (rc != BB_OK) break;
    }
    rc = run_chain(m, &m->dec, m->stage_dev[0][s], dev_in, rows, nullptr, nullptr, norm ? fmin : nullptr,
                   norm ? frange : nullptr, feat_dtype, m->stage_dev[1][s], dev_out, precision, m->s_compute);
    if (rc != BB_OK) break;
    BB_CUDA(cudaEventRecord(m->ev_done[s], m->s_compute));
    BB_CUDA(cudaStreamWaitEvent(m->s_copy_out, m->ev_done[s], 0));
    void* dst = (widen || bounce_out) ? pin_out[s] : (void*)((char*)y_host + (size_t)r0 * F * dtype_size(y_dtype));
    BB_CUDA(cudaMemcpyAsync(dst, m->stage_dev[1][s], (size_t)rows * F * dtype_size(dev_out), cudaMemcpyDeviceToHost, m->s_copy_out));
    BB_CUDA(cudaEventRecord(m->ev_out[s], m->s_copy_out));
  }
  for (int64_t k = std::max<int64_t>(0, n_chunks - 2); k < n_chunks && rc == BB_OK; ++k) rc = finish_chunk(k);
  cudaStreamSynchronize(m->s_compute);
  cudaStreamSynchronize(m->s_copy_out);
  if (rc == BB_OK && precision == BB_PREC_AUTO && chain_has_tc(&m->dec)) {
    int tripped = 0;
    rc = bb_model_range_flag(m, 1, &tripped);
    if (rc == BB_OK && tripped)
      return decompress_host(m, z_host, z_dtype, n_rows, features_host, feat_dtype, y_host, y_dtype, BB_PREC_FP32, q);
  }
  return rc;
}

}  // namespace

extern "C" {

int bb_compress_host(bb_model* m, const float* x_host, int64_t n_rows, float* features_host,
                     int recompute_minmax, void* z_host, int z_dtype, int precision) {
  return compress_host(m, x_host, BB_F32, n_rows, features_host, recompute_minmax, z_host, z_dtype, precision);
}

int bb_decompress_host(bb_model* m, const void* z_host, int z_dtype, int64_t n_rows,
                       const float* features_host, void* y_host, int y_dtype, int precision) {
  return decompress_host(m, z_host, z_dtype, n_rows, features_host, BB_F32, y_host, y_dtype, precision);
}

int bb_compress_host_f64(bb_model* m, const double* x_host, int64_t n_rows, double* features_host,
                         int recompute_minmax, double* z_host) {
  return compress_host(m, x_host, BB_F64, n_rows, features_host, recompute_minmax, z_host, BB_F64, BB_PREC_FP64);
}

int bb_decompress_host_f64(bb_model* m, const double* z_host, int64_t n_rows, const double* features_host,
                           double* y_host) {
  return decompress_host(m, z_host, BB_F64, n_rows, features_host, BB_F64, y_host, BB_F64, BB_PREC_FP64);
}

int bb_compress_host_packed(bb_model* m, const float* x_host, int64_t n_rows, float* features_host, int recompute_minmax,
                            int bits, uint8_t* codes_host, float* lo_host, float* step_host, int precision) {
  const QHost q{bits, codes_host, lo_host, step_host};
  return compress_host(m, x_host, BB_F32, n_rows, features_host, recompute_minmax, nullptr, BB_F32, precision, &q);
}

int bb_decompress_host_packed(bb_model* m, int bits, const uint8_t* codes_host, const float* lo_host, const float* step_host,
                              int64_t n_rows, const float* features_host, void* y_host, int y_dtype, int precision) {
  const QHost q{bits, const_cast<uint8_t*>(codes_host), const_cast<float*>(lo_host), const_cast<float*>(step_host)};
  return decompress_host(m, nullptr, BB_F32, n_rows, features_host, BB_F32, y_host, y_dtype, precision, &q);
}

int bb_compress_host_q8(bb_model* m, const float* x_host, int64_t n_rows, float* features_host, int recompute_minmax,
                        uint8_t* codes_host, float* lo_host, float* step_host, int precision) {
  return bb_compress_host_packed(m, x_host, n_rows, features_host, recompute_minmax, 8, codes_host, lo_host, step_host,
                                 precision);
}

int bb_decompress_host_q8(bb_model* m, const uint8_t* codes_host, const float* lo_host, const float* step_host, int64_t n_rows,
                          const float* features_host, void* y_host, int y_dtype, int precision) {
  return bb_decompress_host_packed(m, 8, codes_host, lo_host, step_host, n_rows, features_host, y_host, y_dtype, precision);
}

}  // extern "C"

// ------------------------------------------------------------------ host tables streamed through a device window

struct HostWindow {
  cudaStream_t copy = nullptr;
  cudaEvent_t landed[2] = {nullptr, nullptr};    // slot's upload complete (copy stream)
  cudaEvent_t consumed[2] = {nullptr, nullptr};  // slot's kernels complete (caller's stream)
  cudaEvent_t staged[2] = {nullptr, nullptr};    // pinned buffer's upload complete (copy stream)
  void* dev[2] = {nullptr, nullptr};
  size_t dev_bytes = 0;
  void* pin[2] = {nullptr, nullptr};
  size_t pin_bytes = 0;
};

namespace {
// pinned staging of a pageable table: 2 x 64 MiB, whatever the window (the window's size is bounded by device memory, the
// staging by what page-locking a shared host can spare)
constexpr size_t WINDOW_STAGE_BYTES = (size_t)64 << 20;

int window_create(HostWindow* w) {
  BB_CUDA(cudaStreamCreateWithFlags(&w->copy, cudaStreamNonBlocking));
  for (int i = 0; i < 2; ++i) {
    BB_CUDA(cudaEventCreateWithFlags(&w->landed[i], cudaEventDisableTiming));
    BB_CUDA(cudaEventCreateWithFlags(&w->consumed[i], cudaEventDisableTiming));
    BB_CUDA(cudaEventCreateWithFlags(&w->staged[i], cudaEventDisableTiming));
  }
  return BB_OK;
}

// upload `bytes` of the host table at src into dst on the copy stream (after whatever the copy stream already waits for)
int window_upload(HostWindow* w, void* dst, const char* src, size_t bytes, bool pinned, unsigned* stage_k) {
  if (pinned) {
    BB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, w->copy));
    return BB_OK;
  }
  for (size_t off = 0; off < bytes; off += w->pin_bytes) {
    const size_t n = std::min(w->pin_bytes, bytes - off);
    const int p = (int)((*stage_k)++ & 1u);
    BB_CUDA(cudaEventSynchronize(w->staged[p]));  // the buffer's previous upload has left it (never recorded: returns)
    copy_parallel(w->pin[p], src + off, n);
    BB_CUDA(cudaMemcpyAsync((char*)dst + off, w->pin[p], n, cudaMemcpyHostToDevice, w->copy));
    BB_CUDA(cudaEventRecord(w->staged[p], w->copy));
  }
  return BB_OK;
}
}  // namespace

void bb_host_window_free(HostWindow* w) {
  if (!w) return;
  if (w->copy) cudaStreamSynchronize(w->copy);
  for (int i = 0; i < 2; ++i) {
    if (w->dev[i]) cudaFree(w->dev[i]);
    if (w->pin[i]) cudaFreeHost(w->pin[i]);
    if (w->landed[i]) cudaEventDestroy(w->landed[i]);
    if (w->consumed[i]) cudaEventDestroy(w->consumed[i]);
    if (w->staged[i]) cudaEventDestroy(w->staged[i]);
  }
  if (w->copy) cudaStreamDestroy(w->copy);
  delete w;
}

int bb_host_window_run(HostWindow** win, const void* x_host, size_t row_bytes, int64_t n_rows, int64_t window_rows,
                       cudaStream_t s, const std::function<int(const void*, int64_t)>& body) {
  if (!win || !x_host || row_bytes == 0 || n_rows < 1 || window_rows < 1) return BB_ERR_INVALID;
  if (!*win) {
    HostWindow* w = new (std::nothrow) HostWindow();
    if (!w) return BB_ERR_NOMEM;
    const int rc = window_create(w);
    if (rc != BB_OK) {
      bb_host_window_free(w);
      return rc;
    }
    *win = w;
  }
  HostWindow* w = *win;
  const int64_t rows_per = std::min(window_rows, n_rows);
  const size_t slot_bytes = (size_t)rows_per * row_bytes;
  if (w->dev_bytes < slot_bytes) {
    BB_CUDA(cudaStreamSynchronize(w->copy));
    for (int i = 0; i < 2; ++i) {
      if (w->dev[i]) cudaFree(w->dev[i]);  // (waits for the kernels still reading it)
      w->dev[i] = nullptr;
    }
    w->dev_bytes = 0;
    for (int i = 0; i < 2; ++i)
      if (cudaMalloc(&w->dev[i], slot_bytes) != cudaSuccess) { cudaGetLastError(); return BB_ERR_NOMEM; }
    w->dev_bytes = slot_bytes;
  }
  const bool pinned = host_pinned(x_host);
  const size_t stage = std::min(WINDOW_STAGE_BYTES, slot_bytes);
  if (!pinned && w->pin_bytes < stage) {
    BB_CUDA(cudaStreamSynchronize(w->copy));
    for (int i = 0; i < 2; ++i) {
      if (w->pin[i]) cudaFreeHost(w->pin[i]);
      w->pin[i] = nullptr;
    }
    w->pin_bytes = 0;
    for (int i = 0; i < 2; ++i)
      if (cudaMallocHost(&w->pin[i], stage) != cudaSuccess) { cudaGetLastError(); return BB_ERR_NOMEM; }
    w->pin_bytes = stage;
  }
  // the slots' previous users (an earlier call on another stream) are done before this call writes them
  for (int i = 0; i < 2; ++i) BB_CUDA(cudaEventRecord(w->consumed[i], s));
  const char* x = (const char*)x_host;
  unsigned stage_k = 0;
  int rc = BB_OK;
  for (int64_t k = 0, r0 = 0; r0 < n_rows && rc == BB_OK; ++k, r0 += rows_per) {
    const int slot = (int)(k & 1);
    const int64_t rows = std::min(rows_per, n_rows - r0);
    rc = (int)cudaStreamWaitEvent(w->copy, w->consumed[slot], 0);  // the kernels of window k - 2 are done with the slot
    if (rc == BB_OK) rc = window_upload(w, w->dev[slot], x + (size_t)r0 * row_bytes, (size_t)rows * row_bytes, pinned, &stage_k);
    if (rc == BB_OK) rc = (int)cudaEventRecord(w->landed[slot], w->copy);
    if (rc == BB_OK) rc = (int)cudaStreamWaitEvent(s, w->landed[slot], 0);
    if (rc == BB_OK) rc = body(w->dev[slot], rows);
    if (rc == BB_OK) rc = (int)cudaEventRecord(w->consumed[slot], s);
  }
  const cudaError_t sync = cudaStreamSynchronize(w->copy);  // (the staging buffers are free again when this returns)
  return rc != BB_OK ? rc : (int)sync;
}
