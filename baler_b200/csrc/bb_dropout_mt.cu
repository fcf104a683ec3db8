// AE_Dropout_BN dropout masks from torch's CPU generator, drawn on the device.
//
// The reference draws every dropout mask with Tensor.bernoulli_(1 - p) on torch's default CPU generator, a 32-bit
// MT19937.  For a float64 tensor bernoulli_ takes one random64 per element, two consecutive words with the first one
// high, and keeps the element when (random64 & (2^53 - 1)) * 2^-53 < 1 - p.  A batch of AE_Dropout_BN draws the four
// encoder masks in layer order, each [rows][N_l] row-major.  This kernel continues the twister from a state the host
// read out of torch.Generator.get_state() and produces exactly those keep-bits, so a float64 run uses the reference's
// own masks and leaves the generator where the reference's would be.
//
// One CTA of 1024 threads.  The state lives in two shared-memory buffers of 624 words.  Each iteration the first 8
// warps twist the next block out of place (three dependent rounds of at most 227 words: word i needs words i + 1 and
// i + 397 of the old block, or i - 227 of the new one) while the other 24 warps temper the current block and turn
// word pairs into keep-bits.  An element whose two words straddle two blocks takes its high word from the previous
// iteration through `carry`.
#include "bb_train_f64.cuh"

namespace {

constexpr int MT_N = 624, MT_M = 397, MT_R1 = MT_N - MT_M;  // 227
constexpr int NT_MT = 1024, NT_TWIST = 256;

__device__ __forceinline__ uint32_t mt_twist(uint32_t u, uint32_t v, uint32_t m) {
  const uint32_t y = (u & 0x80000000u) | (v & 0x7fffffffu);
  return m ^ (y >> 1) ^ ((v & 1u) ? 0x9908b0dfu : 0u);
}

__device__ __forceinline__ uint32_t mt_temper(uint32_t y) {
  y ^= y >> 11;
  y ^= (y << 7) & 0x9d2c5680u;
  y ^= (y << 15) & 0xefc60000u;
  return y ^ (y >> 18);
}

__device__ __forceinline__ void twist_bar() { asm volatile("bar.sync 1, %0;" ::"n"(NT_TWIST) : "memory"); }

struct MtArgs {
  int rows;
  int n[4];
  double keep[4];
  unsigned char* out[4];
};

__global__ void __launch_bounds__(NT_MT) mt_dropout_kernel(uint32_t* __restrict__ state, const __grid_constant__ MtArgs a) {
  __shared__ uint32_t buf[2][MT_N];
  __shared__ uint32_t carry[2];
  const int tid = threadIdx.x;
  for (int i = tid; i < MT_N; i += NT_MT) buf[0][i] = state[i];
  int p_start = (int)state[MT_N];
  __syncthreads();
  long long off[5];
  off[0] = 0;
  for (int l = 0; l < 4; ++l) off[l + 1] = off[l] + (long long)a.rows * a.n[l];
  const long long total = 2 * off[4];  // words of this batch
  long long c = 0;                     // words consumed before the current block
  int cur = 0, it = 0;
  while (true) {
    const int use = (int)min((long long)(MT_N - p_start), total - c);
    const bool need_next = c + use < total;
    if (tid < NT_TWIST) {
      if (need_next) {
        const uint32_t* o = buf[cur];
        uint32_t* nw = buf[cur ^ 1];
        if (tid < MT_R1) nw[tid] = mt_twist(o[tid], o[tid + 1], o[tid + MT_M]);
        twist_bar();
        if (tid < MT_R1) { const int i = MT_R1 + tid; nw[i] = mt_twist(o[i], o[i + 1], nw[i - MT_R1]); }
        twist_bar();
        if (tid < MT_N - 2 * MT_R1) {
          const int i = 2 * MT_R1 + tid;
          nw[i] = mt_twist(o[i], i + 1 < MT_N ? o[i + 1] : nw[0], nw[i - MT_R1]);
        }
      }
    } else {
      const uint32_t* o = buf[cur];
      for (int w = p_start + tid - NT_TWIST; w < p_start + use; w += NT_MT - NT_TWIST) {
        const long long gw = c + (w - p_start);
        if (gw & 1) {
          const uint32_t hi = w > p_start ? mt_temper(o[w - 1]) : carry[(it + 1) & 1];
          const uint32_t lo = mt_temper(o[w]);
          const unsigned long long r = (((unsigned long long)hi << 32) | lo) & ((1ull << 53) - 1);
          const long long e = gw >> 1;
          const int l = e < off[1] ? 0 : e < off[2] ? 1 : e < off[3] ? 2 : 3;
          a.out[l][e - off[l]] = (double)r * 0x1p-53 < a.keep[l] ? 1 : 0;
        } else if (w == p_start + use - 1) {
          carry[it & 1] = mt_temper(o[w]);  // high word of an element whose low word opens the next block
        }
      }
    }
    __syncthreads();
    c += use;
    if (!need_next) { p_start += use; break; }
    cur ^= 1;
    p_start = 0;
    ++it;
  }
  for (int i = tid; i < MT_N; i += NT_MT) state[i] = buf[cur][i];
  if (tid == 0) state[MT_N] = (uint32_t)p_start;
}

}  // namespace

int bb_mt_dropout_launch(uint32_t* state_dev, int rows, const int* widths_4, const double* keep_4,
                         unsigned char* const* out_4, cudaStream_t s) {
  if (!state_dev || rows < 1 || !widths_4 || !keep_4 || !out_4) return BB_ERR_INVALID;
  MtArgs a;
  a.rows = rows;
  for (int l = 0; l < 4; ++l) { a.n[l] = widths_4[l]; a.keep[l] = keep_4[l]; a.out[l] = out_4[l]; }
  mt_dropout_kernel<<<1, NT_MT, 0, s>>>(state_dev, a);
  return (int)cudaGetLastError();
}
