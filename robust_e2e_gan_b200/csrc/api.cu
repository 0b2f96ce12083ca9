// C-ABI bookkeeping: version, build info, error strings, launch counter.
#include <cuda_runtime.h>

#include "common.cuh"

#include <atomic>
#include <map>
#include <mutex>
#include <utility>

namespace re2e {
std::atomic<unsigned long long> g_launches{0};

// the attribute is per (device, function): a process driving several GPUs must set it on each of them
int ensure_smem(const void *func, size_t bytes) {
  static std::mutex mu;
  static std::map<std::pair<int, const void *>, size_t> seen;
  if (bytes > 227 * 1024) return RE2E_E_UNSUPPORTED;
  if (bytes <= 48 * 1024) return RE2E_OK;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return (int)e;
  std::lock_guard<std::mutex> lk(mu);
  auto key = std::make_pair(dev, func);
  auto it = seen.find(key);
  if (it != seen.end() && it->second >= bytes) return RE2E_OK;
  e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) return (int)e;
  seen[key] = bytes;
  return RE2E_OK;
}

int num_sms() {
  static std::mutex mu;
  static std::map<int, int> cache;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  std::lock_guard<std::mutex> lk(mu);
  auto it = cache.find(dev);
  if (it != cache.end()) return it->second;
  int sms = 148;
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) sms = 148;
  cache[dev] = sms;
  return sms;
}
}  // namespace re2e

namespace re2e {
namespace {
// Column sums of a row-major matrix (bias gradients of the dense layers: db = sum over rows of dY), deterministic:
//   pass 1  block (cb, rb): 128 columns x kColRows rows -> partial[rb][c]   (coalesced 512 B row segments, 8 rows
//           in flight per thread)
//   pass 2  out[c] = sum_rb partial[rb][c] in a fixed order
constexpr int kColRows = 128;
__global__ void __launch_bounds__(128) colsum_partial_kernel(const float *__restrict__ X, long long ld, int rows,
                                                              int cols, float *__restrict__ partial) {
  const int c = blockIdx.x * 128 + threadIdx.x;
  const int r0 = blockIdx.y * kColRows, r1 = min(rows, r0 + kColRows);
  if (c >= cols) return;
  const float *p = X + (size_t)r0 * ld + c;
  float a[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) a[i] = 0.0f;
  int r = r0;
  for (; r + 8 <= r1; r += 8) {
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] += __ldg(p + (size_t)i * ld);
    p += (size_t)8 * ld;
  }
  for (; r < r1; ++r) { a[0] += __ldg(p); p += ld; }
  partial[(size_t)blockIdx.y * cols + c] = ((a[0] + a[1]) + (a[2] + a[3])) + ((a[4] + a[5]) + (a[6] + a[7]));
}
__global__ void __launch_bounds__(128) colsum_final_kernel(const float *__restrict__ partial, int nrb, int cols,
                                                            float *__restrict__ out) {
  const int c = blockIdx.x * 128 + threadIdx.x;
  if (c >= cols) return;
  float s = 0.0f;
  for (int rb = 0; rb < nrb; ++rb) s += partial[(size_t)rb * cols + c];
  out[c] = s;
}
}  // namespace
}  // namespace re2e

extern "C" int re2e_colsum_blocks(int rows) { return rows > 0 ? (rows + re2e::kColRows - 1) / re2e::kColRows : 0; }

extern "C" int re2e_colsum(const float *X, long long ld, int rows, int cols, float *partial, float *out,
                           void *stream) {
  RE2E_CHECK_ARG(X && partial && out && rows > 0 && cols > 0 && ld >= cols);
  using namespace re2e;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int nrb = re2e_colsum_blocks(rows);
  dim3 grid((cols + 127) / 128, nrb);
  colsum_partial_kernel<<<grid, 128, 0, st>>>(X, ld, rows, cols, partial);
  colsum_final_kernel<<<(cols + 127) / 128, 128, 0, st>>>(partial, nrb, cols, out);
  count_launch(2);
  return launch_status();
}

extern "C" int re2e_abi_version(void) { return 8; }

extern "C" const char *re2e_build_info(void) {
  return "re2e_b200 sm_100a nvcc " __DATE__ " " __TIME__
#if RE2E_HAS_TCGEN05
         " tcgen05"
#endif
      ;
}

extern "C" const char *re2e_error_string(int code) {
  switch (code) {
    case RE2E_OK: return "ok";
    case RE2E_E_ARG: return "re2e: bad argument (null pointer, non-positive size or misaligned buffer)";
    case RE2E_E_UNSUPPORTED: return "re2e: shape not supported by the sm_100a kernels";
    case RE2E_E_WORKSPACE: return "re2e: workspace too small";
    default: break;
  }
  if (code > 0) return cudaGetErrorString(static_cast<cudaError_t>(code));
  return "re2e: unknown error";
}

extern "C" unsigned long long re2e_launch_count(void) { return re2e::g_launches.load(std::memory_order_relaxed); }
