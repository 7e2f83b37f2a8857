// population_copy_ab.cu -- which copy form population_copy_kernel (csrc/mlp.cu) should use, measured rather than guessed.
// A standalone program: k pairs (dst, src) of agent rows, three arrays (weights, Adam m, Adam v) of `stride` floats each, copied
//   ldg128  as population_copy_kernel: CTAs of 256 threads, each thread 4 independent 16-byte loads in flight before its stores
//   bulk    cp.async.bulk through shared memory: one thread per CTA moves a 16 KB chunk global -> shared (mbarrier) -> global
// for the default networks (stride 6 152) and a 128-wide actor (stride 19 592), alternating the two forms.  Every time is a median
// of CUDA-event intervals over one launch after warm-up, with a 256 MB write between launches (the 126 MB L2 holds no row).
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o /tmp/copy_ab scripts/population_copy_ab.cu && /tmp/copy_ab
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <numeric>
#include <random>
#include <vector>

#include <cuda_runtime.h>

#define CK(x)                                                                                    \
  do {                                                                                           \
    cudaError_t e_ = (x);                                                                        \
    if (e_ != cudaSuccess) {                                                                     \
      fprintf(stderr, "%s:%d %s: %s\n", __FILE__, __LINE__, #x, cudaGetErrorString(e_));         \
      return 1;                                                                                  \
    }                                                                                            \
  } while (0)

constexpr int kThreads = 256, kIlp = 4, kBulkBytes = 16384;

__global__ void __launch_bounds__(kThreads) copy_ldg128(float* p, float* m, float* v, const int32_t* pairs, int stride) {
  constexpr int kChunk = kThreads * kIlp;
  const int row4 = stride / 4, chunks = (row4 + kChunk - 1) / kChunk;
  const int pair = blockIdx.x / chunks, first = (blockIdx.x - pair * chunks) * kChunk + threadIdx.x;
  float* base = blockIdx.y == 0 ? p : blockIdx.y == 1 ? m : v;
  const float4* from = reinterpret_cast<const float4*>(base + (size_t)pairs[2 * pair + 1] * stride);
  float4* to = reinterpret_cast<float4*>(base + (size_t)pairs[2 * pair] * stride);
  float4 r[kIlp];
#pragma unroll
  for (int k = 0; k < kIlp; k++)
    if (first + k * kThreads < row4) r[k] = from[first + k * kThreads];
#pragma unroll
  for (int k = 0; k < kIlp; k++)
    if (first + k * kThreads < row4) to[first + k * kThreads] = r[k];
}

__device__ __forceinline__ uint32_t smem_u32(const void* q) { return (uint32_t)__cvta_generic_to_shared(q); }

__global__ void __launch_bounds__(32) copy_bulk(float* p, float* m, float* v, const int32_t* pairs, int stride) {
  __shared__ alignas(128) char buf[kBulkBytes];
  __shared__ alignas(8) unsigned long long bar;
  const int row_bytes = stride * 4, chunks = (row_bytes + kBulkBytes - 1) / kBulkBytes;
  const int pair = blockIdx.x / chunks, off = (blockIdx.x - pair * chunks) * kBulkBytes;
  const uint32_t bytes = (uint32_t)min(kBulkBytes, row_bytes - off);
  float* base = blockIdx.y == 0 ? p : blockIdx.y == 1 ? m : v;
  const char* from = reinterpret_cast<const char*>(base + (size_t)pairs[2 * pair + 1] * stride) + off;
  char* to = reinterpret_cast<char*>(base + (size_t)pairs[2 * pair] * stride) + off;
  if (threadIdx.x != 0) return;
  asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&bar)) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&bar)), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(buf)),
               "l"(from), "r"(bytes), "r"(smem_u32(&bar))
               : "memory");
  uint32_t ok = 0;
  while (!ok)
    asm volatile("{\n\t.reg .pred q;\n\tmbarrier.try_wait.parity.shared::cta.b64 q, [%1], 0;\n\tselp.b32 %0, 1, 0, q;\n\t}"
                 : "=r"(ok)
                 : "r"(smem_u32(&bar))
                 : "memory");
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(to), "r"(smem_u32(buf)), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

int main() {
  const int P = 32768;
  const int strides[2] = {6152, 19592};
  const int ks[4] = {1, 148, 1024, 16384};
  const int reps = 40;
  float* flush = nullptr;
  CK(cudaMalloc(&flush, 256u << 20));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, 0));
  printf("device %s\n", prop.name);
  printf("stride k form median_us min_us GB/s share_of_7.7TBps\n");
  for (int stride : strides) {
    const size_t bytes = sizeof(float) * (size_t)P * stride;
    float *p, *m, *v;
    CK(cudaMalloc(&p, bytes));
    CK(cudaMalloc(&m, bytes));
    CK(cudaMalloc(&v, bytes));
    std::vector<float> init((size_t)P * stride);
    for (size_t i = 0; i < init.size(); i++) init[i] = (float)(i % 9973);
    CK(cudaMemcpy(p, init.data(), bytes, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(m, init.data(), bytes, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(v, init.data(), bytes, cudaMemcpyHostToDevice));
    for (int k : ks) {
      std::vector<int> perm(P);
      std::iota(perm.begin(), perm.end(), 0);
      std::shuffle(perm.begin(), perm.end(), std::mt19937(k));
      std::vector<int32_t> pairs(2 * k);
      for (int i = 0; i < k; i++) pairs[2 * i] = perm[i], pairs[2 * i + 1] = perm[k + i];
      int32_t* d_pairs;
      CK(cudaMalloc(&d_pairs, sizeof(int32_t) * 2 * k));
      CK(cudaMemcpy(d_pairs, pairs.data(), sizeof(int32_t) * 2 * k, cudaMemcpyHostToDevice));
      const int ldg_chunks = (stride / 4 + kThreads * kIlp - 1) / (kThreads * kIlp);
      const int bulk_chunks = (stride * 4 + kBulkBytes - 1) / kBulkBytes;
      std::vector<float> ms[2];
      for (int r = 0; r < reps + 3; r++)
        for (int form = 0; form < 2; form++) {
          CK(cudaMemset(flush, r & 0xff, 256u << 20));
          cudaEvent_t a, b;
          CK(cudaEventCreate(&a));
          CK(cudaEventCreate(&b));
          CK(cudaEventRecord(a));
          if (form == 0)
            copy_ldg128<<<dim3(k * ldg_chunks, 3), kThreads>>>(p, m, v, d_pairs, stride);
          else
            copy_bulk<<<dim3(k * bulk_chunks, 3), 32>>>(p, m, v, d_pairs, stride);
          CK(cudaGetLastError());
          CK(cudaEventRecord(b));
          CK(cudaEventSynchronize(b));
          float t;
          CK(cudaEventElapsedTime(&t, a, b));
          if (r >= 3) ms[form].push_back(t);
          CK(cudaEventDestroy(a));
          CK(cudaEventDestroy(b));
        }
      // every dst row equals its src row in the three arrays
      std::vector<float> row_d(stride), row_s(stride);
      for (float* base : {p, m, v})
        for (int i = 0; i < k; i += std::max(1, k / 16)) {
          CK(cudaMemcpy(row_d.data(), base + (size_t)pairs[2 * i] * stride, sizeof(float) * stride, cudaMemcpyDeviceToHost));
          CK(cudaMemcpy(row_s.data(), base + (size_t)pairs[2 * i + 1] * stride, sizeof(float) * stride, cudaMemcpyDeviceToHost));
          if (memcmp(row_d.data(), row_s.data(), sizeof(float) * stride) != 0) {
            fprintf(stderr, "stride %d k %d pair %d: dst differs from src\n", stride, k, i);
            return 1;
          }
        }
      const double moved = 2.0 * 3 * sizeof(float) * stride * (double)k;  // read + write of three rows per pair
      for (int form = 0; form < 2; form++) {
        std::sort(ms[form].begin(), ms[form].end());
        const double med = ms[form][ms[form].size() / 2] * 1e-3;
        printf("%d %d %s %.2f %.2f %.1f %.3f\n", stride, k, form == 0 ? "ldg128" : "bulk", med * 1e6, ms[form][0] * 1e3, moved / med * 1e-9,
               moved / med / 7.7e12);
      }
      CK(cudaFree(d_pairs));
    }
    CK(cudaFree(p));
    CK(cudaFree(m));
    CK(cudaFree(v));
  }
  return 0;
}
