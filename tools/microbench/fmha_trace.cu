// Timeline dump of the FMHA kernel (CTA 0): build with
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 --expt-relaxed-constexpr -DLN3_FMHA_TRACE \
//        -Iinclude -Iln3diff_b200/csrc tools/microbench/fmha_trace.cu ln3diff_b200/csrc/*.cu -o tools/microbench/fmha_trace
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "ln3b200.h"
namespace ln3 { int fmha_trace_copy(long long* host); }

int main(int argc, char** argv) {
  const int B = 16, H = 16, L = 768, Lkv = argc > 1 ? atoi(argv[1]) : 768;
  const size_t nq = size_t(B) * L * H * 64, nk = size_t(B) * Lkv * H * 64;
  std::vector<__nv_bfloat16> h(nq);
  srand(1);
  for (auto& v : h) v = __float2bfloat16((rand() / float(RAND_MAX) - 0.5f));
  __nv_bfloat16 *q, *k, *v, *o;
  cudaMalloc(&q, nq * 2); cudaMalloc(&k, nk * 2); cudaMalloc(&v, nk * 2); cudaMalloc(&o, nq * 2);
  cudaMemcpy(q, h.data(), nq * 2, cudaMemcpyHostToDevice);
  cudaMemcpy(k, h.data(), nk * 2, cudaMemcpyHostToDevice);
  cudaMemcpy(v, h.data(), nk * 2, cudaMemcpyHostToDevice);
  ln3_fmha_args a = {};
  a.q = q; a.k = k; a.v = v; a.out = o;
  a.B = B; a.H = H; a.Lq = L; a.Lkv = Lkv; a.head_dim = 64;
  a.q_ld = a.k_ld = a.v_ld = a.o_ld = H * 64;
  a.q_bs = a.o_bs = (long long)L * H * 64;
  a.k_bs = a.v_bs = (long long)Lkv * H * 64;
  a.scale = 0.125f;
  for (int i = 0; i < 3; ++i)
    if (ln3_fmha_fwd(&a, nullptr) != 0) { printf("error: %s\n", ln3_last_error()); return 1; }
  cudaDeviceSynchronize();
  // WG slots 0 wait S | 1 S ready | 2 S in regs | 3 max done | 4 o_full(prev) | 6 exps done | 7 P handed |
  // 8-10 epilogue (slot 5 is not recorded); MMA slots 0-2 QK_t issued | 3/5/7 p_full_t seen | 4/6/8 PV_t issued
  static long long tr[4][64][12];
  if (ln3::fmha_trace_copy(&tr[0][0][0])) { printf("trace copy failed\n"); return 1; }
  long long t0 = tr[3][0][0];
  printf("# role blk: slots (cycles since first event)\n");
  for (int g = 0; g < 26; ++g) {
    for (int r = 0; r < 4; ++r) {
      printf("%s g=%2d:", r == 0 ? "WG0" : r == 1 ? "WG1" : r == 2 ? "WG2" : "MMA", g);
      for (int s = 0; s < (r == 3 ? 9 : 11); ++s) {
        const long long v = tr[r][g][s];
        if (v == 0) printf("       -"); else printf(" %7lld", v - t0);
      }
      printf("\n");
    }
  }
  return 0;
}
