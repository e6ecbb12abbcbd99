// Micro-benchmark of the Scc assembly patterns (config 2: 1000 cameras, 100k landmarks x 10 observations).
// atomic: FP64 atomicAdd throughput into 36-double blocks
//   A: one lane per (pair -> block), 36 sequential REDs per lane (32 different sectors per instruction)
//   B: one warp per pair, lanes 0..35 cover the block (9-10 sectors per instruction)
// gather: schur_gather_kernel itself on config 2's pair lists (landmark cameras as synth.ba_scene draws them: random
//   first camera, stride 1..3), reading 288 B of GE records per entry from a 288 MB GE; both work orders, with L2
//   flushed before each launch (cold) and back to back (warm)
// nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a tools/atomic_bench.cu -o tools/atomic_bench
// tools/atomic_bench [atomic|gather]   (default: both)
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <vector>
#include <cuda_runtime.h>
#include "../openmvg_b200/csrc/ba_kernels.cuh"
__global__ void varA(const int *__restrict__ blk, int npairs, double *__restrict__ S) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x; if (p >= npairs) return;
  double *b = S + 36 * (size_t)blk[p];
  #pragma unroll
  for (int e = 0; e < 36; ++e) atomicAdd(b + e, 1.0 + e);
}
__global__ void varB(const int *__restrict__ blk, int npairs, double *__restrict__ S) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31, nw = (gridDim.x * blockDim.x) >> 5;
  for (int p0 = warp * 32; p0 < npairs; p0 += nw * 32) {
    const int mine = p0 + lane < npairs ? blk[p0 + lane] : -1;
    for (int q = 0; q < 32; ++q) {
      const int bi = __shfl_sync(0xffffffffu, mine, q); if (bi < 0) break;
      double *b = S + 36 * (size_t)bi;
      atomicAdd(b + lane, 1.0 + lane);
      if (lane < 4) atomicAdd(b + 32 + lane, 33.0 + lane);
    }
  }
}
static void gather_probe() {
  const int nc = 1000, np = 100000, K = 10; const long long no = (long long)np * K;
  std::mt19937_64 rng(42);
  std::vector<int> cam(no);
  for (int j = 0; j < np; ++j) { const int s0 = (int)(rng() % nc), st = 1 + j % 3; for (int k = 0; k < K; ++k) cam[(size_t)j * K + k] = (s0 + k * st) % nc; }
  // BSR structure of Scc: rows sorted, diagonal always present
  std::vector<std::vector<int>> rows(nc);
  for (int a = 0; a < nc; ++a) rows[a].push_back(a);
  for (int j = 0; j < np; ++j) for (int t = 0; t < K; ++t) for (int u = 0; u < K; ++u) rows[cam[(size_t)j * K + t]].push_back(cam[(size_t)j * K + u]);
  std::vector<int> hp(nc + 1, 0), hcols, brow;
  for (int a = 0; a < nc; ++a) { auto &r = rows[a]; std::sort(r.begin(), r.end()); r.erase(std::unique(r.begin(), r.end()), r.end()); hp[a + 1] = hp[a] + (int)r.size();
    for (int b : r) { hcols.push_back(b); brow.push_back(a); } }
  const int nnzb = hp[nc];
  auto find = [&](int a, int b) { return (int)(std::lower_bound(hcols.begin() + hp[a], hcols.begin() + hp[a + 1], b) - hcols.begin()); };
  double *GE, *FtF, *Scc, *flush; int *d_brow;
  cudaMalloc(&GE, 36 * no * 8); cudaMalloc(&FtF, 36 * nc * 8); cudaMalloc(&Scc, (size_t)nnzb * 36 * 8); cudaMalloc(&flush, 512ull << 20); cudaMalloc(&d_brow, nnzb * 4);
  { std::vector<double> h(36 * no); for (auto &x : h) x = (double)(rng() % 2001) * 1e-3 - 1.0; cudaMemcpy(GE, h.data(), h.size() * 8, cudaMemcpyHostToDevice); }
  cudaMemset(FtF, 0, 36 * nc * 8); cudaMemcpy(d_brow, brow.data(), nnzb * 4, cudaMemcpyHostToDevice);
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  for (int order = 0; order < 2; ++order) {      // 0: diagonal blocks first, then row by row (as ba.cu); 1: row by row, diagonal first in its row
    std::vector<int> wpos(nnzb, -1), gblk, gblkT;
    if (order == 0) for (int a = 0; a < nc; ++a) { const int e = find(a, a); wpos[e] = (int)gblk.size(); gblk.push_back(e); gblkT.push_back(e); }
    for (int a = 0; a < nc; ++a) for (int e = hp[a]; e < hp[a + 1]; ++e) { const int b = hcols[e]; if (b < a || (b == a && order == 0)) continue;
      wpos[e] = (int)gblk.size(); gblk.push_back(e); gblkT.push_back(find(b, a)); }
    const int nwork = (int)gblk.size();
    std::vector<std::vector<int2>> lists(nwork);
    for (int j = 0; j < np; ++j) for (int t = 0; t < K; ++t) for (int u = 0; u < K; ++u) {
      const int tt = j * K + t, uu = j * K + u; if (cam[uu] < cam[tt]) continue;
      lists[wpos[find(cam[tt], cam[uu])]].push_back(make_int2(tt, uu)); }
    std::vector<int> gstart(nwork + 1, 0); std::vector<int2> pairs;
    for (int w = 0; w < nwork; ++w) { pairs.insert(pairs.end(), lists[w].begin(), lists[w].end()); gstart[w + 1] = (int)pairs.size(); }
    int *d_gs, *d_gb, *d_gt; int2 *d_pairs;
    cudaMalloc(&d_gs, (nwork + 1) * 4); cudaMalloc(&d_gb, nwork * 4); cudaMalloc(&d_gt, nwork * 4); cudaMalloc(&d_pairs, pairs.size() * 8);
    cudaMemcpy(d_gs, gstart.data(), (nwork + 1) * 4, cudaMemcpyHostToDevice); cudaMemcpy(d_gb, gblk.data(), nwork * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(d_gt, gblkT.data(), nwork * 4, cudaMemcpyHostToDevice); cudaMemcpy(d_pairs, pairs.data(), pairs.size() * 8, cudaMemcpyHostToDevice);
    const unsigned grid = (unsigned)(((long long)nwork * 32 + omvg::ba::GATHER_THREADS - 1) / omvg::ba::GATHER_THREADS);
    const double bytes = pairs.size() * 288.0;
    for (int cold = 1; cold >= 0; --cold) {
      float best = 1e30f, sum = 0; const int reps = 10;
      for (int rep = 0; rep < reps + 1; ++rep) {
        if (cold) cudaMemset(flush, rep & 1, 512ull << 20);
        float ms;
        cudaEventRecord(e0);
        omvg::ba::schur_gather_kernel<<<grid, omvg::ba::GATHER_THREADS>>>(GE, d_gs, d_pairs, d_gb, d_gt, nwork, d_brow, FtF, Scc);
        cudaEventRecord(e1); cudaEventSynchronize(e1); cudaEventElapsedTime(&ms, e0, e1);
        if (rep == 0) continue;                  // first launch: module load
        best = std::min(best, ms); sum += ms;
      }
      printf("gather order %s, %s L2: %d upper blocks, %zu entries (%.1f MB lists), %.1f GB of GE records: best %.1f us, mean %.1f us, %.2f TB/s L2->SM\n",
             order == 0 ? "diagonal-first" : "row-major     ", cold ? "cold" : "warm", nwork, pairs.size(), pairs.size() * 8e-6, bytes * 1e-9,
             best * 1e3, sum / reps * 1e3, bytes / (best * 1e-3) * 1e-12);
    }
    cudaFree(d_gs); cudaFree(d_gb); cudaFree(d_gt); cudaFree(d_pairs);
  }
  cudaFree(GE); cudaFree(FtF); cudaFree(Scc); cudaFree(flush); cudaFree(d_brow);
}

static void atomic_probe() {
  const int npairs = 5500000, nblocks = 28000;
  std::vector<int> h(npairs); srand(1);
  // pairs of consecutive "points" hit nearby blocks (as in the real scene), otherwise random
  for (int i = 0; i < npairs; ++i) h[i] = (int)(((long long)rand() * 7919 + i / 55) % nblocks);
  int *d; double *S; cudaMalloc(&d, npairs * 4); cudaMalloc(&S, (size_t)nblocks * 36 * 8);
  cudaMemcpy(d, h.data(), npairs * 4, cudaMemcpyHostToDevice); cudaMemset(S, 0, (size_t)nblocks * 36 * 8);
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  for (int rep = 0; rep < 3; ++rep) {
    float ms;
    cudaEventRecord(e0); varA<<<(npairs + 127) / 128, 128>>>(d, npairs, S); cudaEventRecord(e1); cudaEventSynchronize(e1); cudaEventElapsedTime(&ms, e0, e1);
    printf("A lane-per-block : %.3f ms  %.1f G atomics/s\n", ms, npairs * 36.0 / ms / 1e6);
    cudaEventRecord(e0); varB<<<148 * 8, 256>>>(d, npairs, S); cudaEventRecord(e1); cudaEventSynchronize(e1); cudaEventElapsedTime(&ms, e0, e1);
    printf("B warp-per-block : %.3f ms  %.1f G atomics/s\n", ms, npairs * 36.0 / ms / 1e6);
  }
}

int main(int argc, char **argv) {
  const char *mode = argc > 1 ? argv[1] : "all";
  if (strcmp(mode, "gather") != 0) atomic_probe();
  if (strcmp(mode, "atomic") != 0) gather_probe();
  printf("%s\n", cudaGetErrorString(cudaGetLastError()));
  return 0;
}
