/*
 * Plain-C user of the drop-in boundary (include/pa_b200.h): no Python, no
 * torch, no C++ -- what a foreign-language binding (Julia ccall, cgo, ...) sees.
 * One rank, process grid (1,1): x-pencil -> y-pencil (perm (2,3,1)) -> z-pencil
 * (perm (3,2,1)) of a 24x20x12 Float64 array, checked against the definition
 *     parent(u)[perm * I] == global[I]        (arrays.jl:19-31, 327-337)
 * evaluated with naive loops here.  Exit codes: 0 ok, 2 no GPU (the library
 * refused: there is no CPU fallback), 1 anything else.
 * Usage: c_abi_harness FILE -- FILE is the scratch path of the PencilIO check.
 * Built and run by tests/test_c_abi_harness.py.
 */
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <cuda_runtime_api.h>

#include "pa_b200.h"

#define CHECK(call)                                                                      \
  do {                                                                                   \
    pa_status s_ = (call);                                                               \
    if (s_ != PA_OK) {                                                                   \
      fprintf(stderr, "%s -> %s: %s\n", #call, pa_strerror(s_), pa_last_error());        \
      return s_ == PA_ENOGPU ? 2 : 1;                                                    \
    }                                                                                    \
  } while (0)

/* value of the element at 0-based logical index (i,j,k) */
static double val(int64_t i, int64_t j, int64_t k) { return (double)(i + 100 * j + 10000 * k) + 0.5; }

/* offset of logical index I in a parent with memory order perm (1-based), dims n[] */
static int64_t off(const int* perm, const int64_t* n, const int64_t* I) {
  int64_t o = 0, run = 1;
  for (int m = 0; m < 3; ++m) {
    int l = perm[m] - 1;
    o += I[l] * run;
    run *= n[l];
  }
  return o;
}

int main(int argc, char** argv) {
  if (argc != 2) {
    fprintf(stderr, "usage: %s SCRATCH_FILE\n", argv[0]);
    return 1;
  }
  const int64_t n[3] = {24, 20, 12};
  const int64_t pdims[2] = {1, 1};
  const int dx[2] = {2, 3}, dy[2] = {1, 3}, dz[2] = {1, 2};
  const int px[3] = {1, 2, 3}, py[3] = {2, 3, 1}, pz[3] = {3, 2, 1};
  const int64_t N = 24 * 20 * 12;

  printf("%s, %d device(s)\n", pa_version(), pa_device_count());
  pa_topology* topo = NULL;
  pa_pencil *penx = NULL, *peny = NULL, *penz = NULL;
  pa_plan *xy = NULL, *yz = NULL, *bad = NULL;
  CHECK(pa_topology_create(2, pdims, 0, &topo));
  CHECK(pa_pencil_create(topo, 3, n, dx, NULL, NULL, &penx));
  CHECK(pa_pencil_create(topo, 3, n, dy, py, penx, &peny));   /* shares the staging arenas */
  CHECK(pa_pencil_create(topo, 3, n, dz, pz, peny, &penz));
  CHECK(pa_plan_create(penx, peny, 0, NULL, 8, PA_POINT_TO_POINT, &xy));
  CHECK(pa_plan_create(peny, penz, 0, NULL, 8, PA_ALLTOALLV, &yz));
  /* x -> z differs in two decomposed dimensions: ArgumentError (test/transpose.jl:44-45) */
  if (pa_plan_create(penx, penz, 0, NULL, 8, PA_POINT_TO_POINT, &bad) != PA_EINCOMPAT) {
    fprintf(stderr, "x->z should be refused\n");
    return 1;
  }
  pa_plan_info info;
  CHECK(pa_plan_get_info(xy, &info));
  if (info.dim != 1 || info.nproc != 1 || info.length_in != N) return 1;
  int64_t lo[3], hi[3];
  CHECK(pa_pencil_range(peny, NULL, 1, lo, hi)); /* memory order of perm (2,3,1): (20,12,24) */
  if (hi[0] != 20 || hi[1] != 12 || hi[2] != 24) return 1;

  double* h = (double*)malloc(sizeof(double) * N);
  double* g = (double*)malloc(sizeof(double) * N);
  for (int64_t k = 0; k < n[2]; ++k)
    for (int64_t j = 0; j < n[1]; ++j)
      for (int64_t i = 0; i < n[0]; ++i) {
        const int64_t I[3] = {i, j, k};
        h[off(px, n, I)] = val(i, j, k);
      }

  void *ux = NULL, *uy = NULL, *uz = NULL;
  if (pa_device_count() == 0) {
    /* the data path must refuse, not fall back */
    pa_status s = pa_transpose(xy, NULL, h, g, PA_WAITALL, NULL);
    printf("no device: pa_transpose -> %s\n", pa_strerror(s));
    return s == PA_ENOGPU ? 2 : 1;
  }
  CHECK(pa_set_device(0));
  if (cudaMalloc(&ux, sizeof(double) * N) || cudaMalloc(&uy, sizeof(double) * N) ||
      cudaMalloc(&uz, sizeof(double) * N))
    return 1;
  cudaMemcpy(ux, h, sizeof(double) * N, cudaMemcpyHostToDevice);
  CHECK(pa_transpose(xy, NULL, ux, uy, PA_WAITALL, NULL));                   /* fused K3 */
  CHECK(pa_transpose(yz, NULL, uy, uz, PA_WAITALL | PA_STAGE_SELF, NULL));   /* K1 + K2 via recv_buf */
  CHECK(pa_wait(yz, NULL));
  if (cudaDeviceSynchronize() != cudaSuccess) return 1;

  const int* perms[2] = {py, pz};
  void* arrs[2] = {uy, uz};
  for (int a = 0; a < 2; ++a) {
    cudaMemcpy(g, arrs[a], sizeof(double) * N, cudaMemcpyDeviceToHost);
    for (int64_t k = 0; k < n[2]; ++k)
      for (int64_t j = 0; j < n[1]; ++j)
        for (int64_t i = 0; i < n[0]; ++i) {
          const int64_t I[3] = {i, j, k};
          double want = val(i, j, k), got = g[off(perms[a], n, I)];
          if (memcmp(&want, &got, sizeof want) != 0) {
            fprintf(stderr, "mismatch in array %d at (%lld,%lld,%lld)\n", a, (long long)i,
                    (long long)j, (long long)k);
            return 1;
          }
        }
  }
  /* host entry point: H2D + transpose! + D2H */
  memset(g, 0, sizeof(double) * N);
  CHECK(pa_transpose_host(xy, NULL, h, g, PA_WAITALL));
  for (int64_t k = 0; k < n[2]; ++k)
    for (int64_t j = 0; j < n[1]; ++j)
      for (int64_t i = 0; i < n[0]; ++i) {
        const int64_t I[3] = {i, j, k};
        if (g[off(py, n, I)] != val(i, j, k)) return 1;
      }
  /* host chain: x -> y -> z on host arrays, two submits in flight (pa_host_chain_*) */
  {
    pa_plan* chain_plans[2] = {xy, yz};
    pa_host_chain* hc = NULL;
    CHECK(pa_host_chain_create(2, chain_plans, NULL, &hc));
    double* g2 = (double*)malloc(sizeof(double) * N);
    int64_t t0 = -1, t1 = -1;
    CHECK(pa_host_chain_submit(hc, h, g, &t0));
    CHECK(pa_host_chain_submit(hc, h, g2, &t1));
    CHECK(pa_host_chain_wait(hc, t1));
    CHECK(pa_host_chain_wait(hc, -1));
    if (t0 != 0 || t1 != 1) return 1;
    for (int64_t k = 0; k < n[2]; ++k)
      for (int64_t j = 0; j < n[1]; ++j)
        for (int64_t i = 0; i < n[0]; ++i) {
          const int64_t I[3] = {i, j, k};
          if (g[off(pz, n, I)] != val(i, j, k) || g2[off(pz, n, I)] != val(i, j, k)) return 1;
        }
    pa_host_chain_destroy(hc);
    free(g2);
  }
  /* PencilIO layout: the file is the global array in the pencil's MEMORY order
   * (mpi_io.jl:372-380): written from the device, checked byte for byte, read back */
  {
    const char* path = argv[1];
    FILE* f = fopen(path, "wb");
    if (!f) return 1;
    fclose(f);
    int64_t gbytes = 0;
    CHECK(pa_io_sizes(peny, 0, NULL, 8, 0, &gbytes, NULL, NULL, NULL, NULL));
    if (gbytes != (int64_t)sizeof(double) * N) return 1;
    CHECK(pa_io_write(peny, 0, NULL, 8, 0, uy, path, 0));
    f = fopen(path, "rb");
    if (!f || fread(g, sizeof(double), (size_t)N, f) != (size_t)N) return 1;
    fclose(f);
    for (int64_t k = 0; k < n[2]; ++k)
      for (int64_t j = 0; j < n[1]; ++j)
        for (int64_t i = 0; i < n[0]; ++i) {
          const int64_t I[3] = {i, j, k};
          if (g[off(py, n, I)] != val(i, j, k)) return 1;  /* one rank: file == parent(uy) */
        }
    cudaMemset(uz, 0, sizeof(double) * N);
    CHECK(pa_io_read(peny, 0, NULL, 8, 0, uz, path, 0));
    cudaMemcpy(g, uz, sizeof(double) * N, cudaMemcpyDeviceToHost);
    for (int64_t q = 0; q < N; ++q) {
      double a;
      cudaMemcpy(&a, (double*)uy + q, sizeof a, cudaMemcpyDeviceToHost);
      if (memcmp(&a, &g[q], sizeof a) != 0) return 1;
      q += 997;  /* sample */
    }
    remove(path);
  }
  /* the fused unpack+FFT is for ComplexF64 only: a Float64 plan must be refused, not computed */
  if (pa_transpose(xy, NULL, ux, uy, PA_WAITALL | PA_FFT_FORWARD, NULL) != PA_EINVAL) {
    fprintf(stderr, "PA_FFT_FORWARD on Float64 should be refused\n");
    return 1;
  }
  printf("C ABI harness OK: x->y->z bit-exact, %lld kernel launches\n", (long long)pa_launch_count());
  pa_plan_destroy(xy);
  pa_plan_destroy(yz);
  pa_pencil_destroy(penz);
  pa_pencil_destroy(peny);
  pa_pencil_destroy(penx);
  pa_topology_destroy(topo);
  cudaFree(ux);
  cudaFree(uy);
  cudaFree(uz);
  free(h);
  free(g);
  return 0;
}
