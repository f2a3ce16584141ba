// fpop_lat.cu -- the LATENCY kernel (sm_100a): one problem per thread block, one chain per warp.
//
// Compiled with -DPSD_G32: the operators of fpop_warp.cuh then use a whole warp (32 lanes) per
// chain instead of a half-warp, and dp_run_latency() (same header) drives the two warps of a block
// through the problem with one block barrier per row.  Used when a wave has fewer problems than
// the GPU has room for (a sequential search on one long chromosome, config 3; the worst-case
// sequences, config 5; single calls of PeakSegFPOP_disk, config 1), where the one-warp-per-problem
// kernel leaves most of the chip idle and a row is one long chain of dependent fp64 instructions.
// Warps 2 and 3 of the block are HELPERS: when an overlap interval's difference function has two roots,
// the chain's main warp solves get_smaller_root while its helper solves get_larger_root (named barriers,
// a mailbox in shared memory), so the two Newton loops run side by side instead of back to back.
// 128 threads per block leave every thread up to 255 registers: no spills; the piece lists get the
// block's whole shared memory (~630 pieces per function with one block per SM).
// Same arithmetic, same store records, same backtrack kernel as the throughput path.
#include <cuda_runtime.h>
#include "dp_params.h"

#if !defined(PSD_G32)
#error "fpop_lat.cu must be compiled with -DPSD_G32"
#endif

static __device__ const uint64_t d_lat_exp_tab[256] = PSD_EXP_TAB_INIT;
static __device__ const uint64_t d_lat_log_tab[256] = PSD_LOG_TAB_INIT;

static_assert(sizeof(LatShared) <= PSD_LAT_SHARED_BYTES, "PSD_LAT_SHARED_BYTES too small");

__global__ void __launch_bounds__(PSD_LAT_THREADS)
fpop_dp_lat_kernel(const DpKernelParams P) {
  uint64_t* etab = (uint64_t*)psd_smem;
  uint64_t* ltab = etab + 256;
  for (int i = threadIdx.x; i < 256; i += blockDim.x) { etab[i] = d_lat_exp_tab[i]; ltab[i] = d_lat_log_tab[i]; }
  LatShared* sh = (LatShared*)(psd_smem + PSD_TAB_BYTES);
  __syncthreads();
  const int b = (int)blockIdx.x;
  if (b >= P.n_order) return;
  const int id = P.order[b];
  WarpWs ws_s, ws_g;
  ws_s.base = psd_smem + PSD_TAB_BYTES + PSD_LAT_SHARED_BYTES;
  ws_s.scratch = nullptr; ws_s.flags = (int*)ws_s.base; ws_s.cap = P.cap_s; ws_s.ccap = P.ccap_s; ws_s.help = nullptr;
  ws_g.base = P.gws ? P.gws + (unsigned long long)b * P.ws_g_bytes : nullptr;
  ws_g.scratch = nullptr; ws_g.flags = ws_s.flags; ws_g.cap = P.gws ? P.cap_g : 0; ws_g.ccap = P.ccap_g; ws_g.help = nullptr;
  const int warp = (int)(threadIdx.x >> 5);
  if (warp >= PSD_LAT_WARPS) { lat_helper_loop(&sh->help[warp - PSD_LAT_WARPS], warp - PSD_LAT_WARPS); return; }   // only launched when P.lat_help
  const DpProblem pb = P.problems[id];
  dp_run_latency(ws_s, ws_g, pb, &P.results[id], P.pool, sh, P.lat_help != 0);
}

int psd_lat_set_smem(size_t smem_bytes) {
  return (int)cudaFuncSetAttribute(fpop_dp_lat_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
}

int psd_lat_resident_blocks(size_t smem_bytes, int helpers) {
  int nb = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, fpop_dp_lat_kernel, helpers ? PSD_LAT_THREADS : PSD_LAT_WARPS * 32, smem_bytes) != cudaSuccess) return 0;
  return nb;
}

// P.lat_help: 128 threads per block (two helper warps), else 64
int psd_lat_launch(const DpKernelParams& P, int grid, size_t smem_bytes, void* stream) {
  fpop_dp_lat_kernel<<<grid, P.lat_help ? PSD_LAT_THREADS : PSD_LAT_WARPS * 32, smem_bytes, (cudaStream_t)stream>>>(P);
  return (int)cudaGetLastError();
}

#if defined(PSD_TIMING)
#include <cstring>
extern "C" int psd_debug_read_lat(unsigned long long* out, int n, int reset) {
  unsigned long long tmp[32];
  if (cudaMemcpyFromSymbol(tmp, psd_dbg, sizeof tmp) != cudaSuccess) return -1;
  for (int i = 0; i < n && i < 32; i++) out[i] = tmp[i];
  if (reset) { memset(tmp, 0, sizeof tmp); cudaMemcpyToSymbol(psd_dbg, tmp, sizeof tmp); }
  return 0;
}
#endif
