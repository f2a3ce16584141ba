// dp_params.h -- launch parameters shared by the two translation units that instantiate the DP:
// fpop_gpu.cu (throughput kernel: one problem per warp, chains on half-warps) and fpop_lat.cu
// (latency kernel: one problem per block, one chain per warp, compiled with -DPSD_G32).
#pragma once
#include "fpop_warp.cuh"

#define PSD_TAB_BYTES 4096          /* exp + log tables at the start of dynamic shared memory */
#define PSD_LAT_SHARED_BYTES 4992   /* LatShared (incl. the helpers' mailboxes), between the tables and the workspace (latency kernel) */
#define PSD_LAT_WARPS 2             /* main warps of a latency block: the up chain and the down chain */
#define PSD_LAT_THREADS 128         /* + two helper warps that solve the larger Newton roots */

struct DpKernelParams {
  const DpProblem* problems;
  const int* order;           // problem ids, longest first
  int n_order;
  int* queue;                 // atomic cursor into order
  DpResult* results;
  StorePool pool;
  int cap_s, ccap_s;          // shared-memory tier (cap_s = 0: disabled, warps start in the global tier)
  unsigned long long ws_s_bytes;   // per warp (per block in the latency kernel), >= PSD_WS_HDR (the header holds the flag words)
  unsigned char* gws;         // per-warp (per-block) global-memory workspaces (null: none)
  int cap_g, ccap_g;
  unsigned long long ws_g_bytes;
  int lat_help;               // latency kernel: the block has two helper warps (128 threads) that solve the larger Newton roots
};

// fpop_lat.cu: the latency kernel.  Block b solves problem order[b] (no queue).
int psd_lat_set_smem(size_t smem_bytes);                                   // cudaFuncSetAttribute; returns a cudaError_t
int psd_lat_resident_blocks(size_t smem_bytes, int helpers);               // occupancy query: blocks per SM
int psd_lat_launch(const DpKernelParams& P, int grid, size_t smem_bytes, void* stream);   // returns a cudaError_t
