// mhb_sort.cuh -- on-device LSD radix sort of fixed-width records (8-bit digits, one sweep per digit): the pieces the
// stable sort pass (mhb_sort3.cuh) and the unstable partition pass (mhb_part.cuh) share.
//
// Replaces kmlib::kmsort (voutcn/megahit src/kmlib/kmsort.h:43-122, an in-place MSD byte radix +
// insertion sort run per 16-bit bucket on the CPU) with a stable LSD sort over whole-array passes:
// same total order on the key (kmsort_selector.cpp:18-27), ties left in input order.
#pragma once
#include "mhb_kernels.cuh"

namespace mhb {

// exclusive scan of a 256-bin histogram (one block of 256 threads) -> where each digit's records start, as a
// BYTE ADDRESS: out + offset * rec_bytes.  (The pass kernels take per-digit addresses so that the partition pass can
// scatter straight into other GPUs' memory, see mhb_partition_scatter.)
__global__ void k_hist_scan256(const u64 *hist, u64 *bin_addr, u64 out_addr, u32 rec_bytes) {
  __shared__ u64 s[256];
  const u32 t = threadIdx.x;
  s[t] = hist[t];
  __syncthreads();
  for (int d = 1; d < 256; d <<= 1) {
    u64 v = t >= (u32)d ? s[t - d] : 0;
    __syncthreads();
    s[t] += v;
    __syncthreads();
  }
  bin_addr[t] = out_addr + (s[t] - hist[t]) * rec_bytes;
}

// standalone digit histogram (only needed when the producer of the records did not provide one)
template <int WR>
__global__ void k_hist_byte(const u32 *in, u64 n, int byte_idx, u64 *hist) {
  __shared__ u32 s_h[256];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) s_h[i] = 0;
  __syncthreads();
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    u32 r[WR];
    ld_rec<WR>(in, i, r);
    atomicAdd(&s_h[rec_byte<WR>(r, byte_idx)], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 256; i += blockDim.x)
    if (s_h[i]) atomicAdd((unsigned long long *)&hist[i], (unsigned long long)s_h[i]);
}

// digit = byte `bsel` of word `widx` of the record (both warp-uniform, hoisted out of the loops)
template <int WR>
__device__ __forceinline__ u32 rec_digit(const u32 (&r)[WR], u32 widx, u32 bsel) {
  u32 w;
  if constexpr (WR == 1) w = r[0];
  else if constexpr (WR == 2) w = widx ? r[1] : r[0];
  else w = pick<WR>(r, widx);
  return __byte_perm(w, 0, 0x4440u | bsel);
}

}  // namespace mhb
