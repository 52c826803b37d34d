// slg_launch_items.cu — instantiations of the posting-driven items kernel (plain OR queries, k <= 32, <= 8 terms)
#include "slg_launch.h"

namespace slg {
namespace {
template <class K, class... A>
cudaError_t go(K kern, size_t smem, int grid, cudaStream_t st, A... args) {
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  kern<<<grid, kThreads, smem, st>>>(args...);
  return cudaGetLastError();
}
template <class K, class... A>
cudaError_t go_n(K kern, int threads, size_t smem, int grid, cudaStream_t st, A... args) {
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  kern<<<grid, threads, smem, st>>>(args...);
  return cudaGetLastError();
}
}  // namespace

cudaError_t launch_score_items(bool prune, const SegmentDev &sd, const WarpBatchDev &wb, const ItemsDev &it, size_t smem, int grid,
                               cudaStream_t st) {
  return prune ? go(slg_score_items_kernel<true>, smem, grid, st, sd, wb, it) : go(slg_score_items_kernel<false>, smem, grid, st, sd, wb, it);
}
cudaError_t launch_score_sparse(const SegmentDev &sd, const WarpBatchDev &wb, const StreamDev &st_dev, size_t smem, int grid, cudaStream_t st) {
  cudaError_t e = cudaFuncSetAttribute(slg_score_sparse_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  slg_score_sparse_kernel<false><<<grid, kSparseWarps * 32, smem, st>>>(sd, wb, st_dev);
  return cudaGetLastError();
}
cudaError_t launch_score_columns(bool prune, bool pools, const SegmentDev &sd, const WarpBatchDev &wb, const StreamDev &st_dev, size_t smem, int grid,
                                 cudaStream_t st) {
  if (pools)
    return prune ? go_n(slg_score_columns_kernel<true, true>, kColWarps * 32, smem, grid, st, sd, wb, st_dev)
                 : go_n(slg_score_columns_kernel<false, true>, kColWarps * 32, smem, grid, st, sd, wb, st_dev);
  return prune ? go_n(slg_score_columns_kernel<true, false>, kColWarps * 32, smem, grid, st, sd, wb, st_dev)
               : go_n(slg_score_columns_kernel<false, false>, kColWarps * 32, smem, grid, st, sd, wb, st_dev);
}
cudaError_t launch_columns_ordered(bool pools, const SegmentDev &sd, const WarpBatchDev &wb, const StreamDev &st_dev, int grid, cudaStream_t st) {
  if (pools) slg_columns_ordered_kernel<1><<<grid, 256, 0, st>>>(sd, wb, st_dev);
  else slg_columns_ordered_kernel<0><<<grid, 256, 0, st>>>(sd, wb, st_dev);
  return cudaGetLastError();
}
template <bool PRUNE, bool POOLS>
static void launch_scan_pm(bool must, const SegmentDev &sd, const WarpBatchDev &wb, const ScanDev &sc, int grid, cudaStream_t st) {
  if (must) slg_scan_kernel<PRUNE, POOLS, true><<<grid, kScanWarps * 32, 0, st>>>(sd, wb, sc);
  else slg_scan_kernel<PRUNE, POOLS, false><<<grid, kScanWarps * 32, 0, st>>>(sd, wb, sc);
}
cudaError_t launch_scan(bool prune, bool pools, const SegmentDev &sd, const WarpBatchDev &wb, const ScanDev &sc, int grid, cudaStream_t st) {
  const bool must = sc.must_mode != 0u;
  if (pools) {
    if (prune) launch_scan_pm<true, true>(must, sd, wb, sc, grid, st);
    else launch_scan_pm<false, true>(must, sd, wb, sc, grid, st);
  } else {
    if (prune) launch_scan_pm<true, false>(must, sd, wb, sc, grid, st);
    else launch_scan_pm<false, false>(must, sd, wb, sc, grid, st);
  }
  return cudaGetLastError();
}
cudaError_t launch_seed_items(const SegmentDev &sd, const WarpBatchDev &wb, const ItemsDev &it, size_t smem, int grid, cudaStream_t st) {
  return go(slg_seed_items_kernel<0>, smem, grid, st, sd, wb, it);
}
}  // namespace slg
