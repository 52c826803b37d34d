// slg_launch.h — launchers of the scoring kernels.  Each family of template instantiations lives in its own
// translation unit (slg_launch_tiles.cu, slg_launch_warp.cu, slg_launch_items.cu) so that the library builds in
// parallel; the host code selects a variant by flags.
#pragma once
#include "slg_scan_kernel.cuh"

namespace slg {

cudaError_t launch_score_tiles(bool matcher, bool prune, bool stats, bool plan, const SegmentDev &sd, const BatchDev &bd, size_t smem,
                               int grid, cudaStream_t st);
cudaError_t launch_score_warp(bool matcher, bool prune, bool stats, bool staged, bool plan, const SegmentDev &sd, const WarpBatchDev &wb,
                              size_t smem, int grid, cudaStream_t st);
cudaError_t launch_score_items(bool prune, const SegmentDev &sd, const WarpBatchDev &wb, const ItemsDev &it, size_t smem, int grid,
                               cudaStream_t st);
cudaError_t launch_score_sparse(const SegmentDev &sd, const WarpBatchDev &wb, const StreamDev &st_dev, size_t smem, int grid, cudaStream_t st);
cudaError_t launch_score_columns(bool prune, bool pools, const SegmentDev &sd, const WarpBatchDev &wb, const StreamDev &st_dev, size_t smem, int grid, cudaStream_t st);
cudaError_t launch_scan(bool prune, bool pools, const SegmentDev &sd, const WarpBatchDev &wb, const ScanDev &sc, int grid, cudaStream_t st);
cudaError_t launch_columns_ordered(bool pools, const SegmentDev &sd, const WarpBatchDev &wb, const StreamDev &st_dev, int grid, cudaStream_t st);
cudaError_t launch_seed_items(const SegmentDev &sd, const WarpBatchDev &wb, const ItemsDev &it, size_t smem, int grid, cudaStream_t st);

}  // namespace slg
