// kernels.cuh -- launchers of the sm_100a kernels (kernels.cu)
#pragma once
#include <cuda_runtime.h>
#include "device_types.cuh"

namespace b200vis {
void launch_propagate_cull(cudaStream_t st, const Rows &R, const Tile *tiles, uint32_t n_tiles, const CullViews &cvw,
                           const VisibleBufs &vb, DevStats *stats, uint32_t stages, uint32_t static_opt, uint32_t parity,
                           uint32_t *ticket = nullptr, uint32_t *ticket_base = nullptr, bool named_levels_only = false);
void launch_propagate_cull_small(cudaStream_t st, const Rows &R, const Tile *tiles, uint32_t n_tiles, const CullViews &cvw,
                                 const VisibleBufs &vb, DevStats *stats, uint32_t stages, uint32_t static_opt, uint32_t parity);
unsigned long long kernel_launch_count();
bool tile_kernel_is_tma();
bool tile_kernel_is_warp();
bool tile_kernel_publishes_light_snapshot();
void launch_tile_warp(cudaStream_t st, const Rows &R, const WarpTile *tiles, const uint8_t *sched, uint32_t n_tiles, const CullViews &cvw,
                      const VisibleBufs &vb, DevStats *stats, uint32_t stages, uint32_t static_opt, uint32_t parity, uint32_t *counter);
void launch_cull(cudaStream_t st, const Rows &R, const CullViews &cvw, const VisibleBufs &vb, DevStats *stats, uint32_t parity);
void launch_mark_dirty_global(cudaStream_t st, const Rows &R);
void launch_expand_visible(cudaStream_t st, const VisibleBufs &vb, const DiffBufs &db, const uint32_t *row_of_rank, const FrameConsts *fc,
                           DevStats *stats, uint32_t parity, uint32_t n_rows, uint32_t max_views);
void launch_shadow_cull(cudaStream_t st, const Rows &R, const ShadowBufs &sb, const uint32_t *view_sets, uint32_t n_views,
                        uint32_t n_words, uint32_t n_chunks, uint32_t words_stride, uint32_t chunks_stride, DevStats *stats, uint32_t changed_slot);
void launch_pack_cluster_bindings(cudaStream_t st, const FrameConsts *fc, const ClusterBufs &cb, const BindingBufs &bb, uint32_t max_views);
void launch_publish_visible_diff(cudaStream_t st, const VisibleBufs &vb, const DiffBufs &db, uint32_t *host_rows, uint32_t host_stride,
                                 uint32_t *host_counts, uint32_t n_views, uint32_t max_views);
void launch_cluster_assign(cudaStream_t st, const Rows &R, const Lights &L, const FrameConsts *fc, const ClusterBufs &cb,
                           DevStats *stats, uint32_t max_views);
bool cluster_fused_fits(uint32_t n_lights);
bool launch_cluster_fused(cudaStream_t st, const Rows &R, const Lights &L, const FrameConsts *fc, const ClusterBufs &cb,
                          DevStats *stats, uint32_t max_views);
void launch_publish_visible(cudaStream_t st, const VisibleBufs &vb, const DevStats *stats, uint32_t *host_rows, uint32_t host_stride,
                            uint32_t n_rows, uint32_t n_views, uint8_t *host_classes);
void launch_publish_clusters(cudaStream_t st, const FrameConsts *fc, const ClusterBufs &cb, uint32_t *host_offsets, uint32_t *host_indices,
                             uint32_t host_cap, const DevStats *stats, uint32_t *host_stats, uint32_t changed_slot, uint32_t frame, uint32_t max_views);
void launch_tag_lights(cudaStream_t st, const Rows &R, const Lights &L, uint32_t *light_ord, uint32_t *all_tagged);
void launch_snapshot_lights(cudaStream_t st, const Rows &R, const Lights &L, float4 *snap);
void launch_snapshot_objects(cudaStream_t st, const Rows &R, const ClusterObjects &O, float4 *snap, float *range);
void launch_writeback_columns(cudaStream_t st, const Rows &R, float *host_gt, uint32_t stride, uint32_t *host_gt_bits, uint8_t *host_vv,
                              uint32_t *host_vv_bits, uint8_t *vv_shadow);
void launch_record_push(cudaStream_t st, const uint32_t *block, uint32_t block_words, const ClusterBufs &cb);
void launch_slab_push(cudaStream_t st, const FrameConsts *fc, const ClusterBufs &cb, uint32_t *done, uint32_t max_views);
void launch_cluster_lists(cudaStream_t st, const FrameConsts *fc, const ClusterBufs &cb, DevStats *stats, uint32_t max_views);
void launch_unpack_trs(cudaStream_t st, const Rows &R, uint32_t first, uint32_t count, const float *src, int mark_only);
void launch_scatter_trs(cudaStream_t st, const Rows &R, uint32_t count, const uint32_t *rows, const float *src);
void launch_unpack_gt(cudaStream_t st, const Rows &R, uint32_t first, uint32_t count, const float *src);
void launch_pack_gt(cudaStream_t st, const Rows &R, uint32_t first, uint32_t count, float *dst, uint32_t stride);
void launch_unpack_bounds(cudaStream_t st, const Rows &R, uint32_t first, uint32_t count, const float *bounds,
                          const uint8_t *flags, const uint8_t *cls, uint8_t *cls_col);
void launch_unpack_vv(cudaStream_t st, const Rows &R, uint32_t first, uint32_t count, const uint8_t *vv);
void launch_visibility_propagate(cudaStream_t st, const Rows &R, const Tile *tiles, uint32_t n_tiles, const uint8_t *vis, uint8_t *changed);
void launch_pack_inherited(cudaStream_t st, const Rows &R, uint32_t first, uint32_t count, const uint8_t *changed, uint8_t *out);
void launch_pack_ranges(cudaStream_t st, const Rows &R, uint32_t first, uint32_t count, uint32_t *out);
void launch_unpack_range_params(cudaStream_t st, float2 *se, uint8_t *ua, uint32_t first, uint32_t count, const float *src_se, const uint8_t *src_ua);
void launch_pack_state(cudaStream_t st, const Rows &R, uint32_t first, uint32_t count, uint8_t *out, uint32_t changed_bit);
}
