// scene_prep.h — host-side conversion of the reference buffers into the device layout (see scene_prep.cpp).
#pragma once
#include <string>
#include <vector>
#include "host_surface.h"
#include "render_kernel.cuh"

namespace mmk {

struct Prepared {
    std::vector<PairRec> pairs;
    std::vector<RectI> rects;
    std::vector<RectS> shade;
    std::vector<RectA> rects_axis;   // filled when axis_ok
    std::vector<PairRecY> pairs_y;   // filled when fast_ok and the children have at most kMaxYIntervals distinct y-intervals
    std::vector<float4> y_ivals;     // those intervals as (min.y, max.y, max.y, min.y), in first-use order
    uint32_t n_pairs = 0, root_link = 0, root_count = 0, depth = 0, max_leaf = 0;
    bool fast_ok = false;        // box coordinates inside the guarded ranges of the shared-reciprocal slab quotient
    bool rect_fast_ok = false;   // edge lengths inside the guarded range of edge_thresholds
    bool axis_ok = false;        // every rect axis-aligned (or degenerate): the 32-B axis-aligned rect test applies
};

// Interval [lo, up] on x that is equivalent to `0 <= RN(x / L) && RN(x / L) <= L` (see render_kernel.cuh, RectI).
// Returns false when L is outside the guarded range (then the kernel uses the literal divides for the whole scene).
bool edge_thresholds(float L, float *lo, float *up);

// The axis-aligned form of one rectangle (render_kernel.cuh, RectA).  Returns false when the rect is not axis-aligned.
// Exported for tests as mm_axis_rect.
bool axis_rect(const mm_plane &m, RectA *out);

int prepare_scene(const mm_plane *planes, uint32_t n_planes, const mm_bvh_node *nodes, uint32_t n_nodes,
                  const uint32_t *indices, const uint8_t *materials, const mm_float4 *emissions, Prepared &out,
                  std::string &err);

}  // namespace mmk
