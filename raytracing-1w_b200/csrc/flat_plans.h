// flat_plans.h — the group table of the flat scan (kernels.cuh: closest_hit_flat) and its compile-time plans, shared by the
// host (api.cu builds the table at scene commit and matches it against the plans) and the kernels.
#pragma once

#include <stdint.h>

namespace rt1w {

constexpr int kFlatMax = 32;
constexpr int kFlatMaxFrames = 8;
enum FlatGroupKind : int { G_BOXES = 0, G_SPHERES = 1, G_FACES = 2 };

// The scan-order groups of a flat scene (api.cu: flat_groups): group g = scan slots [end[g-1], end[g]) in frame frame[g]
// (-1 = world).  kind[g]: G_BOXES one box per primitive; G_SPHERES plain spheres, screened by an f32 discriminant on top of
// the box; G_FACES rectangles that are faces of ONE box (every slot of the group carries that box): face_slot[g][f] = scan
// slot of face f (2 * axis + (upper plane ? 1 : 0)) or -1, delta[g] = twice the box padding.
struct FlatGroups {
    int32_t end[kFlatMax];
    int32_t frame[kFlatMax];
    int32_t kind[kFlatMax];
    float delta[kFlatMax];
    int8_t face_slot[kFlatMax][8];
    int32_t n_groups;
};

// A scan plan: the layout of a group table without its coordinates.  A scene whose table has this layout (kind, frame,
// slot range and face map of every group) is scanned by the kernels instantiated for the plan, with the group loop unrolled
// at compile time; boxes, deltas, sphere parameters and frames stay in shared memory, so moving a box keeps the plan.
// faces: slot of face f - the group's first slot in the nibble f (bits 4f .. 4f + 3), 15 = the face is not in the group.
struct FlatPlanGroup {
    int kind, frame, begin, end;
    uint32_t faces;
};
constexpr uint32_t kNoFaces = 0xFFFFFFFFu;
struct FlatPlan {
    int n_groups;
    FlatPlanGroup g[4];
};

// The plans the kernels are instantiated for (render.cu: wave_kernel, tail_kernel_of).  Each one adds a k_wave and a k_tail.
constexpr FlatPlan kFlatPlans[] = {
    // 0: the reference's cornel_box (main.rs:451-507): the five walls (face 4, z = 0, is open), the light, the glass sphere,
    // the six sides of the rotated aluminium box
    {4, {{G_FACES, -1, 0, 5, 0xFF4F3210u}, {G_BOXES, -1, 5, 6, kNoFaces}, {G_SPHERES, -1, 6, 7, kNoFaces}, {G_FACES, 0, 7, 13, 0xFF543210u}}},
};
constexpr int kNumFlatPlans = int(sizeof(kFlatPlans) / sizeof(kFlatPlans[0]));

// The plan whose layout the table has, or -1.
inline int match_flat_plan(const FlatGroups &t) {
    for (int p = 0; p < kNumFlatPlans; ++p) {
        const FlatPlan &pl = kFlatPlans[p];
        bool same = t.n_groups == pl.n_groups;
        for (int g = 0; g < pl.n_groups && same; ++g) {
            const FlatPlanGroup &q = pl.g[g];
            same = t.kind[g] == q.kind && t.frame[g] == q.frame && t.end[g] == q.end && (g == 0 ? 0 : t.end[g - 1]) == q.begin;
            for (int f = 0; f < 8 && same; ++f) {
                const uint32_t nib = (q.faces >> (4 * f)) & 15u;
                same = t.face_slot[g][f] == (q.kind == G_FACES && nib != 15u ? q.begin + int(nib) : -1);
            }
        }
        if (same) return p;
    }
    return -1;
}

} // namespace rt1w
