// flat_plans.h — the group table of the flat scan (kernels.cuh: closest_hit_flat) and the compile-time plans of flat scenes,
// shared by the host (api.cu builds the table at scene commit and matches the scene against the plans) and the kernels.
#pragma once

#include <stdint.h>

#include "device_types.h"

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

// A plan: the structure of a flat scene without its coordinates, compiled into the wave and tail kernels (render.cu:
// wave_kernel, tail_kernel_of).  A scene whose table has the plan's group layout (kind, frame, slot range and face map of
// every group), whose scan slots hold the plan's primitive classes, whose wrapper frames run the plan's op kinds and whose
// light list has the plan's kinds, in order, is rendered by the kernels instantiated for the plan: pass 1 of the scan is
// unrolled over the groups, pass 2 solves each candidate by the class of its group, finalize_hit runs the frame's chain
// unrolled, and scatter_lambertian picks and sums the lights by their known kinds.  Boxes, deltas, sphere parameters,
// frames (angles, offsets), light geometry and materials stay in shared memory or the tables, so moving a box keeps the plan.
// faces: slot of face f - the group's first slot in the nibble f (bits 4f .. 4f + 3), 15 = the face is not in the group.
// prims: the class of every slot of the group, for pass 2: rectangles (P_XY_RECT, P_XZ_RECT, P_YZ_RECT; the axis stays
// data, so walls, lights and box sides share one solve) or plain spheres (P_SPHERE).
enum FlatPrimClass : int { C_RECTS = 0, C_SPHERES = 1 };
struct FlatPlanGroup {
    int kind, frame, begin, end;
    uint32_t faces;
    int prims;
};
constexpr uint32_t kNoFaces = 0xFFFFFFFFu;
struct FlatPlanFrame { // DFrame::n_ops and the ChainOpKind of ops[0 .. n_ops), innermost wrapper first
    int n_ops;
    int op[4];
};
// The light count is a constant of the planned kernels, but the weight 1 / n of the light pdf sum is still computed at run
// time from SceneView::n_lights, as in the generic kernels: under -prec-div=false a folded 1.0f / n is correctly rounded and
// a run-time one is MUFU.RCP, which differ for some n.
struct FlatPlan {
    int n_groups;
    FlatPlanGroup g[4];
    int n_frames; // 0 or 1 (plan_chain_kinds)
    FlatPlanFrame frame[1];
    int n_lights;
    int light[2]; // LightKind of lights[0 .. n_lights), in list order
};

// The plans the kernels are instantiated for (render.cu: wave_kernel, tail_kernel_of).  Each one adds a k_wave and a k_tail.
constexpr FlatPlan kFlatPlans[] = {
    // 0: the reference's cornel_box (main.rs:451-507): the five walls (face 4, z = 0, is open), the light, the glass sphere,
    // the six sides of the rotated aluminium box (frame 0: RotateY inside Translate); lights: the ceiling lamp, the sphere
    {4,
     {{G_FACES, -1, 0, 5, 0xFF4F3210u, C_RECTS},
      {G_BOXES, -1, 5, 6, kNoFaces, C_RECTS},
      {G_SPHERES, -1, 6, 7, kNoFaces, C_SPHERES},
      {G_FACES, 0, 7, 13, 0xFF543210u, C_RECTS}},
     1,
     {{2, {OP_ROTATE_Y, OP_TRANSLATE}}},
     2,
     {L_XZ_RECT, L_SPHERE}},
};
constexpr int kNumFlatPlans = int(sizeof(kFlatPlans) / sizeof(kFlatPlans[0]));

#ifdef __CUDACC__
#define RT1W_PLAN_FN __host__ __device__ constexpr // evaluated at compile time inside the planned kernels
#else
#define RT1W_PLAN_FN constexpr
#endif

// The scan slots of class cls of plan p, as a mask.
RT1W_PLAN_FN uint32_t plan_slots(const FlatPlan &p, int cls) {
    uint64_t m = 0;
    for (int g = 0; g < p.n_groups; ++g)
        if (p.g[g].prims == cls) m |= (1ull << p.g[g].end) - (1ull << p.g[g].begin);
    return uint32_t(m);
}
// The wrapper chain of plan p: its op count in bits 0..3, the kind of op i in bits 4i + 4 .. 4i + 7.  Plans have at most one
// frame, so the planned finalize_hit needs no dispatch over frames.
RT1W_PLAN_FN uint32_t plan_chain_kinds(const FlatPlan &p) {
    uint32_t k = p.n_frames > 0 ? uint32_t(p.frame[0].n_ops) : 0u;
    for (int i = 0; p.n_frames > 0 && i < p.frame[0].n_ops; ++i) k |= uint32_t(p.frame[0].op[i]) << (4 * i + 4);
    return k;
}
// The light kinds of plan p, two bits per light in list order.
RT1W_PLAN_FN uint32_t plan_light_kinds(const FlatPlan &p) {
    uint32_t k = 0;
    for (int i = 0; i < p.n_lights; ++i) k |= uint32_t(p.light[i]) << (2 * i);
    return k;
}

// The plan the scene has, or -1.  slot_type: the PrimType of every scan slot; frames, lights: the scene's tables
// (n_lights = 0 for a scene without a light list).
inline int match_flat_plan(const FlatGroups &t, const int *slot_type, const DFrame *frames, int n_frames, const DLight *lights, int n_lights) {
    for (int p = 0; p < kNumFlatPlans; ++p) {
        const FlatPlan &pl = kFlatPlans[p];
        bool same = t.n_groups == pl.n_groups && n_frames == pl.n_frames && n_lights == pl.n_lights;
        for (int g = 0; g < pl.n_groups && same; ++g) {
            const FlatPlanGroup &q = pl.g[g];
            same = t.kind[g] == q.kind && t.frame[g] == q.frame && t.end[g] == q.end && (g == 0 ? 0 : t.end[g - 1]) == q.begin;
            for (int f = 0; f < 8 && same; ++f) {
                const uint32_t nib = (q.faces >> (4 * f)) & 15u;
                same = t.face_slot[g][f] == (q.kind == G_FACES && nib != 15u ? q.begin + int(nib) : -1);
            }
            for (int k = q.begin; k < q.end && same; ++k) {
                const int y = slot_type[k];
                same = q.prims == C_SPHERES ? y == P_SPHERE : (y == P_XY_RECT || y == P_XZ_RECT || y == P_YZ_RECT);
            }
        }
        for (int f = 0; f < pl.n_frames && same; ++f) {
            same = frames[f].n_ops == pl.frame[f].n_ops;
            for (int i = 0; i < pl.frame[f].n_ops && same; ++i) same = frames[f].ops[i].kind == pl.frame[f].op[i];
        }
        for (int i = 0; i < pl.n_lights && same; ++i) same = lights[i].kind == pl.light[i];
        if (same) return p;
    }
    return -1;
}

} // namespace rt1w
