// ray_math.cuh -- per-ray Siddon / trilinear math (host+device; the kernels are thin wrappers around these).
//
// Replaces, per ray, reference renderers.py:34-76 (Siddon.forward), 205-240 (Trilinear.forward) and their
// autograd graphs.  The reference materialises all D0+D1+D2+3 plane alphas per ray, sorts them, builds
// (B,N,M,3) sample grids and calls grid_sample; here one thread walks one ray with a 3-way monotone
// merge, alphas live in registers and nothing of size (B,N,M) ever exists.
#pragma once

#include "common.cuh"

namespace b200drr {

// ===================================================================================================
// Siddon, general walk: visits EVERY plane of the volume like the reference (no clipping), samples the
// nearest voxel at each segment midpoint through the literal normalise / un-normalise chain of
// renderers.py:143-153 + ATen grid_sampler.  Handles align_corners and reduce="max".  Slow path.
// ===================================================================================================
B200_HD float unnormalize(float g, int size, int align_corners)
{
    return align_corners ? ((g + 1.0f) / 2.0f) * (float)(size - 1) : ((g + 1.0f) * (float)size - 1.0f) / 2.0f;
}

B200_HD float siddon_ray_general(const float* vol, const VolDims& dims, const Ray& ray, float L, float shift,
                                 int reduce, int align_corners)
{
    int pos[3], stp[3], left[3];
    float head[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const bool fwd = ray.d[a] > 0.0f;
        pos[a] = fwd ? 0 : dims.d[a];
        stp[a] = fwd ? 1 : -1;
        left[a] = dims.d[a] + 1;
        head[a] = plane_alpha(ray, a, (float)pos[a], shift);
    }
    const int M = dims.d[0] + dims.d[1] + dims.d[2] + 3;
    float acc = 0.0f, aprev = 0.0f;
    bool first = true;
    for (int m = 0; m < M; ++m) {
        // pop the smallest head (ties: lowest axis first, like a stable sort of cat([ax, ay, az]))
        const float h0 = left[0] > 0 ? head[0] : INFINITY;
        const float h1 = left[1] > 0 ? head[1] : INFINITY;
        const float h2 = left[2] > 0 ? head[2] : INFINITY;
        const float acur = fminf(fminf(h0, h1), h2);
        const int best = (left[0] > 0 && h0 == acur) ? 0 : ((left[1] > 0 && h1 == acur) ? 1 : 2);
#pragma unroll
        for (int a = 0; a < 3; ++a)
            if (a == best) {
                pos[a] += stp[a];
                left[a] -= 1;
                if (left[a] > 0) head[a] = plane_alpha(ray, a, (float)pos[a], shift);
            }
        if (m > 0) {
            const float amid = (aprev + acur) / 2.0f;
            bool inb = true;
            int64_t off = 0;
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const float x = add_rn(ray.s[a], mul_rn(amid, ray.d[a]));
                const float g = 2.0f * (x + shift) / (float)dims.d[a] - 1.0f;
                const float rr = rintf(unnormalize(g, dims.d[a], align_corners));
                inb = inb && (rr >= 0.0f) && (rr < (float)dims.d[a]);
                off = off * dims.d[a] + (inb ? (int64_t)rr : 0);
            }
            const float v = inb ? ldg(vol + off) : 0.0f;
            const float term = mul_rn(mul_rn(L, v), acur - aprev);
            if (reduce == 0) acc = add_rn(acc, term);
            else if (first || term > acc) acc = term;
            first = false;
        }
        aprev = acur;
    }
    return acc;
}

// Backward of the general walk (reducefn "sum" with align_corners=True, or reducefn "max"): the same plane-by-plane
// pop, closed form of SURVEY.md 8a-G.  "max": only the FIRST maximal segment carries gradient (torch.max returns the
// first maximal index): +L v at its exit crossing, -L v at its entry crossing.  gL = g * L.
// Returns sum_j v_j len_j ("sum") or v* len* ("max") for the ray-length gradient; g_vol accumulated into when non-null.
B200_HD float siddon_ray_general_bwd(const float* vol, const VolDims& dims, const Ray& ray, float L, float gL, float shift,
                                     int reduce, int align_corners, float* g_vol, float gs[3], float gt[3])
{
    int pos[3], stp[3], left[3];
    float head[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const bool fwd = ray.d[a] > 0.0f;
        pos[a] = fwd ? 0 : dims.d[a];
        stp[a] = fwd ? 1 : -1;
        left[a] = dims.d[a] + 1;
        head[a] = plane_alpha(ray, a, (float)pos[a], shift);
    }
    const int M = dims.d[0] + dims.d[1] + dims.d[2] + 3;
    float A[3] = {0.0f, 0.0f, 0.0f}, C[3] = {0.0f, 0.0f, 0.0f};
    float sumvl = 0.0f, aprev = 0.0f, vbefore = 0.0f;
    int axprev = 0;
    // "max" bookkeeping
    bool first = true;
    float tbest = 0.0f, vbest = 0.0f, a0best = 0.0f, a1best = 0.0f;
    int ax0best = 0, ax1best = 0;
    int64_t offbest = -1;
    for (int m = 0; m < M; ++m) {
        const float h0 = left[0] > 0 ? head[0] : INFINITY;
        const float h1 = left[1] > 0 ? head[1] : INFINITY;
        const float h2 = left[2] > 0 ? head[2] : INFINITY;
        const float acur = fminf(fminf(h0, h1), h2);
        const int best = (left[0] > 0 && h0 == acur) ? 0 : ((left[1] > 0 && h1 == acur) ? 1 : 2);
#pragma unroll
        for (int a = 0; a < 3; ++a)
            if (a == best) {
                pos[a] += stp[a];
                left[a] -= 1;
                if (left[a] > 0) head[a] = plane_alpha(ray, a, (float)pos[a], shift);
            }
        if (m > 0) {
            const float amid = (aprev + acur) / 2.0f;
            bool inb = true;
            int64_t off = 0;
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const float x = add_rn(ray.s[a], mul_rn(amid, ray.d[a]));
                const float gn = 2.0f * (x + shift) / (float)dims.d[a] - 1.0f;
                const float rr = rintf(unnormalize(gn, dims.d[a], align_corners));
                inb = inb && (rr >= 0.0f) && (rr < (float)dims.d[a]);
                off = off * dims.d[a] + (inb ? (int64_t)rr : 0);
            }
            const float v = inb ? ldg(vol + off) : 0.0f;
            const float len = acur - aprev;
            if (reduce == 0) {
                const float coef = vbefore - v;  // crossing m-1 (axis axprev, alpha aprev) separates the two segments
#pragma unroll
                for (int a = 0; a < 3; ++a)
                    if (a == axprev) {
                        A[a] = fmaf(coef, aprev, A[a]);
                        C[a] += coef;
                    }
                sumvl = fmaf(v, len, sumvl);
                if (g_vol && inb) red_add(g_vol + off, gL * len);
                vbefore = v;
            } else {
                const float term = mul_rn(mul_rn(L, v), len);
                if (first || term > tbest) {
                    tbest = term;
                    vbest = v;
                    a0best = aprev;
                    ax0best = axprev;
                    a1best = acur;
                    ax1best = best;
                    offbest = inb ? off : -1;
                }
                first = false;
            }
        }
        aprev = acur;
        axprev = best;
    }
    if (reduce == 0) {
#pragma unroll
        for (int a = 0; a < 3; ++a)
            if (a == axprev) {  // last crossing: v_last -> 0
                A[a] = fmaf(vbefore, aprev, A[a]);
                C[a] += vbefore;
            }
    } else {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            if (a == ax1best) {
                A[a] = fmaf(vbest, a1best, A[a]);
                C[a] += vbest;
            }
            if (a == ax0best) {
                A[a] = fmaf(-vbest, a0best, A[a]);
                C[a] -= vbest;
            }
        }
        sumvl = vbest * (a1best - a0best);
        if (g_vol && offbest >= 0) red_add(g_vol + offbest, gL * (a1best - a0best));
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        gt[a] = -gL * A[a] * ray.inv[a];
        gs[a] = gL * (A[a] - C[a]) * ray.inv[a];
    }
    return sumvl;
}

// ===================================================================================================
// Siddon, fast walk (align_corners = False): clipped to the volume's box, incremental voxel index.
// In "plane space" q = x + shift, voxel k of axis a spans q in [k, k+1] and the reference's plane i
// (x = i - shift, renderers.py:97-99) sits at q = i.  Every reference segment outside
// [alpha_in, alpha_out] samples zero padding, so clipping to the box is exact; alphas are NOT clipped to
// [0,1] (quirk Q1).  Plane alphas are fma(i, 1/d, c) from the integer plane index (never accumulated),
// c = -(shift + s)/d.
// ===================================================================================================
struct Walk {
    float an[3];   // alpha of the next plane crossing per axis
    float nf[3];   // how many planes of this axis have been crossed so far (float counter)
    float da[3];   // alpha distance between consecutive planes of this axis, |1/d|
    float a0[3];   // alpha of the FIRST plane crossing per axis: an = fma(nf, da, a0)
    float nx[3];   // value of nf at which the ray crosses the boundary plane of the box (leaves it)
    float p0[3];   // index of the first plane crossed per axis
    float inv[3];  // 1/d
    int idx[3];    // entry voxel
    int sti[3];    // +1 / -1
    float a_in, a_out;
    int entry_axis;
    bool hit;
};

// alpha of plane p on axis a in the reference's own difference form ((p - shift) - s) / d: the small
// difference is formed first, so the result is accurate to ~1 ulp even when d is tiny (the fused form
// fma(p, 1/d, -(shift+s)/d) cancels two huge terms there and loses ~1e-2 voxel along the ray).
B200_HD float plane_alpha_acc(const Ray& ray, int a, float p, float shift) { return ((p - shift) - ray.s[a]) * ray.inv[a]; }

// Conservative pre-test for the slab-major kernels (a ray crosses only 1-3 of the ~11 slabs; the rest of its threads
// used to pay the full walk set-up just to find that out): true ONLY when the line certainly stays clear of the box
// [lo, hi), with a margin three orders above fp32 rounding, so every borderline ray still goes through
// the exact set-up, which alone decides hits.  inf / NaN alphas compare false (never skipped).
B200_HD bool box_surely_missed(const Ray& ray, const int lo_v[3], const int hi_v[3], float shift)
{
    float a_in = -INFINITY, a_out = INFINITY;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float a0 = plane_alpha_acc(ray, a, (float)lo_v[a], shift), a1 = plane_alpha_acc(ray, a, (float)hi_v[a], shift);
        a_in = fmaxf(a_in, fminf(a0, a1));
        a_out = fminf(a_out, fmaxf(a0, a1));
    }
    // alphas carry ~1e-7 relative rounding; 1e-4 of their magnitude is three orders above that and still a fraction of a
    // voxel (one voxel is ~7e-4 in alpha at 512^3)
    const float margin = 1e-4f * (1.0f + fabsf(a_in) + fabsf(a_out));
    return a_in > a_out + margin;
}

// Piece `piece` of `pieces` of the volume along the ray's OWN major axis (largest |d|): the ray crosses that axis' planes at the
// highest rate, so the pieces carry about equal shares of its voxel visits whatever the pose is (slabs along a FIXED axis give a
// ray that runs across them one to three pieces only).  Splitting at voxel planes is exact, and each ray may pick its own axis.
// Returns false for an empty piece (pieces does not divide the axis).  Used for batches of one or two poses, where a thread per
// (ray, piece) is what fills the machine: 65 536 rays are 21 % of a B200's thread slots.
B200_HD bool major_axis_piece(const Ray& ray, const VolDims& dims, int piece, int pieces, int lo_v[3], int hi_v[3])
{
    const float a0 = fabsf(ray.d[0]), a1 = fabsf(ray.d[1]), a2 = fabsf(ray.d[2]);
    const int M = (a0 >= a1 && a0 >= a2) ? 0 : (a1 >= a2 ? 1 : 2);
    bool any = true;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const int len = (dims.d[a] + pieces - 1) / pieces;
        const bool m = a == M;
        lo_v[a] = m ? piece * len : 0;
        const int top = (piece + 1) * len;
        hi_v[a] = (m && top < dims.d[a]) ? top : dims.d[a];
        any = any && lo_v[a] < hi_v[a];
    }
    return any;
}

// Walk restricted to the sub-box of voxels [lo_a, hi_a) per axis (planes lo_a .. hi_a); the whole volume is
// lo = 0, hi = dims.  Splitting a ray at voxel planes is exact: every Siddon segment ends on a plane anyway.
// Crossing alphas are generated as fma(n, |1/d|, alpha_first) from an integer crossing count n (never
// accumulated), with alpha_first in the accurate difference form.
B200_HD Walk start_walk_box(const Ray& ray, const int lo_v[3], const int hi_v[3], float shift)
{
    Walk w;
    float lo[3];
    w.a_in = -INFINITY;
    float a_hi = INFINITY;
    w.entry_axis = 0;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        w.inv[a] = ray.inv[a];
        w.da[a] = fabsf(ray.inv[a]);
        const float a0 = plane_alpha_acc(ray, a, (float)lo_v[a], shift);
        const float a1 = plane_alpha_acc(ray, a, (float)hi_v[a], shift);
        lo[a] = fminf(a0, a1);
        a_hi = fminf(a_hi, fmaxf(a0, a1));
        const bool better = lo[a] > w.a_in;
        w.a_in = better ? lo[a] : w.a_in;
        w.entry_axis = better ? a : w.entry_axis;
    }
    w.hit = w.a_in < a_hi;  // false for NaN as well
    w.a_out = INFINITY;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const bool fwd = ray.d[a] > 0.0f;
        w.sti[a] = fwd ? 1 : -1;
        const int lo_i = lo_v[a], hi_i = hi_v[a] - 1;
        int i = (int)floorf(fmaf(w.a_in, ray.d[a], ray.s[a] + shift));
        i = i < lo_i ? lo_i : (i > hi_i ? hi_i : i);
        // Make the start voxel consistent with the ORDER of the crossing alphas (floor() of a position that sits
        // within round-off of a plane is a coin toss): the plane behind must have alpha < a_in, and a plane that
        // ties with the entry face counts as not crossed yet.  Straight-line selects, no branches.
        const float a_behind = plane_alpha_acc(ray, a, (float)(fwd ? i : i + 1), shift);
        const float a_ahead = plane_alpha_acc(ray, a, (float)(fwd ? i + 1 : i), shift);
        const bool back = (a_behind >= w.a_in) && (fwd ? i > lo_i : i < hi_i);
        const bool ahead = !(a_behind >= w.a_in) && (a_ahead < w.a_in) && (fwd ? i < hi_i : i > lo_i);
        i += back ? -w.sti[a] : (ahead ? w.sti[a] : 0);
        i = (lo[a] >= w.a_in) ? (fwd ? lo_i : hi_i) : i;  // entering through a face of this axis
        w.idx[a] = i;
        w.p0[a] = (float)(fwd ? i + 1 : i);
        w.nx[a] = fwd ? (float)hi_v[a] - w.p0[a] : w.p0[a] - (float)lo_v[a];
        w.a0[a] = plane_alpha_acc(ray, a, w.p0[a], shift);
        w.nf[a] = 0.0f;
        w.an[a] = w.a0[a];
        // the exit alpha is produced by the SAME expression the walk uses for its crossings, so that
        // "crossing alpha == a_out" identifies the exit plane exactly
        w.a_out = fminf(w.a_out, fmaf(w.nx[a], w.da[a], w.a0[a]));
    }
    return w;
}

// Same as start_walk_box, but every alpha (crossings AND box faces) is generated from ONE per-ray frame anchored at
// the ray's entry into the whole VOLUME:  alpha_a(p) = fma(|p - pref_a|, |1/d_a|, alpha_acc(pref_a)).  All slabs a
// ray is cut into then see bit-identical alphas for the same plane, so a slab's exit alpha equals the next slab's
// entry alpha and (near-)ties between a slab face and another axis' plane are ordered the same way on both sides.
// The backward pass needs this: an inconsistent order drops or doubles one crossing coefficient (the forward sum
// does not care, the affected segment has ~zero length).
// CUT = true (boxes cut along an axis other than 0: the major-axis pieces): the exit tail of the lean backward / sensitivities
// walks takes the crossings that TIE with the exit alpha on axes BELOW the exit axis before it leaves (stable order, lowest axis
// first), and leaves the ties on higher axes to the next box.  The entry rule below must mirror that at an INTERIOR face, or a
// tied crossing of a lower axis is counted by both boxes (its coefficient doubled on that axis and taken off the face axis: the
// sum of the coefficients still telescopes, their attribution does not -- found as 3-13 rays per 10^6 that run through a voxel
// edge exactly on a cut, 4e-3 of the largest gradient).  Slabs along axis 0 have no lower axis, so CUT = false is exact for them
// (and keeps the production slab kernels' code unchanged).
template <bool CUT = false>
B200_HD Walk start_walk_frame(const Ray& ray, const VolDims& dims, const int lo_v[3], const int hi_v[3], float shift)
{
    Walk w;
    // ---- frame: entry into the whole volume ----------------------------------------------------------------
    float vlo[3];
    float av_in = -INFINITY, av_out = INFINITY;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        w.inv[a] = ray.inv[a];
        w.da[a] = fabsf(ray.inv[a]);
        w.sti[a] = ray.d[a] > 0.0f ? 1 : -1;
        const float a0 = plane_alpha_acc(ray, a, 0.0f, shift), a1 = plane_alpha_acc(ray, a, (float)dims.d[a], shift);
        vlo[a] = fminf(a0, a1);
        av_in = fmaxf(av_in, vlo[a]);
        av_out = fminf(av_out, fmaxf(a0, a1));
    }
    float pref[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        // straight-line (select-only) version of: floor the entry position, then move one voxel back/forward if the
        // plane behind is not strictly before av_in / the plane ahead is already before it
        const bool fwd = w.sti[a] > 0;
        const int hi_i = dims.d[a] - 1;
        int i = (int)floorf(fmaf(av_in, ray.d[a], ray.s[a] + shift));
        i = i < 0 ? 0 : (i > hi_i ? hi_i : i);
        const float a_behind = plane_alpha_acc(ray, a, (float)(fwd ? i : i + 1), shift);
        const float a_ahead = plane_alpha_acc(ray, a, (float)(fwd ? i + 1 : i), shift);
        const bool back = (a_behind >= av_in) && (fwd ? i > 0 : i < hi_i);
        const bool ahead = !(a_behind >= av_in) && (a_ahead < av_in) && (fwd ? i < hi_i : i > 0);
        i += back ? -w.sti[a] : (ahead ? w.sti[a] : 0);
        i = (vlo[a] >= av_in) ? (fwd ? 0 : hi_i) : i;  // entering through a face of this axis
        pref[a] = (float)(fwd ? i + 1 : i);
        w.a0[a] = plane_alpha_acc(ray, a, pref[a], shift);
    }
    // ---- clip to the box with frame alphas -----------------------------------------------------------------
    float lo[3];
    w.a_in = -INFINITY;
    w.a_out = INFINITY;
    w.entry_axis = 0;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float sg = (float)w.sti[a];
        const float a0 = fmaf(((float)lo_v[a] - pref[a]) * sg, w.da[a], w.a0[a]);
        const float a1 = fmaf(((float)hi_v[a] - pref[a]) * sg, w.da[a], w.a0[a]);
        lo[a] = fminf(a0, a1);
        const bool better = lo[a] > w.a_in;
        w.a_in = better ? lo[a] : w.a_in;
        w.entry_axis = better ? a : w.entry_axis;
        w.a_out = fminf(w.a_out, fmaxf(a0, a1));
    }
    // a_in == a_out is a (zero-length) hit here: the voxel touched still takes part in the crossing bookkeeping
    w.hit = (av_in < av_out) && (w.a_in <= w.a_out);
    // CUT: the un-cut walk processes the events of one alpha in this order -- entry into the volume, then the crossings lowest
    // axis first, the exit at its axis' turn (tied crossings on higher axes are dropped) -- and a cut on axis M is the M-crossing
    // of that list: everything before it belongs to the box that is left, everything after it to the box that is entered.  So
    //  * a cut face that TIES with an entry face of the whole volume is the entry face of this box (the box before it was
    //    entered through the volume face and counts as touched: a_in <= a_out above);
    //  * a box that is entered through a cut and left at the same alpha was reached only if the cut comes before that exit in
    //    axis order (otherwise the previous box's tail already left the volume through the lower axis' face);
    //  * ties with a_in on axes below the cut were crossed by the previous box's tail (prev_took_ties below).
    bool interior = false;
    if constexpr (CUT) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const int p = w.sti[a] > 0 ? lo_v[a] : hi_v[a];
            const bool cut_face = p > 0 && p < dims.d[a];
            const bool take = cut_face && lo[a] == w.a_in;
            w.entry_axis = take ? a : w.entry_axis;
            interior = interior || take;
        }
        int exit_axis = 3;
#pragma unroll
        for (int a = 2; a >= 0; --a) {  // lowest axis whose exit plane is at a_out (same expressions as above: bit-identical alphas)
            const float sg = (float)w.sti[a];
            const float a0 = fmaf(((float)lo_v[a] - pref[a]) * sg, w.da[a], w.a0[a]);
            const float a1 = fmaf(((float)hi_v[a] - pref[a]) * sg, w.da[a], w.a0[a]);
            exit_axis = (fmaxf(a0, a1) == w.a_out) ? a : exit_axis;
        }
        w.hit = w.hit && !(interior && w.a_in == w.a_out && exit_axis < w.entry_axis);
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const bool fwd = w.sti[a] > 0;
        const float sg = (float)w.sti[a];
        const int lo_i = lo_v[a], hi_i = hi_v[a] - 1;
        int i = (int)floorf(fmaf(w.a_in, ray.d[a], ray.s[a] + shift));
        i = i < lo_i ? lo_i : (i > hi_i ? hi_i : i);
        const float a_behind = fmaf(((float)(fwd ? i : i + 1) - pref[a]) * sg, w.da[a], w.a0[a]);
        const float a_ahead = fmaf(((float)(fwd ? i + 1 : i) - pref[a]) * sg, w.da[a], w.a0[a]);
        bool back, ahead;
        if constexpr (CUT) {
            // ties with a_in on this axis were already crossed by the previous box's tail (see CUT above)
            const bool prev_took_ties = interior && a < w.entry_axis;
            const bool behind_is_ours = prev_took_ties ? (a_behind > w.a_in) : (a_behind >= w.a_in);
            const bool ahead_is_theirs = prev_took_ties ? (a_ahead <= w.a_in) : (a_ahead < w.a_in);
            back = behind_is_ours && (fwd ? i > lo_i : i < hi_i);
            ahead = !behind_is_ours && ahead_is_theirs && (fwd ? i < hi_i : i > lo_i);
        } else {
            back = (a_behind >= w.a_in) && (fwd ? i > lo_i : i < hi_i);
            ahead = !(a_behind >= w.a_in) && (a_ahead < w.a_in) && (fwd ? i < hi_i : i > lo_i);
        }
        i += back ? -w.sti[a] : (ahead ? w.sti[a] : 0);
        i = (lo[a] >= w.a_in) ? (fwd ? lo_i : hi_i) : i;
        w.idx[a] = i;
        w.p0[a] = (float)(fwd ? i + 1 : i);
        w.nf[a] = (w.p0[a] - pref[a]) * sg;                                     // crossings already behind us
        w.nx[a] = ((fwd ? (float)hi_v[a] : (float)lo_v[a]) - pref[a]) * sg;      // count of the box's exit plane
        w.an[a] = fmaf(w.nf[a], w.da[a], w.a0[a]);
    }
    return w;
}

B200_HD Walk start_walk(const Ray& ray, const VolDims& dims, float shift)
{
    const int lo_v[3] = {0, 0, 0};
    return start_walk_box(ray, lo_v, dims.d, shift);
}

// Advance the walk across the plane at alpha `anext` (= min of w.an); returns the axis crossed and sets
// `inside` to whether the new voxel is still in the volume.
B200_HD int step_walk(Walk& w, const VolDims& dims, float anext, int64_t& off, const int64_t so[3], bool& inside)
{
    int ax;
    if (w.an[0] == anext) ax = 0;
    else if (w.an[1] == anext) ax = 1;
    else ax = 2;
#pragma unroll
    for (int a = 0; a < 3; ++a)
        if (a == ax) {
            w.idx[a] += w.sti[a];
            inside = (unsigned)w.idx[a] < (unsigned)dims.d[a];
            off += so[a];
            w.nf[a] += 1.0f;
            w.an[a] = fmaf(w.nf[a], w.da[a], w.a0[a]);
        }
    return ax;
}

// Sum of v * (alpha_{j+1} - alpha_j) over the voxels the line crosses (multiply by raylen outside).
// COUNT=true skips the loads and returns the number of voxels visited instead.
template <bool COUNT>
B200_HD float siddon_ray_fast(const float* vol, const VolDims& dims, const Ray& ray, float shift, int* visits)
{
    Walk w = start_walk(ray, dims, shift);
    if (!w.hit) {
        if (COUNT) *visits = 0;
        return 0.0f;
    }
    const int64_t s1 = dims.d[2], s0 = (int64_t)dims.d[1] * dims.d[2];
    int64_t off = ((int64_t)w.idx[0] * dims.d[1] + w.idx[1]) * dims.d[2] + w.idx[2];
    const int64_t so[3] = {w.sti[0] * s0, w.sti[1] * s1, (int64_t)w.sti[2]};
    float acur = w.a_in, acc = 0.0f;
    int count = 0;
    bool inside = true;
    while (inside) {
        const float v = COUNT ? 0.0f : ldg(vol + off);
        const float anext = fminf(fminf(w.an[0], w.an[1]), w.an[2]);
        acc = fmaf(anext - acur, v, acc);
        acur = anext;
        ++count;
        step_walk(w, dims, anext, off, so, inside);
    }
    if (COUNT) *visits = count;
    return acc;
}

// Same sum as siddon_ray_fast, software-pipelined: U walk steps are resolved (index + segment length) before their
// U voxel loads are issued together, so every thread keeps U independent loads in flight (the walk itself never
// depends on loaded data).
template <int U>
B200_HD float siddon_ray_fast_ilp(const float* vol, const VolDims& dims, const Ray& ray, float shift)
{
    Walk w = start_walk(ray, dims, shift);
    if (!w.hit) return 0.0f;
    const int64_t s1 = dims.d[2], s0 = (int64_t)dims.d[1] * dims.d[2];
    int64_t off = ((int64_t)w.idx[0] * dims.d[1] + w.idx[1]) * dims.d[2] + w.idx[2];
    const int64_t so[3] = {w.sti[0] * s0, w.sti[1] * s1, (int64_t)w.sti[2]};
    float acur = w.a_in, acc = 0.0f;
    bool inside = true;
    while (inside) {
        float len[U];
        int64_t offs[U];
#pragma unroll
        for (int k = 0; k < U; ++k) {
            offs[k] = off;
            len[k] = 0.0f;
            if (inside) {
                const float anext = fminf(fminf(w.an[0], w.an[1]), w.an[2]);
                len[k] = anext - acur;
                acur = anext;
                step_walk(w, dims, anext, off, so, inside);
            } else {
                offs[k] = -1;
            }
        }
        float v[U];
#pragma unroll
        for (int k = 0; k < U; ++k) v[k] = offs[k] >= 0 ? ldg(vol + offs[k]) : 0.0f;
#pragma unroll
        for (int k = 0; k < U; ++k) acc = fmaf(len[k], v[k], acc);
    }
    return acc;
}

// ---------------------------------------------------------------------------------------------------
// Lean walk: the same sum again with a branch-free step of ~19 instructions.
//   * termination by alpha: the exit plane's alpha is computed by the very expression that produces the
//     walk's own crossing alphas (fma(n, |1/d|, alpha_first)), so `anext < a_out` is exact and no per-axis
//     index/bounds bookkeeping is needed -- the only per-ray state is (an[3], nf[3], off, acur, acc);
//   * all axes whose next plane ties with the minimum step together (the zero-length segments in between
//     contribute nothing), which removes the else-chain;
//   * the final crossing (anext == a_out) is not taken, so `off` never leaves the volume and the U loads of
//     a group can be issued unconditionally.
// Needs D0*D1*D2 < 2^31 (32-bit element offsets); the launcher falls back to siddon_ray_fast_ilp otherwise.
// ---------------------------------------------------------------------------------------------------
B200_HD float min3f(float a, float b, float c)
{
#if defined(__CUDA_ARCH__)
    float r;
    asm("min.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));  // FMNMX3 on sm_100a
    return r;
#else
    return fminf(fminf(a, b), c);
#endif
}

struct LeanState {
    float an0, an1, an2;  // alpha of the next plane per axis
    float nf0, nf1, nf2;  // crossing counters (see Walk)
    float acur;           // alpha reached so far
    int off;              // element offset of the current voxel
};

struct LeanConst {
    float da0, da1, da2, a00, a01, a02, a_out;
    int so0, so1, so2;
};

// One walk step: returns the length (in alpha) of the segment inside the current voxel and moves to the next voxel.
// 17 issue slots on sm_100a: FMNMX3, FADD, FSETP x4, 3 x (@p FADD, @p FFMA, @p IADD).
B200_HD float lean_step(LeanState& s, const LeanConst& k)
{
    float len;
#if defined(__CUDA_ARCH__)
    asm("{\n\t"
        ".reg .pred q, p0, p1, p2;\n\t"
        ".reg .f32 nx;\n\t"
        "min.f32 nx, %0, %1, %2;\n\t"
        "sub.f32 %8, nx, %6;\n\t"
        "mov.f32 %6, nx;\n\t"
        "setp.lt.f32 q, nx, %9;\n\t"
        "setp.eq.and.f32 p0, %0, nx, q;\n\t"
        "setp.eq.and.f32 p1, %1, nx, q;\n\t"
        "setp.eq.and.f32 p2, %2, nx, q;\n\t"
        "@p0 add.f32 %3, %3, 0f3F800000;\n\t"
        "@p1 add.f32 %4, %4, 0f3F800000;\n\t"
        "@p2 add.f32 %5, %5, 0f3F800000;\n\t"
        "@p0 fma.rn.f32 %0, %3, %10, %13;\n\t"
        "@p1 fma.rn.f32 %1, %4, %11, %14;\n\t"
        "@p2 fma.rn.f32 %2, %5, %12, %15;\n\t"
        "@p0 add.s32 %7, %7, %16;\n\t"
        "@p1 add.s32 %7, %7, %17;\n\t"
        "@p2 add.s32 %7, %7, %18;\n\t"
        "}"
        : "+f"(s.an0), "+f"(s.an1), "+f"(s.an2), "+f"(s.nf0), "+f"(s.nf1), "+f"(s.nf2), "+f"(s.acur), "+r"(s.off),
          "=f"(len)
        : "f"(k.a_out), "f"(k.da0), "f"(k.da1), "f"(k.da2), "f"(k.a00), "f"(k.a01), "f"(k.a02), "r"(k.so0), "r"(k.so1),
          "r"(k.so2));
#else
    const float nx = fminf(fminf(s.an0, s.an1), s.an2);
    len = nx - s.acur;
    s.acur = nx;
    const bool q = nx < k.a_out;
    const bool p0 = q && s.an0 == nx, p1 = q && s.an1 == nx, p2 = q && s.an2 == nx;
    if (p0) { s.nf0 += 1.0f; s.an0 = fmaf(s.nf0, k.da0, k.a00); s.off += k.so0; }
    if (p1) { s.nf1 += 1.0f; s.an1 = fmaf(s.nf1, k.da1, k.a01); s.off += k.so1; }
    if (p2) { s.nf2 += 1.0f; s.an2 = fmaf(s.nf2, k.da2, k.a02); s.off += k.so2; }
#endif
    return len;
}

B200_HD void lean_init(const Walk& w, int st0, int st1, int st2, LeanState& s, LeanConst& k)
{
    k.da0 = w.da[0]; k.da1 = w.da[1]; k.da2 = w.da[2];
    k.a00 = w.a0[0]; k.a01 = w.a0[1]; k.a02 = w.a0[2];
    k.a_out = w.a_out;
    k.so0 = w.sti[0] * st0; k.so1 = w.sti[1] * st1; k.so2 = w.sti[2] * st2;
    s.an0 = w.an[0]; s.an1 = w.an[1]; s.an2 = w.an[2];
    s.nf0 = w.nf[0]; s.nf1 = w.nf[1]; s.nf2 = w.nf[2];
    s.acur = w.hit ? w.a_in : w.a_out;  // a miss has nothing to walk
    s.off = w.idx[0] * st0 + w.idx[1] * st1 + w.idx[2] * st2;
}

// Lean walk over the sub-box [lo, hi) of a volume whose element strides are (st0, st1, st2).
template <int U>
B200_HD float siddon_ray_lean_box(const float* vol, const int lo_v[3], const int hi_v[3], int st0, int st1, int st2,
                                  const Ray& ray, float shift)
{
    const Walk w = start_walk_box(ray, lo_v, hi_v, shift);
    if (!w.hit) return 0.0f;
    LeanConst k;
    LeanState s;
    lean_init(w, st0, st1, st2, s, k);
    float acc = 0.0f;
    while (s.acur < k.a_out) {
        float len[U], v[U];
        int offs[U];
#pragma unroll
        for (int j = 0; j < U; ++j) {
            offs[j] = s.off;
            len[j] = lean_step(s, k);
        }
#pragma unroll
        for (int j = 0; j < U; ++j) v[j] = ldg(vol + offs[j]);
#pragma unroll
        for (int j = 0; j < U; ++j) acc = fmaf(len[j], v[j], acc);
    }
    return acc;
}

// ---- EXPERIMENT (opt-in, b200drr_x_siddon_fwd_chunk): per-lane chunk reuse ------------------------------------------
// The lean walk over a copy of the volume whose FASTEST axis is the rays' major axis: consecutive visits of a ray then
// mostly sit next to each other in memory, so a lane fetches an aligned W-voxel chunk (W = 2 or 4: one LDG.64 / LDG.128)
// and serves the following visits from registers until a minor-axis crossing moves it to another row.  CPU emulation of
// the bench rays: 0.45 chunk loads per visit at W = 4 instead of ~0.9 sectors per visit -- the L1 gather machinery is what
// bounds the forward kernel (DESIGN.md 4.1).  Same voxels, same lengths, same summation order as siddon_ray_lean_box:
// results are bitwise identical.  `volT` must be padded by W floats (the last chunk may read past the last voxel).
template <int W>
struct Chunk;
template <>
struct Chunk<4> {
    float v[4];
    B200_HD static Chunk load(const float* base, int c)
    {
        Chunk q;
#if defined(__CUDA_ARCH__)
        const float4 t = __ldg(reinterpret_cast<const float4*>(base) + c);
        q.v[0] = t.x; q.v[1] = t.y; q.v[2] = t.z; q.v[3] = t.w;
#else
        for (int i = 0; i < 4; ++i) q.v[i] = base[4 * (long)c + i];
#endif
        return q;
    }
    B200_HD float pick(int i) const { return i < 2 ? (i == 0 ? v[0] : v[1]) : (i == 2 ? v[2] : v[3]); }
};
template <>
struct Chunk<2> {
    float v[2];
    B200_HD static Chunk load(const float* base, int c)
    {
        Chunk q;
#if defined(__CUDA_ARCH__)
        const float2 t = __ldg(reinterpret_cast<const float2*>(base) + c);
        q.v[0] = t.x; q.v[1] = t.y;
#else
        for (int i = 0; i < 2; ++i) q.v[i] = base[2 * (long)c + i];
#endif
        return q;
    }
    B200_HD float pick(int i) const { return i == 0 ? v[0] : v[1]; }
};

template <int U, int W>
B200_HD float siddon_ray_lean_box_chunk(const float* volT, const int lo_v[3], const int hi_v[3], int st0, int st1, int st2,
                                        const Ray& ray, float shift)
{
    constexpr int SH = W == 4 ? 2 : 1;
    const Walk w = start_walk_box(ray, lo_v, hi_v, shift);
    if (!w.hit) return 0.0f;
    LeanConst k;
    LeanState s;
    lean_init(w, st0, st1, st2, s, k);
    float acc = 0.0f;
    int ccur = -1;  // id of the chunk held in `cur`
    Chunk<W> cur;
#pragma unroll
    for (int i = 0; i < W; ++i) cur.v[i] = 0.0f;
    while (s.acur < k.a_out) {
        float len[U];
        int offs[U];
#pragma unroll
        for (int j = 0; j < U; ++j) {
            offs[j] = s.off;
            len[j] = lean_step(s, k);
        }
        Chunk<W> q[U];
        bool need[U];
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int c = offs[j] >> SH;
            need[j] = c != (j == 0 ? ccur : (offs[j - 1] >> SH));
            if (need[j]) q[j] = Chunk<W>::load(volT, c);
        }
#pragma unroll
        for (int j = 0; j < U; ++j) {
            if (need[j]) cur = q[j];
            acc = fmaf(len[j], cur.pick(offs[j] & (W - 1)), acc);
        }
        ccur = offs[U - 1] >> SH;
    }
    return acc;
}

template <int U>
B200_HD float siddon_ray_lean(const float* vol, const VolDims& dims, const Ray& ray, float shift)
{
    const int lo_v[3] = {0, 0, 0};
    return siddon_ray_lean_box<U>(vol, lo_v, dims.d, dims.d[1] * dims.d[2], dims.d[2], 1, ray, shift);
}

// Lean step for the backward walk: additionally reports which axis' plane ends the current voxel
// (0/1/2; 3 when the walk has reached the exit plane and no crossing is taken).  Unlike lean_step, planes that
// tie are crossed ONE PER STEP (lowest axis first, like a stable sort of the reference's cat([ax, ay, az])): the
// zero-length voxel in between carries no mass but it decides how the crossing coefficient v_before - v_after is
// split between the two axes' gradients.  (Ties are not rare: regular detector grids produce exact edge hits.)
B200_HD float lean_step_ax(LeanState& s, const LeanConst& k, int& ax)
{
    float len;
#if defined(__CUDA_ARCH__)
    asm("{\n\t"
        ".reg .pred q, p0, p1, p2;\n\t"
        ".reg .f32 nx;\n\t"
        "min.f32 nx, %0, %1, %2;\n\t"
        "sub.f32 %8, nx, %6;\n\t"
        "mov.f32 %6, nx;\n\t"
        "setp.lt.f32 q, nx, %10;\n\t"
        "setp.eq.and.f32 p0, %0, nx, q;\n\t"
        "setp.eq.and.f32 p1, %1, nx, q;\n\t"
        "setp.eq.and.f32 p2, %2, nx, q;\n\t"
        "and.pred p1, p1, !p0;\n\t"
        "or.pred q, p0, p1;\n\t"
        "and.pred p2, p2, !q;\n\t"
        "selp.s32 %9, 2, 3, p2;\n\t"
        "selp.s32 %9, 1, %9, p1;\n\t"
        "selp.s32 %9, 0, %9, p0;\n\t"
        "@p0 add.f32 %3, %3, 0f3F800000;\n\t"
        "@p1 add.f32 %4, %4, 0f3F800000;\n\t"
        "@p2 add.f32 %5, %5, 0f3F800000;\n\t"
        "@p0 fma.rn.f32 %0, %3, %11, %14;\n\t"
        "@p1 fma.rn.f32 %1, %4, %12, %15;\n\t"
        "@p2 fma.rn.f32 %2, %5, %13, %16;\n\t"
        "@p0 add.s32 %7, %7, %17;\n\t"
        "@p1 add.s32 %7, %7, %18;\n\t"
        "@p2 add.s32 %7, %7, %19;\n\t"
        "}"
        : "+f"(s.an0), "+f"(s.an1), "+f"(s.an2), "+f"(s.nf0), "+f"(s.nf1), "+f"(s.nf2), "+f"(s.acur), "+r"(s.off),
          "=f"(len), "=r"(ax)
        : "f"(k.a_out), "f"(k.da0), "f"(k.da1), "f"(k.da2), "f"(k.a00), "f"(k.a01), "f"(k.a02), "r"(k.so0), "r"(k.so1),
          "r"(k.so2));
#else
    const float nx = fminf(fminf(s.an0, s.an1), s.an2);
    len = nx - s.acur;
    s.acur = nx;
    const bool q = nx < k.a_out;
    const bool p0 = q && s.an0 == nx, p1 = q && !p0 && s.an1 == nx, p2 = q && !p0 && !p1 && s.an2 == nx;
    ax = p0 ? 0 : (p1 ? 1 : (p2 ? 2 : 3));
    if (p0) { s.nf0 += 1.0f; s.an0 = fmaf(s.nf0, k.da0, k.a00); s.off += k.so0; }
    if (p1) { s.nf1 += 1.0f; s.an1 = fmaf(s.nf1, k.da1, k.a01); s.off += k.so1; }
    if (p2) { s.nf2 += 1.0f; s.an2 = fmaf(s.nf2, k.da2, k.a02); s.off += k.so2; }
#endif
    return len;
}

// mask_to_channels (reference renderers.py:77-89): the same lean walk, but every segment's term goes to the channel
// given by the label volume at the same voxel.  Labels are piecewise constant along a ray, so the walk keeps a running
// sum per label RUN and flushes it to out[label] when the label changes (few flushes per ray; each (pose, ray) column of
// `out` belongs to exactly one thread, so a plain += suffices).  `out_n` points at out[b][0][n]; channels are `cstride`
// floats apart.  Labels outside [0, C) are dropped (the reference's scatter_add_ would raise).
template <int U, bool ATOMIC>
B200_HD void siddon_ray_lean_mask_box(const float* vol, const float* mask, const int lo_v[3], const int hi_v[3], int st0, int st1,
                                      int st2, const Ray& ray, float shift, float L, float* out_n, int64_t cstride, int C)
{
    const Walk w = start_walk_box(ray, lo_v, hi_v, shift);
    if (!w.hit) return;
    LeanConst k;
    LeanState s;
    lean_init(w, st0, st1, st2, s, k);
    int cur = -1;
    float run = 0.0f;
    // ATOMIC: several CTAs (one per slab of the volume) own pieces of the same ray -> red.global.add instead of +=
    auto flush = [&](int c, float v) {
        if (v != 0.0f && (unsigned)c < (unsigned)C) {
            if (ATOMIC)
                red_add(out_n + (int64_t)c * cstride, L * v);
            else
                out_n[(int64_t)c * cstride] += L * v;
        }
    };
    while (s.acur < k.a_out) {
        float len[U], v[U], lab[U];
        int offs[U];
#pragma unroll
        for (int j = 0; j < U; ++j) {
            offs[j] = s.off;
            len[j] = lean_step(s, k);
        }
#pragma unroll
        for (int j = 0; j < U; ++j) {
            v[j] = ldg(vol + offs[j]);
            lab[j] = ldg(mask + offs[j]);
        }
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int c = (int)lab[j];
            if (c != cur) {
                flush(cur, run);
                cur = c;
                run = 0.0f;
            }
            run = fmaf(len[j], v[j], run);
        }
    }
    flush(cur, run);
}

template <int U>
B200_HD void siddon_ray_lean_mask(const float* vol, const float* mask, const VolDims& dims, const Ray& ray, float shift,
                                  float L, float* out_n, int64_t cstride, int C)
{
    const int lo_v[3] = {0, 0, 0};
    siddon_ray_lean_mask_box<U, false>(vol, mask, lo_v, dims.d, dims.d[1] * dims.d[2], dims.d[2], 1, ray, shift, L, out_n, cstride,
                                       C);
}

// Trilinear with a label mask (reference renderers.py:242-252): density sampled trilinearly, label sampled NEAREST at
// the same point (round-half-even per axis, zero padding -> label 0).  `scale` = raylen * step.
B200_HD void trilinear_ray_fwd_mask(const float* vol, const float* mask, const VolDims& dims, const Ray& ray, float shift,
                                    int P, float amin, float amax, int align_corners, float scale, float* out_n,
                                    int64_t cstride, int C);

// A[ax] += coef * alpha;  C[ax] += coef   for ax in {0,1,2} (nothing for ax == 3), without branches.
B200_HD void axis_accumulate(int ax, float coef, float alpha, float& A0, float& A1, float& A2, float& C0, float& C1,
                             float& C2)
{
#if defined(__CUDA_ARCH__)
    asm("{\n\t"
        ".reg .pred q0, q1, q2;\n\t"
        "setp.eq.s32 q0, %6, 0;\n\t"
        "setp.eq.s32 q1, %6, 1;\n\t"
        "setp.eq.s32 q2, %6, 2;\n\t"
        "@q0 fma.rn.f32 %0, %7, %8, %0;\n\t"
        "@q1 fma.rn.f32 %1, %7, %8, %1;\n\t"
        "@q2 fma.rn.f32 %2, %7, %8, %2;\n\t"
        "@q0 add.f32 %3, %3, %7;\n\t"
        "@q1 add.f32 %4, %4, %7;\n\t"
        "@q2 add.f32 %5, %5, %7;\n\t"
        "}"
        : "+f"(A0), "+f"(A1), "+f"(A2), "+f"(C0), "+f"(C1), "+f"(C2)
        : "r"(ax), "f"(coef), "f"(alpha));
#else
    if (ax == 0) { A0 = fmaf(coef, alpha, A0); C0 += coef; }
    if (ax == 1) { A1 = fmaf(coef, alpha, A1); C1 += coef; }
    if (ax == 2) { A2 = fmaf(coef, alpha, A2); C2 += coef; }
#endif
}

// ---- two-axis bookkeeping for the sensitivities walk ---------------------------------------------------------------
// Over one box the crossing coefficients telescope:  sum_a C_a = 0  and  sum_a A_a = sum_j v_j len_j  (Abel summation,
// box faces counted against 0).  So only TWO axes need per-crossing accumulation; the third follows from the totals.
// The derived axis is the ray's MAJOR axis M (most crossings -> most work saved; and its gradient is divided by the
// largest |d|, so the subtraction costs no accuracy).  LOCAL axis index: 0 = first minor axis, 1 = second, 2 = neither.
template <int M>
struct MinorAxes {
    static constexpr int U = M == 0 ? 1 : 0;
    static constexpr int V = M == 2 ? 1 : 2;
    B200_HD static int local(int axis) { return axis == U ? 0 : (axis == V ? 1 : 2); }
};

// The sensitivities walk's state: lean_step_ax's (an, nf, acur, off) with the two MINOR axes' alphas and counters held as
// pairs (u, v), so that one packed f32x2 instruction updates both (FADD2 / FFMA2 on sm_100a).
struct SensState {
    Pair an_uv, nf_uv;  // minor axes
    float an_m, nf_m;   // major axis
    float acur;
    int off;
};
struct SensConst {
    Pair da_uv, a0_uv;
    float da_m, a0_m, a_out;
    int so0, so1, so2;
};

// |1/d| of the minor axes as a pair of their own.  Left alone, the compiler folds them into an |abs| modifier on the 1/d
// registers the ray keeps for after the walk; for major axes 1 and 2 those are not adjacent and every FFMA2 of the walk
// would first copy them into a register pair.  (x + 0 is x here: |1/d| is never -0.)
B200_HD Pair own_pair(float a, float b)
{
#if defined(__CUDA_ARCH__)
    float ra, rb;
    asm("add.rn.f32 %0, %1, 0f00000000;" : "=f"(ra) : "f"(a));
    asm("add.rn.f32 %0, %1, 0f00000000;" : "=f"(rb) : "f"(b));
    return Pair{ra, rb};
#else
    return Pair{a, b};
#endif
}

template <int M>
B200_HD void sens_init(const Walk& w, int st0, int st1, int st2, SensState& s, SensConst& k)
{
    using Ax = MinorAxes<M>;
    k.da_uv = own_pair(w.da[Ax::U], w.da[Ax::V]);
    k.a0_uv = Pair{w.a0[Ax::U], w.a0[Ax::V]};
    k.da_m = w.da[M];
    k.a0_m = w.a0[M];
    k.a_out = w.a_out;
    k.so0 = w.sti[0] * st0; k.so1 = w.sti[1] * st1; k.so2 = w.sti[2] * st2;
    s.an_uv = Pair{w.an[Ax::U], w.an[Ax::V]};
    s.nf_uv = Pair{w.nf[Ax::U], w.nf[Ax::V]};
    s.an_m = w.an[M];
    s.nf_m = w.nf[M];
    s.acur = w.hit ? w.a_in : w.a_out;
    s.off = w.idx[0] * st0 + w.idx[1] * st1 + w.idx[2] * st2;
}

// alpha of the next plane on global axis A
template <int M, int A>
B200_HD float sens_an(const SensState& s)
{
    return A == M ? s.an_m : (A == MinorAxes<M>::U ? s.an_uv.x : s.an_uv.y);
}
// crossing counter of global axis A
template <int M, int A>
B200_HD float sens_nf(const SensState& s)
{
    return A == M ? s.nf_m : (A == MinorAxes<M>::U ? s.nf_uv.x : s.nf_uv.y);
}

// One step of the sensitivities walk: lean_step_ax's crossing -- the same alphas and the same sequential tie order (lowest
// axis first; nothing is crossed at the exit alpha) -- with the crossed axis reported as the mask pair m = (crossed u,
// crossed v) in {0, 1}^2 ((0, 0): the major axis or no crossing).  The minor axes are updated without a predicate:
// nf_uv += m, an_uv = fma(nf_uv, da_uv, a0_uv) recomputes an unchanged alpha bit for bit (the walk's set-up forms every `an`
// by that same expression), up to the sign of a zero counter.  Ties:
//   q = nx < a_out;   p0 = q & (an0 == nx), x = q & !(an0 == nx);   p1 = x & (an1 == nx), p2 = x & !(an1 == nx)
// (when q holds and neither axis 0 nor 1 attains the minimum, axis 2 does; `neu` is !(==) also for a NaN alpha).
// sm_100a: FMNMX3, 5 FSETP, 2 FSEL, predicated FADD + FFMA (major), FADD2 + FFMA2 (minor), 3 predicated IADD (one of them
// as IADD + SEL).
#define B200_SENS_STEP_ASM(PM, PU, PV)                                                                                 \
    asm("{\n\t"                                                                                                    \
        ".reg .pred q, x, p0, p1, p2;\n\t"                                                                          \
        ".reg .f32 nx;\n\t"                                                                                         \
        "min.f32 nx, %6, %7, %8;\n\t"                                                                               \
        "mov.f32 %2, nx;\n\t"                                                                                       \
        "setp.lt.f32 q, nx, %9;\n\t"                                                                               \
        "setp.eq.and.f32 p0, %6, nx, q;\n\t"                                                                        \
        "setp.neu.and.f32 x, %6, nx, q;\n\t"                                                                        \
        "setp.eq.and.f32 p1, %7, nx, x;\n\t"                                                                        \
        "setp.neu.and.f32 p2, %7, nx, x;\n\t"                                                                       \
        "selp.f32 %4, 0f3F800000, 0f00000000, " PU ";\n\t"                                                          \
        "selp.f32 %5, 0f3F800000, 0f00000000, " PV ";\n\t"                                                          \
        "@" PM " add.rn.f32 %1, %1, 0f3F800000;\n\t"                                                                \
        "@" PM " fma.rn.f32 %0, %1, %10, %11;\n\t"                                                                  \
        "@p2 add.s32 %3, %3, %14;\n\t"                                                                              \
        "@p1 add.s32 %3, %3, %13;\n\t"                                                                              \
        "@p0 add.s32 %3, %3, %12;\n\t"                                                                              \
        "}"                                                                                                         \
        : "+f"(s.an_m), "+f"(s.nf_m), "=f"(s.acur), "+r"(s.off), "=f"(m.x), "=f"(m.y)                                 \
        : "f"(sens_an<M, 0>(s)), "f"(sens_an<M, 1>(s)), "f"(sens_an<M, 2>(s)), "f"(k.a_out), "f"(k.da_m), "f"(k.a0_m), \
          "r"(k.so0), "r"(k.so1), "r"(k.so2))

template <int M>
B200_HD void sens_step(SensState& s, const SensConst& k, Pair& m)
{
#if defined(__CUDA_ARCH__)
    if (M == 0) B200_SENS_STEP_ASM("p0", "p1", "p2");       // minor axes (1, 2)
    else if (M == 1) B200_SENS_STEP_ASM("p1", "p0", "p2");  // minor axes (0, 2)
    else B200_SENS_STEP_ASM("p2", "p0", "p1");              // minor axes (0, 1)
#else
    const float a0 = sens_an<M, 0>(s), a1 = sens_an<M, 1>(s), a2 = sens_an<M, 2>(s);
    const float nx = fminf(fminf(a0, a1), a2);
    s.acur = nx;
    const bool q = nx < k.a_out;
    const bool p[3] = {q && a0 == nx, q && !(a0 == nx) && a1 == nx, q && !(a0 == nx) && !(a1 == nx)};
    m = Pair{p[MinorAxes<M>::U] ? 1.0f : 0.0f, p[MinorAxes<M>::V] ? 1.0f : 0.0f};
    if (p[M]) { s.nf_m += 1.0f; s.an_m = fmaf(s.nf_m, k.da_m, k.a0_m); }
    if (p[0]) s.off += k.so0;
    if (p[1]) s.off += k.so1;
    if (p[2]) s.off += k.so2;
#endif
    s.nf_uv = add2_rn(s.nf_uv, m);
    s.an_uv = fma2_rn(s.nf_uv, k.da_uv, k.a0_uv);
}

// (Au, Av) += coef*alpha * m, (Cu, Cv) += coef * m: the crossing's coefficient goes to the minor axis its mask selects; the
// other one gets an exact 0 added (FMUL2, FFMA2, FADD2).
B200_HD void minor_accumulate(Pair m, float coef, float alpha, Pair& A, Pair& C)
{
    const Pair cm = mul2_rn(m, Pair{coef, coef});
    A = fma2_rn(cm, Pair{alpha, alpha}, A);
    C = add2_rn(C, cm);
}

// mask pair of a LOCAL index of MinorAxes<M> (0 = u, 1 = v, 2 = neither)
B200_HD Pair minor_mask(int local) { return Pair{local == 0 ? 1.0f : 0.0f, local == 1 ? 1.0f : 0.0f}; }

// How the sensitivities walk fetches its voxels: one scalar load per visit from the volume as stored (production), or --
// EXPERIMENT, see siddon_ray_lean_box_chunk -- W-voxel chunks from a major-axis-fastest copy, re-used across visits.
struct LoadPlain {
    template <int U>
    B200_HD void batch(const float* vol, const int (&offs)[U], float (&v)[U])
    {
#pragma unroll
        for (int j = 0; j < U; ++j) v[j] = ldg(vol + offs[j]);
    }
    B200_HD float at(const float* vol, int off) const { return ldg(vol + off); }
};

template <int W>
struct LoadChunk {
    Chunk<W> cur;
    int ccur = -1;
    template <int U>
    B200_HD void batch(const float* volT, const int (&offs)[U], float (&v)[U])
    {
        constexpr int SH = W == 4 ? 2 : 1;
        Chunk<W> q[U];
        bool need[U];
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int c = offs[j] >> SH;
            need[j] = c != (j == 0 ? ccur : (offs[j - 1] >> SH));
            if (need[j]) q[j] = Chunk<W>::load(volT, c);
        }
#pragma unroll
        for (int j = 0; j < U; ++j) {
            if (need[j]) cur = q[j];
            v[j] = cur.pick(offs[j] & (W - 1));
        }
        ccur = offs[U - 1] >> SH;
    }
    B200_HD float at(const float* volT, int off) const { return ldg(volT + off); }
};

// The sensitivities walk of one ray restricted to a box, for a ray whose major axis is M: same walk, tie order and
// tail as siddon_ray_bwd_lean_box, two accumulated axes + the telescoping identities.  A, C accumulated INTO.
template <int U, int M, class Load = LoadPlain, bool CUT = false>
B200_HD float siddon_ray_sens_box_m(const float* vol, const VolDims& dims, const int lo_v[3], const int hi_v[3], int st0,
                                    int st1, int st2, const Ray& ray, float shift, float A[3], float C[3])
{
    using Ax = MinorAxes<M>;
    Load loader;
    const Walk w = start_walk_frame<CUT>(ray, dims, lo_v, hi_v, shift);
    if (!w.hit) return 0.0f;
    SensConst k;
    SensState s;
    sens_init<M>(w, st0, st1, st2, s, k);
    Pair Auv = {0.0f, 0.0f}, Cuv = {0.0f, 0.0f};
    float acc = 0.0f;
    Pair prev = {0.0f, w.a_in};  // (value of the voxel before, alpha of the crossing that left it)
    Pair mprev = minor_mask(Ax::local(w.entry_axis));
    if (!(s.acur < k.a_out)) {  // the box is only touched (a_in == a_out): the entry crossing leads into the one voxel
        prev.x = loader.at(vol, s.off);
        minor_accumulate(mprev, -prev.x, w.a_in, Auv, Cuv);
    }
    while (s.acur < k.a_out) {
        float v[U];
        int offs[U];
        Pair m[U], va[U];
#pragma unroll
        for (int j = 0; j < U; ++j) {
            offs[j] = s.off;
            sens_step<M>(s, k, m[j]);
            va[j].y = s.acur;
        }
        loader.template batch<U>(vol, offs, v);
#pragma unroll
        for (int j = 0; j < U; ++j) {
            // crossing (mprev, prev.y) led into voxel j; padding steps after the exit carry the mask (0, 0) and length 0.
            // One FADD2 forms (v_j - v_before, alpha_j - alpha_before) = (-coef, segment length): the same two
            // subtractions, the first with its operands swapped, which negates it exactly.
            va[j].x = v[j];
            const Pair d = sub2_rn(va[j], prev);
            minor_accumulate(mprev, -d.x, prev.y, Auv, Cuv);
            acc = fmaf(d.y, va[j].x, acc);
            prev = va[j];
            mprev = m[j];
        }
    }
    float vprev = prev.x;
    // Tail: identical to siddon_ray_bwd_lean_box (ties with the exit alpha, lowest axis first)
    int ax_exit = 3;
    {
        const float an0 = sens_an<M, 0>(s), an1 = sens_an<M, 1>(s), an2 = sens_an<M, 2>(s);
        const bool t0 = an0 <= k.a_out, t1 = an1 <= k.a_out, t2 = an2 <= k.a_out;
        const bool b0 = sens_nf<M, 0>(s) == w.nx[0], b1 = sens_nf<M, 1>(s) == w.nx[1], b2 = sens_nf<M, 2>(s) == w.nx[2];
        if (t0 && b0) ax_exit = 0;
        if (ax_exit == 3 && t0) {
            s.off += k.so0;
            const float vm = loader.at(vol, s.off);
            minor_accumulate(minor_mask(Ax::local(0)), vprev - vm, k.a_out, Auv, Cuv);
            vprev = vm;
        }
        if (ax_exit == 3 && t1 && b1) ax_exit = 1;
        if (ax_exit == 3 && t1) {
            s.off += k.so1;
            const float vm = loader.at(vol, s.off);
            minor_accumulate(minor_mask(Ax::local(1)), vprev - vm, k.a_out, Auv, Cuv);
            vprev = vm;
        }
        if (ax_exit == 3 && t2 && b2) ax_exit = 2;
        if (ax_exit == 3) ax_exit = (an0 <= an1 && an0 <= an2) ? 0 : (an1 <= an2 ? 1 : 2);
    }
    minor_accumulate(minor_mask(Ax::local(ax_exit)), vprev, k.a_out, Auv, Cuv);
    const float Au = Auv.x, Av = Auv.y, Cu = Cuv.x, Cv = Cuv.y;
    A[Ax::U] += Au;
    A[Ax::V] += Av;
    A[M] += acc - Au - Av;  // sum_a A_a = sum_j v_j len_j over the box
    C[Ax::U] += Cu;
    C[Ax::V] += Cv;
    C[M] -= Cu + Cv;        // sum_a C_a = 0 over the box
    return acc;
}

// Dispatch on the ray's major axis (uniform per warp except for rays near a 45-degree direction).
template <int U, class Load = LoadPlain, bool CUT = false>
B200_HD float siddon_ray_sens_box(const float* vol, const VolDims& dims, const int lo_v[3], const int hi_v[3], int st0,
                                  int st1, int st2, const Ray& ray, float shift, float A[3], float C[3])
{
    const float a0 = fabsf(ray.d[0]), a1 = fabsf(ray.d[1]), a2 = fabsf(ray.d[2]);
    if (a0 >= a1 && a0 >= a2)
        return siddon_ray_sens_box_m<U, 0, Load, CUT>(vol, dims, lo_v, hi_v, st0, st1, st2, ray, shift, A, C);
    if (a1 >= a2) return siddon_ray_sens_box_m<U, 1, Load, CUT>(vol, dims, lo_v, hi_v, st0, st1, st2, ray, shift, A, C);
    return siddon_ray_sens_box_m<U, 2, Load, CUT>(vol, dims, lo_v, hi_v, st0, st1, st2, ray, shift, A, C);
}

// Backward of one ray restricted to the sub-box [lo, hi) (closed form, see siddon_ray_bwd below for the algebra).
// Crossing m between voxel values (before, after) on axis a at alpha contributes coef = before - after to
//   A_a += coef * alpha,  C_a += coef;  box faces count as crossings against 0, which telescopes correctly when a
// ray is split into slabs (the two halves of an interior face add up to the true coefficient).
// Returns sum_j v_j len_j; adds gL*len_j to g_vol[voxel_j] when g_vol != nullptr.  A, C are accumulated INTO.
template <int U, bool WANT_VOL>
B200_HD float siddon_ray_bwd_lean_box(const float* vol, const VolDims& dims, const int lo_v[3], const int hi_v[3], int st0,
                                      int st1, int st2, const Ray& ray, float shift, float gL, float* g_vol, float A[3],
                                      float C[3])
{
    const Walk w = start_walk_frame(ray, dims, lo_v, hi_v, shift);
    if (!w.hit) return 0.0f;
    LeanConst k;
    LeanState s;
    lean_init(w, st0, st1, st2, s, k);
    float A0 = 0.0f, A1 = 0.0f, A2 = 0.0f, C0 = 0.0f, C1 = 0.0f, C2 = 0.0f;
    float acc = 0.0f, vprev = 0.0f, aprev = w.a_in;
    int axprev = w.entry_axis;
    bool any = false;
    while (s.acur < k.a_out) {
        float len[U], aend[U], v[U];
        int offs[U], ax[U];
#pragma unroll
        for (int j = 0; j < U; ++j) {
            offs[j] = s.off;
            len[j] = lean_step_ax(s, k, ax[j]);
            aend[j] = s.acur;
        }
#pragma unroll
        for (int j = 0; j < U; ++j) v[j] = ldg(vol + offs[j]);
#pragma unroll
        for (int j = 0; j < U; ++j) {
            // crossing (axprev, aprev) led into voxel j; after the exit the padding steps carry axprev == 3 (matches no
            // axis) and len == 0, so they fall through without a branch
            axis_accumulate(axprev, vprev - v[j], aprev, A0, A1, A2, C0, C1, C2);
            acc = fmaf(len[j], v[j], acc);
            if (WANT_VOL) {
                if (len[j] != 0.0f) red_add(g_vol + offs[j], gL * len[j]);
            }
            any = any || (axprev < 3);
            vprev = v[j];
            axprev = ax[j];
            aprev = aend[j];
        }
    }
    if (!any) {  // the box is only touched (a_in == a_out, e.g. the ray enters the volume exactly on a slab face)
        const float v0 = ldg(vol + s.off);
        axis_accumulate(w.entry_axis, -v0, w.a_in, A0, A1, A2, C0, C1, C2);
        vprev = v0;
    }
    // Tail: crossings that TIE with the exit alpha are taken lowest axis first (stable-sort order) until the first
    // boundary plane is met; interior planes among them lead through zero-length voxels that only matter for how the
    // exit coefficient is split between the axes.  (Regular detector grids hit voxel edges exactly, so this is common.)
    int ax_exit = 3;
    {
        const bool t0 = s.an0 <= k.a_out, t1 = s.an1 <= k.a_out, t2 = s.an2 <= k.a_out;
        const bool b0 = s.nf0 == w.nx[0], b1 = s.nf1 == w.nx[1], b2 = s.nf2 == w.nx[2];
        if (t0 && b0) ax_exit = 0;
        if (ax_exit == 3 && t0) {  // interior plane of axis 0 at the exit alpha
            s.off += k.so0;
            const float vm = ldg(vol + s.off);
            axis_accumulate(0, vprev - vm, k.a_out, A0, A1, A2, C0, C1, C2);
            vprev = vm;
        }
        if (ax_exit == 3 && t1 && b1) ax_exit = 1;
        if (ax_exit == 3 && t1) {
            s.off += k.so1;
            const float vm = ldg(vol + s.off);
            axis_accumulate(1, vprev - vm, k.a_out, A0, A1, A2, C0, C1, C2);
            vprev = vm;
        }
        if (ax_exit == 3 && t2 && b2) ax_exit = 2;
        if (ax_exit == 3) ax_exit = (s.an0 <= s.an1 && s.an0 <= s.an2) ? 0 : (s.an1 <= s.an2 ? 1 : 2);
    }
    axis_accumulate(ax_exit, vprev, k.a_out, A0, A1, A2, C0, C1, C2);
    A[0] += A0; A[1] += A1; A[2] += A2;
    C[0] += C0; C[1] += C1; C[2] += C2;
    return acc;
}

// Closed-form backward of one ray (SURVEY.md 8a-G).  With v_j the voxel of segment j and crossing m on
// axis a:  dI/dalpha_m = L (v_{m-1} - v_m),  dalpha/ds_a = (alpha - 1)/d_a,  dalpha/dt_a = -alpha/d_a.
// Per axis accumulate A_a = sum coef*alpha, C_a = sum coef with coef = v_before - v_after; then
//   g_t[a] = -g L A_a / d_a,   g_s[a] = g L (A_a - C_a) / d_a.
// Returns sum_j v_j len_j (for g_raylen); g_vol[voxel_j] += gL * len_j when g_vol != nullptr.
// `fetch(off, gj)` returns the EFFECTIVE voxel value gj * V[off] and the per-voxel upstream factor gj: 1 for the plain
// renderer; with a label mask (mask_to_channels, renderers.py:77-89) gj = gout[b][label(off)][n], the gradient of the
// channel the segment was scattered to -- everything else is unchanged (v_j -> g_j v_j, g = 1).
struct FetchPlain {
    const float* vol;
    B200_HD float operator()(int64_t off, float& gj) const
    {
        gj = 1.0f;
        return ldg(vol + off);
    }
};

struct FetchMasked {
    const float* vol;
    const float* mask;
    const float* gch;  // gout[b][0][n]; channels are cstride floats apart
    int64_t cstride;
    int C;
    B200_HD float operator()(int64_t off, float& gj) const
    {
        const int c = (int)ldg(mask + off);
        gj = (unsigned)c < (unsigned)C ? ldg(gch + (int64_t)c * cstride) : 0.0f;
        return gj * ldg(vol + off);
    }
};

template <class Fetch>
B200_HD float siddon_ray_bwd_f(const Fetch& fetch, const VolDims& dims, const Ray& ray, float shift, float gL, float* g_vol,
                               float gs[3], float gt[3])
{
    Walk w = start_walk(ray, dims, shift);
    float A[3] = {0.0f, 0.0f, 0.0f}, C[3] = {0.0f, 0.0f, 0.0f};
    float acc = 0.0f;
    if (w.hit) {
        const int64_t s1 = dims.d[2], s0 = (int64_t)dims.d[1] * dims.d[2];
        int64_t off = ((int64_t)w.idx[0] * dims.d[1] + w.idx[1]) * dims.d[2] + w.idx[2];
        const int64_t so[3] = {w.sti[0] * s0, w.sti[1] * s1, (int64_t)w.sti[2]};
        float acur = w.a_in, vprev = 0.0f;
        int axis_in = w.entry_axis;
        bool inside = true;
        while (inside) {
            float gj;
            const float v = fetch(off, gj);
            const float coef = vprev - v;  // crossing into this voxel at acur through axis_in
#pragma unroll
            for (int a = 0; a < 3; ++a)
                if (a == axis_in) {
                    A[a] = fmaf(coef, acur, A[a]);
                    C[a] += coef;
                }
            const float anext = fminf(fminf(w.an[0], w.an[1]), w.an[2]);
            const float len = anext - acur;
            acc = fmaf(len, v, acc);
            if (g_vol) red_add(g_vol + off, (gL * gj) * len);
            acur = anext;
            vprev = v;
            axis_in = step_walk(w, dims, anext, off, so, inside);
        }
        // exit crossing: v_last -> 0 through axis_in at acur
#pragma unroll
        for (int a = 0; a < 3; ++a)
            if (a == axis_in) {
                A[a] = fmaf(vprev, acur, A[a]);
                C[a] += vprev;
            }
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        gt[a] = -gL * A[a] * ray.inv[a];
        gs[a] = gL * (A[a] - C[a]) * ray.inv[a];
    }
    return acc;
}

B200_HD float siddon_ray_bwd(const float* vol, const VolDims& dims, const Ray& ray, float shift, float gL, float* g_vol,
                             float gs[3], float gt[3])
{
    return siddon_ray_bwd_f(FetchPlain{vol}, dims, ray, shift, gL, g_vol, gs, gt);
}

// ===================================================================================================
// Trilinear ray marching.  Continuous voxel coordinate as a linear function of alpha:
//   pix_a = p0_a + alpha * dp_a,   from x = s + alpha d,  g = 2 (x + shift)/D - 1  (renderers.py:148-152) and
//   ATen's un-normalisation: align_corners=False -> pix = x + shift - 0.5;  True -> pix = (x + shift)(D-1)/D.
// Interpolation weights are plain fp32 (no texture-unit fixed-point filtering: it would break 1e-4).
// ===================================================================================================
struct PixLine {
    float p0[3], dp[3], ka[3];
};

B200_HD PixLine make_pixline(const Ray& ray, const VolDims& dims, float shift, int align_corners)
{
    PixLine pl;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float ka = align_corners ? (float)(dims.d[a] - 1) / (float)dims.d[a] : 1.0f;
        const float kb = align_corners ? shift * ka : shift - 0.5f;
        pl.ka[a] = ka;
        pl.p0[a] = fmaf(ray.s[a], ka, kb);
        pl.dp[a] = ray.d[a] * ka;
    }
    return pl;
}

// torch.linspace(0, 1, P)[m] exactly as ATen evaluates it in fp32 (symmetric halves, fused end - step*k).
B200_HD float linspace01(int m, int P, float step)
{
    return (m < P / 2) ? mul_rn(step, (float)m) : fmaf(-step, (float)(P - 1 - m), 1.0f);
}

// Sample index range [m_lo, m_hi] whose points can touch the volume (pix in (-1, D) on every axis);
// samples outside it interpolate only zero padding.  One sample of slack on both sides.
B200_HD void sample_range(const PixLine& pl, const VolDims& dims, float amin, float range, int P, int& m_lo, int& m_hi)
{
    float lo = -INFINITY, hi = INFINITY;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float inv = 1.0f / pl.dp[a];
        const float a0 = (-1.0f - pl.p0[a]) * inv, a1 = ((float)dims.d[a] - pl.p0[a]) * inv;
        lo = fmaxf(lo, fminf(a0, a1));
        hi = fminf(hi, fmaxf(a0, a1));
    }
    if (!(range > 0.0f)) {  // degenerate range: march everything
        m_lo = 0;
        m_hi = P - 1;
        return;
    }
    if (!(lo <= hi)) {  // the line misses the (padded) volume
        m_lo = 1;
        m_hi = 0;
        return;
    }
    const float scale = (float)(P - 1) / range;
    const float f_lo = floorf((lo - amin) * scale) - 1.0f, f_hi = ceilf((hi - amin) * scale) + 1.0f;
    m_lo = (int)fmaxf(0.0f, fminf(f_lo, (float)P));
    m_hi = (int)fminf((float)(P - 1), fmaxf(f_hi, -1.0f));
}

// Narrow [m_lo, m_hi] to the samples whose BASE voxel along axis 0 (floor(pix0)) can lie in [s_lo, s_hi): the
// slab-major trilinear kernels cut the volume into such slabs; the loop re-checks every sample exactly, so each
// sample is counted by exactly one slab.  One sample of slack on both sides.
B200_HD void sample_range_slab(const PixLine& pl, float amin, float range, int P, float s_lo, float s_hi, int& m_lo,
                               int& m_hi)
{
    if (!(range > 0.0f) || m_lo > m_hi) return;
    const float inv = 1.0f / pl.dp[0];
    const float a0 = (s_lo - pl.p0[0]) * inv, a1 = (s_hi - pl.p0[0]) * inv;
    const float lo = fminf(a0, a1), hi = fmaxf(a0, a1);
    if (!(lo <= hi)) return;  // dp0 == 0 (NaN): the ray runs inside one slab, keep the whole range
    const float scale = (float)(P - 1) / range;
    const float f_lo = floorf((lo - amin) * scale) - 1.0f, f_hi = ceilf((hi - amin) * scale) + 1.0f;
    const int n_lo = (int)fmaxf(0.0f, fminf(f_lo, (float)P)), n_hi = (int)fminf((float)(P - 1), fmaxf(f_hi, -1.0f));
    m_lo = m_lo > n_lo ? m_lo : n_lo;
    m_hi = m_hi < n_hi ? m_hi : n_hi;
}

struct Corner8 {
    float v[8];
    float f[3];
    int64_t base;   // offset of corner (0,0,0); only dereferenced where the in-bounds mask is set
    unsigned mask;  // bit c = corner c in bounds, c = o0 | o1<<1 | o2<<2 (o_a = offset along volume axis a)
};

B200_HD int64_t corner_off(const VolDims& dims, int c)
{
    return (int64_t)(c & 1) * dims.d[1] * dims.d[2] + (int64_t)((c >> 1) & 1) * dims.d[2] + ((c >> 2) & 1);
}

B200_HD Corner8 gather8(const float* vol, const VolDims& dims, const float pix[3])
{
    Corner8 k;
    int i0[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float fl = floorf(pix[a]);
        k.f[a] = pix[a] - fl;
        i0[a] = (int)fl;
    }
    k.base = ((int64_t)i0[0] * dims.d[1] + i0[1]) * dims.d[2] + i0[2];
    const bool interior = (unsigned)i0[0] < (unsigned)(dims.d[0] - 1) && (unsigned)i0[1] < (unsigned)(dims.d[1] - 1) &&
                          (unsigned)i0[2] < (unsigned)(dims.d[2] - 1);
    if (interior) {
        k.mask = 0xffu;
#pragma unroll
        for (int c = 0; c < 8; ++c) k.v[c] = ldg(vol + k.base + corner_off(dims, c));
    } else {
        k.mask = 0u;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const int x = i0[0] + (c & 1), y = i0[1] + ((c >> 1) & 1), z = i0[2] + ((c >> 2) & 1);
            const bool inb = (unsigned)x < (unsigned)dims.d[0] && (unsigned)y < (unsigned)dims.d[1] &&
                             (unsigned)z < (unsigned)dims.d[2];
            k.v[c] = inb ? ldg(vol + k.base + corner_off(dims, c)) : 0.0f;
            k.mask |= inb ? (1u << c) : 0u;
        }
    }
    return k;
}

// Gather policies for the trilinear marchers: 8 scalar loads from the plain volume, or one 32-byte read from the
// packed-corner copy (see trilinear_ray_fwd_packed).
struct GatherPlain {
    const float* vol;
    B200_HD Corner8 operator()(const VolDims& dims, const float pix[3]) const { return gather8(vol, dims, pix); }
};

struct GatherPacked {
    const float4* packed;
    B200_HD Corner8 operator()(const VolDims& dims, const float pix[3]) const
    {
        Corner8 k;
        int i0[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float fl = floorf(pix[a]);
            k.f[a] = pix[a] - fl;
            i0[a] = (int)fl + 1;  // the packed array starts at base index -1
        }
        const int64_t p1 = dims.d[2] + 1, p0 = (int64_t)(dims.d[1] + 1) * p1;
        const float4* cell = packed + 2 * ((int64_t)i0[0] * p0 + (int64_t)i0[1] * p1 + i0[2]);
#if defined(__CUDA_ARCH__)
        const float4 lo = __ldg(cell), hi = __ldg(cell + 1);
#else
        const float4 lo = cell[0], hi = cell[1];
#endif
        k.v[0] = lo.x; k.v[1] = lo.y; k.v[2] = lo.z; k.v[3] = lo.w;
        k.v[4] = hi.x; k.v[5] = hi.y; k.v[6] = hi.z; k.v[7] = hi.w;
        k.base = 0;
        k.mask = 0u;  // no per-corner addresses: the packed path never scatters a volume gradient
        return k;
    }
};

B200_HD bool outside_padded(const float pix[3], const VolDims& dims)
{
    return pix[0] <= -1.0f || pix[1] <= -1.0f || pix[2] <= -1.0f || pix[0] >= (float)dims.d[0] ||
           pix[1] >= (float)dims.d[1] || pix[2] >= (float)dims.d[2];
}

// value of the interpolant; axis 2 is the memory-fastest axis
B200_HD float lerp8(const Corner8& k)
{
    const float f0 = k.f[0], f1 = k.f[1], f2 = k.f[2];
    const float c00 = fmaf(f2, k.v[4] - k.v[0], k.v[0]);  // o0=0 o1=0
    const float c10 = fmaf(f2, k.v[5] - k.v[1], k.v[1]);  // o0=1 o1=0
    const float c01 = fmaf(f2, k.v[6] - k.v[2], k.v[2]);  // o0=0 o1=1
    const float c11 = fmaf(f2, k.v[7] - k.v[3], k.v[3]);  // o0=1 o1=1
    const float c0 = fmaf(f1, c01 - c00, c00);
    const float c1 = fmaf(f1, c11 - c10, c10);
    return fmaf(f0, c1 - c0, c0);
}

// sum (or max) over the samples of tri(V, x_m); multiply by raylen * step outside.
B200_HD float trilinear_ray_fwd(const float* vol, const VolDims& dims, const Ray& ray, float shift, int P, float amin,
                                float amax, int reduce, int align_corners)
{
    const PixLine pl = make_pixline(ray, dims, shift, align_corners);
    const float range = amax - amin;
    const float lstep = 1.0f / (float)(P - 1);
    int m_lo, m_hi;
    sample_range(pl, dims, amin, range, P, m_lo, m_hi);
    float acc = 0.0f;
    bool have = false;
    for (int m = m_lo; m <= m_hi; ++m) {
        const float alpha = add_rn(mul_rn(linspace01(m, P, lstep), range), amin);
        float pix[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) pix[a] = fmaf(alpha, pl.dp[a], pl.p0[a]);
        float val = 0.0f;
        if (!outside_padded(pix, dims)) val = lerp8(gather8(vol, dims, pix));
        if (reduce == 0) acc += val;
        else acc = have ? fmaxf(acc, val) : val;
        have = true;
    }
    // samples skipped by sample_range are exact zeros: they take part in a max
    if (reduce != 0 && (m_lo > 0 || m_hi < P - 1 || !have)) acc = have ? fmaxf(acc, 0.0f) : 0.0f;
    return acc;
}

B200_HD void trilinear_ray_fwd_mask(const float* vol, const float* mask, const VolDims& dims, const Ray& ray, float shift,
                                    int P, float amin, float amax, int align_corners, float scale, float* out_n,
                                    int64_t cstride, int C)
{
    const PixLine pl = make_pixline(ray, dims, shift, align_corners);
    const float range = amax - amin;
    const float lstep = 1.0f / (float)(P - 1);
    int m_lo, m_hi;
    sample_range(pl, dims, amin, range, P, m_lo, m_hi);
    int cur = -1;
    float run = 0.0f;
    for (int m = m_lo; m <= m_hi; ++m) {
        const float alpha = add_rn(mul_rn(linspace01(m, P, lstep), range), amin);
        float pix[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) pix[a] = fmaf(alpha, pl.dp[a], pl.p0[a]);
        if (outside_padded(pix, dims)) continue;
        const float val = lerp8(gather8(vol, dims, pix));
        bool inb = true;
        int64_t flat = 0;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float rr = rintf(pix[a]);
            inb = inb && rr >= 0.0f && rr < (float)dims.d[a];
            flat = flat * dims.d[a] + (inb ? (int64_t)rr : 0);
        }
        const int c = inb ? (int)ldg(mask + flat) : 0;
        if (c != cur) {
            if (run != 0.0f && (unsigned)cur < (unsigned)C) out_n[(int64_t)cur * cstride] += scale * run;
            cur = c;
            run = 0.0f;
        }
        run += val;
    }
    if (run != 0.0f && (unsigned)cur < (unsigned)C) out_n[(int64_t)cur * cstride] += scale * run;
}

// ---- packed-corner volume: packed[(i0+1)][(i1+1)][(i2+1)][8] holds the 8 corner values of the interpolation cell
// whose base voxel is (i0, i1, i2), i in [-1, D-1], zero padding included, corner c = o0 | o1<<1 | o2<<2.  One sample is
// then ONE aligned 32-byte read (two LDG.128) instead of 8 scalar gathers -- exactly the 32 algorithmic bytes/sample.
B200_HD float trilinear_ray_fwd_packed(const float4* packed, const VolDims& dims, const Ray& ray, float shift, int P,
                                       float amin, float amax, float s_lo = -INFINITY, float s_hi = INFINITY)
{
    const PixLine pl = make_pixline(ray, dims, shift, 0);
    const float range = amax - amin;
    const float lstep = 1.0f / (float)(P - 1);
    int m_lo, m_hi;
    sample_range(pl, dims, amin, range, P, m_lo, m_hi);
    sample_range_slab(pl, amin, range, P, s_lo, s_hi, m_lo, m_hi);
    const GatherPacked gather{packed};
    float acc = 0.0f;
    for (int m = m_lo; m <= m_hi; ++m) {
        const float alpha = add_rn(mul_rn(linspace01(m, P, lstep), range), amin);
        float pix[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) pix[a] = fmaf(alpha, pl.dp[a], pl.p0[a]);
        if (outside_padded(pix, dims) || !(pix[0] >= s_lo && pix[0] < s_hi)) continue;
        acc += lerp8(gather(dims, pix));
    }
    return acc;
}

struct TriGrad {
    float gs[3], gt[3];  // d/d source, d/d target  (already scaled by g L step)
    float sumV;          // sum of sampled values
    float ga0, ga1;      // d/d alphamin, d/d alphamax
};

// Closed-form backward of one ray (SURVEY.md 8a-G).  G = gradient of the interpolant w.r.t. pix (zero-padded):
//   g_s = g L step sum (1-alpha_m) G_m ka,  g_t = g L step sum alpha_m G_m ka,  g_L = g step sum V_m,
//   g_amin = g L [-sum V/(P-1) + step sum (1-lin_m) G_m.dp],  g_amax = g L [+sum V/(P-1) + step sum lin_m G_m.dp],
//   g_V[corner] += g L step w_corner.
// Per-sample upstream factor: 1 for the plain renderer; with a label mask (renderers.py:242-252) the gradient of the
// channel the sample was scattered to, label sampled NEAREST at the sample point (zero padding -> label 0).
struct SampleGradOne {
    B200_HD float operator()(const VolDims&, const float*) const { return 1.0f; }
};

struct SampleGradMasked {
    const float* mask;
    const float* gch;  // gout[b][0][n]; channels are cstride floats apart
    int64_t cstride;
    int C;
    B200_HD float operator()(const VolDims& dims, const float pix[3]) const
    {
        bool inb = true;
        int64_t flat = 0;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float rr = rintf(pix[a]);
            inb = inb && rr >= 0.0f && rr < (float)dims.d[a];
            flat = flat * dims.d[a] + (inb ? (int64_t)rr : 0);
        }
        const int c = inb ? (int)ldg(mask + flat) : 0;
        return (unsigned)c < (unsigned)C ? ldg(gch + (int64_t)c * cstride) : 0.0f;
    }
};

template <class Gather, class SampleGrad = SampleGradOne>
B200_HD TriGrad trilinear_ray_bwd_g(const Gather& gather, const VolDims& dims, const Ray& ray, float shift, int P,
                                    float amin, float amax, int align_corners, float g, float L, float* g_vol,
                                    float s_lo = -INFINITY, float s_hi = INFINITY,
                                    const SampleGrad& sample_grad = SampleGrad(), int m_only = -1)
{
    const PixLine pl = make_pixline(ray, dims, shift, align_corners);
    const float range = amax - amin;
    const float step = range / (float)(P - 1);
    const float lstep = 1.0f / (float)(P - 1);
    int m_lo, m_hi;
    sample_range(pl, dims, amin, range, P, m_lo, m_hi);
    sample_range_slab(pl, amin, range, P, s_lo, s_hi, m_lo, m_hi);
    if (m_only != -1) {  // reducefn="max": the gradient of ONE sample (m_only < -1: none at all)
        m_lo = m_lo > m_only ? m_lo : m_only;
        m_hi = m_only < -1 ? m_lo - 1 : (m_hi < m_only ? m_hi : m_only);
    }
    const float gLs = g * L * step;
    float sumV = 0.0f, S[3] = {0.0f, 0.0f, 0.0f}, T[3] = {0.0f, 0.0f, 0.0f}, E0 = 0.0f, E1 = 0.0f;
    for (int m = m_lo; m <= m_hi; ++m) {
        const float lin = linspace01(m, P, lstep);
        const float alpha = add_rn(mul_rn(lin, range), amin);
        float pix[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) pix[a] = fmaf(alpha, pl.dp[a], pl.p0[a]);
        if (outside_padded(pix, dims) || !(pix[0] >= s_lo && pix[0] < s_hi)) continue;
        const Corner8 k = gather(dims, pix);
        const float f0 = k.f[0], f1 = k.f[1], f2 = k.f[2];
        const float e0 = 1.0f - f0, e1 = 1.0f - f1, e2 = 1.0f - f2;
        const float c00 = fmaf(f2, k.v[4] - k.v[0], k.v[0]), c10 = fmaf(f2, k.v[5] - k.v[1], k.v[1]);
        const float c01 = fmaf(f2, k.v[6] - k.v[2], k.v[2]), c11 = fmaf(f2, k.v[7] - k.v[3], k.v[3]);
        const float c0 = fmaf(f1, c01 - c00, c00), c1 = fmaf(f1, c11 - c10, c10);
        const float gm = sample_grad(dims, pix);  // == 1.0f exactly for the plain renderer (products below are exact)
        sumV += gm * fmaf(f0, c1 - c0, c0);
        float G[3];
        G[0] = gm * (c1 - c0);
        G[1] = gm * (e0 * (c01 - c00) + f0 * (c11 - c10));
        G[2] = gm * (e0 * (e1 * (k.v[4] - k.v[0]) + f1 * (k.v[6] - k.v[2])) +
                     f0 * (e1 * (k.v[5] - k.v[1]) + f1 * (k.v[7] - k.v[3])));
        float Gd = 0.0f;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            S[a] = fmaf(1.0f - alpha, G[a], S[a]);
            T[a] = fmaf(alpha, G[a], T[a]);
            Gd = fmaf(G[a], pl.dp[a], Gd);
        }
        E0 = fmaf(1.0f - lin, Gd, E0);
        E1 = fmaf(lin, Gd, E1);
        if (g_vol) {
#pragma unroll
            for (int c = 0; c < 8; ++c)
                if (k.mask & (1u << c)) {
                    const float w = ((c & 1) ? f0 : e0) * (((c >> 1) & 1) ? f1 : e1) * (((c >> 2) & 1) ? f2 : e2);
                    red_add(g_vol + k.base + corner_off(dims, c), (gLs * gm) * w);
                }
        }
    }
    TriGrad out;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        out.gs[a] = gLs * pl.ka[a] * S[a];
        out.gt[a] = gLs * pl.ka[a] * T[a];
    }
    out.sumV = sumV;
    const float gLv = g * L * sumV / (float)(P - 1);
    out.ga0 = -gLv + gLs * E0;
    out.ga1 = gLv + gLs * E1;
    return out;
}

B200_HD TriGrad trilinear_ray_bwd(const float* vol, const VolDims& dims, const Ray& ray, float shift, int P, float amin,
                                  float amax, int align_corners, float g, float L, float* g_vol)
{
    return trilinear_ray_bwd_g(GatherPlain{vol}, dims, ray, shift, P, amin, amax, align_corners, g, L, g_vol);
}

// reducefn="max" (renderers.py:175-183 on Trilinear.forward): I = max_m (L V_m) step; the gradient flows through the
// FIRST maximal sample only (torch.max).  Samples skipped by sample_range are exact zeros and take part in the max: if
// one of them is the (first) maximum nothing has a gradient.  L, step > 0, so the order of the terms is that of V_m.
B200_HD TriGrad trilinear_ray_bwd_max(const float* vol, const VolDims& dims, const Ray& ray, float shift, int P, float amin,
                                      float amax, int align_corners, float g, float L, float* g_vol)
{
    const PixLine pl = make_pixline(ray, dims, shift, align_corners);
    const float range = amax - amin;
    const float lstep = 1.0f / (float)(P - 1);
    int m_lo, m_hi;
    sample_range(pl, dims, amin, range, P, m_lo, m_hi);
    int mbest = -2;  // -2: a skipped (zero, gradient-free) sample holds the maximum
    float best = 0.0f;
    bool have = m_lo > 0;  // samples before m_lo are zeros and come first
    for (int m = m_lo; m <= m_hi; ++m) {
        const float alpha = add_rn(mul_rn(linspace01(m, P, lstep), range), amin);
        float pix[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) pix[a] = fmaf(alpha, pl.dp[a], pl.p0[a]);
        float val = 0.0f;
        if (!outside_padded(pix, dims)) val = lerp8(gather8(vol, dims, pix));
        if (!have || val > best) {
            best = val;
            mbest = m;
        }
        have = true;
    }
    if (have && m_hi < P - 1 && best < 0.0f) mbest = -2;  // a trailing zero beats an all-negative march
    if (!have) mbest = -2;
    return trilinear_ray_bwd_g(GatherPlain{vol}, dims, ray, shift, P, amin, amax, align_corners, g, L, g_vol, -INFINITY,
                               INFINITY, SampleGradOne(), mbest);
}

B200_HD TriGrad trilinear_ray_bwd_packed(const float4* packed, const VolDims& dims, const Ray& ray, float shift, int P,
                                         float amin, float amax, float g, float L, float s_lo = -INFINITY,
                                         float s_hi = INFINITY)
{
    return trilinear_ray_bwd_g(GatherPacked{packed}, dims, ray, shift, P, amin, amax, 0, g, L, nullptr, s_lo, s_hi);
}

// ===================================================================================================
// Siddon with mode="bilinear" (reference renderers.py:18,66): the density of a segment is the TRILINEAR interpolant T at the
// segment midpoint instead of the nearest voxel; everything else is the general plane-by-plane walk above.  Slow path.
//   I = L sum_j len_j T(x_j)                    (reduce "max": max_j instead of sum_j, forward only)
// GRAD (reduce "sum"): closed-form backward, pinned to the reference's autograd through the oracle:
//   dI/dalpha_m = L [ (T_{m-1} - T_m) + (len_{m-1} G_{m-1}.d + len_m G_m.d)/2 ],  G = grad T w.r.t. x
//   dI/ds += L sum_j len_j (1 - abar_j) G_j,  dI/dt += L sum_j len_j abar_j G_j,  dI/dL = sum_j len_j T_j,
//   dI/dV[corner] += L len_j w_corner.   stop_grad (stop_gradients_through_grid_sample): T is a constant, only the
//   (T_{m-1} - T_m) terms remain.  gs/gt come back already multiplied by g; returns the image value; sum_tl = sum len T.
// ===================================================================================================
template <bool GRAD>
B200_HD float siddon_ray_bilinear(const float* vol, const VolDims& dims, const Ray& ray, float L, float shift, int reduce,
                                  int align_corners, float g, bool stop_grad, float* g_vol, float gs[3], float gt[3],
                                  float& sum_tl)
{
    int pos[3], stp[3], left[3];
    float head[3], ka[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const bool fwd = ray.d[a] > 0.0f;
        pos[a] = fwd ? 0 : dims.d[a];
        stp[a] = fwd ? 1 : -1;
        left[a] = dims.d[a] + 1;
        head[a] = plane_alpha(ray, a, (float)pos[a], shift);
        ka[a] = align_corners ? (float)(dims.d[a] - 1) / (float)dims.d[a] : 1.0f;
    }
    const int M = dims.d[0] + dims.d[1] + dims.d[2] + 3;
    const float gL = g * L;
    float acc = 0.0f, aprev = 0.0f;
    bool first = true;
    float A[3] = {0.0f, 0.0f, 0.0f}, C[3] = {0.0f, 0.0f, 0.0f}, S[3] = {0.0f, 0.0f, 0.0f}, Tt[3] = {0.0f, 0.0f, 0.0f};
    float Tprev = 0.0f, hprev = 0.0f;  // value and len*G.d/2 of the segment before the previous crossing
    int axprev = 0;
    sum_tl = 0.0f;
    for (int m = 0; m < M; ++m) {
        const float h0 = left[0] > 0 ? head[0] : INFINITY;
        const float h1 = left[1] > 0 ? head[1] : INFINITY;
        const float h2 = left[2] > 0 ? head[2] : INFINITY;
        const float acur = fminf(fminf(h0, h1), h2);
        const int best = (left[0] > 0 && h0 == acur) ? 0 : ((left[1] > 0 && h1 == acur) ? 1 : 2);
#pragma unroll
        for (int a = 0; a < 3; ++a)
            if (a == best) {
                pos[a] += stp[a];
                left[a] -= 1;
                if (left[a] > 0) head[a] = plane_alpha(ray, a, (float)pos[a], shift);
            }
        if (m > 0) {
            const float amid = (aprev + acur) / 2.0f, len = acur - aprev;
            float pix[3];
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const float x = add_rn(ray.s[a], mul_rn(amid, ray.d[a]));
                pix[a] = unnormalize(2.0f * (x + shift) / (float)dims.d[a] - 1.0f, dims.d[a], align_corners);
            }
            float T = 0.0f, half = 0.0f;
            if (!outside_padded(pix, dims)) {
                const Corner8 k = gather8(vol, dims, pix);
                const float f0 = k.f[0], f1 = k.f[1], f2 = k.f[2];
                const float e0 = 1.0f - f0, e1 = 1.0f - f1, e2 = 1.0f - f2;
                const float c00 = fmaf(f2, k.v[4] - k.v[0], k.v[0]), c10 = fmaf(f2, k.v[5] - k.v[1], k.v[1]);
                const float c01 = fmaf(f2, k.v[6] - k.v[2], k.v[2]), c11 = fmaf(f2, k.v[7] - k.v[3], k.v[3]);
                const float c0 = fmaf(f1, c01 - c00, c00), c1 = fmaf(f1, c11 - c10, c10);
                T = fmaf(f0, c1 - c0, c0);
                if (GRAD && !stop_grad) {
                    float G[3];
                    G[0] = (c1 - c0) * ka[0];
                    G[1] = (e0 * (c01 - c00) + f0 * (c11 - c10)) * ka[1];
                    G[2] = (e0 * (e1 * (k.v[4] - k.v[0]) + f1 * (k.v[6] - k.v[2])) +
                            f0 * (e1 * (k.v[5] - k.v[1]) + f1 * (k.v[7] - k.v[3]))) * ka[2];
                    float Gd = 0.0f;
#pragma unroll
                    for (int a = 0; a < 3; ++a) {
                        S[a] = fmaf(len * (1.0f - amid), G[a], S[a]);
                        Tt[a] = fmaf(len * amid, G[a], Tt[a]);
                        Gd = fmaf(G[a], ray.d[a], Gd);
                    }
                    half = 0.5f * len * Gd;
                    if (g_vol) {
#pragma unroll
                        for (int c = 0; c < 8; ++c)
                            if (k.mask & (1u << c)) {
                                const float w = ((c & 1) ? f0 : e0) * (((c >> 1) & 1) ? f1 : e1) * (((c >> 2) & 1) ? f2 : e2);
                                red_add(g_vol + k.base + corner_off(dims, c), gL * len * w);
                            }
                    }
                }
            }
            const float term = mul_rn(mul_rn(L, T), len);
            if (reduce == 0) acc = add_rn(acc, term);
            else if (first || term > acc) acc = term;
            first = false;
            if (GRAD) {
                sum_tl = fmaf(T, len, sum_tl);
                const float coef = (Tprev - T) + (hprev + half);  // crossing m-1 (axis axprev, alpha aprev)
#pragma unroll
                for (int a = 0; a < 3; ++a)
                    if (a == axprev) {
                        A[a] = fmaf(coef, aprev, A[a]);
                        C[a] += coef;
                    }
                Tprev = T;
                hprev = half;
            }
        }
        aprev = acur;
        axprev = best;
    }
    if (GRAD) {
        const float coef = Tprev + hprev;  // last crossing: T_last -> 0
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            if (a == axprev) {
                A[a] = fmaf(coef, aprev, A[a]);
                C[a] += coef;
            }
            gt[a] = gL * (Tt[a] - A[a] * ray.inv[a]);
            gs[a] = gL * (S[a] + (A[a] - C[a]) * ray.inv[a]);
        }
    }
    return acc;
}

}  // namespace b200drr
