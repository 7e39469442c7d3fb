// ort_beam.cuh -- conservative beam start for camera frames (round 2): skip the part of every ray's walk that runs
// through space the whole 8 x 4 pixel tile provably sees as empty, without changing a single output bit.
//
// Where the rounds go.  On the bench frames (depth 12, 4K) 60 % of the rays leave the cube without a hit and the others
// spend 35-58 % of their PUSH rounds in levels 1-3: the walk from the camera through the coarse empty cells above the
// terrain.  Those rounds are the same for all rays of a tile, but SIMT already issues them once per warp -- only not
// running them saves anything (tools/beam/beam_model.py: 19.7 / 30.3 / 37.6 rounds per ray -> 6.7 / 17.0 / 21.8).
//
// Three pieces.
//
// (1) Re-entry (LeanWalker::start_at).  For a ray of the lean tier (no degenerate axis, no negative t, finite bias) let
//     e_1 <= e_2 <= ... be the exit times the reference computes in its STEPs at the empty slots S_1, S_2, ... it visits
//     (och_h_octree.h:378-406).  t_a(X) = fma(X, coef_a, bias_a) is a non-increasing function of the plane coordinate X
//     (rounding is monotone), and every exit plane of the cell entered after a STEP has t >= the STEP's tmin, so the e_i
//     never decrease.  Take any tau > 0 that is not later than the ray's hit time (its cube exit time for a MISS) and let i
//     be the first index with e_i >= tau.  Descending from the root with the reference's own child test `t_mid >= tmin`
//     (:363-373) at tmin = tau reaches exactly S_i, through the same nodes:
//       - where the reference's cell is the upper half on axis a (mid plane m not crossed): t_a(m) >= t_a(exit plane of
//         S_i on a) >= e_i >= tau, so the test picks the upper half;
//       - where it is the lower half, the reference either failed the test at some earlier tmin (t_a(m) < e_q <= e_{i-1}
//         < tau, or t_a(m) < 0 during the first descents), or stepped across m at e_q = t_a(m) <= e_{i-1} < tau, or the
//         half was picked from the origin's bits at level 1 (:320-324: m = 1.5 lies behind the origin, t_a(m) <= 0 < tau):
//         the test picks the lower half.
//     So the slot word, the position, the cell size and every parent-stack entry (the slot word of each ancestor) are
//     the reference's; the STEP that follows overwrites tmin and min_t_idx before anything reads them, and from there on
//     the two walks are the same instruction stream.  tau beyond the cube exit time means the ray ends as a MISS without
//     a round.  A re-entry that reaches a voxel without a single STEP can only mean tau was later than the hit time:
//     the kernel then walks the ray again from the start (a guard; the bound below rules it out).
//
// (2) The bound (beam_march).  The reference does not trace the ray (o, d) but, up to 2^-22 in space, the straight ray
//     (o, d') with d'_a = 1 / |coef_a|: RCPPS is a 12-bit reciprocal (relative error eps_r, measured from the table).  At
//     its hit time the point o + t_hit d' lies within 2^-22 of the hit voxel (every entry plane of the voxel has t <=
//     t_hit, every exit plane t >= t_hit).  Let R bound |d' - d_c| over the rays of a tile, d_c the direction through the
//     tile's centre: R = (half diagonal of the tile in the image plane) / fov + eps_r + rounding.  A level-k grid cell has
//     size s = 2^-k; take the largest k with t_max R + slack <= 0.7 s (t_max = the distance from the origin to the farthest
//     corner of the cube, widened by eps_r: no ray stays longer in it).  Then, at equal parameter t, every ray of the
//     tile is in one of the 27 cells around the cell of the central ray.  `skip` holds, for every level-k cell, 0 if any of its 27 neighbours contains a non-empty level-k cell
//     of the DAG ("dilated-occupied"), else the coarsest level j <= k whose cell around it is dilated-empty throughout.
//     Marching the central ray through that grid (one load per step, the steps as large as the empty cells) gives the
//     first parameter tau_c at which it is inside a dilated-occupied cell: no ray of the tile can hit anything before
//     tau_c.  The march samples 2^-19 past every exit plane instead of tracking cell indices, and lets the ray drift up to
//     a 16th of a cell into a neighbour it runs along; the cells it can miss that way are clipped by less than the slack
//     (0.3 s).  tau = tau_c (1 - 2^-12) - 2^-17.
//
//     The condition on t_max is stronger than the argument needs: it uses the bound only at the times t < tau_c, and
//     there every ray of the tile stays within R t <= R tau_c of the central ray.  t_max was only ever an upper bound of
//     tau_c.  So a tile may march on from its level-k stop t_k on the finer level-8 grid (beam_tile_start, refinement) and
//     stop at t_8: for t < t_k the level-k march answers as before (R t <= R t_max fits level k), for t_k <= t < t_8 every
//     ray is within R t_8 of the central ray, inside one of the 27 level-8 cells around the central ray's cell, as long as
//     R t_8 + slack <= 0.7 2^-8.  That is checked per tile at t_8, where the march stops (the beam only widens with t), as
//     t_8 <= t_fine = (0.7 2^-8 - slack) / R, rounded down on the host.  A tile that fails it keeps t_k.  A march that
//     leaves the cube stops at the sample that is more than a level-8 cell outside, and the same check at that time lets
//     its tile see nothing (+inf, item 3 with level-8 cells).
//
// (3) Tiles that see nothing.  When the central ray has left the cube by more than a cell without meeting a marked cell,
//     every ray of the tile has left it too: tau = +inf.  If all rays of the tile are certain to be lean-tier rays
//     (beam_tile_start), the trace kernel writes 32 MISSes and is done -- no camera ray, no reciprocals.
//
// What this buys is measured in profiles/ (r2_final_beam_ncu_full.md, r2_bench_n1.json) and argued in DESIGN.md 4b; what it
// costs is one byte grid per DAG version and level in use (built lazily: occupancy, dilation, k - 1 pyramid levels, skip
// levels; 8^k bytes; the level-8 grid of the refinement is built with the launch's level) and one march per tile (a
// separate launch, one thread per tile).
// Tested claim by claim: tests/test_beam.py (this header compiled for the host) and tests/test_gpu_beam.py; the level-8
// refinement in tests/test_beam_refine.py and tests/test_gpu_beam_refine.py.
#pragma once

#include <cmath>

#include "ort_trace.cuh"

namespace ort {

constexpr int kBeamMinLevel = 3;      // below this the grid says nothing (8 cells per axis)
constexpr int kBeamMaxLevel = 7;      // 128^3 bytes = 2 MiB: the finest level a whole launch is bounded with
constexpr int kBeamFineLevel = 8;     // 256^3 bytes = 16 MiB: the grid tiles refine their start on (item 2)
constexpr int kBeamMaxSteps = 64;       // a march that needs more ends early: its tile starts where the march stood

struct BeamGrid
{
	const uint8_t* skip;   // (2^k)^3 bytes, index (z * N + y) * N + x, world axes
	int k;
};

// Level for a launch: the largest k in [kBeamMinLevel, min(depth, kBeamMaxLevel)] whose cells are wider than the tile's
// beam wherever a ray of this origin can be inside the cube, or 0.  tile_radius = R above, t_max = the longest stay of a
// ray in the cube (host side, double precision).
inline int beam_level_for(double tile_radius, int depth, double t_max = 1.75)
{
	const int hi = depth < kBeamMaxLevel ? depth : kBeamMaxLevel;
	for (int k = hi; k >= kBeamMinLevel; --k)
		if (t_max * tile_radius + 3e-5 <= 0.7 / static_cast<double>(1 << k))
			return k;
	return 0;
}

// Refinement of a launch at level k (host side): t_fine, the latest stop time of the level-8 march at which a tile's beam
// still fits a level-8 cell, rounded down to a float; 0 = no refinement.  Only launches at level kBeamMaxLevel get it: a
// coarser launch level means R t_max > 0.7 2^-7, so the level-8 bound would hold over less than about half of the
// longest stay in the cube, too little to pay for the 16 MiB grid.
inline float beam_fine_t_limit(double tile_radius, int depth, int k)
{
	if (k != kBeamMaxLevel || depth < kBeamFineLevel || !(tile_radius > 0.0)) return 0.0f;
	const double cell = 1.0 / static_cast<double>(1 << kBeamFineLevel), t = (0.7 * cell - 3e-5) / tile_radius;
	if (!(t >= cell)) return 0.0f;
	float f = static_cast<float>(t);
	if (static_cast<double>(f) > t) f = std::nextafter(f, 0.0f);
	return f;
}

// Longest stay in the cube [1,2]^3 of a ray from (ox, oy, oz) inside it: the distance to the farthest corner, widened
// for the reference's clock (t = length / |d'|, |d'| within eps_r of 1).
inline double beam_t_max(double ox, double oy, double oz, double rcp_eps)
{
	const double fx = ox - 1.0 > 2.0 - ox ? ox - 1.0 : 2.0 - ox, fy = oy - 1.0 > 2.0 - oy ? oy - 1.0 : 2.0 - oy, fz = oz - 1.0 > 2.0 - oz ? oz - 1.0 : 2.0 - oz;
	return std::sqrt(fx * fx + fy * fy + fz * fz) * (1.0 + 2.0 * rcp_eps + 1e-5) + 1e-5;
}

// R for the 8 x 4 pixel tiles of a camera frame.  The rays are M (u, v, fov)^T normalised (camera_ray), M the caller's
// rotation: with M orthonormal to 1e-3 two rays differ by at most 1.01 |(du, dv)| / fov.  Returns a negative number
// when the camera gives no bound (fov <= 0, M not a rotation).
inline double beam_tile_radius(const Camera& c, double rcp_eps)
{
	if (!(c.fov > 0.0f)) return -1.0;
	for (int i = 0; i < 3; ++i)
		for (int j = 0; j < 3; ++j)
		{
			double dot = 0;                                   // columns i, j of M
			for (int r = 0; r < 3; ++r) dot += static_cast<double>(c.r[3 * r + i]) * c.r[3 * r + j];
			const double dev = dot - (i == j ? 1.0 : 0.0);
			if (!(dev < 1e-3 && dev > -1e-3)) return -1.0;
		}
	const double du = 3.5 * static_cast<double>(c.aspect) * c.vfx, dv = 1.5 * static_cast<double>(c.vfy);   // tile centre to the farthest pixel centre: 3.5 x 1.5 pixels
	return 1.01 * std::sqrt(du * du + dv * dv) / c.fov + rcp_eps + 1e-6;
}

// Largest relative error of a reciprocal table over its bins: entry i serves the mantissas [i, i + 1) / n of [1, 2).
inline double rcp_table_rel_error(const uint32_t* tab, int log2n)
{
	const size_t n = static_cast<size_t>(1) << log2n;
	double worst = 0;
	for (size_t i = 0; i < n; ++i)
	{
		uint32_t b = tab[i];
		float r;
#ifdef ORT_HOST_EMU
		r = __uint_as_float(b);
#else
		memcpy(&r, &b, 4);
#endif
		const double lo = 1.0 + static_cast<double>(i) / n, hi = 1.0 + static_cast<double>(i + 1) / n;
		const double e0 = r * lo - 1.0, e1 = r * hi - 1.0;
		const double e = (e0 < 0 ? -e0 : e0) > (e1 < 0 ? -e1 : e1) ? (e0 < 0 ? -e0 : e0) : (e1 < 0 ? -e1 : e1);
		if (e > worst) worst = e;
	}
	return worst;
}

// March of the ray o + t d (|d| = 1, o inside the cube) from t on (0: from the origin) to the first parameter at which it
// is inside a dilated-occupied cell of the grid.  Returns that parameter, or with `left` set the time of the first sample
// that lies more than a cell outside the cube with nothing met before; 0 when the march cannot start (NaN, the origin
// outside); a time later than t_end as soon as it is clear that the march stops after t_end (the caller only wants to
// know whether it stops by then).  Outside the cube the grid continues as one ring of virtual cells that inherit the flag
// of the boundary cell next to them (the inside cells around a virtual cell are among the 27 around that boundary cell):
// the tile's other rays may still be inside while the central ray is up to one cell out, and not once it is further.
__device__ __forceinline__ float beam_march(const BeamGrid g, float ox, float oy, float oz, float dx, float dy, float dz, float t, float t_end, bool& left, int* steps)
{
	const int N = 1 << g.k;
	const float fN = static_cast<float>(N), cell = 1.0f / fN;
	const float inf = __uint_as_float(0x7F800000u);
	const float ix_ = dx != 0.0f ? __fdiv_rn(1.0f, dx) : inf, iy_ = dy != 0.0f ? __fdiv_rn(1.0f, dy) : inf, iz_ = dz != 0.0f ? __fdiv_rn(1.0f, dz) : inf;
	const float delta = 0x1p-19f;
	left = false;
	for (int it = 0; it < kBeamMaxSteps; ++it)
	{
		const float ts = t > 0.0f ? __fadd_rn(t, delta) : 0.0f;
		const float qx = __fmul_rn(__fsub_rn(__fmaf_rn(ts, dx, ox), 1.0f), fN), qy = __fmul_rn(__fsub_rn(__fmaf_rn(ts, dy, oy), 1.0f), fN),
		            qz = __fmul_rn(__fsub_rn(__fmaf_rn(ts, dz, oz), 1.0f), fN);                      // position in cells
		const float lim = __fadd_rn(fN, 1.0f);
		if (!(qx >= -1.0f && qx < lim && qy >= -1.0f && qy < lim && qz >= -1.0f && qz < lim))
		{
			left = t > 0.0f;                               // more than a cell outside (at the origin: NaN, no beam start)
			return left ? ts : 0.0f;
		}
		const int cx = static_cast<int>(floorf(qx)), cy = static_cast<int>(floorf(qy)), cz = static_cast<int>(floorf(qz));      // -1 .. N
		const int bx = min(max(cx, 0), N - 1), by = min(max(cy, 0), N - 1), bz = min(max(cz, 0), N - 1);
		const int s = g.skip[(static_cast<size_t>(bz) * N + by) * N + bx];
		if (steps) ++*steps;
		if (s == 0)
			break;
		// leave the level-s cell around the sample point (a virtual cell: that cell alone) through its nearest exit plane
		const int sh = (cx == bx && cy == by && cz == bz) ? g.k - s : 0;
		const int keep = ~((1 << sh) - 1);                 // (a mask, not shifts: virtual cells have index -1)
		const float lx = __fmaf_rn(static_cast<float>(cx & keep), cell, 1.0f), ly = __fmaf_rn(static_cast<float>(cy & keep), cell, 1.0f),
		            lz = __fmaf_rn(static_cast<float>(cz & keep), cell, 1.0f);
		const float w = static_cast<float>(1 << sh) * cell;
		// Exit times of the three axes.  One that is not in the future (<= t) belongs to a plane the sample point sits on within
		// rounding: the ray runs along it (or has just crossed it and the next sample will say so).  It is no exit; but while
		// the ray may be drifting into the cell beyond that plane the step is kept so short that the drift stays below a 16th
		// of a cell -- part of the slack of the bound, like the 2^-19 the samples are set past every plane.
		const float ex = dx != 0.0f ? __fmul_rn(__fsub_rn(dx > 0.0f ? __fadd_rn(lx, w) : lx, ox), ix_) : inf;
		const float ey = dy != 0.0f ? __fmul_rn(__fsub_rn(dy > 0.0f ? __fadd_rn(ly, w) : ly, oy), iy_) : inf;
		const float ez = dz != 0.0f ? __fmul_rn(__fsub_rn(dz > 0.0f ? __fadd_rn(lz, w) : lz, oz), iz_) : inf;
		const float drift = cell * 0.0625f;
		float te = inf;
		te = fminf(te, ex > t ? ex : __fmaf_rn(drift, fabsf(ix_), t));
		te = fminf(te, ey > t ? ey : __fmaf_rn(drift, fabsf(iy_), t));
		te = fminf(te, ez > t ? ez : __fmaf_rn(drift, fabsf(iz_), t));
		t = te > t ? te : __fadd_rn(t, delta);             // always forward
		if (t > t_end) break;
	}
	// inside a dilated-occupied cell from t on (or out of steps): nothing before t
	return t;
}

// A tile whose march ends with +inf has nothing in sight; if, on top of that, every ray of the tile is certain to be in
// the lean tier, the trace kernel can end the whole tile as MISSes without setting up a single ray (kBeamAllMiss).
// Certain means: the origin lies off the finest grid on all three axes (Ray::t0or stays 0; the host knows) and no
// direction component of any ray of the tile can be zero or denormal -- every component of the central direction is at
// least min_comp = 1.5 R + 1e-4 away from zero, R the tile radius.  Tiles that see nothing but cannot be certified get
// kBeamNoneInSight: later than any cube exit time, so their lean-tier rays still end as a MISS one by one.
constexpr uint32_t kBeamAllMissBits = 0x7F800000u;        // +inf
constexpr float kBeamNoneInSight = 3.0e38f;

// start time of the 8 x 4 pixel tile whose first pixel is (x0, y0) of the frame: the ray through the tile's centre, marched
// on the launch's grid g and then, if the stop time is not later than fine_t (> 0: refinement on), on the level-8 grid
// `fine` -- kept where that march also stops by fine_t.  min_comp <= 0: never certify.  steps: grid lookups (statistics).
__device__ __forceinline__ float beam_tile_start(const BeamGrid g, const Camera& c, int x0, int y0, float min_comp = 0.0f, int* steps = nullptr,
                                                 const BeamGrid fine = BeamGrid{ nullptr, 0 }, float fine_t = 0.0f)
{
	const float xc = static_cast<float>(x0) + 3.5f, yc = static_cast<float>(y0) + 1.5f;
	const float u = __fmul_rn(c.aspect, __fsub_rn(__fmul_rn(c.vfx, xc), 1.0f));
	const float v = __fsub_rn(__fmul_rn(c.vfy, yc), 1.0f);
	const float ru = __fadd_rn(__fadd_rn(__fmul_rn(u, c.r[0]), __fmul_rn(v, c.r[1])), __fmul_rn(c.fov, c.r[2]));
	const float rv = __fadd_rn(__fadd_rn(__fmul_rn(u, c.r[3]), __fmul_rn(v, c.r[4])), __fmul_rn(c.fov, c.r[5]));
	const float rw = __fadd_rn(__fadd_rn(__fmul_rn(u, c.r[6]), __fmul_rn(v, c.r[7])), __fmul_rn(c.fov, c.r[8]));
	const float s = __fadd_rn(__fadd_rn(__fmul_rn(ru, ru), __fmul_rn(rv, rv)), __fmul_rn(rw, rw));
	const float rm = __fdiv_rn(1.0f, __fsqrt_rn(s));
	const float dx = __fmul_rn(rw, rm), dy = __fmul_rn(ru, rm), dz = __fmul_rn(-rv, rm);
	bool left;
	float t = beam_march(g, c.ox, c.oy, c.oz, dx, dy, dz, 0.0f, __uint_as_float(0x7F800000u), left, steps);
	if (!left && fine_t > 0.0f && t <= fine_t)
	{
		bool left_fine;
		const float tf = beam_march(fine, c.ox, c.oy, c.oz, dx, dy, dz, t, fine_t, left_fine, steps);
		if (tf <= fine_t)
		{
			t = tf;
			left = left_fine;
		}
	}
	if (!left)
	{
		const float tau = __fsub_rn(__fmul_rn(t, 1.0f - 0x1p-12f), 0x1p-17f);
		return tau > 0.0f ? tau : 0.0f;
	}
	const bool certain = min_comp > 0.0f && fminf(fabsf(dx), fminf(fabsf(dy), fabsf(dz))) >= min_comp;
	return certain ? __uint_as_float(kBeamAllMissBits) : kBeamNoneInSight;
}

// significant bits of a float's mantissa (1 for a power of two, 24 at most)
inline int float_sig_bits(float f)
{
	uint32_t b;
#ifdef ORT_HOST_EMU
	b = __float_as_uint(f);
#else
	memcpy(&b, &f, 4);
#endif
	uint32_t m = (b & 0x7FFFFFu) | 0x800000u;
	int tz = 0;
	while (!(m & 1u)) { m >>= 1; ++tz; }
	return 24 - tz;
}

// largest number of significant bits among the entries of a reciprocal table (Intel's RCPPS: 12)
inline int rcp_table_sig_bits(const uint32_t* tab, int log2n)
{
	int worst = 1;
	for (size_t i = 0; i < (static_cast<size_t>(1) << log2n); ++i)
	{
		uint32_t m = (tab[i] & 0x7FFFFFu) | 0x800000u;
		int tz = 0;
		while (!(m & 1u)) { m >>= 1; ++tz; }
		if (24 - tz > worst) worst = 24 - tz;
	}
	return worst;
}

// min_comp for a camera (host side), 0 = never certify.  An origin coordinate on the finest grid puts a cell plane through
// the origin; its t is the rounding residue of bias = -(coef * o) and a negative one sends the ray to another tier
// (Ray::t0or).  That cannot happen when the product is exact: coef has at most rcp_sig_bits significant bits (a property
// of the table), the mirrored coordinate (o or 3 - o) a few, and a product of at most 24 bits is not rounded -- the residue
// is +0 for every ray.  Otherwise the tier depends on the ray and the tile cannot be certified.
inline float beam_certify_min_comp(const Camera& c, double tile_radius, int rcp_sig_bits)
{
	const float o[3] = { c.ox, c.oy, c.oz };
	for (int a = 0; a < 3; ++a)
		if (c.origin_flags & (1u << a))
		{
			const int so = float_sig_bits(o[a]), sm = float_sig_bits(3.0f - o[a]);      // 3 - o is exact for o in [1, 2)
			if ((so > sm ? so : sm) + rcp_sig_bits > 24) return 0.0f;
		}
	return static_cast<float>(1.5 * tile_radius + 1e-4);
}

// The lean tier with a beam start: `tau` as beam_tile_start() gave it for the ray's tile (0: none).  Returns true when
// the result is already known (a MISS: the tile sees nothing before the ray has left the cube); otherwise the walker
// stands at the re-entry state (or at the ordinary start).  beam_used tells the caller to check the guard afterwards.
template<bool COUNT>
__device__ __forceinline__ bool lean_start(LeanWalker<COUNT>& w, uint32_t root, const Ray& r, float tau, float miss_t, bool& beam_used)
{
	beam_used = false;
	if (tau > 0.0f && fmaxf(r.bx, fmaxf(r.by, r.bz)) < __uint_as_float(0x7F800000u))
	{
		w.start_at(root, r, tau);
		if (tau > w.cube_exit_time())
		{
			w.hit.voxel = 0;
			w.hit.face = 6;
			w.hit.t = miss_t;
			return true;
		}
		beam_used = true;
		return false;
	}
	w.start(root, r);
	return false;
}

}  // namespace ort
