// beam_model.c -- offline model (CPU, statistics only) of a conservative "beam start" for the trace:
// how many PUSH rounds of the reference walk happen before a tile-wide conservative start time t0, and at which
// level the walk is at that moment (the cost of re-entering the walk there).  Plain float arithmetic with exact
// reciprocals: this is a counting model, not the bit-exact path (that is csrc/ort_trace.cuh).
#include <math.h>
#include <stdint.h>
#include <string.h>
#include <stddef.h>

static inline uint32_t f2u(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
static inline float u2f(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }

// nodes8: node id i (1-based) at nodes8[8*(i-1)..]; slot bit a set = upper half in world coordinates on axis a
void beam_walk(const uint32_t* nodes8, uint32_t root, int depth, const float* o, const float* d, const float* t0, size_t n,
               int32_t* rounds, int32_t* at_round, int32_t* at_level, float* t_hit)
{
	for (size_t r = 0; r < n; ++r)
	{
		float coef[3], bias[3];
		uint32_t pos[3], inv = 0, idx = 0;
		for (int a = 0; a < 3; ++a)
		{
			const float da = d[3 * r + a];
			const int sg = 0.0f < da;
			inv |= (uint32_t)sg << a;
			const float oa = fabsf((sg ? 3.0f : 0.0f) - o[a]);
			coef[a] = -1.0f / fabsf(da);
			bias[a] = -(coef[a] * oa);
			pos[a] = f2u(oa) & 0x3FC00000u;
			idx |= (uint32_t)(pos[a] == 0x3FC00000u) << a;
		}
		uint32_t node = root, dim = 1u << 22, stack[24];
		int level = 1, np = 0, found = 0;
		float tmin = 0.0f;
		rounds[r] = 0; at_round[r] = -1; at_level[r] = -1; t_hit[r] = INFINITY;
		for (;;)
		{
			++np;
			const uint32_t child = nodes8[8 * (size_t)(node - 1) + ((idx ^ inv) & 7u)];
			if (child)
			{
				if (level == depth) { t_hit[r] = tmin; break; }
				stack[level - 1] = node;
				++level; node = child; dim >>= 1;
				idx = 0;
				for (int a = 0; a < 3; ++a)
				{
					const float t = fmaf(u2f(pos[a] | dim), coef[a], bias[a]);
					if (t >= tmin) { idx |= 1u << a; pos[a] |= dim; }
				}
				continue;
			}
			int miss = 0;
			for (;;)
			{
				float t[3];
				for (int a = 0; a < 3; ++a) t[a] = fmaf(u2f(pos[a]), coef[a], bias[a]);
				const float tm = fminf(t[0], fminf(t[1], t[2]));
				const uint32_t mti = t[0] == tm ? 1u : (t[1] == tm ? 2u : 4u);
				tmin = tm;
				if (!found && tm >= t0[r]) { found = 1; at_round[r] = np - 1; at_level[r] = level; }
				if (idx & mti)
				{
					for (int a = 0; a < 3; ++a) if (mti >> a & 1u) pos[a] &= ~dim;
					idx ^= mti;
					break;
				}
				if (--level == 0) { miss = 1; break; }
				node = stack[level - 1];
				for (int a = 0; a < 3; ++a) pos[a] &= ~dim;
				dim <<= 1;
				idx = 0;
				for (int a = 0; a < 3; ++a) idx |= (uint32_t)((pos[a] & dim) != 0u) << a;
			}
			if (miss) break;
		}
		rounds[r] = np;
	}
}

// Entry parameter of the first occupied cell of a (dilated) level-k bitmap along the ray o + t * d (world coordinates,
// cube [1,2)^3) from t0[r] on (NULL: from 0), plain 3-D DDA in double precision; +inf when the ray leaves the cube first,
// and then t_exit[r] (if not NULL) = the parameter at which it leaves.  occ: (2^k)^3 bytes, index (z * N + y) * N + x.
void beam_dda(const uint8_t* occ, int k, const float* o, const double* d, const double* t0, size_t n, double* t_entry, double* t_exit)
{
	const int N = 1 << k;
	for (size_t r = 0; r < n; ++r)
	{
		int c[3], step[3];
		double tnext[3], dt[3];
		const double ts = t0 ? t0[r] : 0.0;
		for (int a = 0; a < 3; ++a)
		{
			const double da = d[3 * r + a];
			const double p = ((double)o[a] + ts * da - 1.0) * N;
			c[a] = (int)floor(p);
			if (c[a] < 0) c[a] = 0;
			if (c[a] >= N) c[a] = N - 1;
			step[a] = da > 0 ? 1 : -1;
			if (da == 0.0) { tnext[a] = INFINITY; dt[a] = INFINITY; }
			else
			{
				const double edge = da > 0 ? (c[a] + 1) : c[a];
				tnext[a] = ts + (edge - p) / (da * N);
				dt[a] = 1.0 / (fabs(da) * N);
			}
		}
		double t = ts;
		if (t_exit) t_exit[r] = INFINITY;
		for (;;)
		{
			if (occ[((size_t)c[2] * N + c[1]) * N + c[0]]) { t_entry[r] = t; break; }
			const int a = tnext[0] <= tnext[1] ? (tnext[0] <= tnext[2] ? 0 : 2) : (tnext[1] <= tnext[2] ? 1 : 2);
			t = tnext[a];
			c[a] += step[a];
			tnext[a] += dt[a];
			if (c[a] < 0 || c[a] >= N) { t_entry[r] = INFINITY; if (t_exit) t_exit[r] = t; break; }
		}
	}
}
