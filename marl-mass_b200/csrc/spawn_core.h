// spawn_core.h — the reference's seed-exact scene construction (spawn.spawn_scene) as host+device code (mm_reset_seeded).
//
// What it is: `MergeEnv._make_vehicles` (highway_env/envs/merge_env_v1.py:180-211, 265-364, 476-495) after
// `np.random.seed(seed)` (abstract.py:176-199), i.e. every draw it takes from numpy's legacy MT19937 stream, restated
// so that the SAME source compiles for the host (g++, the CPU parity test against spawn.spawn_scene through
// spawn_host.cpp) and for sm_100a (the seeded reset kernel of merge_step.cu, one thread per env).  numpy's legacy
// algorithms, as RandomState uses them:
//   seeding        mt19937_seed: init_genrand of a 32-bit seed (RandomState(int) accepts [0, 2^32))
//   randint/choice random_bounded_uint64_fill for a range below 2^32: masked rejection on single 32-bit words
//   choice(k, replace=False) = permutation(pop)[:k]; permutation = legacy shuffle (_shuffle_raw) from the last index
//                  down with random_interval (masked rejection); the draws are taken even when k == 0
//   rand           random_sample: ((a >> 5) * 67108864 + (b >> 6)) / 2^53
// The state is the full 624-word array: rejection may in principle need more words than one twist provides.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define MM_SP_HD __host__ __device__
#else
#define MM_SP_HD
#endif

namespace mmspawn {

constexpr int MT_N = 624, MT_M = 397;
constexpr int MAX_SCENE = 12;     // one road holds 6 spawn points: at most 12 vehicles before the reference raises
constexpr int KIND_CAV = 1, KIND_HDV = 2;                                        // MM_KIND_*
constexpr int TRAFFIC_CAV = 0, TRAFFIC_MIXED = 1, TRAFFIC_AV = 2, TRAFFIC_HDV = 3;   // MM_TRAFFIC_*
// spawn_scene outcome: OK, the reference raises (ValueError: a larger sample than the road's free spawn points), or the
// scene is built but holds more vehicles than an env slot set (mm_set_state rejects it)
enum { SPAWN_OK = 0, SPAWN_RAISES = 1, SPAWN_TOO_MANY = 2 };

struct MT19937 {
    uint32_t key[MT_N];
    int pos;
};

MM_SP_HD inline void mt_seed(MT19937 &s, uint32_t seed) {
    for (int i = 0; i < MT_N; ++i) {
        s.key[i] = seed;
        seed = 1812433253u * (seed ^ (seed >> 30)) + (uint32_t)(i + 1);
    }
    s.pos = MT_N;
}

MM_SP_HD inline void mt_twist(MT19937 &s) {
    int i = 0;
    uint32_t y;
    for (; i < MT_N - MT_M; ++i) {
        y = (s.key[i] & 0x80000000u) | (s.key[i + 1] & 0x7fffffffu);
        s.key[i] = s.key[i + MT_M] ^ (y >> 1) ^ ((0u - (y & 1u)) & 0x9908b0dfu);
    }
    for (; i < MT_N - 1; ++i) {
        y = (s.key[i] & 0x80000000u) | (s.key[i + 1] & 0x7fffffffu);
        s.key[i] = s.key[i + (MT_M - MT_N)] ^ (y >> 1) ^ ((0u - (y & 1u)) & 0x9908b0dfu);
    }
    y = (s.key[MT_N - 1] & 0x80000000u) | (s.key[0] & 0x7fffffffu);
    s.key[MT_N - 1] = s.key[MT_M - 1] ^ (y >> 1) ^ ((0u - (y & 1u)) & 0x9908b0dfu);
    s.pos = 0;
}

MM_SP_HD inline uint32_t mt_next32(MT19937 &s) {
    if (s.pos == MT_N) mt_twist(s);
    uint32_t y = s.key[s.pos++];
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= y >> 18;
    return y;
}

// a uniform integer in [0, max] by masked rejection (random_interval; also buffered_bounded_masked_uint32, the same
// loop, for randint(0, max + 1)): no word is drawn when max == 0
MM_SP_HD inline uint32_t mt_interval(MT19937 &s, uint32_t max) {
    if (max == 0) return 0;
    uint32_t mask = max;
    mask |= mask >> 1; mask |= mask >> 2; mask |= mask >> 4; mask |= mask >> 8; mask |= mask >> 16;
    uint32_t v;
    while ((v = (mt_next32(s) & mask)) > max) {}
    return v;
}

// random_sample: 53 random bits; every operation is exact (no rounding, so a fused multiply-add changes nothing)
MM_SP_HD inline double mt_double(MT19937 &s) {
    const uint32_t a = mt_next32(s) >> 5, b = mt_next32(s) >> 6;
    return ((double)a * 67108864.0 + (double)b) / 9007199254740992.0;
}

// u * scale + offset with both operations rounded separately, as numpy's `rand(n) * scale + offset` does
MM_SP_HD inline double scale_add(double u, double scale, double offset) {
#if defined(__CUDA_ARCH__)
    return __dadd_rn(__dmul_rn(u, scale), offset);
#else
    volatile double p = u * scale;      // kept apart from the add whatever the host compiler's contraction setting
    return p + offset;
#endif
}

// choice(points[0..n), k, replace=False) = points[permutation(n)[:k]]; writes the k picks to out and removes them from
// points (list.remove keeps the order of the rest)
MM_SP_HD inline void choice_without_replacement(MT19937 &s, int *points, int &n, int k, int *out) {
    int perm[6];
    for (int i = 0; i < n; ++i) perm[i] = i;
    for (int i = n - 1; i >= 1; --i) {
        const int j = (int)mt_interval(s, (uint32_t)i);
        const int t = perm[i]; perm[i] = perm[j]; perm[j] = t;
    }
    bool taken[6] = {false, false, false, false, false, false};
    for (int i = 0; i < k; ++i) { out[i] = points[perm[i]]; taken[perm[i]] = true; }
    int m = 0;
    for (int i = 0; i < n; ++i)
        if (!taken[i]) points[m++] = points[i];
    n = m;
}

// lo_c, lo_h of _num_vehicles (merge_env_v1.py:180-211): the counts are lo + choice(3)
MM_SP_HD inline int density_lo_cav(int density) { return density == 1 ? 1 : density == 2 ? 2 : 4; }
MM_SP_HD inline int density_lo_hdv(int density) { return density == 1 ? 1 : density == 2 ? 2 : 3; }

// The vehicle counts of spawn.num_vehicles: (num_CAV, num_HDV) after the traffic_type rule.  num_cav == 0 draws it.
MM_SP_HD inline void spawn_counts(MT19937 &s, int density, int traffic, int num_cav, int &n_cav, int &n_hdv) {
    int c = num_cav;
    if (c == 0) c = density_lo_cav(density) + (int)mt_interval(s, 2);
    int h = density_lo_hdv(density) + (int)mt_interval(s, 2);
    if (traffic == TRAFFIC_CAV) { c = c + h; h = 0; }
    else if (traffic == TRAFFIC_AV) { h = c + h - 1; c = 1; }
    else if (traffic == TRAFFIC_HDV) { h = c + h; c = 0; }
    n_cav = c;
    n_hdv = h;
}

struct Scene {
    int n_veh, n_cav, n_merge;
    int kind[MAX_SCENE];
    double x[MAX_SCENE], y[MAX_SCENE], speed[MAX_SCENE];
};

// spawn.spawn_scene(seed, density, traffic_type, num_CAV): the vehicles in road.vehicles order (CAVs on the main road,
// CAVs on the ramp, HDVs on the main road, HDVs on the ramp), every speed drawn before every position noise.  Returns
// SPAWN_* (out is complete only for SPAWN_OK and SPAWN_TOO_MANY).  num_cav in [0, 11]; the caller checks the range.
MM_SP_HD inline int spawn_scene(uint32_t seed, int density, int traffic, int num_cav, Scene &out, MT19937 &s) {
    mt_seed(s, seed);
    int n_c, n_h;
    spawn_counts(s, density, traffic, num_cav, n_c, n_h);
    int pts_s[6] = {10, 60, 110, 160, 210, 260}, pts_m[6] = {5, 55, 105, 155, 205, 255};
    int free_s = 6, free_m = 6;
    const int s_c = n_c != 1 ? n_c / 2 : (int)mt_interval(s, 1);
    const int m_c = n_c - s_c;
    if (s_c > free_s) return SPAWN_RAISES;
    int sp_s_c[6], sp_m_c[6], sp_s_h[6], sp_m_h[6];
    choice_without_replacement(s, pts_s, free_s, s_c, sp_s_c);
    if (m_c > free_m) return SPAWN_RAISES;
    choice_without_replacement(s, pts_m, free_m, m_c, sp_m_c);
    const int s_h = n_h != 1 ? n_h / 2 : (int)mt_interval(s, 1);
    const int m_h = n_h - s_h;
    if (s_h > free_s) return SPAWN_RAISES;
    choice_without_replacement(s, pts_s, free_s, s_h, sp_s_h);
    if (m_h > free_m) return SPAWN_RAISES;
    choice_without_replacement(s, pts_m, free_m, m_h, sp_m_h);
    const int n = n_c + n_h;
    for (int i = 0; i < n; ++i) out.speed[i] = scale_add(mt_double(s), 2.0, 25.0);      // initial_speed
    for (int i = 0; i < n; ++i) out.x[i] = scale_add(mt_double(s), 8.0, -4.0);          // loc_noise, added below
    int v = 0;
    for (int i = 0; i < s_c; ++i, ++v) { out.kind[v] = KIND_CAV; out.x[v] += (double)sp_s_c[i]; out.y[v] = 0.0; }
    for (int i = 0; i < m_c; ++i, ++v) { out.kind[v] = KIND_CAV; out.x[v] += (double)sp_m_c[i]; out.y[v] = 10.5; }
    for (int i = 0; i < s_h; ++i, ++v) { out.kind[v] = KIND_HDV; out.x[v] += (double)sp_s_h[i]; out.y[v] = 0.0; }
    for (int i = 0; i < m_h; ++i, ++v) { out.kind[v] = KIND_HDV; out.x[v] += (double)sp_m_h[i]; out.y[v] = 10.5; }
    out.n_veh = n;
    out.n_cav = n_c;
    out.n_merge = m_c;
    return n > MAX_SCENE - 1 ? SPAWN_TOO_MANY : SPAWN_OK;
}

// Whether spawn_scene(seed, density, traffic, num_cav) succeeds with at most 11 vehicles, for 0 <= num_cav <= 11.  Only
// the total count decides (at most 11 always fits the two roads' 6 + 6 points, 13 or more never does, 12 either raises or
// does not fit an env), and it depends on the seed only through the HDV-count draw: the seed is replayed that far only
// when the density's HDV range straddles the limit.
MM_SP_HD inline bool spawn_fits(uint32_t seed, int density, int num_cav, MT19937 &s) {
    if (num_cav == 0) return true;       // drawn counts: at most (lo_c + 2) + (lo_h + 2) = 11
    const int lo_h = density_lo_hdv(density);
    if (num_cav + lo_h + 2 <= MAX_SCENE - 1) return true;
    if (num_cav + lo_h > MAX_SCENE - 1) return false;
    mt_seed(s, seed);
    return num_cav + lo_h + (int)mt_interval(s, 2) <= MAX_SCENE - 1;
}

}  // namespace mmspawn
