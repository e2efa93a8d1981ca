// Host harness of spawn_core.h for the CPU parity test (tests/test_spawn_seeded_cpu.py): n seeds in, n scenes out.
// g++ -O2 -ffp-contract=off -shared -fPIC spawn_host.cpp -o libspawn_host.so   (not part of the product library)
#include "spawn_core.h"

// status[i]: SPAWN_*; fits[i]: spawn_fits; scene rows [n][12] (kind 0 beyond n_veh), filled unless the spawn raises
extern "C" int mm_spawn_host(const uint32_t *seeds, const int32_t *num_cav, int n, int density, int traffic, int32_t *status,
                             uint8_t *fits, int32_t *n_veh, int32_t *n_cav, int32_t *n_merge, int32_t *kind, double *x,
                             double *y, double *speed) {
    using namespace mmspawn;
    if (n < 0 || density < 1 || density > 3 || traffic < TRAFFIC_CAV || traffic > TRAFFIC_HDV) return 1;
    static MT19937 s;
    for (int i = 0; i < n; ++i) {
        if (num_cav[i] < 0 || num_cav[i] > 11) return 1;
        Scene sc{};
        status[i] = spawn_scene(seeds[i], density, traffic, num_cav[i], sc, s);
        fits[i] = spawn_fits(seeds[i], density, num_cav[i], s) ? 1 : 0;
        n_veh[i] = status[i] == SPAWN_RAISES ? 0 : sc.n_veh;
        n_cav[i] = sc.n_cav;
        n_merge[i] = sc.n_merge;
        for (int j = 0; j < MAX_SCENE; ++j) {
            const bool live = j < n_veh[i];
            kind[i * MAX_SCENE + j] = live ? sc.kind[j] : 0;
            x[i * MAX_SCENE + j] = live ? sc.x[j] : 0.0;
            y[i * MAX_SCENE + j] = live ? sc.y[j] : 0.0;
            speed[i * MAX_SCENE + j] = live ? sc.speed[j] : 0.0;
        }
    }
    return 0;
}
