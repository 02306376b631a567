// TEST INFRASTRUCTURE — host build of the device functions of the power-mode light table (csrc/restir_core.cuh:
// light_slots_log2 .. slot_sel), run in the order of csrc/geometry.cu: build_light_slots, one loop per kernel, so that
// `pytest -m "not gpu"` checks the CUDA path's arithmetic against the CPU specification (tests/lights/light_port.cpp).
#include <algorithm>
#include <cstring>
#include <numeric>
#include <vector>

#include "../../include/cedecrt.h"
#include "restir_core.cuh"

using namespace crt;

extern "C" long emu_light_table(const float* tris60, const uint32_t* lights, int nlights, int log2_slots, float* out,
                                long cap, uint32_t* starts)
{
    const uint32_t n = (uint32_t)nlights;
    const int k = n ? light_slots_log2(n, log2_slots) : -1;
    if (k < 0) return -1;
    const uint32_t K = 1u << k;
    std::vector<float> power(n);
    uint32_t pmax = 0;
    for (uint32_t i = 0; i < n; i++)  // k_light_power
    {
        power[i] = light_power(tris60, lights[i]);
        pmax = std::max(pmax, f2u(power[i]));
    }
    std::vector<unsigned long long> q(n + 1), prefix(n + 1);
    for (uint32_t i = 0; i < n; i++) q[i] = light_quantum(power[i], u2f(pmax));  // k_light_quantise
    q[n] = 0;
    std::exclusive_scan(q.begin(), q.end(), prefix.begin(), 0ull);
    std::vector<uint32_t> start(n + 1);
    for (uint32_t i = 0; i < n; i++) start[i] = light_start(i, n, K, prefix[i], prefix[n]);  // k_light_starts
    start[n] = K;
    if (starts) memcpy(starts, start.data(), start.size() * sizeof(uint32_t));
    if (!out) return K;
    if (cap < (long)K) return -1;
    for (uint32_t s = 0; s < K; s++)  // k_light_slots
    {
        const uint32_t i = slot_owner(start.data(), n, s);
        const LightRec r = light_rec(tris60, lights[i], slot_sel(start[i + 1] - start[i], K));
        memcpy(out + 16 * (size_t)s, &r, sizeof r);
    }
    return K;
}
