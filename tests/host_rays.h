// tests/host_rays.h -- TEST SCAFFOLDING: the ray and line tables of obf::flips_for / obf::flips_lut for the host
// builds of the kernels' headers.  The kernels stage the same words (ob::kRayTable) in shared memory; here the table
// is a compile-time constant, so it needs no initialisation and any number of threads may read it.
#pragma once
#include "../subproc_b200/csrc/fastboard.cuh"

struct HostRayTable {
    unsigned long long v[obf::kRayTable64];
    constexpr HostRayTable() : v()
    {
        for (int i = 0; i < obf::kRayTable64; i++) v[i] = obf::make_table_word(i);
    }
};
static constexpr HostRayTable kHostRays;

struct Rays {
    unsigned long long operator()(int d, int s) const { return kHostRays.v[d * 64 + s]; }
    unsigned long long word(unsigned i) const { return kHostRays.v[i]; }
    unsigned byte(unsigned i) const { return ((const unsigned char *)kHostRays.v)[i]; }     // (little-endian host)
};
