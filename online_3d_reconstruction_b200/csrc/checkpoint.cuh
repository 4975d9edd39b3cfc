// checkpoint.cuh — export and import of the resident accumulators (o3r_cloud_export_cells / o3r_cloud_import_cells):
// the structure-of-arrays shard (res_keys, res_acc, res_rgb) packed into o3r_cell records, and the validation of records that
// come back from outside the program before they are merged.
#pragma once
#include "voxel.cuh"

namespace o3r {

// failure classes of an imported record (bits of the check result; host_checkpoint.cuh names them)
enum : uint32_t {
    kCkKeyBit63 = 1u, kCkKeyRange = 2u, kCkZeroCount = 4u, kCkNotFinite = 8u, kCkColour = 16u, kCkPad = 32u, kCkOwner = 64u
};

// resident shard -> o3r_cell records, ascending key (the shard's order).  Launched over the host's upper bound of the
// resident count; the exact count is read from the device.
__global__ void __launch_bounds__(kThreads) k_cells_pack(const uint32_t* __restrict__ n_res_ptr, const uint64_t* __restrict__ res_keys,
                                                         const float4* __restrict__ res_acc, const uint4* __restrict__ res_rgb,
                                                         o3r_cell* __restrict__ out) {
    const uint32_t n_res = *n_res_ptr;
    for (uint32_t i = blockIdx.x * kThreads + threadIdx.x; i < n_res; i += gridDim.x * kThreads) {
        const float4 a = res_acc[i];
        const uint4 c = res_rgb[i];
        o3r_cell r;
        r.key = res_keys[i];
        r.sx = a.x; r.sy = a.y; r.sz = a.z; r.n = __float_as_uint(a.w);
        r.sr = c.x; r.sg = c.y; r.sb = c.z; r.pad = 0u;
        out[i] = r;
    }
}

// Validates n imported records.  res[0] (u64) = min over bad records of (index << 32 | that record's failure classes), so
// the first bad index comes with its own reasons; res[1] (u32 pair) = OR of every record's failure classes.  res[0] must
// start at ~0, res[1] at 0.  world = 0: no ownership check.
__global__ void __launch_bounds__(kThreads) k_cells_check(const o3r_cell* __restrict__ cells, uint32_t n, uint32_t world,
                                                          uint32_t rank, unsigned long long* __restrict__ res) {
    uint32_t all = 0u;
    for (uint32_t i = blockIdx.x * kThreads + threadIdx.x; i < n; i += gridDim.x * kThreads) {
        const o3r_cell c = cells[i];
        uint32_t f = 0u;
        if (c.key >> 63) f |= kCkKeyBit63;
        // a 21-bit field of 0 is cell -2^20, outside +-(2^20 - 1)
        if ((c.key & 0x1fffffull) == 0ull || ((c.key >> 21) & 0x1fffffull) == 0ull || ((c.key >> 42) & 0x1fffffull) == 0ull)
            f |= kCkKeyRange;
        if (c.n == 0u) f |= kCkZeroCount;
        if (!isfinite(c.sx) || !isfinite(c.sy) || !isfinite(c.sz)) f |= kCkNotFinite;
        const unsigned long long lim = 255ull * c.n;
        if (c.sr > lim || c.sg > lim || c.sb > lim) f |= kCkColour;
        if (c.pad != 0u) f |= kCkPad;
        if (world && (uint32_t)(hash64(c.key) % world) != rank) f |= kCkOwner;
        if (f) {
            atomicMin(&res[0], ((unsigned long long)i << 32) | f);
            all |= f;
        }
    }
    all = __reduce_or_sync(kFull, all);
    if ((threadIdx.x & 31) == 0 && all) atomicOr(&res[1], (unsigned long long)all);
}

}  // namespace o3r
