// gmap.cu -- GPU-resident global keypoint map (SURVEY 8a row a9 / 8f "next" #2).
//
// Replaces the reference's host map on the hot path: Keypoint::createKeypoint (src/keypoint.cpp:23-32: position snapped
// to the 10 mm lattice by truncation), Map::addKeypoint (src/mymap.cpp:4-26: 10 m blocks; a keypoint is rejected when a
// stored keypoint of its block lies within 800 mm and is at least as salient; otherwise inserted, or overwrites the entry
// at exactly the same position), LidarOdometry::updateMap (src/lidar_odometry.cpp:343-358: every keypoint of the frame,
// in keypoint order, transformed by the frame pose) and Map::getKeypoints (src/mymap.cpp:28-74: all keypoints of the
// blocks in the +-range cube around a position, blocks visited x-outermost / z-innermost).  The gathered descriptors
// land straight in the matcher's target buffer, followed by the reference frame's descriptors
// (src/lidar_odometry.cpp:197-206) -- no host re-assembly, no PCIe upload of the target set.
//
// Order inside a block: the reference iterates an unordered_map (implementation defined, SURVEY 3.3); here, as in the
// host mirror (host/mymap.h) and the oracle (orc_map_*), it is INSERTION order (an overwrite keeps its slot).
//
// Layout: entries are append-only SoA arrays (position + seg-ratio as float4, 48-byte descriptor); a block is a hash
// table slot {key, count, first chunk, last chunk} plus a chain of 32-index chunks, so a warp reads a block 32 entries
// at a time.  Admission is sequential per block (the rule is order dependent) and parallel across blocks: one warp per
// block touched by the frame walks the frame's keypoints in order.
#include <algorithm>
#include <cmath>

#include "common.cuh"
#include "stages.h"

namespace bshot {

constexpr unsigned GM_PREC = 10000;          // block edge (mm), src/mymap.h:49
constexpr float GM_LATTICE = 10.0f;          // position lattice (mm), src/keypoint.cpp:25
constexpr float GM_REJECT_MM = 800.0f;       // src/mymap.cpp:17
constexpr unsigned long long GM_OCC = 1ull << 63;
// A storable position: every coordinate finite and within +-2.1e9 mm (2100 km), so the lattice snap
// (|int(trunc(v / 10))| * 10 <= 2^31 - 1) and the block id (|roundf(v / 10 m)| * 10 m <= 2^31 - 1, up to 2.147485e9 mm)
// stay inside int32.  Tested on the unsnapped coordinates: a float made from an int is always finite, and a
// saturated int32 times 10 wraps near the origin
constexpr float GM_MAX_MM = 2.1e9f;

__host__ __device__ __forceinline__ bool gm_storable(float x, float y, float z) {
    return fabsf(x) <= GM_MAX_MM && fabsf(y) <= GM_MAX_MM && fabsf(z) <= GM_MAX_MM;   // false for NaN
}

struct GmapBlock {
    unsigned long long key;   // GM_OCC | block id (21 bits per axis), 0 = free
    unsigned count, first, last, touched;
};

// block id of a position: every axis rounded to the 10 m lattice, 21 bits each (src/mymap.cpp:103-112)
__host__ __device__ __forceinline__ unsigned long long gm_block_id(float x, float y, float z) {
    const int gx = (int)roundf(x / (float)GM_PREC) * (int)GM_PREC, gy = (int)roundf(y / (float)GM_PREC) * (int)GM_PREC,
              gz = (int)roundf(z / (float)GM_PREC) * (int)GM_PREC;
    return (((unsigned long long)(long long)gx & 0x1FFFFFull) << 42) | (((unsigned long long)(long long)gy & 0x1FFFFFull) << 21) |
           ((unsigned long long)(long long)gz & 0x1FFFFFull);
}

__device__ __forceinline__ unsigned gm_hash(unsigned long long k, unsigned mask) {
    k ^= k >> 33; k *= 0xFF51AFD7ED558CCDull; k ^= k >> 33;
    return (unsigned)k & mask;
}

// slot of the block, optionally creating it; 0xFFFFFFFF = absent (lookup) / table full (insert)
__device__ __forceinline__ unsigned gm_find(GmapBlock* tab, unsigned mask, unsigned long long id, bool create) {
    const unsigned long long key = GM_OCC | id;
    unsigned h = gm_hash(id, mask);
    for (unsigned probe = 0; probe <= mask; ++probe, h = (h + 1) & mask) {
        unsigned long long cur = *reinterpret_cast<volatile unsigned long long*>(&tab[h].key);
        if (cur == key) return h;
        if (cur == 0ull) {
            if (!create) return 0xFFFFFFFFu;
            cur = atomicCAS(&tab[h].key, 0ull, key);
            if (cur == 0ull || cur == key) return h;
        }
    }
    return 0xFFFFFFFFu;
}

// Keypoint::createKeypoint: int(trunc(pos / prec)) * prec on every axis, for a storable position
__device__ __forceinline__ float3 gm_snap(float3 p) {
    return make_float3((float)((int)truncf(p.x / GM_LATTICE) * (int)GM_LATTICE), (float)((int)truncf(p.y / GM_LATTICE) * (int)GM_LATTICE),
                       (float)((int)truncf(p.z / GM_LATTICE) * (int)GM_LATTICE));
}

// ---- update (addKeypoint for a whole frame) --------------------------------------------------------------------------
// world position, lattice snap, block slot of every keypoint; first toucher of a block lists it
__global__ void gm_prepare_kernel(const float4* __restrict__ kp, const float* __restrict__ ratio, const int* __restrict__ count_dev,
                                  unsigned n_cap, const float* __restrict__ pose, int have_pose, GmapBlock* tab, unsigned mask,
                                  float4* __restrict__ world, unsigned* __restrict__ blk_of, unsigned* __restrict__ touched_list,
                                  unsigned* __restrict__ ctl, unsigned epoch, unsigned update, float* __restrict__ traj) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 12) traj[(size_t)update * 12 + i] = have_pose ? pose[i] : (i % 5 == 0 ? 1.0f : 0.0f);   // the pose this update uses
    const unsigned n = count_dev ? min(n_cap, (unsigned)max(*count_dev, 0)) : n_cap;
    if (i >= n) return;
    const float4 p = kp[i];
    float3 w = have_pose ? pose_apply_rn(pose, p.x, p.y, p.z) : make_float3(p.x, p.y, p.z);
    // a keypoint that is not storable (a non-finite position or pose, or beyond GM_MAX_MM) is skipped; it is not a drop
    if (!gm_storable(w.x, w.y, w.z)) { blk_of[i] = 0xFFFFFFFFu; return; }
    w = gm_snap(w);
    world[i] = make_float4(w.x, w.y, w.z, ratio[i]);
    const unsigned slot = gm_find(tab, mask, gm_block_id(w.x, w.y, w.z), true);
    blk_of[i] = slot;
    if (slot == 0xFFFFFFFFu) { atomicAdd(&ctl[3], 1u); return; }  // table full: counted, reported by the host
    if (atomicExch(&tab[slot].touched, epoch) != epoch) touched_list[atomicAdd(&ctl[1], 1u)] = slot;
}

// one warp per touched block: the frame's keypoints of that block, in keypoint order, through the admission rule
__global__ void __launch_bounds__(128)
gm_admit_kernel(const float4* __restrict__ world, const unsigned* __restrict__ blk_of, const uint64_t* __restrict__ bits,
                const int* __restrict__ count_dev, unsigned n_cap, GmapBlock* tab, const unsigned* __restrict__ touched_list,
                unsigned* __restrict__ ctl, float4* __restrict__ e_pos, uint64_t* __restrict__ e_desc, unsigned* __restrict__ e_tag,
                unsigned* __restrict__ chunks, unsigned max_entries, unsigned max_chunks, unsigned update) {
    const unsigned lane = threadIdx.x & 31, w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (w >= ctl[1]) return;
    const unsigned slot = touched_list[w];
    const unsigned n = count_dev ? min(n_cap, (unsigned)max(*count_dev, 0)) : n_cap;
    unsigned cnt = tab[slot].count, first = tab[slot].first, last = tab[slot].last;
    for (unsigned base = 0; base < n; base += 32) {
        const unsigned i = base + lane;
        unsigned members = __ballot_sync(0xffffffffu, i < n && blk_of[i] == slot);
        while (members) {
            const unsigned k = base + (unsigned)(__ffs(members) - 1);
            members &= members - 1u;
            const float4 p = world[k];  // (x, y, z, seg-ratio) of the new keypoint
            // walk the stored entries of the block, 32 at a time
            bool reject = false;
            unsigned same = 0xFFFFFFFFu;
            unsigned c = first;
            for (unsigned j0 = 0; j0 < cnt; j0 += 32, c = chunks[c * 33u + 32u]) {
                const unsigned j = j0 + lane;
                bool rj = false;
                unsigned sm = 0xFFFFFFFFu;
                if (j < cnt) {
                    const unsigned e = chunks[c * 33u + lane];
                    const float4 q = e_pos[e];
                    const float dx = __fsub_rn(p.x, q.x), dy = __fsub_rn(p.y, q.y), dz = __fsub_rn(p.z, q.z);
                    const float dist = sqrtf(dot3_rn(dx, dy, dz, dx, dy, dz));
                    rj = dist < GM_REJECT_MM && p.w <= q.w;   // src/mymap.cpp:17-18
                    if (q.x == p.x && q.y == p.y && q.z == p.z) sm = e;
                }
                reject = reject || __any_sync(0xffffffffu, rj);
                const unsigned who = __ballot_sync(0xffffffffu, sm != 0xFFFFFFFFu);
                if (who) same = __shfl_sync(0xffffffffu, sm, __ffs(who) - 1);
            }
            if (reject) continue;
            unsigned e = same;  // keypoints_[block][position] = keypoint: overwrite at an equal position, else insert
            if (e == 0xFFFFFFFFu) {
                // the chunk first, then the entry: an entry index below max_entries cannot be given back (another warp
                // may already hold the next one), a chunk that is not linked is only unused
                unsigned nc = 0xFFFFFFFFu;
                if ((cnt & 31u) == 0u) {  // new chunk
                    if (lane == 0) nc = atomicAdd(&ctl[2], 1u);
                    nc = __shfl_sync(0xffffffffu, nc, 0);
                    if (nc >= max_chunks) { if (lane == 0) atomicAdd(&ctl[3], 1u); continue; }
                }
                if (lane == 0) e = atomicAdd(&ctl[0], 1u);
                e = __shfl_sync(0xffffffffu, e, 0);
                if (e >= max_entries) { if (lane == 0) { atomicAdd(&ctl[3], 1u); atomicSub(&ctl[0], 1u); } continue; }
                if (nc != 0xFFFFFFFFu) {
                    if (lane == 0) {
                        chunks[nc * 33u + 32u] = 0xFFFFFFFFu;
                        if (cnt == 0u) first = nc; else chunks[last * 33u + 32u] = nc;
                    }
                    first = __shfl_sync(0xffffffffu, first, 0);
                    last = nc;
                }
                if (lane == 0) chunks[last * 33u + (cnt & 31u)] = e;
                ++cnt;
            }
            if (lane == 0) { e_pos[e] = p; e_tag[e] = update; }   // an overwrite takes this update's tag: its descriptor is this scan's
            if (lane < 6) e_desc[(size_t)e * 6 + lane] = bits[(size_t)k * 6 + lane];
            __syncwarp();
            __threadfence_block();
        }
    }
    if (lane == 0) { tab[slot].count = cnt; tab[slot].first = first; tab[slot].last = last; }
}

// ---- gather (getKeypoints) ----------------------------------------------------------------------------------------------
struct GmapCube { int x0, y0, z0, nx, ny, nz; };

__host__ __device__ inline GmapCube gm_cube(float px, float py, float pz, float range) {
    GmapCube c;
    const float prec = (float)GM_PREC;
    c.x0 = (int)roundf((px - range) / prec); c.nx = (int)roundf((px + range) / prec) - c.x0 + 1;
    c.y0 = (int)roundf((py - range) / prec); c.ny = (int)roundf((py + range) / prec) - c.y0 + 1;
    c.z0 = (int)roundf((pz - range) / prec); c.nz = (int)roundf((pz + range) / prec) - c.z0 + 1;
    return c;
}

// one step of a running exclusive scan over a CTA of 1024 threads: *carry (shared, 0 before the first step) + the exclusive
// prefix of v over this step's threads; *carry then holds the running total.  Every thread must call it
__device__ __forceinline__ unsigned cta_scan_1024(unsigned v, unsigned* ws, unsigned* carry) {
    const unsigned tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    unsigned inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned up = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (unsigned)o) inc += up;
    }
    if (lane == 31) ws[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        const unsigned u = ws[lane];
        unsigned winc = u;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned up = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= (unsigned)o) winc += up;
        }
        ws[lane] = winc - u;
    }
    __syncthreads();
    const unsigned excl = *carry + ws[wid] + inc - v;
    __syncthreads();
    if (tid == 1023) *carry = excl + v;
    __syncthreads();
    return excl;
}

// one CTA: counts of the probed blocks in loop order (x outermost, z innermost), exclusive scan -> offsets
__global__ void __launch_bounds__(1024)
gm_probe_kernel(const GmapBlock* __restrict__ tab, unsigned mask, GmapCube cube, const float* __restrict__ dev_pose, float range,
                unsigned* __restrict__ probe_slot, unsigned* __restrict__ probe_off, unsigned* __restrict__ ctl, unsigned max_probe) {
    __shared__ unsigned ws[32];
    __shared__ unsigned carry;
    const unsigned tid = threadIdx.x;
    if (dev_pose) {   // position = translation of the row-major [R|T]; a non-finite pose probes nothing
        cube = gm_cube(dev_pose[3], dev_pose[7], dev_pose[11], range);
        if (cube.nx <= 0 || cube.ny <= 0 || cube.nz <= 0) cube.nx = cube.ny = cube.nz = 0;
    }
    const unsigned np = min((unsigned)(cube.nx * cube.ny * cube.nz), max_probe);
    if (tid == 0) carry = 0;
    __syncthreads();
    for (unsigned base = 0; base < np; base += 1024) {
        const unsigned p = base + tid;
        unsigned cnt = 0, slot = 0xFFFFFFFFu;
        if (p < np) {
            const int iz = (int)(p % (unsigned)cube.nz), iy = (int)((p / (unsigned)cube.nz) % (unsigned)cube.ny), ix = (int)(p / ((unsigned)cube.nz * (unsigned)cube.ny));
            const float x = (float)((cube.x0 + ix) * (int)GM_PREC), y = (float)((cube.y0 + iy) * (int)GM_PREC), z = (float)((cube.z0 + iz) * (int)GM_PREC);
            slot = gm_find(const_cast<GmapBlock*>(tab), mask, gm_block_id(x, y, z), false);
            if (slot != 0xFFFFFFFFu) cnt = tab[slot].count;
            probe_slot[p] = slot;
        }
        const unsigned excl = cta_scan_1024(cnt, ws, &carry);
        if (p < np) probe_off[p] = excl;
    }
    if (tid == 0) { ctl[4] = carry; ctl[5] = np; }
}

// one warp per listed block (*d_np of them): entries in insertion order -> out[offset + j]
__global__ void __launch_bounds__(128)
gm_collect_kernel(const GmapBlock* __restrict__ tab, const unsigned* __restrict__ probe_slot, const unsigned* __restrict__ probe_off,
                  const unsigned* __restrict__ d_np, const unsigned* __restrict__ chunks, const float4* __restrict__ e_pos,
                  const uint64_t* __restrict__ e_desc, float4* __restrict__ out_pos, uint64_t* __restrict__ out_desc, unsigned out_cap,
                  const unsigned* __restrict__ e_tag, unsigned* __restrict__ out_tag) {
    const unsigned lane = threadIdx.x & 31;
    const unsigned np = *d_np;
    for (unsigned p = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; p < np; p += (gridDim.x * blockDim.x) >> 5) {
        const unsigned slot = probe_slot[p];
        if (slot == 0xFFFFFFFFu) continue;
        const unsigned cnt = tab[slot].count, off = probe_off[p];
        unsigned c = tab[slot].first;
        for (unsigned j0 = 0; j0 < cnt; j0 += 32, c = chunks[c * 33u + 32u]) {
            const unsigned j = j0 + lane;
            if (j < cnt && off + j < out_cap) {
                const unsigned e = chunks[c * 33u + lane];
                out_pos[off + j] = e_pos[e];
                if (out_tag) out_tag[off + j] = e_tag[e];
#pragma unroll
                for (int k = 0; k < 6; ++k) out_desc[(size_t)(off + j) * 6 + k] = e_desc[(size_t)e * 6 + k];
            }
        }
    }
}

// appends the reference frame: positions transformed by its pose (pcl::transformPointCloud, :202), descriptors as they are
__global__ void gm_append_ref_kernel(const float4* __restrict__ ref_kp, const uint64_t* __restrict__ ref_bits, const int* __restrict__ ref_count,
                                     unsigned n_cap, const float* __restrict__ pose, int have_pose, const unsigned* __restrict__ ctl,
                                     float4* __restrict__ out_pos, uint64_t* __restrict__ out_desc, unsigned out_cap, unsigned* __restrict__ total_out) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned n = ref_count ? min(n_cap, (unsigned)max(*ref_count, 0)) : n_cap;
    const unsigned base = min(ctl[4], out_cap);
    if (i == 0) *total_out = min(base + n, out_cap);
    if (i >= n || base + i >= out_cap) return;
    const float4 p = ref_kp[i];
    const float3 w = have_pose ? pose_apply_rn(pose, p.x, p.y, p.z) : make_float3(p.x, p.y, p.z);
    out_pos[base + i] = make_float4(w.x, w.y, w.z, 0.0f);
#pragma unroll
    for (int k = 0; k < 6; ++k) out_desc[(size_t)(base + i) * 6 + k] = ref_bits[(size_t)i * 6 + k];
}

// ---- the whole map in map order (gmap_gather_all), and the import's rebuild ---------------------------------------------
// Map order: occupied blocks in ascending lattice coordinates (x outermost, z innermost: the order gm_probe_kernel visits
// them), entries of a block in insertion order.  A block's coordinates are roundf(p / 10 m) of any of its entries (the
// block id was computed from that same stored position).  actl: [0] listed blocks, [1] entries gathered, [2] import
// error bits (1 position not storable, 2 table / chunks full), [3] import entries.
constexpr unsigned GM_AXIS_BIAS = 1u << 20;

__device__ __forceinline__ unsigned long long gm_order_key(float4 p) {
    const unsigned kx = ((unsigned)(int)roundf(p.x / (float)GM_PREC) + GM_AXIS_BIAS) & 0x1FFFFFu;
    const unsigned ky = ((unsigned)(int)roundf(p.y / (float)GM_PREC) + GM_AXIS_BIAS) & 0x1FFFFFu;
    const unsigned kz = ((unsigned)(int)roundf(p.z / (float)GM_PREC) + GM_AXIS_BIAS) & 0x1FFFFFu;
    return ((unsigned long long)kx << 42) | ((unsigned long long)ky << 21) | (unsigned long long)kz;
}

// occupied, non-empty slots -> (order key, slot); the list's order is irrelevant (the keys are distinct and get sorted)
__global__ void gm_list_blocks_kernel(const GmapBlock* __restrict__ tab, unsigned tab_cap, const unsigned* __restrict__ chunks,
                                      const float4* __restrict__ e_pos, unsigned long long* __restrict__ keys, unsigned* __restrict__ slots,
                                      unsigned* __restrict__ actl) {
    const unsigned s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= tab_cap || tab[s].key == 0ull || tab[s].count == 0u) return;
    const unsigned long long k = gm_order_key(e_pos[chunks[tab[s].first * 33u]]);
    const unsigned i = atomicAdd(&actl[0], 1u);
    keys[i] = k;
    slots[i] = s;
}

// one CTA: entry offsets of the listed blocks in their sorted order; actl[1] = entries
__global__ void __launch_bounds__(1024)
gm_block_offsets_kernel(const GmapBlock* __restrict__ tab, const unsigned* __restrict__ slots, unsigned* __restrict__ off, unsigned* __restrict__ actl) {
    __shared__ unsigned ws[32];
    __shared__ unsigned carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const unsigned nb = actl[0];
    for (unsigned base = 0; base < nb; base += 1024) {
        const unsigned i = base + threadIdx.x;
        const unsigned cnt = i < nb ? tab[slots[i]].count : 0u;
        const unsigned excl = cta_scan_1024(cnt, ws, &carry);
        if (i < nb) off[i] = excl;
    }
    if (threadIdx.x == 0) actl[1] = carry;
}

// import: the entries already sit at pool index = input index (*d_n of them, n_cap without a device count).  Block slot
// of every entry (created when new), its count, and (slot, input index) for the stable sort by slot.  Tags from tag_src
// (null: 0); with traj the trajectory's update 0 becomes the identity
__global__ void gm_import_find_kernel(const float4* __restrict__ e_pos, unsigned n_cap, const unsigned* __restrict__ d_n, GmapBlock* tab, unsigned mask,
                                      unsigned long long* __restrict__ keys, unsigned* __restrict__ idx, unsigned* __restrict__ actl,
                                      const unsigned* __restrict__ tag_src, unsigned* __restrict__ e_tag, float* __restrict__ traj) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned n = d_n ? min(*d_n, n_cap) : n_cap;
    if (i == 0) actl[3] = n;
    if (traj && i < 12) traj[i] = (i % 5 == 0) ? 1.0f : 0.0f;   // the import is update 0, in the map frame
    if (i >= n) return;
    e_tag[i] = tag_src ? tag_src[i] : 0u;
    const float4 p = e_pos[i];
    unsigned slot = 0xFFFFFFFFu;
    if (!gm_storable(p.x, p.y, p.z)) atomicOr(&actl[2], 1u);
    else if ((slot = gm_find(tab, mask, gm_block_id(p.x, p.y, p.z), true)) == 0xFFFFFFFFu) atomicOr(&actl[2], 2u);
    else atomicAdd(&tab[slot].count, 1u);
    keys[i] = slot;
    idx[i] = i;
}

// import, one CTA over every table slot in slot order: first entry of the slot in the slot-sorted list (start) and
// ceil(count / 32) consecutive chunks, first / last of the block; then the entry and chunk counts (the dropped count
// ctl[3] stays: a re-anchor keeps it, an import starts from a reset map)
__global__ void __launch_bounds__(1024)
gm_import_blocks_kernel(GmapBlock* tab, unsigned tab_cap, unsigned* __restrict__ start, unsigned* __restrict__ ctl, unsigned* __restrict__ actl,
                        unsigned max_chunks) {
    __shared__ unsigned ws[32];
    __shared__ unsigned carry_e, carry_c;
    if (threadIdx.x == 0) carry_e = carry_c = 0;
    __syncthreads();
    for (unsigned base = 0; base < tab_cap; base += 1024) {
        const unsigned s = base + threadIdx.x;
        const unsigned cnt = (s < tab_cap && tab[s].key != 0ull) ? tab[s].count : 0u, nch = (cnt + 31u) / 32u;
        const unsigned e0 = cta_scan_1024(cnt, ws, &carry_e);
        const unsigned c0 = cta_scan_1024(nch, ws, &carry_c);
        if (s < tab_cap) start[s] = e0;
        if (cnt) { tab[s].first = c0; tab[s].last = c0 + nch - 1u; }
    }
    if (threadIdx.x == 0) {
        if (carry_c > max_chunks) actl[2] |= 2u;
        ctl[0] = carry_e;
        ctl[2] = carry_c;
    }
}

// import: sorted position j -> rank r in its block -> chunk first + r / 32, lane r % 32; a chunk's first entry links it.
// *d_n entries (gm_import_find_kernel's count)
__global__ void gm_import_chain_kernel(const unsigned long long* __restrict__ slot_of, const unsigned* __restrict__ idx, const unsigned* __restrict__ d_n,
                                       const GmapBlock* __restrict__ tab, unsigned tab_cap, const unsigned* __restrict__ start,
                                       unsigned* __restrict__ chunks, unsigned max_chunks) {
    const unsigned j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= *d_n) return;
    const unsigned long long s = slot_of[j];
    if (s >= tab_cap) return;   // an entry without a block: the import fails
    const unsigned r = j - start[s], cnt = tab[s].count, ch = tab[s].first + r / 32u;
    if (ch >= max_chunks) return;
    chunks[ch * 33u + (r & 31u)] = idx[j];
    if ((r & 31u) == 0u) chunks[ch * 33u + 32u] = r + 32u < cnt ? ch + 1u : 0xFFFFFFFFu;
}

// re-anchor: the whole map in map order (*d_n entries), each entry of a changed update u moved by that update's correction
// C_u (row-major 3x4) and snapped to the lattice as gm_prepare_kernel moves and snaps a keypoint; the entries of
// unchanged updates are copied as they are.  Written straight into the entry pool at pool index = map-order index, with
// their descriptors, where the rebuild reads them; *n_out = the count, for the rebuild
__global__ void gm_reanchor_move_kernel(const float4* __restrict__ apos, const uint64_t* __restrict__ adesc, const unsigned* __restrict__ atag,
                                        const unsigned* __restrict__ d_n, unsigned n_cap, const float* __restrict__ corr, const unsigned* __restrict__ changed,
                                        unsigned n_upd, float4* __restrict__ e_pos, uint64_t* __restrict__ e_desc, unsigned* __restrict__ n_out) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned n = min(*d_n, n_cap);
    if (i == 0) *n_out = n;
    if (i >= n) return;
#pragma unroll
    for (int k = 0; k < 6; ++k) e_desc[(size_t)i * 6 + k] = adesc[(size_t)i * 6 + k];
    const float4 p = apos[i];
    const unsigned u = atag[i];
    if (u >= n_upd || !changed[u]) { e_pos[i] = p; return; }
    float3 w = pose_apply_rn(corr + (size_t)u * 12, p.x, p.y, p.z);
    // an entry moved out of the storable range stays unsnapped: the rebuild rejects it and the map is restored
    if (gm_storable(w.x, w.y, w.z)) w = gm_snap(w);
    e_pos[i] = make_float4(w.x, w.y, w.z, p.w);
}

// ---- host side -----------------------------------------------------------------------------------------------------------
int gmap_create(Ctx* c, size_t max_entries, size_t max_blocks) {
    Gmap& g = c->gmap;
    if (g.d_tab) return BSHOT_OK;
    unsigned cap = 1024;
    while (cap < 2 * max_blocks) cap <<= 1;
    g.tab_cap = cap;
    g.max_entries = (unsigned)max_entries;
    g.max_chunks = (unsigned)(max_entries / 32 + max_blocks + 64);
    g.max_probe = 32768;
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_tab, sizeof(GmapBlock) * cap));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_epos, sizeof(float4) * max_entries));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_edesc, 48 * max_entries));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_chunks, sizeof(unsigned) * 33 * g.max_chunks));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_world, sizeof(float4) * c->max_kp));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_blk_of, sizeof(unsigned) * c->max_kp));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_touched, sizeof(unsigned) * c->max_kp));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_probe_slot, sizeof(unsigned) * g.max_probe));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_probe_off, sizeof(unsigned) * g.max_probe));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_ctl, sizeof(unsigned) * 8));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_pose, sizeof(float) * 24));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_tpos, sizeof(float4) * c->max_targets));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_etag, sizeof(unsigned) * max_entries));
    g.traj_cap = 1024;
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_traj, sizeof(float) * 12 * g.traj_cap));
    return gmap_reset(c);
}

void gmap_free(Ctx* c) {
    Gmap& g = c->gmap;
    void* ptrs[] = {g.d_tab, g.d_epos, g.d_edesc, g.d_chunks, g.d_world, g.d_blk_of, g.d_touched, g.d_probe_slot, g.d_probe_off, g.d_ctl, g.d_pose, g.d_tpos,
                    g.d_apos, g.d_adesc, g.d_skeys[0], g.d_skeys[1], g.d_svals[0], g.d_svals[1], g.d_shist, g.d_boff, g.d_actl,
                    g.d_etag, g.d_traj, g.d_atag, g.d_lpos, g.d_ldesc, g.d_ltag, g.d_ltile, g.d_lctl, g.d_rtraj, g.d_rcorr, g.d_rchg};
    for (void* p : ptrs) if (p) cudaFree(p);
    g = Gmap();
}

int gmap_reset(Ctx* c) {
    Gmap& g = c->gmap;
    if (!g.d_tab) return BSHOT_OK;
    BSHOT_CUDA_TRY(cudaMemsetAsync(g.d_tab, 0, sizeof(GmapBlock) * g.tab_cap, c->stream));
    BSHOT_CUDA_TRY(cudaMemsetAsync(g.d_ctl, 0, sizeof(unsigned) * 8, c->stream));
    g.epoch = 0;
    g.n_gathered = 0;
    g.entries_upper = 0;
    g.n_updates = 0;
    g.last_by_scan = false;
    return BSHOT_OK;
}

void gmap_record_update(Ctx* c, size_t n_cap, bool by_scan) {
    Gmap& g = c->gmap;
    g.entries_upper += n_cap;
    ++g.n_updates;
    g.last_by_scan = by_scan;
}

// ctl: [0] entries, [1] touched blocks of the current update, [2] chunks, [3] dropped (capacity), [4] gathered map entries, [5] probes
int gmap_update(Ctx* c, const float4* d_kp, const float* d_ratio, const uint64_t* d_bits, const int* d_count, size_t n_cap, const float* pose12, bool pose_on_device) {
    Gmap& g = c->gmap;
    if (!g.d_tab) { set_error("map: bshot_gmap_create first"); return BSHOT_E_STATE; }
    if (n_cap == 0) return BSHOT_OK;
    if (n_cap > c->max_kp) { set_error("map update: %zu keypoints > capacity %zu", n_cap, c->max_kp); return BSHOT_E_CAPACITY; }
    if (g.n_updates >= g.traj_cap) {   // the trajectory doubles; gmap_record_update advances n_updates once the update succeeded
        float* grown = nullptr;
        BSHOT_CUDA_TRY(cudaMalloc((void**)&grown, sizeof(float) * 24 * g.traj_cap));
        BSHOT_CUDA_TRY(cudaMemcpyAsync(grown, g.d_traj, sizeof(float) * 12 * g.traj_cap, cudaMemcpyDeviceToDevice, c->stream));
        BSHOT_CUDA_TRY(cudaStreamSynchronize(c->stream));
        BSHOT_CUDA_TRY(cudaFree(g.d_traj));
        g.d_traj = grown;
        g.traj_cap *= 2;
    }
    if (pose12) BSHOT_CUDA_TRY(cudaMemcpyAsync(g.d_pose, pose12, sizeof(float) * 12, pose_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, c->stream));
    BSHOT_CUDA_TRY(cudaMemsetAsync(g.d_ctl + 1, 0, sizeof(unsigned), c->stream));
    ++g.epoch;
    const unsigned n = (unsigned)n_cap;
    gm_prepare_kernel<<<(n + 255) / 256, 256, 0, c->stream>>>(d_kp, d_ratio, d_count, n, g.d_pose, pose12 ? 1 : 0, reinterpret_cast<GmapBlock*>(g.d_tab),
                                                             g.tab_cap - 1, g.d_world, g.d_blk_of, g.d_touched, g.d_ctl, g.epoch, g.n_updates, g.d_traj);
    // at most n blocks are touched: one warp each (warps beyond the device-side count exit)
    gm_admit_kernel<<<(n * 32 + 127) / 128, 128, 0, c->stream>>>(g.d_world, g.d_blk_of, d_bits, d_count, n, reinterpret_cast<GmapBlock*>(g.d_tab), g.d_touched,
                                                                g.d_ctl, g.d_epos, g.d_edesc, g.d_etag, g.d_chunks, g.max_entries, g.max_chunks,
                                                                g.n_updates);
    count_launch(c, 2);
    return check_launch("map update kernels");
}

// target set of featureMatching in RUN status: map keypoints within `range` of `pos`, then the reference frame
// (d_ref_* may be null).  Descriptors -> d_t_out (the matcher's target buffer), positions -> g.d_tpos; *d_total = count.
int gmap_gather(Ctx* c, const float pos[3], float range, const float4* d_ref_kp, const uint64_t* d_ref_bits, const int* d_ref_count,
                size_t ref_cap, const float* ref_pose12, uint64_t* d_t_out, size_t out_cap, unsigned* d_total, bool pose_on_device) {
    Gmap& g = c->gmap;
    if (!g.d_tab) { set_error("map: bshot_gmap_create first"); return BSHOT_E_STATE; }
    GmapCube cube = {0, 0, 0, 0, 0, 0};
    if (pose_on_device) {
        // position = translation of the device-side pose: the cube is computed by the probe kernel.  Its edge is at most
        // round((p + r) / 10 m) - round((p - r) / 10 m) + 1 <= 2 r / 10 m + 3 blocks (rounding included), whatever p is
        const double edge = std::floor(2.0 * (double)range / (double)GM_PREC) + 3.0;
        if (!ref_pose12 || edge * edge * edge > (double)g.max_probe) { set_error("map gather: range %.0f probes more than %u blocks", range, g.max_probe); return BSHOT_E_CAPACITY; }
    } else {
        cube = gm_cube(pos[0], pos[1], pos[2], range);
        if ((long long)cube.nx * cube.ny * cube.nz > (long long)g.max_probe) { set_error("map gather: range %.0f probes more than %u blocks", range, g.max_probe); return BSHOT_E_CAPACITY; }
    }
    if (ref_pose12)
        BSHOT_CUDA_TRY(cudaMemcpyAsync(g.d_pose + 12, ref_pose12, sizeof(float) * 12, pose_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, c->stream));
    gm_probe_kernel<<<1, 1024, 0, c->stream>>>(reinterpret_cast<const GmapBlock*>(g.d_tab), g.tab_cap - 1, cube, pose_on_device ? g.d_pose + 12 : nullptr, range,
                                               g.d_probe_slot, g.d_probe_off, g.d_ctl, g.max_probe);
    gm_collect_kernel<<<(unsigned)c->sm_count * 2u, 128, 0, c->stream>>>(reinterpret_cast<const GmapBlock*>(g.d_tab), g.d_probe_slot, g.d_probe_off, g.d_ctl + 5, g.d_chunks,
                                                                        g.d_epos, g.d_edesc, g.d_tpos, d_t_out, (unsigned)out_cap, nullptr, nullptr);
    const unsigned nref = d_ref_bits ? (unsigned)ref_cap : 0u;
    gm_append_ref_kernel<<<(std::max(nref, 1u) + 255) / 256, 256, 0, c->stream>>>(d_ref_kp, d_ref_bits, d_ref_count, nref, g.d_pose + 12, ref_pose12 ? 1 : 0, g.d_ctl,
                                                                                g.d_tpos, d_t_out, (unsigned)out_cap, d_total);
    count_launch(c, 3);
    return check_launch("map gather kernels");
}

// buffers of the whole-map gather and the import (entry-sized), allocated by the first call that needs them
static int gmap_all_alloc(Ctx* c) {
    Gmap& g = c->gmap;
    if (g.d_apos) return BSHOT_OK;
    const size_t m = std::max<size_t>(g.tab_cap, g.max_entries);
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_apos, sizeof(float4) * g.max_entries));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_adesc, 48 * (size_t)g.max_entries));
    for (int k = 0; k < 2; ++k) {
        BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_skeys[k], sizeof(unsigned long long) * m));
        BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_svals[k], sizeof(unsigned) * m));
    }
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_shist, sizeof(unsigned) * radix_hist_words(m)));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_boff, sizeof(unsigned) * g.tab_cap));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_actl, sizeof(unsigned) * 8));
    BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_atag, sizeof(unsigned) * g.max_entries));
    return BSHOT_OK;
}

int gmap_gather_all(Ctx* c, size_t* nt_cap_out, bool with_tags) {
    Gmap& g = c->gmap;
    if (!g.d_tab) { set_error("map: bshot_gmap_create first"); return BSHOT_E_STATE; }
    BSHOT_TRY(gmap_all_alloc(c));
    const size_t nt_cap = std::min<size_t>(g.entries_upper, g.max_entries);
    *nt_cap_out = nt_cap;
    BSHOT_CUDA_TRY(cudaMemsetAsync(g.d_actl, 0, sizeof(unsigned) * 8, c->stream));
    if (nt_cap == 0) return BSHOT_OK;
    GmapBlock* tab = reinterpret_cast<GmapBlock*>(g.d_tab);
    gm_list_blocks_kernel<<<(g.tab_cap + 255) / 256, 256, 0, c->stream>>>(tab, g.tab_cap, g.d_chunks, g.d_epos, g.d_skeys[0], g.d_svals[0], g.d_actl);
    count_launch(c);
    BSHOT_TRY(check_launch("gm_list_blocks_kernel"));
    // 63-bit keys: 8 passes, the result is back in buffer 0
    BSHOT_TRY(radix_sort_pairs(c, g.d_skeys, g.d_svals, g.d_shist, g.d_actl, std::min<size_t>(g.tab_cap, nt_cap), 8));
    gm_block_offsets_kernel<<<1, 1024, 0, c->stream>>>(tab, g.d_svals[0], g.d_boff, g.d_actl);
    gm_collect_kernel<<<(unsigned)c->sm_count * 2u, 128, 0, c->stream>>>(tab, g.d_svals[0], g.d_boff, g.d_actl, g.d_chunks, g.d_epos, g.d_edesc, g.d_apos,
                                                                        g.d_adesc, g.max_entries, g.d_etag, with_tags ? g.d_atag : nullptr);
    count_launch(c, 2);
    return check_launch("map gather-all kernels");
}

int gmap_export(Ctx* c, float* xyzr_out, uint64_t* desc_out, size_t cap, size_t* n_out) {
    Gmap& g = c->gmap;
    size_t nt_cap;
    BSHOT_TRY(gmap_gather_all(c, &nt_cap));
    unsigned* h = reinterpret_cast<unsigned*>(&c->h_scratch[48]);
    BSHOT_CUDA_TRY(cudaMemcpyAsync(h, g.d_actl, sizeof(unsigned) * 4, cudaMemcpyDeviceToHost, c->stream));
    BSHOT_CUDA_TRY(cudaStreamSynchronize(c->stream));
    const size_t n = h[1], m = std::min(n, cap);
    if (n_out) *n_out = n;
    if (xyzr_out && m) BSHOT_CUDA_TRY(cudaMemcpyAsync(xyzr_out, g.d_apos, sizeof(float4) * m, cudaMemcpyDeviceToHost, c->stream));
    if (desc_out && m) BSHOT_CUDA_TRY(cudaMemcpyAsync(desc_out, g.d_adesc, 48 * m, cudaMemcpyDeviceToHost, c->stream));
    BSHOT_CUDA_TRY(cudaStreamSynchronize(c->stream));
    if (n > cap) { set_error("bshot_gmap_export: %zu entries > capacity %zu", n, cap); return BSHOT_E_CAPACITY; }
    return BSHOT_OK;
}

int gmap_import_dev(Ctx* c, const float4* d_pos, const uint64_t* d_desc, const unsigned* d_tag, size_t n_cap, const unsigned* d_n, const char* who) {
    Gmap& g = c->gmap;
    BSHOT_TRY(gmap_all_alloc(c));
    const unsigned nn = (unsigned)n_cap;
    GmapBlock* tab = reinterpret_cast<GmapBlock*>(g.d_tab);
    BSHOT_CUDA_TRY(cudaMemsetAsync(g.d_tab, 0, sizeof(GmapBlock) * g.tab_cap, c->stream));
    BSHOT_CUDA_TRY(cudaMemsetAsync(g.d_actl, 0, sizeof(unsigned) * 8, c->stream));
    if (d_pos != g.d_epos) BSHOT_CUDA_TRY(cudaMemcpyAsync(g.d_epos, d_pos, sizeof(float4) * n_cap, cudaMemcpyDeviceToDevice, c->stream));
    if (d_desc != g.d_edesc) BSHOT_CUDA_TRY(cudaMemcpyAsync(g.d_edesc, d_desc, 48 * n_cap, cudaMemcpyDeviceToDevice, c->stream));
    gm_import_find_kernel<<<(nn + 255) / 256, 256, 0, c->stream>>>(g.d_epos, nn, d_n, tab, g.tab_cap - 1, g.d_skeys[0], g.d_svals[0], g.d_actl, d_tag, g.d_etag,
                                                                    d_tag ? nullptr : g.d_traj);
    count_launch(c);
    BSHOT_TRY(check_launch("gm_import_find_kernel"));
    // stable by slot: the input order survives inside a block.  Slots are < tab_cap (a power of two)
    unsigned bits = 0;
    while ((1u << bits) < g.tab_cap) ++bits;
    const unsigned passes = (bits + 7) / 8;
    BSHOT_TRY(radix_sort_pairs(c, g.d_skeys, g.d_svals, g.d_shist, g.d_actl + 3, n_cap, passes));
    gm_import_blocks_kernel<<<1, 1024, 0, c->stream>>>(tab, g.tab_cap, g.d_boff, g.d_ctl, g.d_actl, g.max_chunks);
    gm_import_chain_kernel<<<(nn + 255) / 256, 256, 0, c->stream>>>(g.d_skeys[passes & 1], g.d_svals[passes & 1], g.d_actl + 3, tab, g.tab_cap, g.d_boff,
                                                                    g.d_chunks, g.max_chunks);
    count_launch(c, 2);
    BSHOT_TRY(check_launch("map import kernels"));
    unsigned* h = reinterpret_cast<unsigned*>(&c->h_scratch[48]);
    BSHOT_CUDA_TRY(cudaMemcpyAsync(h, g.d_actl, sizeof(unsigned) * 4, cudaMemcpyDeviceToHost, c->stream));
    BSHOT_CUDA_TRY(cudaStreamSynchronize(c->stream));
    if (h[2] & 1u) { set_error("%s: a position is not finite or beyond +-2.1e9 mm", who); return BSHOT_E_INVALID; }
    if (h[2]) { set_error("%s: more blocks or chunks than the map holds (%u slots, %u chunks)", who, g.tab_cap, g.max_chunks); return BSHOT_E_CAPACITY; }
    return BSHOT_OK;
}

int gmap_import(Ctx* c, const float* xyzr, const uint64_t* desc, size_t n) {
    Gmap& g = c->gmap;
    if (!g.d_tab) { set_error("map: bshot_gmap_create first"); return BSHOT_E_STATE; }
    BSHOT_TRY(gmap_reset(c));
    if (n > g.max_entries) {
        BSHOT_CUDA_TRY(cudaStreamSynchronize(c->stream));
        set_error("bshot_gmap_import: %zu entries > max_entries %u", n, g.max_entries);
        return BSHOT_E_CAPACITY;
    }
    if (n == 0) { BSHOT_CUDA_TRY(cudaStreamSynchronize(c->stream)); return BSHOT_OK; }
    BSHOT_CUDA_TRY(cudaMemcpyAsync(g.d_epos, xyzr, sizeof(float4) * n, cudaMemcpyHostToDevice, c->stream));
    BSHOT_CUDA_TRY(cudaMemcpyAsync(g.d_edesc, desc, 48 * n, cudaMemcpyHostToDevice, c->stream));
    const int rc = gmap_import_dev(c, g.d_epos, g.d_edesc, nullptr, n, nullptr, "bshot_gmap_import");
    if (rc == BSHOT_E_INVALID || rc == BSHOT_E_CAPACITY) {   // an empty map
        BSHOT_TRY(gmap_reset(c));
        BSHOT_CUDA_TRY(cudaStreamSynchronize(c->stream));
        return rc;
    }
    BSHOT_TRY(rc);
    gmap_record_update(c, n, /*by_scan=*/false);   // update 0
    return BSHOT_OK;
}

// re-anchor (bshot_gmap_reanchor): the whole map in map order with its tags, every entry moved by the correction of the
// update that wrote it into the entry pool, and the table rebuilt from there in that order.  When the moved map does not
// fit, the table is rebuilt from the untouched gather buffers: export order makes that the map as it was.  Then the trajectory
// becomes poses3x4 and the pose d_pose (16 floats) the one reanchor_corrections derived
int gmap_reanchor(Ctx* c, const float* poses3x4, size_t n, float* d_pose, float* pose_out) {
    Gmap& g = c->gmap;
    if (n) {
        if (g.rcap < n) {   // sized like the trajectory, which grows by doubling
            const size_t cap = std::max<size_t>(g.traj_cap, n);
            void* old[] = {g.d_rtraj, g.d_rcorr, g.d_rchg};
            for (void* p : old) if (p) cudaFree(p);
            g.d_rtraj = g.d_rcorr = nullptr;
            g.d_rchg = nullptr;
            g.rcap = 0;
            BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_rtraj, sizeof(float) * 12 * cap));
            BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_rcorr, sizeof(float) * (12 * cap + 16)));
            BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_rchg, sizeof(unsigned) * (cap + 1)));
            g.rcap = cap;
        }
        float* d_pose_new = g.d_rcorr + 12 * g.rcap;
        unsigned* d_count = g.d_rchg + g.rcap;
        BSHOT_CUDA_TRY(cudaMemcpyAsync(g.d_rtraj, poses3x4, sizeof(float) * 12 * n, cudaMemcpyHostToDevice, c->stream));
        BSHOT_TRY(reanchor_corrections(c, g.d_traj, g.d_rtraj, (unsigned)n, g.d_rcorr, g.d_rchg, d_pose, d_pose_new));
        size_t nt_cap;
        BSHOT_TRY(gmap_gather_all(c, &nt_cap, /*with_tags=*/true));
        if (nt_cap) {
            const unsigned nn = (unsigned)nt_cap;
            gm_reanchor_move_kernel<<<(nn + 255) / 256, 256, 0, c->stream>>>(g.d_apos, g.d_adesc, g.d_atag, g.d_actl + 1, nn, g.d_rcorr, g.d_rchg, (unsigned)n,
                                                                              g.d_epos, g.d_edesc, d_count);
            count_launch(c);
            BSHOT_TRY(check_launch("gm_reanchor_move_kernel"));
            const int rc = gmap_import_dev(c, g.d_epos, g.d_edesc, g.d_atag, nt_cap, d_count, "bshot_gmap_reanchor");
            if (rc == BSHOT_E_INVALID || rc == BSHOT_E_CAPACITY) {
                BSHOT_TRY(gmap_import_dev(c, g.d_apos, g.d_adesc, g.d_atag, nt_cap, d_count, "bshot_gmap_reanchor (restoring the map)"));
                if (rc == BSHOT_E_INVALID) set_error("bshot_gmap_reanchor: a moved entry is not finite or beyond +-2.1e9 mm; nothing changed");
                else set_error("bshot_gmap_reanchor: the moved map needs more blocks or chunks than the map holds (%u slots, %u chunks); nothing changed",
                               g.tab_cap, g.max_chunks);
                return rc;
            }
            BSHOT_TRY(rc);
        }
        BSHOT_CUDA_TRY(cudaMemcpyAsync(g.d_traj, g.d_rtraj, sizeof(float) * 12 * n, cudaMemcpyDeviceToDevice, c->stream));
        BSHOT_CUDA_TRY(cudaMemcpyAsync(d_pose, d_pose_new, sizeof(float) * 16, cudaMemcpyDeviceToDevice, c->stream));
    }
    if (pose_out) BSHOT_CUDA_TRY(cudaMemcpyAsync(pose_out, d_pose, sizeof(float) * 16, cudaMemcpyDeviceToHost, c->stream));
    BSHOT_CUDA_TRY(cudaStreamSynchronize(c->stream));
    return BSHOT_OK;
}

// ---- loop closure: entry tags, trajectory, candidate selection (loop_run, odometry.cu) ----------------------------------
int gmap_scans(Ctx* c, uint32_t* entry_scan_out, size_t entry_cap, float* poses3x4_out, size_t pose_cap, size_t* n_entries_out, size_t* n_scans_out) {
    Gmap& g = c->gmap;
    size_t n = 0;
    if (entry_scan_out || n_entries_out) {   // the tags need the whole-map gather; the trajectory alone does not
        size_t nt_cap;
        BSHOT_TRY(gmap_gather_all(c, &nt_cap, /*with_tags=*/true));
        unsigned* h = reinterpret_cast<unsigned*>(&c->h_scratch[48]);
        BSHOT_CUDA_TRY(cudaMemcpyAsync(h, g.d_actl, sizeof(unsigned) * 4, cudaMemcpyDeviceToHost, c->stream));
        BSHOT_CUDA_TRY(cudaStreamSynchronize(c->stream));
        n = h[1];
    }
    const size_t m = std::min(n, entry_cap), ns = g.n_updates, ms = std::min(ns, pose_cap);
    if (n_entries_out) *n_entries_out = n;
    if (n_scans_out) *n_scans_out = ns;
    if (entry_scan_out && m) BSHOT_CUDA_TRY(cudaMemcpyAsync(entry_scan_out, g.d_atag, sizeof(unsigned) * m, cudaMemcpyDeviceToHost, c->stream));
    if (poses3x4_out && ms) BSHOT_CUDA_TRY(cudaMemcpyAsync(poses3x4_out, g.d_traj, sizeof(float) * 12 * ms, cudaMemcpyDeviceToHost, c->stream));
    BSHOT_CUDA_TRY(cudaStreamSynchronize(c->stream));
    if ((entry_scan_out && n > entry_cap) || (poses3x4_out && ns > pose_cap)) {
        set_error("bshot_gmap_scans: %zu entries / %zu scans > capacities %zu / %zu", n, ns, entry_cap, pose_cap);
        return BSHOT_E_CAPACITY;
    }
    return BSHOT_OK;
}

// A stable selection of *d_n entries in three launches: count per 1024-entry tile, one CTA scans the tile counts, each tile
// writes its selected entries at its offset in their order.  mode 0 keeps the loop candidates (tag + min_gap <= scan),
// mode 1 the entries whose block lattice coordinates lie in the +-range cube around the translation of the device pose T
// (gmap_gather's block test).  ctl_out[0] = min(selected, out_cap), ctl_out[1] = selected; with err, more than out_cap
// selected sets *err = BSHOT_E_CAPACITY
struct GmSelect { int mode; unsigned scan, min_gap; const float* T; float range; };

__device__ __forceinline__ bool gm_selected(const GmSelect& s, const float4* __restrict__ pos, const unsigned* __restrict__ tag, unsigned e) {
    if (s.mode == 0) return (unsigned long long)tag[e] + s.min_gap <= s.scan;
    const GmapCube cube = gm_cube(s.T[3], s.T[7], s.T[11], s.range);
    if (cube.nx <= 0 || cube.ny <= 0 || cube.nz <= 0) return false;   // a non-finite pose selects nothing
    const float4 p = pos[e];
    const int bx = (int)roundf(p.x / (float)GM_PREC), by = (int)roundf(p.y / (float)GM_PREC), bz = (int)roundf(p.z / (float)GM_PREC);
    return bx >= cube.x0 && bx < cube.x0 + cube.nx && by >= cube.y0 && by < cube.y0 + cube.ny && bz >= cube.z0 && bz < cube.z0 + cube.nz;
}

__global__ void __launch_bounds__(1024)
gm_select_count_kernel(GmSelect s, const float4* __restrict__ pos, const unsigned* __restrict__ tag, const unsigned* __restrict__ d_n, unsigned* __restrict__ tile_cnt) {
    const unsigned e = blockIdx.x * 1024u + threadIdx.x;
    const unsigned n = *d_n;
    if (blockIdx.x * 1024u >= n) return;   // the whole tile is past the count
    const int cnt = __syncthreads_count(e < n && gm_selected(s, pos, tag, e));
    if (threadIdx.x == 0) tile_cnt[blockIdx.x] = (unsigned)cnt;
}

__global__ void __launch_bounds__(1024)
gm_select_scan_kernel(const unsigned* __restrict__ d_n, const unsigned* __restrict__ tile_cnt, unsigned* __restrict__ tile_off, unsigned* __restrict__ ctl_out,
                      unsigned out_cap, int* err) {
    __shared__ unsigned ws[32];
    __shared__ unsigned carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const unsigned nt = (*d_n + 1023u) / 1024u;
    for (unsigned base = 0; base < nt; base += 1024) {
        const unsigned t = base + threadIdx.x;
        const unsigned excl = cta_scan_1024(t < nt ? tile_cnt[t] : 0u, ws, &carry);
        if (t < nt) tile_off[t] = excl;
    }
    if (threadIdx.x == 0) {
        ctl_out[0] = min(carry, out_cap);
        ctl_out[1] = carry;
        if (err && carry > out_cap) *err = BSHOT_E_CAPACITY;
    }
}

__global__ void __launch_bounds__(1024)
gm_select_scatter_kernel(GmSelect s, const float4* __restrict__ pos, const uint64_t* __restrict__ desc, const unsigned* __restrict__ tag,
                         const unsigned* __restrict__ d_n, const unsigned* __restrict__ tile_off, float4* __restrict__ out_pos, uint64_t* __restrict__ out_desc,
                         unsigned* __restrict__ out_tag, unsigned out_cap) {
    __shared__ unsigned wcnt[32];
    const unsigned e = blockIdx.x * 1024u + threadIdx.x, lane = threadIdx.x & 31u, wid = threadIdx.x >> 5;
    const unsigned n = *d_n;
    if (blockIdx.x * 1024u >= n) return;
    const bool sel = e < n && gm_selected(s, pos, tag, e);
    const unsigned m = __ballot_sync(0xffffffffu, sel);
    if (lane == 0) wcnt[wid] = __popc(m);
    __syncthreads();
    if (!sel) return;
    unsigned o = tile_off[blockIdx.x] + __popc(m & ((1u << lane) - 1u));
    for (unsigned w = 0; w < wid; ++w) o += wcnt[w];
    if (o >= out_cap) return;
    out_pos[o] = pos[e];
    if (out_tag) out_tag[o] = tag[e];
    if (out_desc)
#pragma unroll
        for (int k = 0; k < 6; ++k) out_desc[(size_t)o * 6 + k] = desc[(size_t)e * 6 + k];
}

static int gm_select(Ctx* c, const GmSelect& s, const float4* pos, const uint64_t* desc, const unsigned* tag, const unsigned* d_n, size_t n_cap, float4* out_pos,
                     uint64_t* out_desc, unsigned* out_tag, unsigned out_cap, unsigned* ctl_out, int* err) {
    Gmap& g = c->gmap;
    if (n_cap == 0) {
        BSHOT_CUDA_TRY(cudaMemsetAsync(ctl_out, 0, sizeof(unsigned) * 2, c->stream));
        return BSHOT_OK;
    }
    const unsigned tiles = (unsigned)((n_cap + 1023) / 1024);
    gm_select_count_kernel<<<tiles, 1024, 0, c->stream>>>(s, pos, tag, d_n, g.d_ltile);
    gm_select_scan_kernel<<<1, 1024, 0, c->stream>>>(d_n, g.d_ltile, g.d_ltile + g.ltile_cap, ctl_out, out_cap, err);
    gm_select_scatter_kernel<<<tiles, 1024, 0, c->stream>>>(s, pos, desc, tag, d_n, g.d_ltile + g.ltile_cap, out_pos, out_desc, out_tag, out_cap);
    count_launch(c, 3);
    return check_launch("map selection kernels");
}

int gmap_loop_candidates(Ctx* c, unsigned scan, unsigned min_gap, size_t* nc_cap_out) {
    Gmap& g = c->gmap;
    if (!g.d_lpos) {
        g.ltile_cap = (g.max_entries + 1023) / 1024;
        BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_lpos, sizeof(float4) * g.max_entries));
        BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_ldesc, 48 * (size_t)g.max_entries));
        BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_ltag, sizeof(unsigned) * g.max_entries));
        BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_ltile, sizeof(unsigned) * 2 * g.ltile_cap));
        BSHOT_CUDA_TRY(cudaMalloc((void**)&g.d_lctl, sizeof(unsigned) * 4));
    }
    size_t nm_cap = 0;
    // no entry can be min_gap updates older than the scan: nothing to gather
    if ((unsigned long long)scan >= min_gap) BSHOT_TRY(gmap_gather_all(c, &nm_cap, /*with_tags=*/true));
    *nc_cap_out = nm_cap;
    const GmSelect s = {0, scan, min_gap, nullptr, 0.0f};
    return gm_select(c, s, g.d_apos, g.d_adesc, g.d_atag, g.d_actl + 1, nm_cap, g.d_lpos, g.d_ldesc, g.d_ltag, g.max_entries, g.d_lctl, nullptr);
}

int gmap_loop_icp_targets(Ctx* c, const float* d_T, float range, size_t nc_cap, int* d_err) {
    Gmap& g = c->gmap;
    const GmSelect s = {1, 0u, 0u, d_T, range};
    return gm_select(c, s, g.d_lpos, nullptr, nullptr, g.d_lctl, nc_cap, g.d_tpos, nullptr, nullptr, (unsigned)c->max_targets, g.d_lctl + 2, d_err);
}

}  // namespace bshot
