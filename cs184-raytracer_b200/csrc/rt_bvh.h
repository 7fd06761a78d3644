// rt_bvh.h — LBVH build entry point (see rt_bvh.cu).
#pragma once
#include "rt_device.cuh"

namespace rt {

// Bump allocator over one persistent device buffer: scene uploads and LBVH builds take their
// temporaries from it, so a steady-state rt_scene_upload performs no cudaMalloc/cudaFree
// (both are synchronising and, right after another process released memory, very slow).
struct DeviceArena {
    char* base = nullptr;
    size_t cap = 0, used = 0;
    ~DeviceArena() { if (base) cudaFree(base); }
    cudaError_t reserve(size_t bytes) {      // call with the arena empty
        used = 0;
        if (bytes <= cap) return cudaSuccess;
        if (base) cudaFree(base);
        base = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&base, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    template <typename T>
    T* take(size_t count) {
        size_t bytes = (count * sizeof(T) + 255) & ~(size_t)255;
        if (used + bytes > cap) return nullptr;
        T* p = reinterpret_cast<T*>(base + used);
        used += bytes;
        return p;
    }
    void reset() { used = 0; }
    static size_t padded(size_t bytes) { return (bytes + 255) & ~(size_t)255; }
};

// scratch bytes build_lbvh takes from the arena for n primitives
inline size_t lbvh_scratch_bytes(size_t n) {
    return 4 * DeviceArena::padded(12 * n) + 12 * DeviceArena::padded(4 * n) + 2 * DeviceArena::padded(16 * n) + DeviceArena::padded(4 * 256 * 4097 /* radix-sort histograms, SORT_MAX_BLOCKS + 1 */) + 4096;
}

// Builds one LBVH per primitive group over the n primitive codes in d_codes (device;
// group_first_code[g] = first code of group g, all the host side needs to know), groups being consecutive ranges of sizes group_sizes[0..ngroups), and
// joins them under super nodes so that node 0 is always the root, written to `nodes`
// (caller-allocated).  n < 2 builds nothing (*out_count = 0).  Temporaries come from `arena`.  extra_abs: largest |coordinate| of ray origins outside the
// primitives (the camera eye) and of the primitives kept OUT of the LBVH (flat list), folded into the box padding.
// node_level (device, one int per node slot) receives the wide level of every node, root or super node = 0, and -1
// for slots that hold no node; *out_levels the number of levels.  Both are what refit_lbvh needs.
// Returns RT_OK, RT_ERR_CUDA or RT_ERR_LIMIT (too many nodes / tree deeper than the traversal stack).
int build_lbvh(const DScene& S, const int* d_codes, const int* group_first_code, int n, const int* group_sizes, int ngroups,
               float extra_abs, cudaStream_t stream, DeviceArena& arena, BvhNode* nodes /* >= n + ngroups */,
               size_t* out_count, int* launches, char* err, int errlen,
               float* centroid_bounds /* [6] or null: min xyz, max xyz of the primitive centroids */,
               float* out_pad_scale /* or null: the largest |coordinate| the box padding covers */,
               int* node_level /* >= n + ngroups */, int* out_levels);

// Recomputes every box of the node array build_lbvh wrote over the same n primitive codes, whose geometry (S) may
// have changed, and keeps its topology: one bounds pass over d_codes (new M = largest |coordinate|, folded with
// extra_abs as in the build, and the centroid bounds), then one launch per level, deepest first.  The padding is
// the build's, so refitting unchanged primitives rewrites the node array byte for byte.  Takes 24 B per primitive and
// per node from `arena`; synchronises `stream` once, after the bounds pass (M is needed on the host), and leaves the
// level launches enqueued.  Returns RT_OK or RT_ERR_CUDA.
int refit_lbvh(const DScene& S, const int* d_codes, int n, const int* node_level, int levels, size_t node_count,
               float extra_abs, cudaStream_t stream, DeviceArena& arena, BvhNode* nodes, int* launches, char* err,
               int errlen, float* centroid_bounds /* [6] */, float* out_pad_scale);

}  // namespace rt
