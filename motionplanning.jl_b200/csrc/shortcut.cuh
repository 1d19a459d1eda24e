// shortcut.cuh -- what the two phases of mpb200_shortcut_paths share (specification in include/mpb200.h and DESIGN.md
// section 10c): the per-path descriptor in device scratch and the lookup from a global node (= visibility row) to its path.
#pragma once
#include "common.cuh"

namespace mpb {

// Path q of a call: its nodes are global nodes node0 .. node0 + M - 1 (nodes, best, pred and the output rows are indexed
// by global node); its input states start at row y0 of the uploaded states; row b of its visibility bits holds the words
// bits + bit0 + b * words (bit a = free(a, b), words = ceil(M / 32)).  Entry npaths is a sentinel with node0 = total nodes.
struct ShortcutPath {
    int64_t node0, y0, bit0;
    int32_t M, L, words, pad;
};
// Per-path results, read back in one copy: the output length and cost, and the segment tests of the visibility pass
// (zeroed by the node kernel, summed with one atomicAdd per warp and path).
struct ShortcutResult {
    long long len;
    double cost;
    unsigned long long checks;
};

// the path holding global node g (paths[0].node0 = 0 <= g < paths[npaths].node0)
__device__ __forceinline__ int shortcut_path_of(const ShortcutPath *__restrict__ paths, int npaths, int64_t g) {
    int lo = 0, hi = npaths - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (paths[mid].node0 <= g) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

// phase 1 (collide.cu): argument checks of the space / obstacle pair, then the visibility pass
int shortcut_check_space(const mpb200_obstacles *o, const mpb200_space_desc *ss, int d);
int shortcut_visibility_device(const ShortcutPath *paths, int npaths, int64_t nodes_total, const double *nodes, int d,
                               const mpb200_obstacles *o, const mpb200_space_desc *ss, uint32_t *bits,
                               ShortcutResult *results);

}  // namespace mpb
