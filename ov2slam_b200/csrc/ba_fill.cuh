// Tile-level symbolic Cholesky of the reduced camera system of a large local-BA window (ba_large.cu).
//
// The reduced system S (n = 6 x optimised keyframes, keyframes in trajectory order) is stored as the upper triangle of a
// dense n x n array cut into TILE x TILE tiles.  Keyframe pair (lo, hi) is a 6 x 6 block of S when a landmark touches
// both (anchor x observer, observer x observer); over a trajectory that is a band plus the loop-closure blocks.  The
// factorisation A = U'U only ever reads and writes the tiles U can make non-zero; this header finds them: the tiles the
// keyframe blocks cover, closed under the right-looking update (tile (i, j) is filled when some earlier tile row k holds
// both (k, i) and (k, j)).  Host-only code, compiled into the library and, on its own, by tests/test_ba_large_fill.py.
#pragma once
#include <stdint.h>
#include <vector>

namespace bafill {

constexpr int TILE = 32;

// Marks the tiles (row <= column) covered by the 6 x 6 block of keyframe slots lo <= hi.  T: nt x nt, row-major.
inline void mark_block(int nt, uint8_t* T, int lo, int hi) {
    const int r0 = 6 * lo / TILE, r1 = (6 * lo + 5) / TILE, c0 = 6 * hi / TILE, c1 = (6 * hi + 5) / TILE;
    for (int r = r0; r <= r1; ++r)
        for (int c = c0; c <= c1; ++c)
            if (r <= c) T[(size_t)r * nt + c] = 1;
}

// Right-looking symbolic Cholesky on the tile pattern T (upper triangle used, diagonal always kept): on return T holds
// every tile of U that can be non-zero.
inline void symbolic_fill(int nt, uint8_t* T) {
    std::vector<int> row;
    for (int k = 0; k < nt; ++k) {
        T[(size_t)k * nt + k] = 1;
        row.clear();
        for (int j = k + 1; j < nt; ++j)
            if (T[(size_t)k * nt + j]) row.push_back(j);
        for (size_t a = 0; a < row.size(); ++a)
            for (size_t b = a; b < row.size(); ++b) T[(size_t)row[a] * nt + row[b]] = 1;
    }
}

}  // namespace bafill
