// ccu_layout.h - commit-time layout builders (host C++): the value-carrying octree layout, the march ("air") layout and
// the BVH stage layout.  Included by chunkycu.cu only.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <unordered_map>
#include <vector>

#include "ccu_device.cuh"
#include "ccu_march.cuh"

// ------------------------------------------------------------------------------------------------------
// commit-time traversal layout (see DScene::top / DScene::wide)
// ------------------------------------------------------------------------------------------------------
namespace {
struct WideLayout {
    std::vector<unsigned> top, wide;
    int cell_level = 0, top_log2 = 0;
    bool ok = true;
};

inline unsigned wide_leaf(int word, int level, bool &ok) {
    long long v = -(long long)word;
    unsigned val;
    if (v == 0x7FFFFFFELL) val = CCU_WIDE_ANY;
    else if (v >= 0 && v < (long long)CCU_WIDE_ANY) val = (unsigned)v;
    else { ok = false; val = 0; }
    return CCU_WIDE_LEAF | ((unsigned)level << 26) | val;
}

unsigned wide_node(const int *tree, size_t n, int word, int lvl, WideLayout &b) {
    if (lvl < 2 || (size_t)word + 7 >= n) { b.ok = false; return wide_leaf(0, 0, b.ok); }
    const size_t idx = b.wide.size() / 64;
    if (idx >= 0x7FFFFFFFu) { b.ok = false; return wide_leaf(0, 0, b.ok); }
    b.wide.resize(b.wide.size() + 64);
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < 4; j++)
            for (int k = 0; k < 4; k++) {
                unsigned e;
                int c1 = tree[(size_t)word + ((((i >> 1) & 1) << 2) | (((j >> 1) & 1) << 1) | ((k >> 1) & 1))];
                if (c1 <= 0) {
                    e = wide_leaf(c1, lvl - 1, b.ok);
                } else if ((size_t)c1 + 7 >= n) {
                    b.ok = false;
                    e = wide_leaf(0, 0, b.ok);
                } else {
                    int c2 = tree[(size_t)c1 + (((i & 1) << 2) | ((j & 1) << 1) | (k & 1))];
                    e = c2 <= 0 ? wide_leaf(c2, lvl - 2, b.ok) : wide_node(tree, n, c2, lvl - 2, b);
                }
                b.wide[idx * 64 + ((i << 4) | (j << 2) | k)] = e;
            }
    return (unsigned)idx;
}

// "Air layout" for the march loop (ccu_march.cuh): top table over cells of level `cell_level` (>= 4), 64-ary nodes down to
// level 4 for deep worlds, and one 2-KiB brick of 4-bit voxel codes per 16^3 cell that is not a single leaf (in shallow
// worlds the single-leaf cells share one constant brick per leaf level).  The march loop needs nothing else (octree.h:89-106:
// an air leaf is left through its cube, anything else goes to the block test); a leaf lookup is one table load plus at most
// one brick load.
struct AirLayout {
    std::vector<unsigned> top, wide, bricks;
    std::vector<unsigned char> wide_level;     // level of every 64-ary node (its entries sit two levels below)
    int cell_level = 4, top_log2 = 0;
    bool ok = true;
};

constexpr size_t AIR_MAX_BRICKS = 0x400000;   // brick word offsets stay below the leaf bit (CCU_WIDE_LEAF)

// The top table is filled slab by slab (x ranges) on several host threads; every thread appends to vectors of its own, and the
// indices it handed out are shifted by the sizes of the slabs before it when the parts are joined.
inline int layout_threads(int dim) {
    if (dim < 8) return 1;
    if (const char *e = getenv("CCU_COMMIT_THREADS")) return std::max(1, std::min(dim, atoi(e)));
    const unsigned hw = std::thread::hardware_concurrency();
    return (int)std::max(1u, std::min({hw ? hw : 4u, (unsigned)dim, 16u}));
}

inline unsigned air_leaf(int word, int level) { return CCU_WIDE_LEAF | ((word == 0 ? (unsigned)level : 31u) << 26); }
inline int oct_child(int x, int y, int z) { return ((x & 1) << 2) | ((y & 1) << 1) | (z & 1); }

// brick code of a leaf word (octree.h: 0 = air) of the given level
inline unsigned air_code(int word, int level) { return word == 0 ? (unsigned)level : (unsigned)CCU_AIR_SOLID; }
inline void air_brick_set(unsigned *brick, int x, int y, int z, unsigned code) {
    brick[ccu::air_brick_word(x, y, z)] |= code << ((z & 7) * 4);
}

// brick of the 16^3 cell rooted at the branch node `word` (level 4); returns its word offset
unsigned air_brick(const int *tree, size_t n, int word, AirLayout &b) {
    const size_t idx = b.bricks.size() / CCU_BRICK_WORDS;
    if (idx >= AIR_MAX_BRICKS || (size_t)word + 7 >= n) { b.ok = false; return air_leaf(1, 0); }
    b.bricks.resize(b.bricks.size() + CCU_BRICK_WORDS, 0u);
    unsigned *brick = &b.bricks[idx * CCU_BRICK_WORDS];
    // descend level 3 .. 0 and write the code of the leaf every voxel lies in
    for (int x = 0; x < 16; x++)
        for (int y = 0; y < 16; y++)
            for (int z = 0; z < 16; z++) {
                int level = 4, w = word;
                while (w > 0 && level > 0) {
                    if ((size_t)w + 7 >= n) { b.ok = false; w = -1; break; }
                    level--;
                    w = tree[(size_t)w + oct_child(x >> level, y >> level, z >> level)];
                }
                if (w > 0) { b.ok = false; w = -1; }                  // deeper than the declared depth
                air_brick_set(brick, x, y, z, air_code(w, level));
            }
    return (unsigned)(idx * CCU_BRICK_WORDS);
}

// word offset of the constant brick of a leaf (every voxel has its code), added on first use
unsigned air_const_brick(AirLayout &b, std::vector<unsigned> &made, unsigned code) {
    if (made[code] == ~0u) {
        made[code] = (unsigned)b.bricks.size();
        b.bricks.resize(b.bricks.size() + CCU_BRICK_WORDS, code * 0x11111111u);
    }
    return made[code];
}

unsigned air_node(const int *tree, size_t n, int word, int lvl, AirLayout &b) {
    if (lvl == 4) return air_brick(tree, n, word, b);
    if (lvl < 6 || (size_t)word + 7 >= n) { b.ok = false; return air_leaf(1, 0); }
    const size_t idx = b.wide.size() / 64;
    if (idx >= 0x1FFFFFFu) { b.ok = false; return air_leaf(1, 0); }
    b.wide.resize(b.wide.size() + 64);
    b.wide_level.push_back((unsigned char)lvl);
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < 4; j++)
            for (int k = 0; k < 4; k++) {
                unsigned e;
                const int c1 = tree[(size_t)word + oct_child(i >> 1, j >> 1, k >> 1)];
                if (c1 <= 0) {
                    e = air_leaf(c1, lvl - 1);
                } else if ((size_t)c1 + 7 >= n) {
                    b.ok = false;
                    e = air_leaf(1, 0);
                } else {
                    const int c2 = tree[(size_t)c1 + oct_child(i, j, k)];
                    e = c2 <= 0 ? air_leaf(c2, lvl - 2) : air_node(tree, n, c2, lvl - 2, b);
                }
                b.wide[idx * 64 + ((i << 4) | (j << 2) | k)] = e;
            }
    return (unsigned)idx;
}

// Octrees shallower than a brick (depth < 4): one brick whose corner [0, 2^depth)^3 holds the tree, filled voxel by voxel
// from the root descent (octree.h:81-88); the march loop never looks outside the cube (bounds check octree.h:76-78).
void air_small_brick(const int *tree, size_t n, int depth, AirLayout &b) {
    b.bricks.assign(CCU_BRICK_WORDS, 0u);
    const int size = 1 << depth;
    for (int x = 0; x < 16; x++)
        for (int y = 0; y < 16; y++)
            for (int z = 0; z < 16; z++) {
                int level = depth, word = tree[0];
                if (x >= size || y >= size || z >= size) word = -1;
                while (word > 0 && level > 0) {
                    level--;
                    const size_t at = (size_t)word + oct_child(x >> level, y >> level, z >> level);
                    if (at >= n) { b.ok = false; word = -1; break; }
                    word = tree[at];
                }
                if (word > 0) { b.ok = false; word = -1; }
                air_brick_set(b.bricks.data(), x, y, z, air_code(word, level));
            }
}

// cells [x0, x1) of the top table, into `b` (indices local to b)
inline void air_fill_slab(const int *tree, size_t n, int depth, int cl, int dim, int x0, int x1, unsigned *top, AirLayout &b) {
    for (int x = x0; x < x1 && b.ok; x++)
        for (int y = 0; y < dim; y++)
            for (int z = 0; z < dim; z++) {
                int level = depth;
                int word = tree[0];
                while (word > 0 && level > cl) {
                    level--;
                    const int sh = level - cl;
                    const size_t at = (size_t)word + oct_child(x >> sh, y >> sh, z >> sh);
                    if (at >= n) { b.ok = false; word = 0; break; }
                    word = tree[at];
                }
                top[((size_t)x * dim + y) * dim + z] = word <= 0 ? air_leaf(word, level) : air_node(tree, n, word, cl, b);
            }
}

AirLayout build_air_layout(const int *tree, size_t n, int depth) {
    AirLayout b;
    if (depth < 4) {
        b.cell_level = 4;
        b.top_log2 = 0;
        if (tree[0] <= 0) b.top.assign(1, air_leaf(tree[0], depth));
        else { b.top.assign(1, 0u); air_small_brick(tree, n, depth, b); }
    } else {
        int cl = std::max(depth - 7, 4);             // top table of at most 128^3 cells
        if (cl & 1) cl++;
        if (cl > depth) cl = depth & ~1;
        b.cell_level = cl;
        b.top_log2 = depth - cl;
        const int dim = 1 << b.top_log2;
        b.top.assign((size_t)dim * dim * dim, 0u);
        const int nt = layout_threads(dim);
        if (nt == 1) {
            air_fill_slab(tree, n, depth, cl, dim, 0, dim, b.top.data(), b);
        } else {
            std::vector<AirLayout> part(nt);
            std::vector<std::thread> th;
            for (int t = 0; t < nt; t++)
                th.emplace_back([&, t] { air_fill_slab(tree, n, depth, cl, dim, dim * t / nt, dim * (t + 1) / nt, b.top.data(), part[t]); });
            for (auto &t : th) t.join();
            for (int t = 0; t < nt; t++) {
                const unsigned wide_off = (unsigned)(b.wide.size() / 64), brick_off = (unsigned)(b.bricks.size() / CCU_BRICK_WORDS);
                AirLayout &p = part[t];
                b.ok = b.ok && p.ok;
                // entries below the leaf bit are indices: of bricks where they sit at level 4, of 64-ary nodes above that
                for (size_t j = 0; j < p.wide_level.size(); j++) {
                    const unsigned off = p.wide_level[j] - 2 == 4 ? brick_off * CCU_BRICK_WORDS : wide_off;
                    for (int e = 0; e < 64; e++)
                        if (!(p.wide[j * 64 + e] & CCU_WIDE_LEAF)) p.wide[j * 64 + e] += off;
                }
                const unsigned top_off = cl == 4 ? brick_off * CCU_BRICK_WORDS : wide_off;
                const size_t c0 = (size_t)(dim * t / nt) * dim * dim, c1 = (size_t)(dim * (t + 1) / nt) * dim * dim;
                for (size_t c = c0; c < c1; c++)
                    if (!(b.top[c] & CCU_WIDE_LEAF)) b.top[c] += top_off;
                b.wide.insert(b.wide.end(), p.wide.begin(), p.wide.end());
                b.wide_level.insert(b.wide_level.end(), p.wide_level.begin(), p.wide_level.end());
                b.bricks.insert(b.bricks.end(), p.bricks.begin(), p.bricks.end());
            }
            if (b.wide.size() / 64 >= 0x1FFFFFFu || b.bricks.size() / CCU_BRICK_WORDS >= AIR_MAX_BRICKS) b.ok = false;
        }
    }
    if (b.cell_level == 4 && b.top_log2 < 4) {
        // a smaller world's table is padded to 16^3 cells, which the wavefront kernel's march step indexes with immediate
        // shifts (the padding cells, not air, are never looked up for a voxel inside the octree cube)
        const int dim = 1 << b.top_log2;
        std::vector<unsigned> t((size_t)16 * 16 * 16, air_leaf(1, 0));
        for (int x = 0; x < dim; x++)
            for (int y = 0; y < dim; y++)
                for (int z = 0; z < dim; z++) t[(size_t)((x << 8) | (y << 4) | z)] = b.top[((size_t)x * dim + y) * dim + z];
        b.top.swap(t);
        b.top_log2 = 4;
    }
    if (b.cell_level == 4) {
        // shallow worlds: the cells that are one leaf refer to the constant brick of that leaf
        std::vector<unsigned> made(16, ~0u);
        for (unsigned &e : b.top)
            if (e & CCU_WIDE_LEAF) {
                const unsigned level = (e >> 26) & 31u;
                e = air_const_brick(b, made, level == 31 ? (unsigned)CCU_AIR_SOLID : level);
            }
        if (b.bricks.size() / CCU_BRICK_WORDS >= AIR_MAX_BRICKS) b.ok = false;
    }
    if (b.wide.empty()) b.wide.assign(64, air_leaf(1, 0));
    if (b.bricks.empty()) b.bricks.assign(CCU_BRICK_WORDS, CCU_AIR_SOLID * 0x11111111u);
    return b;
}

// Traversal layout of a packed BVH (PackedBvhNode.java:22-31: 7 ints per node, first child at node + 7, second child at
// node[0]) for the BVH stage of ccu_queue.cuh: one 64-byte record per inner node holding BOTH children's boxes
// (bvh.h:73-91 fetches exactly those at every inner node) and a reference per child, and 16-byte aligned triangle
// blocks.  ref >= 0: record index; ref < 0: leaf, -(1 + offset of its block in `tris`, in units of 8 words).
struct BvhLayout {
    std::vector<int> rec;
    int root = 0;
    bool ok = true;
};
// Both entity BVHs, which share the triangle blocks (build_bvh_stage).
struct BvhStage {
    BvhLayout world, actor;
    std::vector<int> tris;                       // per leaf: {count, 0 x 7} + count x (20 words (PackedTriangle.java:46-78) + 4 pad)
    std::unordered_map<int, int> leaf_at;        // palette offset -> block: a leaf both BVHs reference is stored once
    bool ok = true;
    // block of the leaf at triangle-palette offset `prim`, in units of 32 bytes
    int leaf(const std::vector<int> &trigs, int prim, bool &valid) {
        auto [at, fresh] = leaf_at.try_emplace(prim, 0);
        if (!fresh) return at->second;
        if (prim < 0 || (size_t)prim >= trigs.size()) { valid = false; return 0; }
        const int count = trigs[(size_t)prim];
        if (count < 0 || (size_t)prim + 1 + (size_t)count * 20 > trigs.size()) { valid = false; return 0; }
        at->second = (int)(tris.size() / 8);
        tris.push_back(count);
        tris.insert(tris.end(), 7, 0);
        for (int i = 0; i < count; i++) {
            tris.insert(tris.end(), trigs.begin() + prim + 1 + (size_t)i * 20, trigs.begin() + prim + 1 + (size_t)(i + 1) * 20);
            tris.insert(tris.end(), 4, 0);
        }
        return at->second;
    }
};

int bvh_ref(const std::vector<int> &bvh, const std::vector<int> &trigs, size_t node, int depth, BvhLayout &b, BvhStage &s) {
    if (!b.ok) return -1;
    // deeper than the traversal stack of the reference (int nodesToVisit[64], bvh.h:38): undefined there, refused here
    if (node + 6 >= bvh.size() || depth >= 64) { b.ok = false; return -1; }
    const int head = bvh[node];
    if (head <= 0) return -(1 + s.leaf(trigs, -head, b.ok));
    const size_t left = node + 7, right = (size_t)head;
    if (left + 6 >= bvh.size() || right + 6 >= bvh.size()) { b.ok = false; return -1; }
    const size_t r = b.rec.size() / 16;
    b.rec.resize(b.rec.size() + 16, 0);
    // two 32-byte halves of the same shape: {box (6 floats), ref, 0} of the first child, then of the second child
    for (int i = 0; i < 6; i++) {
        b.rec[r * 16 + i] = bvh[left + 1 + i];
        b.rec[r * 16 + 8 + i] = bvh[right + 1 + i];
    }
    const int rl = bvh_ref(bvh, trigs, left, depth + 1, b, s);
    const int rr = bvh_ref(bvh, trigs, right, depth + 1, b, s);
    b.rec[r * 16 + 6] = rl;
    b.rec[r * 16 + 14] = rr;
    return (int)r;
}

inline bool bvh_is_empty(const std::vector<int> &bvh) {   // bvh.h:23-32
    if (bvh.size() < 7) return true;
    if (bvh[0] != 0) return false;
    for (int i = 1; i < 7; i++) {
        float f;
        memcpy(&f, &bvh[i], 4);
        if (!std::isnan(f)) return false;
    }
    return true;
}

// The BVH stage layout of the world and actor BVHs.  When either cannot be held (malformed, or deeper than the 64 entries of
// the reference's traversal stack, bvh.h:38), ok is false and the records and triangle blocks are empty.
inline BvhStage build_bvh_stage(const std::vector<int> &world, const std::vector<int> &actor, const std::vector<int> &trigs) {
    BvhStage s;
    if (!bvh_is_empty(world)) s.world.root = bvh_ref(world, trigs, 0, 0, s.world, s);
    if (!bvh_is_empty(actor)) s.actor.root = bvh_ref(actor, trigs, 0, 0, s.actor, s);
    s.ok = s.world.ok && s.actor.ok;
    if (!s.ok) { s.world.rec.clear(); s.actor.rec.clear(); s.tris.clear(); }
    s.tris.insert(s.tris.end(), 8, 0);      // the leaf stage reads the 32 bytes behind a count word before it looks at the count
    return s;
}

inline void wide_fill_slab(const int *tree, size_t n, int depth, int cl, int dim, int x0, int x1, unsigned *top, WideLayout &b) {
    for (int x = x0; x < x1 && b.ok; x++)
        for (int y = 0; y < dim; y++)
            for (int z = 0; z < dim; z++) {
                int level = depth;
                int word = tree[0];
                while (word > 0 && level > cl) {
                    level--;
                    int sh = level - cl;
                    size_t at = (size_t)word + ((((x >> sh) & 1) << 2) | (((y >> sh) & 1) << 1) | ((z >> sh) & 1));
                    if (at >= n) { b.ok = false; word = 0; break; }
                    word = tree[at];
                }
                top[((size_t)x * dim + y) * dim + z] = word <= 0 ? wide_leaf(word, level, b.ok) : wide_node(tree, n, word, cl, b);
            }
}

WideLayout build_wide_layout(const int *tree, size_t n, int depth) {
    WideLayout b;
    int cl = std::max(depth - 7, 4);
    if (const char *e = getenv("CCU_CELL_LEVEL")) cl = std::max(0, atoi(e));   // tuning knob: level of the top table's cells
    if (cl & 1) cl++;
    if (cl > depth) cl = depth & ~1;
    b.cell_level = cl;
    b.top_log2 = depth - cl;
    const int dim = 1 << b.top_log2;
    b.top.assign((size_t)dim * dim * dim, 0u);
    const int nt = layout_threads(dim);
    if (nt == 1) {
        wide_fill_slab(tree, n, depth, cl, dim, 0, dim, b.top.data(), b);
    } else {
        std::vector<WideLayout> part(nt);
        std::vector<std::thread> th;
        for (int t = 0; t < nt; t++)
            th.emplace_back([&, t] { wide_fill_slab(tree, n, depth, cl, dim, dim * t / nt, dim * (t + 1) / nt, b.top.data(), part[t]); });
        for (auto &t : th) t.join();
        for (int t = 0; t < nt; t++) {
            const unsigned off = (unsigned)(b.wide.size() / 64);
            WideLayout &p = part[t];
            b.ok = b.ok && p.ok;
            for (unsigned &e : p.wide)
                if (!(e & CCU_WIDE_LEAF)) e += off;           // every index refers to a 64-ary node
            const size_t c0 = (size_t)(dim * t / nt) * dim * dim, c1 = (size_t)(dim * (t + 1) / nt) * dim * dim;
            for (size_t c = c0; c < c1; c++)
                if (!(b.top[c] & CCU_WIDE_LEAF)) b.top[c] += off;
            b.wide.insert(b.wide.end(), p.wide.begin(), p.wide.end());
        }
        if (b.wide.size() / 64 >= 0x7FFFFFFFu) b.ok = false;
    }
    if (b.wide.empty()) b.wide.assign(64, wide_leaf(0, 0, b.ok));
    return b;
}

// 16-byte-vectorised palettes (DScene::block_rec / mat_rec / quad_rec / aabb_rec): the reference's scalar int[] palettes
// (PackedBlock.java:79-85, PackedMaterial.java:74-100, PackedQuad.java:41-66, PackedAabb.java:75-102) re-laid out so that a
// block test reads whole records with 128-bit loads.  A block-palette position whose entry cannot be translated (model pointer
// outside its palette) keeps type 0x7FFFFFFF, which no branch of intersect_block accepts - the same miss the reference's
// out-of-range read would most likely produce, but defined.
struct PaletteRecs {
    std::vector<int> block, mat, quad, aabb;
    bool ok = true;
};

inline PaletteRecs build_palette_recs(const std::vector<int> &bp, const std::vector<int> &mp, const std::vector<int> &quads,
                                      const std::vector<int> &aabbs) {
    PaletteRecs r;
    const size_t n_mat = mp.size() / 6;
    r.mat.assign(std::max<size_t>(n_mat, 1) * 8, 0);
    for (size_t i = 0; i < n_mat; i++)
        for (int k = 0; k < 6; k++) r.mat[i * 8 + k] = mp[i * 6 + k];
    std::unordered_map<int, int> quad_at, aabb_at;     // model pointer -> offset in units of 16 bytes
    auto model = [&](const std::vector<int> &src, int ptr, int words, std::vector<int> &dst, std::unordered_map<int, int> &at, int &out) {
        auto it = at.find(ptr);
        if (it != at.end()) { out = it->second; return true; }
        if (ptr < 0 || (size_t)ptr >= src.size()) return false;
        const int count = src[ptr];
        if (count < 0 || (size_t)ptr + 1 + (size_t)count * words > src.size()) return false;
        out = (int)(dst.size() / 4);
        dst.push_back(count); dst.push_back(0); dst.push_back(0); dst.push_back(0);
        for (int i = 0; i < count; i++) {
            for (int k = 0; k < 16; k++) dst.push_back(k < words ? src[(size_t)ptr + 1 + (size_t)i * words + k] : 0);
        }
        at.emplace(ptr, out);
        return true;
    };
    const size_t n_pos = bp.size() >= 2 ? bp.size() - 1 : 0;
    r.block.assign(std::max<size_t>(n_pos, 1) * 8, 0);
    for (size_t b = 0; b < n_pos; b++) {
        int *rec = &r.block[b * 8];
        const int type = bp[b], ptr = bp[b + 1];
        rec[0] = type;
        rec[1] = ptr;
        if (type == 1) {
            // full cube: the six material words travel with the entry
            if (ptr >= 0 && (size_t)ptr + 5 < mp.size()) {
                for (int k = 0; k < 6; k++) rec[2 + k] = mp[(size_t)ptr + k];
            } else {
                rec[0] = 0x7FFFFFFF;
            }
        } else if (type == 2) {
            if (!model(aabbs, ptr, 13, r.aabb, aabb_at, rec[1])) rec[0] = 0x7FFFFFFF;
        } else if (type == 3) {
            if (!model(quads, ptr, 15, r.quad, quad_at, rec[1])) rec[0] = 0x7FFFFFFF;
        }
    }
    if (r.quad.empty()) r.quad.assign(4, 0);
    if (r.aabb.empty()) r.aabb.assign(4, 0);
    return r;
}

// ------------------------------------------------------------------------------------------------------
// emitter table of CCU_RENDER_EMITTER_SAMPLING (DESIGN §10; DScene::emit ...)
// ------------------------------------------------------------------------------------------------------
constexpr int EMIT_SHIFT0 = 3;                  // cells of G = 8 voxels to start with
constexpr long long EMIT_CELL_BUDGET = 1 << 21; // G doubles until the cell box has at most this many cells
constexpr long long EMIT_MAX = 1 << 18;         // a scene with more emitter voxels gets no table (the flag changes nothing)

struct EmitterGrid {
    std::vector<int> emit;        // {x, y, z, block} per emitter, sorted by (x, y, z)
    std::vector<int> off, list;   // CSR cell lists
    int g0[3] = {0, 0, 0}, dim[3] = {0, 0, 0}, shift = EMIT_SHIFT0;
};

// An emitter block: a palette position whose fused record (build_palette_recs) is a full cube whose material has textured
// emittance (flag bit 1) or a non-zero emittance byte.
inline bool block_emits(const std::vector<int> &block_rec, int b) {
    if (b < 0 || (size_t)b * 8 + 7 >= block_rec.size()) return false;
    const int *r = &block_rec[(size_t)b * 8];
    return r[0] == 1 && ((r[2] & 2) || (r[6] & 0xFF));
}

// The emitter primitives of CCU_RENDER_EMITTER_MODELS (DESIGN §12; EmitView::mhead / mprim): per block palette position the
// int4 index of its header in `prim`, or -1 when it is no model emitter.  A model emitter is a quad model with a quad whose
// material emits, or an AABB model with an emitting box face (the material and flags textured_box assigns to it; +z: material
// 0, flags 0; a face with the no-hit bit never emits).  Header {m, bbox (6 float bits: xmin, xmax, ymin, ymax, zmin, zmax of
// the emitting primitives, block-local), 0}, then per primitive, in model order (boxes: faces -x, +x, -y, +y, -z, +z),
// {kind, material, face flags, 13 words}: kind 6 a quad with its 13 geometry / uv words, kind axis * 2 + (1 for +) a box face
// with the box's 6 words.
struct ModelEmitters {
    std::vector<int> head, prim;
    bool any = false;
};

// Whether material pointer p of the raw material palette emits: textured emittance (flag bit 1) or an emittance byte.
inline bool material_emits(const std::vector<int> &mp, int p) {
    return p >= 0 && (size_t)p + 5 < mp.size() && ((mp[(size_t)p] & 2) || (mp[(size_t)p + 4] & 0xFF));
}

inline ModelEmitters build_model_emitters(const PaletteRecs &pr, const std::vector<int> &mp) {
    ModelEmitters me;
    const size_t n_pos = pr.block.size() / 8;
    me.head.assign(n_pos, -1);
    auto as_f = [](int w) { float f; memcpy(&f, &w, 4); return f; };
    auto as_i = [](float f) { int w; memcpy(&w, &f, 4); return w; };
    for (size_t b = 0; b < n_pos; b++) {
        const int type = pr.block[b * 8], ref = pr.block[b * 8 + 1];
        if (type != 2 && type != 3) continue;
        std::vector<int> recs;
        float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
        auto grow = [&](const float *p) {
            for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], p[a]); hi[a] = std::max(hi[a], p[a]); }
        };
        const std::vector<int> &src = type == 2 ? pr.aabb : pr.quad;
        const int count = src[(size_t)ref * 4];
        for (int i = 0; i < count; i++) {
            const int *w = &src[(size_t)(ref + 1 + 4 * i) * 4];
            if (type == 3) {
                if (!material_emits(mp, w[13])) continue;
                recs.push_back(6); recs.push_back(w[13]); recs.push_back(0);
                for (int k = 0; k < 13; k++) recs.push_back(w[k]);
                const float o[3] = {as_f(w[0]), as_f(w[1]), as_f(w[2])}, x[3] = {as_f(w[3]), as_f(w[4]), as_f(w[5])},
                            y[3] = {as_f(w[6]), as_f(w[7]), as_f(w[8])};
                const float ox[3] = {o[0] + x[0], o[1] + x[1], o[2] + x[2]}, oy[3] = {o[0] + y[0], o[1] + y[1], o[2] + y[2]};
                const float oxy[3] = {ox[0] + y[0], ox[1] + y[1], ox[2] + y[2]};
                grow(o); grow(ox); grow(oy); grow(oxy);
                continue;
            }
            const float bx[6] = {as_f(w[0]), as_f(w[1]), as_f(w[2]), as_f(w[3]), as_f(w[4]), as_f(w[5])};
            // faces -x, +x, -y, +y, -z, +z: material word and flag shift of textured_box
            const int mat[6] = {w[10], w[8], w[12], w[11], w[9], 0}, shift[6] = {12, 4, 20, 16, 8, -1};
            for (int f = 0; f < 6; f++) {
                const int fl = shift[f] < 0 ? 0 : (w[6] >> shift[f]) & 15;
                if ((fl & 8) || !material_emits(mp, mat[f])) continue;
                recs.push_back(f); recs.push_back(mat[f]); recs.push_back(fl);
                for (int k = 0; k < 13; k++) recs.push_back(k < 6 ? w[k] : 0);
                const int axis = f >> 1;
                float c0[3] = {bx[0], bx[2], bx[4]}, c1[3] = {bx[1], bx[3], bx[5]};
                c0[axis] = c1[axis] = bx[2 * axis + (f & 1)];
                grow(c0); grow(c1);
            }
        }
        if (recs.empty()) continue;
        me.any = true;
        me.head[b] = (int)(me.prim.size() / 4);
        const int m = (int)(recs.size() / 16);
        const int hd[8] = {m, as_i(lo[0]), as_i(hi[0]), as_i(lo[1]), as_i(hi[1]), as_i(lo[2]), as_i(hi[2]), 0};
        me.prim.insert(me.prim.end(), hd, hd + 8);
        me.prim.insert(me.prim.end(), recs.begin(), recs.end());
    }
    return me;
}

// The table over the voxels whose leaf value b satisfies emits(b) (block_emits for DESIGN §10; with model emitters for §12).
template <class Emits>
inline EmitterGrid build_emitter_grid(const int *tree, size_t n, int depth, Emits emits) {
    EmitterGrid g;
    if (n == 0 || depth < 0 || depth > 30) return g;
    struct Leaf { int x, y, z, level, block; };
    std::vector<Leaf> leaves;
    long long count = 0;
    // depth-first over the reference's node array (ClSceneLoader.java:56-59); a malformed pointer ends its branch
    struct Item { size_t node; int x, y, z, level; };
    std::vector<Item> stack{{0, 0, 0, 0, depth}};
    while (!stack.empty()) {
        const Item it = stack.back();
        stack.pop_back();
        const int data = tree[it.node];
        if (data > 0) {
            if (it.level == 0 || (size_t)data + 7 >= n) continue;
            for (int k = 7; k >= 0; k--)
                stack.push_back({(size_t)data + k, (it.x << 1) | (k >> 2), (it.y << 1) | ((k >> 1) & 1), (it.z << 1) | (k & 1), it.level - 1});
            continue;
        }
        if (data == INT32_MIN || !emits(-data)) continue;
        if (it.level > 6) return EmitterGrid{};   // 8^7 voxels alone exceed EMIT_MAX
        count += 1ll << (3 * it.level);
        if (count > EMIT_MAX) return EmitterGrid{};
        leaves.push_back({it.x << it.level, it.y << it.level, it.z << it.level, it.level, -data});
    }
    if (leaves.empty()) return g;
    std::vector<int4> e;
    e.reserve((size_t)count);
    for (const Leaf &l : leaves) {
        const int s = 1 << l.level;
        for (int x = 0; x < s; x++)
            for (int y = 0; y < s; y++)
                for (int z = 0; z < s; z++) e.push_back(make_int4(l.x + x, l.y + y, l.z + z, l.block));
    }
    std::sort(e.begin(), e.end(), [](const int4 &a, const int4 &b) {
        return a.x != b.x ? a.x < b.x : (a.y != b.y ? a.y < b.y : a.z < b.z);
    });
    int lo[3] = {INT32_MAX, INT32_MAX, INT32_MAX}, hi[3] = {0, 0, 0};
    for (const int4 &v : e) {
        const int c[3] = {v.x, v.y, v.z};
        for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], c[a]); hi[a] = std::max(hi[a], c[a]); }
    }
    // the cell box: the emitters' cells and one more cell on every side
    for (;; g.shift++) {
        long long cells = 1;
        for (int a = 0; a < 3; a++) {
            const int c0 = (lo[a] >> g.shift) - 1, c1 = (hi[a] >> g.shift) + 1;
            g.g0[a] = c0 * (1 << g.shift);
            g.dim[a] = c1 - c0 + 1;
            cells *= g.dim[a];
        }
        if (cells <= EMIT_CELL_BUDGET) break;
    }
    const size_t n_cells = (size_t)g.dim[0] * g.dim[1] * g.dim[2];
    g.off.assign(n_cells + 1, 0);
    auto each_cell = [&](const int4 &v, auto f) {
        const int cx = (v.x - g.g0[0]) >> g.shift, cy = (v.y - g.g0[1]) >> g.shift, cz = (v.z - g.g0[2]) >> g.shift;
        for (int dx = -1; dx <= 1; dx++)
            for (int dy = -1; dy <= 1; dy++)
                for (int dz = -1; dz <= 1; dz++) f(((size_t)(cx + dx) * g.dim[1] + (size_t)(cy + dy)) * g.dim[2] + (size_t)(cz + dz));
    };
    for (const int4 &v : e) each_cell(v, [&](size_t c) { g.off[c + 1]++; });
    for (size_t c = 0; c < n_cells; c++) g.off[c + 1] += g.off[c];
    g.list.resize((size_t)g.off[n_cells]);
    std::vector<int> fill(g.off.begin(), g.off.end() - 1);
    for (size_t i = 0; i < e.size(); i++) each_cell(e[i], [&](size_t c) { g.list[(size_t)fill[c]++] = (int)i; });
    g.emit.resize(e.size() * 4);
    for (size_t i = 0; i < e.size(); i++) {
        g.emit[4 * i] = e[i].x; g.emit[4 * i + 1] = e[i].y; g.emit[4 * i + 2] = e[i].z; g.emit[4 * i + 3] = e[i].w;
    }
    return g;
}

// The wider table of DESIGN §12: the full-cube emitters and the model emitters of `me`; empty when no model emitter is in it
// (or it exceeds the limits of build_emitter_grid).
inline EmitterGrid build_model_grid(const int *tree, size_t n, int depth, const PaletteRecs &pr, const ModelEmitters &me) {
    if (!me.any) return EmitterGrid{};
    const auto is_model = [&](int b) { return b >= 0 && (size_t)b < me.head.size() && me.head[(size_t)b] >= 0; };
    EmitterGrid g = build_emitter_grid(tree, n, depth, [&](int b) { return block_emits(pr.block, b) || is_model(b); });
    for (size_t i = 3; i < g.emit.size(); i += 4)
        if (is_model(g.emit[i])) return g;
    return EmitterGrid{};
}

// ------------------------------------------------------------------------------------------------------
// biome colours of CCU_RENDER_BIOME_TINT (BiomeView, DESIGN §13)
// ------------------------------------------------------------------------------------------------------
// chunks: n x {cx, cz}; rgb: n x 3 planes x 256 texels x 3 floats, as ccu_scene_set_biome_colors takes them (already checked
// there).  The grid covers the chunks' bounding box: gx x gz chunk indices from chunk (x0, z0), index (cx - x0) * gz + (cz - z0),
// -1 = no tile; tiles: the same texels as {r, g, b, 0}.  status: 0 built; 1 chunk `bad` lies outside the octree's `extent` x
// `extent` chunks (extent = max(1, 2^depth / 16)); 2 the bounding box has more than CCU_BIOME_GRID_MAX cells (nothing built).
#define CCU_BIOME_GRID_MAX (1ll << 24)   // grid cells (64 MiB): every chunk of a depth-16 octree
struct BiomeLayout {
    int x0 = 0, z0 = 0, gx = 0, gz = 0;
    int64_t extent = 1;
    std::vector<int> grid;
    std::vector<float> tiles;   // float4 per texel
    int status = 0;
    int64_t bad = -1;
};
inline BiomeLayout build_biome_layout(const int32_t *chunks, const float *rgb, int64_t n, int depth) {
    BiomeLayout b;
    b.extent = depth > 4 ? 1ll << (depth - 4) : 1;
    if (n == 0) return b;
    int64_t lx = INT64_MAX, lz = INT64_MAX, hx = -1, hz = -1;
    for (int64_t i = 0; i < n; i++) {
        const int64_t cx = chunks[2 * i], cz = chunks[2 * i + 1];
        if (cx >= b.extent || cz >= b.extent) {
            b.status = 1;
            b.bad = i;
            return b;
        }
        lx = std::min(lx, cx); hx = std::max(hx, cx);
        lz = std::min(lz, cz); hz = std::max(hz, cz);
    }
    if ((hx - lx + 1) * (hz - lz + 1) > CCU_BIOME_GRID_MAX) {
        b.status = 2;
        return b;
    }
    b.x0 = (int)lx; b.z0 = (int)lz; b.gx = (int)(hx - lx + 1); b.gz = (int)(hz - lz + 1);
    b.grid.assign((size_t)b.gx * b.gz, -1);
    b.tiles.assign((size_t)n * 3 * 256 * 4, 0.0f);
    for (int64_t i = 0; i < n; i++) {
        b.grid[(size_t)(chunks[2 * i] - b.x0) * b.gz + (size_t)(chunks[2 * i + 1] - b.z0)] = (int)i;
        for (size_t t = 0; t < 3 * 256; t++)
            for (int c = 0; c < 3; c++) b.tiles[((size_t)i * 3 * 256 + t) * 4 + c] = rgb[((size_t)i * 3 * 256 + t) * 3 + c];
    }
    return b;
}

}  // namespace
