// Huffman table construction ON THE DEVICE, for batches of frames (SURVEY.md 8(f)1).
//
// Produces exactly what the reference's generateHuffmanCode(text) produces (src/Huffman.cpp:3-66,
// include/Huffman.hpp:114-174), like the host build in host/huffman_build.cpp, from the same inputs (K2's symbol
// histogram and first-occurrence keys).  The host build gets the two library-defined orders the result depends on --
// std::unordered_map<int,int> iteration order and std::priority_queue's heap layout (SURVEY.md H2) -- by driving the
// real libstdc++ containers; device code cannot, so both are restated here on plain arrays:
//   * OrderedMap: libstdc++'s _Hashtable for int keys (identity hash): one forward list threaded through the buckets,
//     a new node goes to the front of its bucket (or, for an empty bucket, to the front of the whole list),
//     _Prime_rehash_policy growth (1 -> 13 -> 29 -> 59 -> 127 -> 257 -> 541 buckets), _M_rehash_aux re-threading;
//   * heap_push / heap_pop: std::push_heap / std::pop_heap (bits/stl_heap.h: __push_heap, __adjust_heap) with the
//     reference's comparator "weight greater" (Huffman.hpp:117-119).
// tests/test_gpu_parity.py compares the result with the host build on every test image and on random histograms.
//
// Why it exists: a 1080p frame costs 38 us of host CPU for its four tables.  With one GPU and 16 cores that hides
// behind the other pipeline lanes' kernels; on an 8-GPU box with 32 cores it is what limits a batch (8 x fewer
// cores per GPU).  On the device a table is a serial chain of ~6 k (27 symbols) to ~50 k (162 symbols) dependent heap
// steps -- one thread, ~40 ns per step -- but all 4 * F tables of a pass run side by side (one warp each, lane 0
// working) and the other lanes' kernels fill the SMs meanwhile.  A single image keeps the host build: 16 us there
// against >= 250 us here.
#include <cstring>

#include "common.cuh"

namespace jpgenc {

namespace {

constexpr int kMaxSyms = 256;
constexpr int kMaxBuckets = 600;
constexpr int kLimit = 15;                                     // package_merge(symbol_frequency, 15)
constexpr int kMaxNodes = kMaxSyms * (kLimit + 2) + 16;        // leaves + at most one package per pair of items per level
constexpr int kBeforeBegin = -2;

struct HeapItem {
    long long w;
    int node;
};
struct Node {
    short left, right, sym;                                    // sym >= 0: leaf
    short pad;
};

struct OrderedMap {                                            // libstdc++ unordered_map<int, T> iteration order
    short key[kMaxSyms], nxt[kMaxSyms], slot_of[kMaxSyms];
    short bucket[kMaxBuckets];                                 // node BEFORE the bucket's first node; -1 = empty bucket
    int nb, n, next_resize, head;
};

struct TableScratch {
    OrderedMap map;
    short syms[kMaxSyms];
    unsigned freq[kMaxSyms];
    unsigned short len_of[kMaxSyms], cnt[kMaxSyms];
    unsigned char per_len[18][kMaxSyms];
    int per_len_n[18];
    HeapItem blueprint[kMaxSyms], heap_a[2 * kMaxSyms + 16], heap_b[2 * kMaxSyms + 16];
    Node nodes[kMaxNodes];
    unsigned char order[kMaxSyms];
};

__host__ __device__ void um_init(OrderedMap& m) {
    m.nb = 1; m.n = 0; m.next_resize = 0; m.head = -1;
    for (int i = 0; i < kMaxSyms; ++i) m.slot_of[i] = -1;
    m.bucket[0] = -1;
}

__host__ __device__ int um_next_bkt(OrderedMap& m, int want) {         // _Prime_rehash_policy::_M_next_bkt
    const unsigned char fast[14] = {2, 2, 2, 3, 5, 5, 7, 7, 11, 11, 11, 11, 13, 13};
    const short primes[46] = {17,  19,  23,  29,  31,  37,  41,  43,  47,  53,  59,  61,  67,  71,  73,  79,
                              83,  89,  97,  103, 109, 113, 127, 137, 139, 149, 157, 167, 179, 193, 199, 211,
                              227, 241, 257, 277, 293, 313, 337, 359, 383, 409, 439, 467, 503, 541};
    if (want < 14) {
        if (want == 0) return 1;
        m.next_resize = fast[want];
        return fast[want];
    }
    for (int i = 0; i < 46; ++i)
        if (primes[i] >= want) { m.next_resize = primes[i]; return primes[i]; }
    m.next_resize = 541;
    return 541;                                                // unreachable: at most 256 keys
}

__host__ __device__ int um_get_next(const OrderedMap& m, int node) { return node == kBeforeBegin ? m.head : m.nxt[node]; }
__host__ __device__ void um_set_next(OrderedMap& m, int node, int v) { if (node == kBeforeBegin) m.head = v; else m.nxt[node] = static_cast<short>(v); }

__host__ __device__ void um_rehash(OrderedMap& m, int nb) {            // _M_rehash_aux(n, true_type)
    int p = m.head, bbegin_bkt = 0;
    for (int i = 0; i < nb; ++i) m.bucket[i] = -1;
    m.head = -1;
    while (p >= 0) {
        const int next = m.nxt[p];
        const int bkt = m.key[p] % nb;
        if (m.bucket[bkt] == -1) {
            m.nxt[p] = static_cast<short>(m.head);
            m.head = p;
            m.bucket[bkt] = kBeforeBegin;
            if (m.nxt[p] >= 0) m.bucket[bbegin_bkt] = static_cast<short>(p);
            bbegin_bkt = bkt;
        } else {
            const int before = m.bucket[bkt];
            m.nxt[p] = static_cast<short>(um_get_next(m, before));
            um_set_next(m, before, p);
        }
        p = next;
    }
    m.nb = nb;
}

// operator[]: the node of `key`, inserted when new
__host__ __device__ int um_touch(OrderedMap& m, int key) {
    if (m.slot_of[key] >= 0) return m.slot_of[key];
    if (m.n + 1 > m.next_resize) {                             // _M_need_rehash(n_bkt, n_elt, 1)
        int min_bkts = m.n + 1;
        if (m.next_resize == 0 && min_bkts < 11) min_bkts = 11;
        if (min_bkts >= m.nb) {
            int want = min_bkts + 1;
            if (want < m.nb * 2) want = m.nb * 2;
            um_rehash(m, um_next_bkt(m, want));
        } else {
            m.next_resize = m.nb;
        }
    }
    const int node = m.n++;
    m.key[node] = static_cast<short>(key);
    m.slot_of[key] = static_cast<short>(node);
    const int bkt = key % m.nb;
    if (m.bucket[bkt] != -1) {                                 // _M_insert_bucket_begin
        const int before = m.bucket[bkt];
        m.nxt[node] = static_cast<short>(um_get_next(m, before));
        um_set_next(m, before, node);
    } else {
        m.nxt[node] = static_cast<short>(m.head);
        m.head = node;
        if (m.nxt[node] >= 0) m.bucket[m.key[m.nxt[node]] % m.nb] = static_cast<short>(node);
        m.bucket[bkt] = kBeforeBegin;
    }
    return node;
}

void heap_push_hole(HeapItem* v, int hole, int top, long long val_w, int val_node) {      // std::__push_heap
    int parent = (hole - 1) / 2;
    while (hole > top && v[parent].w > val_w) {
        v[hole].w = v[parent].w;
        v[hole].node = v[parent].node;
        hole = parent;
        parent = (hole - 1) / 2;
    }
    v[hole].w = val_w;
    v[hole].node = val_node;
}
void heap_push(HeapItem* v, int& n, long long w, int node) { ++n; heap_push_hole(v, n - 1, 0, w, node); }
// top(), then std::pop_heap + pop_back
void heap_pop(HeapItem* v, int& n, long long& top_w, int& top_node) {
    top_w = v[0].w;
    top_node = v[0].node;
    if (n > 1) {
        const int len = n - 1;                                                       // std::__pop_heap -> std::__adjust_heap
        const long long val_w = v[len].w;
        const int val_node = v[len].node;
        int hole = 0, child = 0;
        while (child < (len - 1) / 2) {
            child = 2 * (child + 1);
            if (v[child].w > v[child - 1].w) --child;
            v[hole].w = v[child].w;
            v[hole].node = v[child].node;
            hole = child;
        }
        if ((len & 1) == 0 && child == (len - 2) / 2) {
            child = 2 * (child + 1);
            v[hole].w = v[child - 1].w;
            v[hole].node = v[child - 1].node;
            hole = child - 1;
        }
        heap_push_hole(v, hole, 0, val_w, val_node);
    }
    --n;
}

// occurrences of every symbol among the leaves of package `root`: cnt[] is incremented, the symbols seen are flagged in
// the 256-bit mask
void count_leaves(const Node* nodes, int root, unsigned short* cnt, unsigned (&mask)[8]) {
    int stack[40], sp = 0;                                     // a package is at most kLimit levels deep: <= 17 pending nodes
    stack[sp++] = root;
    while (sp) {
        const int k = stack[--sp];
        const int sym = nodes[k].sym;
        if (sym >= 0) { ++cnt[sym]; mask[sym >> 5] |= 1u << (sym & 31); continue; }
        stack[sp++] = nodes[k].left;
        stack[sp++] = nodes[k].right;
    }
}

__host__ __device__ void write_table(const TableScratch& s, int nsymbols, jpgenc_huff_table* t) {     // generateCodes, src/Huffman.cpp:50-66
    unsigned code = 0;
    int k = 0;
    for (int len = 1; len <= 16; ++len) {
        t->counts[len - 1] = static_cast<uint8_t>(s.per_len_n[len]);
        for (int i = 0; i < s.per_len_n[len]; ++i) {
            const int sym = s.per_len[len][i];
            t->code_msb[sym] = code << (32 - len);
            t->length[sym] = static_cast<uint8_t>(len);
            t->symbols[k++] = static_cast<uint8_t>(sym);
            ++code;
        }
        code <<= 1;
    }
    t->nsymbols = nsymbols;
}

// The one-thread construction: s.order[0..n) = the distinct symbols in order of first appearance, count[256] their
// frequencies; *tab has been zeroed.  Runs on the host, as the reference the CPU tests check the array restatement with.
void build_table_serial(TableScratch& s, const uint32_t* count, int n, jpgenc_huff_table* tab) {
    OrderedMap& map = s.map;
    Node* nodes = s.nodes;
    HeapItem *blueprint = s.blueprint, *heap_a = s.heap_a, *heap_b = s.heap_b;
    unsigned short *len_of = s.len_of, *cnt = s.cnt;
    um_init(map);
    for (int i = 0; i < n; ++i) um_touch(map, s.order[i]);
    int m = 0;
    for (int p = map.head; p >= 0; p = map.nxt[p]) { s.syms[m] = map.key[p]; s.freq[m] = count[map.key[p]]; ++m; }
    for (int l = 0; l < 18; ++l) s.per_len_n[l] = 0;

    if (n == 1) {                                              // src/Huffman.cpp:17-25: the lone symbol gets code "0"
        s.per_len[1][s.per_len_n[1]++] = static_cast<unsigned char>(s.syms[0]);
        write_table(s, n, tab);
        return;
    }
    int nn = 0, nb = 0;
    for (int i = 0; i < n; ++i) {                              // map iteration order feeds the first heap
        nodes[nn] = Node{-1, -1, s.syms[i], 0};
        heap_push(blueprint, nb, static_cast<long long>(static_cast<int>(s.freq[i])), nn);   // the reference counts in int
        ++nn;
    }
    HeapItem *cur = heap_a, *nxt = heap_b;
    int ncur = n, nnxt = 0;
    for (int i = 0; i < n; ++i) cur[i] = blueprint[i];
    for (int lvl = 0; lvl < kLimit; ++lvl) {
        if (lvl + 1 < kLimit) {                                // every level but the last starts as a copy of the leaves
            for (int i = 0; i < n; ++i) nxt[i] = blueprint[i];
            nnxt = n;
        } else {
            nnxt = 0;
        }
        while (ncur > 1) {
            long long aw, bw;
            int an, bn;
            heap_pop(cur, ncur, aw, an);
            heap_pop(cur, ncur, bw, bn);
            nodes[nn] = Node{static_cast<short>(an), static_cast<short>(bn), -1, 0};
            heap_push(nxt, nnxt, aw + bw, nn);
            ++nn;
        }
        HeapItem* sw = cur; cur = nxt; nxt = sw;
        ncur = nnxt;
    }
    // drain the last level: a symbol's code length is the number of times it occurs in the surviving packages; the
    // lengths map is touched package by package, symbols of a package in ascending order
    um_init(map);
    for (int i = 0; i < 256; ++i) { len_of[i] = 0; cnt[i] = 0; }
    while (ncur) {
        long long pw;
        int pn;
        heap_pop(cur, ncur, pw, pn);
        unsigned mask[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        count_leaves(nodes, pn, cnt, mask);
#pragma unroll 1
        for (int w = 0; w < 8; ++w) {                          // ascending symbol order, only the symbols that occur
            unsigned bits = mask[w];
            while (bits) {
                int b = 0;
                while (!((bits >> b) & 1u)) ++b;               // lowest set bit
                const int sym = w * 32 + b;
                bits &= bits - 1;
                um_touch(map, sym);
                len_of[sym] += cnt[sym];
                cnt[sym] = 0;
            }
        }
    }
    for (int p = map.head; p >= 0; p = map.nxt[p]) {
        const int sym = map.key[p], len = len_of[sym];
        s.per_len[len][s.per_len_n[len]++] = static_cast<unsigned char>(sym);
    }
    // preventOnlyOnesCode (src/Huffman.cpp:37-48): the last symbol of the deepest level moves one level down
    int deepest = 16;
    while (deepest > 0 && s.per_len_n[deepest] == 0) --deepest;
    const int moved = s.per_len[deepest][--s.per_len_n[deepest]];
    s.per_len[deepest + 1][s.per_len_n[deepest + 1]++] = static_cast<unsigned char>(moved);
    write_table(s, n, tab);
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------------
// The same construction with the whole warp working on one table.
//
// A table is a chain of heap operations that depend on each other (15 levels x ~2n pops and ~n pushes); one thread spends
// ~400 cycles on a pop because every step of the sift-down is a round trip through shared memory followed by dependent
// address arithmetic (measured: 0.59 ms for the four tables of a 1920x1080 frame, 28 symbols in the luma AC table, 70 % of
// a batched pass).  The operations themselves are easy to spread over the lanes without changing their result:
//   * pop  = libstdc++'s __adjust_heap: the hole at the root walks down to a leaf position, always to the lighter child
//            (the right one on a tie), then the former last element is sifted up from there.  Which child is the lighter
//            one is decided for ALL nodes at once (one 16-byte load per lane, one ballot); the walk is then bit arithmetic
//            on the ballot word, the moves along the path are one load and one store by one lane each, and where the
//            sift-up stops is a ballot over the path.
//   * push = __push_heap: the ancestors of the new position are loaded by one lane each; a ballot tells how far the new
//            element rises.
// Heap items are packed into one 64-bit word (weight << 16 | node) and stored at slot index + 1, so that the two children
// of a node are one aligned 16-byte pair.  The container emulation (unordered_map order) stays on lane 0: n insertions.
// The walk over the final packages (which symbol occurs how often = its code length, and which package touches it first
// = its place in the reference's second unordered_map) runs one package per lane.
// ---------------------------------------------------------------------------------------------------------------------
#ifdef __CUDACC__
namespace {

constexpr int kHeapSlots = 2 * kMaxSyms + 18;                 // element i lives in slot i + 1; +1 so that a pair load never leaves the array

struct WarpShared {
    alignas(16) unsigned long long heap[3][kHeapSlots];
    OrderedMap map;
    short syms[kMaxSyms];                                      // map iteration order -> symbol (= leaf node id -> symbol)
    unsigned freq[kMaxSyms];
    unsigned short cnt[kMaxSyms];                              // occurrences in the final packages = code length
    unsigned short first[kMaxSyms];                            // pop index of the first final package that holds the symbol
    unsigned short root[kMaxSyms];                             // final packages in pop order
    unsigned char order[kMaxSyms];
    unsigned char present[kMaxSyms];
};

__device__ __forceinline__ unsigned long long item_w(unsigned long long it) { return it >> 16; }

// std::push_heap of `item` onto a heap of `len` elements (len grows by one)
__device__ __forceinline__ void warp_push(unsigned long long* H, int& len, unsigned long long item, int lane) {
    const int p = len;                                         // new position
    // lane j >= 1 looks at ancestor j of p: a_j = ((p + 1) >> j) - 1, while it exists
    const int a = static_cast<int>((static_cast<unsigned>(p) + 1u) >> lane) - 1;
    const bool has = lane >= 1 && a >= 0;
    const unsigned long long anc = has ? H[a + 1] : 0ull;
    const unsigned up = __ballot_sync(0xffffffffu, has && item_w(anc) > item_w(item)) >> 1;   // bit j-1: ancestor j is heavier
    const int r = __ffs(~up) - 1;                              // the element rises past r ancestors
    if (has && lane <= r) H[(lane == 1 ? p : static_cast<int>((static_cast<unsigned>(p) + 1u) >> (lane - 1)) - 1) + 1] = anc;   // ancestor j moves to a_{j-1}
    if (lane == 0) H[(r == 0 ? p : static_cast<int>((static_cast<unsigned>(p) + 1u) >> r) - 1) + 1] = item;
    len = p + 1;
    __syncwarp();
}

// top() followed by std::pop_heap + pop_back on a heap of `len` elements (len shrinks by one); returns the top item
__device__ __forceinline__ unsigned long long warp_pop(unsigned long long* H, int& len, int lane) {
    const unsigned long long top = H[1];
    const int m = len - 1;                                     // elements that stay
    len = m;
    if (m == 0) { __syncwarp(); return top; }
    const unsigned long long val = H[m + 1];                   // the former last element looks for its place
    const int k2 = (m - 1) / 2;                                // nodes 0 .. k2-1 have both children among the m elements
    // which child is lighter, for every such node: bit = 1 -> left (the right child is strictly heavier)
    unsigned word0 = 0, mine = 0;                              // ballot of nodes 0..31 (every lane), of nodes 32g .. 32g+31 (lane g)
    for (int g = 0; g * 32 < k2; ++g) {
        const int k = g * 32 + lane;
        bool left = false;
        if (k < k2) {
            const ulonglong2 pair = *reinterpret_cast<const ulonglong2*>(H + 2 * k + 2);   // elements 2k+1 (left), 2k+2 (right)
            left = item_w(pair.y) > item_w(pair.x);
        }
        const unsigned b = __ballot_sync(0xffffffffu, left);
        if (g == 0) word0 = b;
        if (lane == g) mine = b;
    }
    // the hole's way down; lane j remembers step j: the element at `from` moves up to `to`
    int h = 0, steps = 0, from = 0, to = 0;
    while (h < k2) {
        const unsigned w = h < 32 ? word0 : __shfl_sync(0xffffffffu, mine, h >> 5);
        const int c = 2 * h + 2 - static_cast<int>((w >> (h & 31)) & 1u);
        if (lane == steps) { to = h; from = c; }
        h = c;
        ++steps;
    }
    if ((m & 1) == 0 && h == (m - 2) / 2) {                    // a last node with a left child only
        const int c = 2 * h + 1;
        if (lane == steps) { to = h; from = c; }
        h = c;
        ++steps;
    }
    // sift-up of val from the final hole: it passes every moved element that is heavier, from the bottom of the path
    const bool on_path = lane < steps;
    const unsigned long long moved = on_path ? H[from + 1] : 0ull;
    const unsigned heavier = __ballot_sync(0xffffffffu, on_path && item_w(moved) > item_w(val));
    const unsigned stops = ~heavier & (steps >= 32 ? 0xffffffffu : ((1u << steps) - 1u));     // path steps val does NOT pass
    const int jstar = stops ? 32 - __clz(stops) : 0;           // val lands at path[jstar]; steps below it keep their elements
    __syncwarp();
    if (on_path && lane < jstar) H[to + 1] = moved;
    if (lane == jstar) H[(jstar == steps ? h : to) + 1] = val;  // lane jstar < steps holds path[jstar] in `to`; jstar == steps: the final hole
    __syncwarp();
    return top;
}

// ---- heap items: two encodings behind one interface ----------------------------------------------------------------
// Wide: weight << 16 | node (48-bit weights), the general case.  Lean<W>: weight << 32 | node for heaps of at most 64 W
// elements whose weights fit 32 bits -- every table of an ordinary frame (a level holds at most 2 n - 1 items; the sum of
// the packages of a level is at most 15 x the number of symbols in the text) -- with a pop that has no loop at all.
struct WideHeap {
    static __device__ __forceinline__ unsigned long long make(unsigned long long w, unsigned node) { return (w << 16) | node; }
    static __device__ __forceinline__ unsigned long long weight(unsigned long long it) { return it >> 16; }
    static __device__ __forceinline__ unsigned node(unsigned long long it) { return static_cast<unsigned>(it & 0xFFFFu); }
    static __device__ __forceinline__ void push(unsigned long long* H, int& len, unsigned long long item, int lane) { warp_push(H, len, item, lane); }
    static __device__ __forceinline__ unsigned long long pop(unsigned long long* H, int& len, int lane) { return warp_pop(H, len, lane); }
};

// Element i (1-based) lives in slot i; its children are 2 i and 2 i + 1: one aligned 16-byte pair.  Lane l owns the nodes
// k = l + 32 t (t < W) -- that is, it holds node k's two children in registers after ONE load.
//   pop  = __adjust_heap: the hole walks from the root to a leaf, always to the lighter child (the right one on a tie),
//          then the former last element `val` rises from there past every heavier element (__push_heap).
//          Every node decides "left or right" at once (ballot Lw).  Node k lies on the hole's way iff the decisions of its
//          ancestors spell the bits of k below its leading one -- each lane tests that for its own nodes with a few shifts
//          of Lw, no walk.  The lanes whose node is on the way hold the elements that move (their chosen child); a ballot
//          of "heavier than val" over them tells where val stops: the deepest such child that is not heavier.  Children
//          at or above that depth move up into their parent, val takes the place of the deepest mover, the rest stays.
//   push = __push_heap: lane j looks at ancestor j of the new position; a ballot tells how far the new element rises.
template <int W>
struct LeanHeap {
    static constexpr unsigned kFull = 0xffffffffu;
    static constexpr int kDepth = W == 1 ? 4 : 5;              // a node index below 32 W has at most this many bits below its leading one
    static __device__ __forceinline__ unsigned long long make(unsigned long long w, unsigned node) { return (w << 32) | node; }
    static __device__ __forceinline__ unsigned long long weight(unsigned long long it) { return it >> 32; }
    static __device__ __forceinline__ unsigned node(unsigned long long it) { return static_cast<unsigned>(it); }
    static __device__ __forceinline__ unsigned wt(unsigned long long it) { return static_cast<unsigned>(it >> 32); }

    static __device__ __forceinline__ void push(unsigned long long* H, int& len, unsigned long long item, int lane) {
        const int p = len + 1;                                  // the new position
        const int a = p >> lane;                                // lane j >= 1: ancestor j of p (0 = none)
        const bool has = lane >= 1 && a >= 1;
        const unsigned long long anc = has ? H[a] : 0ull;
        const unsigned up = __ballot_sync(kFull, has && wt(anc) > wt(item)) >> 1;   // bit j-1: ancestor j is heavier
        const int r = __ffs(~up) - 1;                           // the element rises past r ancestors
        if (has && lane <= r) H[p >> (lane - 1)] = anc;         // ancestor j moves down to where ancestor j-1 was
        if (lane == 0) H[p >> r] = item;
        len = p;
        __syncwarp();
    }

    static __device__ __forceinline__ unsigned long long pop(unsigned long long* H, int& len, int lane) {
        const unsigned long long top = H[1];
        const int m = len - 1;                                  // elements that stay: 1 .. m
        len = m;
        if (m == 0) { __syncwarp(); return top; }
        const unsigned long long val = H[m + 1];                // the former last element looks for its place
        const unsigned vw = wt(val);
        ulonglong2 pr[W];
        bool left[W];
        unsigned Lw[W];
#pragma unroll
        for (int t = 0; t < W; ++t) {
            const int k = lane + 32 * t;
            pr[t] = *reinterpret_cast<const ulonglong2*>(H + 2 * k);             // children 2k (x) and 2k+1 (y); k = 0 reads slots 0, 1: unused
            const bool hasl = k >= 1 && 2 * k <= m, hasr = 2 * k + 1 <= m;
            left[t] = hasl && (!hasr || wt(pr[t].y) > wt(pr[t].x));              // left only when the right child is strictly heavier (or absent)
            Lw[t] = __ballot_sync(kFull, left[t]);
        }
        unsigned pc[W], hv[W];
        unsigned long long child[W];
        bool onp[W];
#pragma unroll
        for (int t = 0; t < W; ++t) {
            const int k = lane + 32 * t;
            unsigned x = 0;                                     // bit j = "ancestor k >> (j+1) goes left"
#pragma unroll
            for (int j = 0; j < kDepth; ++j) {
                const int a = k >> (j + 1);
                const unsigned word = (W > 1 && a >= 32) ? Lw[W - 1] : Lw[0];
                x |= ((word >> (a & 31)) & 1u) << j;
            }
            const unsigned mask = k >= 1 ? (1u << (31 - __clz(k))) - 1u : 0u;
            // going left means bit 0: the way to k is taken iff every ancestor's decision differs from k's bit
            onp[t] = k >= 1 && 2 * k <= m && (((x ^ static_cast<unsigned>(k)) & mask) == mask);
            child[t] = left[t] ? pr[t].x : pr[t].y;
            pc[t] = __ballot_sync(kFull, onp[t]);
            hv[t] = __ballot_sync(kFull, onp[t] && wt(child[t]) > vw);
        }
        // deepest element on the way that val does not pass (deeper = larger node index); none: val goes to the root
        int kstar = 0;
#pragma unroll
        for (int t = 0; t < W; ++t) {
            const unsigned stops = pc[t] & ~hv[t];
            if (stops) kstar = 32 * t + 31 - __clz(stops);
        }
        __syncwarp();
#pragma unroll
        for (int t = 0; t < W; ++t) {
            const int k = lane + 32 * t;
            if (onp[t] && k <= kstar) H[k] = child[t];          // the chosen child moves up into its parent
            if (onp[t] && k == kstar) H[2 * k + (left[t] ? 0 : 1)] = val;
        }
        if (kstar == 0 && lane == 0) H[1] = val;
        __syncwarp();
        return top;
    }
};

// package_merge (Huffman.hpp:114-160) on the warp's three heaps: leaf i = node i, packages are nodes n, n+1, ... with two
// children; returns the number of packages of the last level and leaves their node ids, in pop order, in ws.root
template <class HP>
__device__ int package_merge_warp(WarpShared& ws, uint32_t* nodes, int n, int lane) {
    unsigned long long *bp = ws.heap[0], *cur = ws.heap[1], *nxt = ws.heap[2];
    int nb = 0;
    for (int i = 0; i < n; ++i)                                // map iteration order feeds the first heap; the reference counts in int
        HP::push(bp, nb, HP::make(static_cast<unsigned long long>(static_cast<unsigned>(static_cast<int>(ws.freq[i]))), static_cast<unsigned>(i)), lane);
    int nn = n, ncur = n, nnxt = 0;
    for (int i = lane; i < n; i += 32) cur[i + 1] = bp[i + 1];
    __syncwarp();
    for (int lvl = 0; lvl < kLimit; ++lvl) {
        if (lvl + 1 < kLimit) {                                // every level but the last starts as a copy of the leaves
            for (int i = lane; i < n; i += 32) nxt[i + 1] = bp[i + 1];
            nnxt = n;
            __syncwarp();
        } else {
            nnxt = 0;
        }
        while (ncur > 1) {
            const unsigned long long a = HP::pop(cur, ncur, lane), b = HP::pop(cur, ncur, lane);
            if (lane == 0) nodes[nn] = HP::node(a) | (HP::node(b) << 16);
            HP::push(nxt, nnxt, HP::make(HP::weight(a) + HP::weight(b), static_cast<unsigned>(nn)), lane);
            ++nn;
        }
        unsigned long long* sw = cur; cur = nxt; nxt = sw;
        ncur = nnxt;
    }
    // ---- drain the last level: packages in pop order ----
    int npk = 0;
    while (ncur) {
        const unsigned long long pk = HP::pop(cur, ncur, lane);
        if (lane == 0) ws.root[npk] = static_cast<unsigned short>(HP::node(pk));
        ++npk;
    }
    return npk;
}

// The table `tab` (zeroed) from count[] / first[]; ws = the warp's shared memory, s = its scratch slab in global memory.
__device__ void build_table_warp(WarpShared& ws, TableScratch& s, const uint32_t* count, const unsigned long long* first,
                                 jpgenc_huff_table* tab, int lane, uint32_t* status) {
    // ---- distinct symbols in order of first appearance (= the order the reference's counting loop creates map entries) ----
    int n = 0;
    for (int base = 0; base < 256; base += 32) {
        const int sym = base + lane;
        const bool here = count[sym] != 0;
        const unsigned b = __ballot_sync(0xffffffffu, here);
        if (here) ws.present[n + __popc(b & ((1u << lane) - 1u))] = static_cast<unsigned char>(sym);
        n += __popc(b);
    }
    __syncwarp();
    if (n == 0) { if (lane == 0) *status = 1; return; }        // the reference asserts text.size() > 0
    if (lane == 0) *status = 0;
    for (int i = lane; i < n; i += 32) {                       // rank among the present symbols (keys are unique)
        const int sym = ws.present[i];
        const unsigned long long k = first[sym];
        int rank = 0;
        for (int o = 0; o < n; ++o) rank += first[ws.present[o]] < k ? 1 : 0;
        ws.order[rank] = static_cast<unsigned char>(sym);
    }
    __syncwarp();
    if (lane == 0) {
        um_init(ws.map);
        for (int i = 0; i < n; ++i) um_touch(ws.map, ws.order[i]);
        int m = 0;
        for (int p = ws.map.head; p >= 0; p = ws.map.nxt[p]) { ws.syms[m] = ws.map.key[p]; ws.freq[m] = count[ws.map.key[p]]; ++m; }
        for (int l = 0; l < 18; ++l) s.per_len_n[l] = 0;
    }
    __syncwarp();
    if (n == 1) {                                              // src/Huffman.cpp:17-25: the lone symbol gets code "0"
        if (lane == 0) {
            s.per_len[1][s.per_len_n[1]++] = static_cast<unsigned char>(ws.syms[0]);
            write_table(s, n, tab);
        }
        return;
    }
    // ---- package-merge (Huffman.hpp:114-160): leaf i = node i; packages are nodes n, n+1, ... with two children ----
    uint32_t* nodes = reinterpret_cast<uint32_t*>(s.nodes);    // left | right << 16
    unsigned long long total = 0;
    for (int i = lane; i < n; i += 32) total += ws.freq[i];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) total += __shfl_xor_sync(0xffffffffu, total, d);
    const bool small_weights = total < (1ull << 28);           // 15 x total (the heaviest a package can get) fits 32 bits
    int npk;
    if (small_weights && n <= 32) npk = package_merge_warp<LeanHeap<1>>(ws, nodes, n, lane);
    else if (small_weights && n <= 64) npk = package_merge_warp<LeanHeap<2>>(ws, nodes, n, lane);
    else npk = package_merge_warp<WideHeap>(ws, nodes, n, lane);
    for (int i = lane; i < n; i += 32) { ws.cnt[i] = 0; ws.first[i] = 0xFFFFu; }
    __syncwarp();
    __threadfence_block();                                     // lane 0's node records are visible to every lane
    // a symbol's code length is the number of times it occurs in the surviving packages; the reference's lengths map is
    // touched package by package (pop order), symbols of a package in ascending order -> remember the first package
    for (int k = lane; k < npk; k += 32) {
        int stack[20], sp = 0;                                 // a package is at most kLimit levels deep
        stack[sp++] = ws.root[k];
        while (sp) {
            const int id = stack[--sp];
            if (id < n) {                                      // leaf: node id = position in map iteration order
                atomicAdd(reinterpret_cast<unsigned*>(ws.cnt) + (id >> 1), (id & 1) ? 0x10000u : 1u);
                unsigned* w = reinterpret_cast<unsigned*>(ws.first) + (id >> 1);
                // 16-bit minimum inside a 32-bit word: compare-and-swap (rarely more than one round)
                unsigned old = *w;
                for (;;) {
                    const unsigned cur16 = (id & 1) ? old >> 16 : old & 0xFFFFu;
                    if (cur16 <= static_cast<unsigned>(k)) break;
                    const unsigned want = (id & 1) ? (old & 0xFFFFu) | (static_cast<unsigned>(k) << 16) : (old & 0xFFFF0000u) | static_cast<unsigned>(k);
                    const unsigned seen = atomicCAS(w, old, want);
                    if (seen == old) break;
                    old = seen;
                }
                continue;
            }
            const uint32_t nd = nodes[id];
            stack[sp++] = static_cast<int>(nd & 0xFFFFu);
            stack[sp++] = static_cast<int>(nd >> 16);
        }
    }
    __syncwarp();
    // touch order of the lengths map: (first package, symbol value) ascending
    for (int i = lane; i < n; i += 32) {
        const unsigned key = (static_cast<unsigned>(ws.first[i]) << 16) | static_cast<unsigned>(ws.syms[i]);
        int rank = 0;
        for (int o = 0; o < n; ++o) rank += ((static_cast<unsigned>(ws.first[o]) << 16) | static_cast<unsigned>(ws.syms[o])) < key ? 1 : 0;
        ws.order[rank] = static_cast<unsigned char>(i);        // leaf ids in touch order
    }
    __syncwarp();
    if (lane == 0) {
        um_init(ws.map);
        for (int i = 0; i < n; ++i) um_touch(ws.map, ws.syms[ws.order[i]]);
        // symbol -> code length: cnt is indexed by leaf id; the map holds symbols
        for (int i = 0; i < n; ++i) s.len_of[ws.syms[i]] = ws.cnt[i];
        for (int p = ws.map.head; p >= 0; p = ws.map.nxt[p]) {
            const int sym = ws.map.key[p], len = s.len_of[sym];
            s.per_len[len][s.per_len_n[len]++] = static_cast<unsigned char>(sym);
        }
        // preventOnlyOnesCode (src/Huffman.cpp:37-48): the last symbol of the deepest level moves one level down
        int deepest = 16;
        while (deepest > 0 && s.per_len_n[deepest] == 0) --deepest;
        const int moved = s.per_len[deepest][--s.per_len_n[deepest]];
        s.per_len[deepest + 1][s.per_len_n[deepest + 1]++] = static_cast<unsigned char>(moved);
        write_table(s, n, tab);
    }
}

}  // namespace
#endif

// One warp per table.  status[table] = 0 ok, 1 = no symbol at all.
// (No __restrict__ on these parameters: with it nvcc 12.9 -O3 treated the two level heaps -- members of one scratch
// object whose pointers swap roles every level -- as never aliasing, and a popped weight read back as 0.  Found by the
// parity test; -G, -Xcicc -O1 and non-inlined heap functions all gave the right tables.)
__global__ void __launch_bounds__(32) build_tables_kernel(const uint8_t* stats, uint32_t stats_stride, uint32_t ntables,
                                                          TableScratch* scratch, jpgenc_huff_table* out, uint32_t* status) {
    const uint32_t table = blockIdx.x, lane = threadIdx.x;
    if (table >= ntables) return;
    const uint32_t frame = table >> 2, t = table & 3;
    const uint32_t* count = reinterpret_cast<const uint32_t*>(stats + static_cast<size_t>(frame) * stats_stride) + t * 256;
    const unsigned long long* first =
        reinterpret_cast<const unsigned long long*>(stats + static_cast<size_t>(frame) * stats_stride + 4096) + t * 256;
    TableScratch& s = scratch[table];
    jpgenc_huff_table* tab = out + table;
    {
        uint32_t* w = reinterpret_cast<uint32_t*>(tab);
        for (uint32_t i = lane; i < sizeof(jpgenc_huff_table) / 4; i += 32) w[i] = 0;
    }
    __shared__ WarpShared ws;
    __syncwarp();
    build_table_warp(ws, s, count, first, tab, static_cast<int>(lane), status + table);
}

size_t table_scratch_bytes() { return sizeof(TableScratch); }

// the same code on the host (no GPU involved): lets the array restatement be checked against the container-driven build
// in the CPU test suite
int build_table_arrays_host(const uint32_t count[256], const uint64_t first_pos[256], jpgenc_huff_table* out) {
    TableScratch* s = new TableScratch;
    std::memset(s, 0xA5, sizeof *s);            // device scratch is not initialised either: nothing may be read before it is written
    std::memset(out, 0, sizeof *out);
    int n = 0;
    for (int sym = 0; sym < 256; ++sym) {
        if (!count[sym]) continue;
        int rank = 0;
        for (int o = 0; o < 256; ++o) rank += (count[o] != 0 && first_pos[o] < first_pos[sym]) ? 1 : 0;
        s->order[rank] = static_cast<unsigned char>(sym);
        ++n;
    }
    if (n) build_table_serial(*s, count, n, out);
    delete s;
    return n ? JPGENC_OK : JPGENC_ERR_ARG;
}

// tables [ntables] (device) from the statistics of ntables / 4 frames laid out as K2 leaves them (stats_stride bytes per
// frame: histogram u32[4][256], first-occurrence keys u64[4][256]); scratch: ntables * table_scratch_bytes()
int launch_build_tables(jpgenc_ctx* c, const uint8_t* d_stats, uint32_t stats_stride, uint32_t ntables, void* d_scratch,
                        jpgenc_huff_table* d_out, uint32_t* d_status) {
    build_tables_kernel<<<ntables, 32, 0, c->stream>>>(d_stats, stats_stride, ntables, static_cast<TableScratch*>(d_scratch), d_out, d_status);
    JPGENC_CUDA(c, cudaGetLastError());
    c->launches += 1;
    return JPGENC_OK;
}

}  // namespace jpgenc
