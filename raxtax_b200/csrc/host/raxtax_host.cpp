// raxtax_host.cpp -- C++ host side of the B200 raxtax hot path (libraxtax_host.so, C ABI in include/raxtax_host.h).
//
// Mirrors the reference's host-side interface around the device boundary:
//   parser::parse_reference_fasta_str / parse_query_fasta_str   src/parser.rs:46-154
//   Tree::new                                                   src/tree.rs:47-140
//   raxtax::raxtax                                              src/raxtax.rs:14-97
//   EvaluationResult::get_output_string / get_tsv_string        src/lineage.rs:17-48, src/utils.rs:62-89
// Data layout is flat (CSR postings, BFS-numbered node arrays, one sequence blob) because it feeds
// rtx_index_upload directly; the per-query numerics all run on the GPU through include/raxtax_b200.h.

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <deque>
#include <exception>
#include <memory>
#include <mutex>
#include <numeric>
#include <stdexcept>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include <sys/stat.h>
#include <zlib.h>

#include "raxtax_host.h"

namespace raxtax {

typedef uint8_t u8;
typedef uint16_t u16;
typedef uint32_t u32;
typedef uint64_t u64;

struct Error : std::runtime_error {
    using std::runtime_error::runtime_error;
};

// ---- threads ----------------------------------------------------------------------------------------------------------------
static size_t host_threads() {
    if (const char* e = getenv("RXH_THREADS")) return (size_t)std::max(1, atoi(e));
    return std::min<size_t>(16, std::max<size_t>(1, std::thread::hardware_concurrency()));
}
// fn(task) for task = 0 .. n-1 on up to host_threads() threads (tasks handed out through a counter); the first exception is re-thrown
template <typename F>
static void parallel_for(size_t n, F&& fn) {
    const size_t T = std::min(host_threads(), n);
    if (T <= 1) {
        for (size_t i = 0; i < n; ++i) fn(i);
        return;
    }
    std::atomic<size_t> next{0};
    std::exception_ptr err;
    std::mutex err_mtx;
    std::vector<std::thread> th;
    for (size_t t = 0; t < T; ++t)
        th.emplace_back([&] {
            for (size_t i; (i = next.fetch_add(1)) < n;) {
                try {
                    fn(i);
                } catch (...) {
                    std::lock_guard<std::mutex> g(err_mtx);
                    if (!err) err = std::current_exception();
                }
            }
        });
    for (auto& t : th) t.join();
    if (err) std::rethrow_exception(err);
}

// ---- parser.rs:11-34 ------------------------------------------------------------------------------------------
struct DnaTable {
    u8 t[256];
    DnaTable() {
        memset(t, 0, sizeof t);
        const u8 a = 1, c = 2, g = 4, tt = 8;
        auto set = [&](char ch, u8 v) {
            t[(unsigned char)ch] = v;
            t[(unsigned char)(ch + 32)] = v;  // to_ascii_uppercase
        };
        set('A', a); set('C', c); set('G', g); set('T', tt);
        set('W', a | tt); set('S', c | g); set('M', a | c); set('K', g | tt); set('R', a | g); set('Y', c | tt);
        set('B', c | g | tt); set('D', a | g | tt); set('H', a | c | tt); set('V', a | c | g); set('N', a | c | g | tt);
    }
};
static const DnaTable kDna;

static inline u8 map_dna_char(char ch) {
    u8 v = kDna.t[(unsigned char)ch];
    if (!v) throw Error(std::string("Unexpected character: ") + ch);  // panic! in the reference (parser.rs:32)
    return v;
}
// one sequence line appended to a code vector: table translation in bulk, the (rare) bad character found afterwards
// std::vector::resize zero-fills: for the code bytes of a FASTA file and the sorted copy of the sequences (650 MB per million 650 bp
// references, written three times on the way from the text to the Tree) that is a pass over memory the real writer behind it overwrites
// entirely.  With this allocator resize leaves the bytes alone.
template <typename T>
struct DefaultInitAlloc : std::allocator<T> {
    template <typename U>
    struct rebind {
        using other = DefaultInitAlloc<U>;
    };
    template <typename U>
    void construct(U* p) noexcept {
        ::new (static_cast<void*>(p)) U;
    }
    template <typename U, typename... A>
    void construct(U* p, A&&... a) {
        ::new (static_cast<void*>(p)) U(std::forward<A>(a)...);
    }
};
using ByteVec = std::vector<u8, DefaultInitAlloc<u8>>;

static inline void append_codes(ByteVec& codes, const char* b, const char* e) {
    const size_t at = codes.size(), n = (size_t)(e - b);
    codes.resize(at + n);
    u8* out = codes.data() + at;
    u8 all = 0xFF;
    for (size_t i = 0; i < n; ++i) {
        const u8 v = kDna.t[(unsigned char)b[i]];
        out[i] = v;
        all &= (u8)(v ? 0xFF : 0x00);
    }
    if (!all)
        for (size_t i = 0; i < n; ++i) map_dna_char(b[i]);  // throws at the first offender, as the reference panics
}

// One logical FASTA line: str::lines() then trim() (parser.rs:53-57).  Returns false at end of input.
struct LineReader {
    const char* p;
    const char* end;
    LineReader(const char* text, size_t len) : p(text), end(text + len) {}
    static bool ws(unsigned char c) { return c == ' ' || (c >= 9 && c <= 13); }
    bool next(const char** b, const char** e) {
        while (p < end) {
            const char* nl = (const char*)memchr(p, '\n', (size_t)(end - p));
            const char* le = nl ? nl : end;
            const char* lb = p;
            p = nl ? nl + 1 : end;
            while (lb < le && ws((unsigned char)*lb)) ++lb;
            while (le > lb && ws((unsigned char)le[-1])) --le;
            if (le > lb && *lb != ';') {  // filter(|l| !l.is_empty() && !l.starts_with(';'))
                *b = lb;
                *e = le;
                return true;
            }
        }
        return false;
    }
};

// regex `tax=([^;]+);` -- leftmost match (parser.rs:50)
static bool capture_tax(const char* b, const char* e, std::string* out) {
    static const char pat[] = "tax=";
    const char* from = b;
    while (true) {
        const char* p = std::search(from, e, pat, pat + 4);
        if (p == e) return false;
        const char* s = p + 4;
        const char* q = s;
        while (q < e && *q != ';') ++q;
        if (q > s && q < e) {
            out->assign(s, q);
            return true;
        }
        from = p + 1;
    }
}

// ---- Tree (tree.rs:36-43) in flat form --------------------------------------------------------------------------
struct Tree {
    size_t num_tips = 0;
    std::vector<std::string> lineages;  // sorted (tree.rs:128-131)
    std::vector<u64> seq_off;           // sorted sequences, 4-bit codes
    ByteVec seq_codes;
    std::vector<u64> csr_off;  // k_mer_map (tree.rs:41): 65537 offsets.  Built on first use (ensure_csr): the device builds its own
    std::vector<u32> csr_ids;  // index from the sorted sequences, so the classification path never needs the lists on the host
    bool has_csr = false;
    std::mutex csr_mtx;
    // sequences (tree.rs:40, `HashMap<Vec<u8>, Vec<u32>>`): open addressing over a 64-bit hash of the code bytes; a slot holds the FIRST
    // reference of a group of identical sequences, the group's other members hang off it in ascending order (ex_next)
    std::vector<u32> ex_head;  // id + 1, 0 = empty
    std::vector<u32> ex_tag;   // high half of the hash of the slot's sequence (pre-filter before the memcmp)
    std::vector<u32> ex_next;  // [num refs] next reference with the same sequence, kNone = last of its group
    size_t ex_mask = 0;
    static constexpr u32 kNone = 0xFFFFFFFFu;
    // Inner / Taxon (and non-leaf Sequence) nodes, BFS order, children contiguous
    std::vector<u32> node_lo, node_hi, child_first, child_count;
    std::vector<u8> node_type;
    std::vector<u8> ref_levels;

    // four independent multiply-xor lanes over 32 bytes per round (a single lane is a 7-cycle dependency chain per 8 bytes: at
    // 650 bytes per query and two hashes per query that alone was a third of the driver's per-query host time)
    static u64 hash_bytes(const u8* p, size_t n) {
        const u64 k0 = 0x9E3779B97F4A7C15ull, k1 = 0xC2B2AE3D27D4EB4Full, k2 = 0x165667B19E3779F9ull, k3 = 0xD6E8FEB86659FD93ull;
        u64 a = k0 ^ (n * 0xff51afd7ed558ccdull), b = k1, c = k2, d = k3;
        auto round = [&](const u64* w) {
            a = (a ^ w[0]) * k1;
            a ^= a >> 29;
            b = (b ^ w[1]) * k2;
            b ^= b >> 29;
            c = (c ^ w[2]) * k3;
            c ^= c >> 29;
            d = (d ^ w[3]) * k0;
            d ^= d >> 29;
        };
        size_t i = 0;
        u64 w[4];
        for (; i + 32 <= n; i += 32) {
            memcpy(w, p + i, 32);
            round(w);
        }
        if (i < n) {
            w[0] = w[1] = w[2] = w[3] = 0;
            memcpy(w, p + i, n - i);
            round(w);
        }
        u64 h = (a ^ ((b << 17) | (b >> 47))) * k2;
        h ^= c ^ ((d << 31) | (d >> 33));
        h *= k1;
        return h ^ (h >> 32);
    }

    bool same_seq(u32 id, const u8* seq, size_t len) const {
        const size_t l = (size_t)(seq_off[id + 1] - seq_off[id]);
        return l == len && (len == 0 || memcmp(seq_codes.data() + seq_off[id], seq, len) == 0);
    }
    // first reference carrying exactly this sequence, or kNone
    u32 exact_head(const u8* seq, size_t len, u64 h) const {
        if (ex_head.empty()) return kNone;
        const u32 tag = (u32)(h >> 32);
        for (size_t at = (size_t)h & ex_mask;; at = (at + 1) & ex_mask) {
            const u32 e = ex_head[at];
            if (!e) return kNone;
            if (ex_tag[at] == tag && same_seq(e - 1, seq, len)) return e - 1;
        }
    }
    // tree.sequences.get(seq) (raxtax.rs:42)
    void exact(const u8* seq, size_t len, std::vector<u32>* out) const { exact_h(seq, len, hash_bytes(seq, len), out); }
    void exact_h(const u8* seq, size_t len, u64 h, std::vector<u32>* out) const {
        out->clear();
        for (u32 id = exact_head(seq, len, h); id != kNone; id = ex_next[id]) out->push_back(id);
    }
    void hash_all(std::vector<u64>& hashes) const;  // hash of every reference sequence, in parallel
    // sequences.entry(sequence).or_default().push(idx) for idx = 0 .. n-1 (tree.rs:109-112)
    void build_exact() {
        const size_t n = seq_off.empty() ? 0 : seq_off.size() - 1;
        size_t cap = 64;
        while (cap < n * 2) cap <<= 1;
        ex_head.assign(cap, 0);
        ex_tag.assign(cap, 0);
        ex_next.assign(n, kNone);
        ex_mask = cap - 1;
        std::vector<u32> tail(n, 0);  // tail[head] = last member of head's group so far
        std::vector<u64> hashes(n);
        hash_all(hashes);
        for (size_t idx = 0; idx < n; ++idx) {
            const u8* sp = seq_codes.data() + seq_off[idx];
            const size_t sl = (size_t)(seq_off[idx + 1] - seq_off[idx]);
            const u64 h = hashes[idx];
            const u32 tag = (u32)(h >> 32);
            for (size_t at = (size_t)h & ex_mask;; at = (at + 1) & ex_mask) {
                const u32 e = ex_head[at];
                if (!e) {
                    ex_head[at] = (u32)idx + 1;
                    ex_tag[at] = tag;
                    tail[idx] = (u32)idx;
                    break;
                }
                if (ex_tag[at] == tag && same_seq(e - 1, sp, sl)) {
                    ex_next[tail[e - 1]] = (u32)idx;
                    tail[e - 1] = (u32)idx;
                    break;
                }
            }
        }
    }
};

void Tree::hash_all(std::vector<u64>& hashes) const {
    const size_t n = hashes.size(), blocks = (n + 16383) / 16384;
    parallel_for(blocks, [&](size_t b) {
        const size_t hi = std::min(n, (b + 1) * 16384);
        for (size_t idx = b * 16384; idx < hi; ++idx)
            hashes[idx] = hash_bytes(seq_codes.data() + seq_off[idx], (size_t)(seq_off[idx + 1] - seq_off[idx]));
    });
}

template <typename F>
static inline void for_each_kmer(const u8* s, size_t n, F&& f);

// k_mer_map as CSR (tree.rs:114-123 windowing, 134-137 unique + sorted): a counting pass and a fill pass over the sorted sequences
static void build_csr(Tree& t) {
    const size_t n = t.num_tips;
    std::vector<u32> kcount(65537, 0), last(65536, 0xFFFFFFFFu);
    for (size_t idx = 0; idx < n; ++idx) {
        for_each_kmer(t.seq_codes.data() + t.seq_off[idx], (size_t)(t.seq_off[idx + 1] - t.seq_off[idx]), [&](u16 k) {
            if (last[k] != (u32)idx) {
                last[k] = (u32)idx;
                kcount[k + 1]++;
            }
        });
    }
    t.csr_off.assign(65537, 0);
    for (u32 k = 0; k < 65536; ++k) t.csr_off[k + 1] = t.csr_off[k] + kcount[k + 1];
    t.csr_ids.resize(t.csr_off[65536]);
    std::vector<u64> pos(t.csr_off.begin(), t.csr_off.end() - 1);
    std::fill(last.begin(), last.end(), 0xFFFFFFFFu);
    for (size_t idx = 0; idx < n; ++idx) {
        for_each_kmer(t.seq_codes.data() + t.seq_off[idx], (size_t)(t.seq_off[idx + 1] - t.seq_off[idx]), [&](u16 k) {
            if (last[k] != (u32)idx) {
                last[k] = (u32)idx;
                t.csr_ids[pos[k]++] = (u32)idx;
            }
        });
    }
    t.has_csr = true;
}
static void ensure_csr(const Tree& ct) {
    Tree& t = const_cast<Tree&>(ct);
    std::lock_guard<std::mutex> g(t.csr_mtx);
    if (!t.has_csr) build_csr(t);
}

struct BNode {  // build-time node (tree.rs:189-194)
    std::string label;
    u32 lo, hi;
    u8 type;  // 0 Inner, 1 Taxon, 2 Sequence
    std::vector<u32> children;  // materialised children only
    bool trailing_seq = false;  // the last child is an implicit (childless) Sequence leaf labelled like this node
};

static inline int two_bit(u8 c) {  // utils.rs:17-25
    switch (c) {
        case 1: return 0;
        case 2: return 1;
        case 4: return 2;
        case 8: return 3;
        default: return -1;
    }
}

template <typename F>
static inline void for_each_kmer(const u8* s, size_t n, F&& f) {  // windows(8) with the None-on-ambiguity fold (utils.rs:29-38)
    u32 val = 0, run = 0;
    for (size_t i = 0; i < n; ++i) {
        int t = two_bit(s[i]);
        if (t < 0) {
            run = 0;
            continue;
        }
        val = ((val << 2) | (u32)t) & 0xFFFFu;
        if (++run >= 8) f((u16)val);
    }
}

// flatten: BFS numbering, children contiguous.  Implicit Sequence leaves are dropped: they can neither be emitted
// nor change a decision of Lineage::eval_recurse (lineage.rs:119-179) because their parent is never Inner.
static void flatten_nodes(const std::vector<BNode>& nodes, Tree& tree) {
    const size_t nn = nodes.size();
    std::vector<u32> bfs;
    bfs.reserve(nn);
    bfs.push_back(0);
    tree.node_lo.reserve(nn);
    for (size_t head = 0; head < bfs.size(); ++head) {
        const BNode& b = nodes[bfs[head]];
        if (b.type == 0 && b.trailing_seq) throw Error("internal: Inner node with a Sequence child");
        tree.node_lo.push_back(b.lo);
        tree.node_hi.push_back(b.hi);
        tree.node_type.push_back(b.type);
        tree.child_first.push_back(b.children.empty() ? 0u : (u32)bfs.size());
        tree.child_count.push_back((u32)b.children.size());
        for (u32 c : b.children) bfs.push_back(c);
    }
}

// Tree::new (tree.rs:47-140)
static std::unique_ptr<Tree> tree_new(std::vector<std::string> lineages, const u64* seq_off, const u8* codes, bool eager_csr = false) {
    const size_t n = lineages.size();
    if (n > 0xFFFFFFFFull)
        throw Error("Too many database sequences to run with 32-bit indices!");  // tree.rs:24-31
    auto tree = std::make_unique<Tree>();
    const bool timing = getenv("RXH_TIMING") != nullptr;  // phase times of the build on stderr
    auto t_prev = std::chrono::steady_clock::now();
    auto lap = [&](const char* what) {
        if (!timing) return;
        auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[rxh tree_new] %-28s %8.3f s\n", what, std::chrono::duration<double>(now - t_prev).count());
        t_prev = now;
    };
    std::vector<u32> order(n);
    std::iota(order.begin(), order.end(), 0u);
    {   // tree.rs:54: stable sort by lineage -- runs sorted in parallel, then merged pairwise (std::inplace_merge is stable)
        auto less = [&](u32 a, u32 b) { return lineages[a].compare(lineages[b]) < 0; };
        size_t runs = 1;
        while (runs < host_threads() && n / (runs * 2) >= 65536) runs *= 2;
        std::vector<size_t> cut(runs + 1);
        for (size_t r = 0; r <= runs; ++r) cut[r] = n * r / runs;
        parallel_for(runs, [&](size_t r) { std::stable_sort(order.begin() + (ptrdiff_t)cut[r], order.begin() + (ptrdiff_t)cut[r + 1], less); });
        for (size_t w = 1; w < runs; w *= 2)
            parallel_for(runs / (2 * w), [&](size_t k) {
                const size_t lo = cut[2 * w * k], mid = cut[2 * w * k + w], hi = cut[2 * w * k + 2 * w];
                std::inplace_merge(order.begin() + (ptrdiff_t)lo, order.begin() + (ptrdiff_t)mid, order.begin() + (ptrdiff_t)hi, less);
            });
    }

    lap("stable sort by lineage");
    std::vector<BNode> nodes;
    nodes.reserve(n / 2 + 16);
    nodes.push_back(BNode{"root", 0, 1, 0, {}, false});
    size_t confidence_idx = 0;
    tree->seq_off.assign(n + 1, 0);
    tree->ref_levels.resize(n);
    for (size_t i = 0; i < n; ++i) tree->seq_off[i + 1] = tree->seq_off[i] + (seq_off[order[i] + 1] - seq_off[order[i]]);
    tree->seq_codes.resize(tree->seq_off[n]);
    {   // the sequences in sorted order (tree.rs:109-112 keeps them as the keys of `sequences`)
        const size_t blocks = (n + 16383) / 16384;
        parallel_for(blocks, [&](size_t b) {
            const size_t hi = std::min(n, (b + 1) * 16384);
            for (size_t idx = b * 16384; idx < hi; ++idx) {
                const u64 o = seq_off[order[idx]], l = seq_off[order[idx] + 1] - o;
                if (l) memcpy(tree->seq_codes.data() + tree->seq_off[idx], codes + o, l);
            }
        });
    }
    lap("sequences copied");
    // the lineages in sorted order (tree.rs:128-131) before the node walk reads them: the walk then goes through them front to back
    // instead of chasing order[] into the input
    tree->lineages.resize(n);
    {
        const size_t blocks = (n + 16383) / 16384;
        parallel_for(blocks, [&](size_t b) {
            const size_t hi = std::min(n, (b + 1) * 16384);
            for (size_t idx = b * 16384; idx < hi; ++idx) tree->lineages[idx] = std::move(lineages[order[idx]]);
        });
    }
    lap("lineages in sorted order");
    // ---- nodes (tree.rs:56-126).  The references are sorted and the reference compares a level's label with the LAST child only
    // (tree.rs:77-96), so which nodes a reference creates is decided by the lineage right before it alone: it re-uses that one's nodes on
    // the leading levels the two share and opens new ones below; when the previous lineage is a prefix of this one, level-wise, its final
    // node still has the implicit Sequence leaf as last child (tree.rs:102-106), and a next level repeating that node's label walks INTO
    // the leaf.  That makes the string work -- levels, shared levels, the repeated-label test -- independent per reference (parallel);
    // what is left for the sequential pass is integer bookkeeping: node ids in creation order, child lists, ranges.
    // RXH_TREE_WALK=1 runs the level-by-level walk of round 1 instead (kept as the statement the tests compare with).
    if (getenv("RXH_TREE_WALK") == nullptr) {
        std::vector<u8> n_lev(n), n_shared(n), degenerate(n);
        std::atomic<bool> too_deep{false};
        {
            const size_t blocks = (n + 16383) / 16384;
            parallel_for(blocks, [&](size_t b) {
                const size_t hi = std::min(n, (b + 1) * 16384);
                for (size_t idx = b * 16384; idx < hi; ++idx) {
                    const std::string& cur = tree->lineages[idx];
                    const size_t levels = (size_t)std::count(cur.begin(), cur.end(), ',') + 1;
                    if (levels > 255) {
                        too_deep.store(true);
                        continue;
                    }
                    n_lev[idx] = (u8)levels;
                    tree->ref_levels[idx] = (u8)levels;
                    size_t shared = 0;
                    bool deg = false;
                    if (idx > 0) {
                        const std::string& prev = tree->lineages[idx - 1];
                        const size_t m = std::min(prev.size(), cur.size());
                        size_t k = 0, last_comma = std::string::npos;  // the last comma inside the common part
                        while (k < m && prev[k] == cur[k]) {
                            if (cur[k] == ',') {
                                ++shared;
                                last_comma = k;
                            }
                            ++k;
                        }
                        if (k == m && prev.size() == cur.size()) {
                            ++shared;  // the same lineage again
                        } else if (k == prev.size() && k < cur.size() && cur[k] == ',') {
                            ++shared;  // the previous lineage is a prefix of this one, level-wise: its final node is on this one's path
                            // label of the previous lineage's last level (= this one's level shared - 1) against this one's next level
                            const size_t a0 = last_comma == std::string::npos ? 0 : last_comma + 1, a1 = k;
                            const size_t b0 = k + 1;
                            size_t b1 = cur.find(',', b0);
                            if (b1 == std::string::npos) b1 = cur.size();
                            deg = (a1 - a0) == (b1 - b0) && cur.compare(a0, a1 - a0, cur, b0, b1 - b0) == 0;
                        }
                    }
                    n_shared[idx] = (u8)std::min<size_t>(shared, 255);
                    degenerate[idx] = deg ? 1 : 0;
                }
            });
        }
        if (too_deep.load()) throw Error("lineage with more than 255 ranks");
        std::vector<u32> path;  // node of every level of the previous reference
        for (size_t idx = 0; idx < n; ++idx) {
            const size_t levels = n_lev[idx];
            const size_t shared = std::min<size_t>(std::min<size_t>(n_shared[idx], path.size()), levels);
            for (size_t l = shared; l < path.size(); ++l) nodes[path[l]].hi = (u32)idx;  // the previous reference's nodes below the shared levels end here
            path.resize(levels);
            for (size_t level = shared; level < levels; ++level) {
                const u32 parent = level == 0 ? 0u : path[level - 1];
                const u32 id = (u32)nodes.size();
                if (level == shared && degenerate[idx])
                    nodes.push_back(BNode{std::string(), (u32)idx - 1, (u32)idx, 2, {}, false});  // the Sequence leaf of the reference before (tree.rs:102-106)
                else
                    nodes.push_back(BNode{std::string(), (u32)idx, (u32)idx + 1, (u8)(level == levels - 1 ? 1 : 0), {}, false});
                nodes[parent].children.push_back(id);
                nodes[parent].trailing_seq = false;
                path[level] = id;
            }
            nodes[path[levels - 1]].trailing_seq = true;  // add_child(Sequence(label, ci-1)) (tree.rs:102-106)
            confidence_idx += 1;
        }
        for (size_t l = 0; l < path.size(); ++l) nodes[path[l]].hi = (u32)n;
    } else {
        struct LevelView {
            const char* p;
            size_t n;
            bool equals(const std::string& s) const { return s.size() == n && (n == 0 || memcmp(s.data(), p, n) == 0); }
            std::string str() const { return std::string(p, n); }
        };
        std::vector<LevelView> levels;
        // The references arrive sorted, so a lineage shares its leading levels with the one before it, and on those levels the walk of
        // tree.rs:77-96 finds "the last child carries my label" -- the node the previous reference went through (it is still the last
        // child: everything added since went below it, and a node with children never has a trailing Sequence leaf).  Those levels only
        // extend the node ranges; label comparisons and the split at ',' start at the first level that differs.
        std::vector<u32> path;       // node of every level of the previous reference
        const std::string* prev = nullptr;
        for (size_t idx = 0; idx < n; ++idx) {  // tree.rs:56-126
            const std::string& lineage = tree->lineages[idx];
            if (idx + 8 < n) __builtin_prefetch(tree->lineages[idx + 8].data());
            size_t shared = 0;  // leading levels equal to the previous lineage's
            if (prev) {
                const size_t m = std::min(prev->size(), lineage.size());
                size_t k = 0;
                while (k < m && (*prev)[k] == lineage[k]) ++k;
                const bool whole = k == m && prev->size() == lineage.size();  // the same lineage again
                for (size_t j = 0; j < k; ++j)
                    if (lineage[j] == ',') ++shared;
                if (whole || (k == prev->size() && k < lineage.size() && lineage[k] == ','))
                    ++shared;  // the same lineage again / the previous one is a strict prefix of this one, level-wise (variable depth)
                shared = std::min(shared, path.size());
            }
            levels.clear();
            {
                size_t start = 0;
                while (true) {
                    size_t p = lineage.find(',', start);
                    if (p == std::string::npos) {
                        levels.push_back(LevelView{lineage.data() + start, lineage.size() - start});
                        break;
                    }
                    levels.push_back(LevelView{lineage.data() + start, p - start});
                    start = p + 1;
                }
            }
            if (levels.size() > 255) throw Error("lineage with more than 255 ranks");
            tree->ref_levels[idx] = (u8)levels.size();
            const size_t last_level = levels.size() - 1;
            shared = std::min(shared, levels.size());
            path.resize(levels.size());
            u32 cur = 0;
            for (size_t level = 0; level < levels.size(); ++level) {
                if (level < shared) {  // the previous reference's node of this level: only its range grows (tree.rs:95-96)
                    nodes[cur].hi = (u32)confidence_idx + 1;
                    if (level == last_level) confidence_idx += 1;
                    cur = path[level];
                    continue;
                }
                const LevelView& label = levels[level];
                const u8 nt = level == last_level ? 1 : 0;
                BNode& c = nodes[cur];
                bool need_new = true;
                u32 next = 0;
                if (c.trailing_seq) {  // last child is the Sequence leaf carrying this node's own label (tree.rs:102-106)
                    if (label.equals(c.label)) {
                        // degenerate lineage (a rank repeats its parent's label): the reference walks INTO the Sequence node
                        BNode s{c.label, c.hi - 1, c.hi, 2, {}, false};
                        next = (u32)nodes.size();
                        nodes.push_back(std::move(s));
                        nodes[cur].children.push_back(next);
                        nodes[cur].trailing_seq = false;
                        need_new = false;
                    }
                } else if (!c.children.empty()) {
                    next = c.children.back();
                    if (label.equals(nodes[next].label)) need_new = false;
                }
                if (need_new) {
                    next = (u32)nodes.size();
                    nodes.push_back(BNode{label.str(), (u32)confidence_idx, (u32)confidence_idx + 1, nt, {}, false});
                    nodes[cur].children.push_back(next);
                    nodes[cur].trailing_seq = false;
                }
                nodes[cur].hi = (u32)confidence_idx + 1;
                if (level == last_level) confidence_idx += 1;
                cur = next;
                path[level] = cur;
            }
            nodes[cur].trailing_seq = true;  // add_child(Sequence(label, ci-1)) (tree.rs:102-106)
            nodes[cur].hi = (u32)confidence_idx;  // tree.rs:107
            prev = &lineage;
        }
    }
    lap("nodes");
    tree->build_exact();  // tree.rs:109-112
    lap("sequence map");
    nodes[0].hi = (u32)confidence_idx;  // tree.rs:127
    tree->num_tips = confidence_idx;    // tree.rs:138

    if (eager_csr) build_csr(*tree);  // tree.rs:114-123,134-137; otherwise on first use
    lap(eager_csr ? "k_mer_map (CSR), 2 passes" : "k_mer_map deferred");
    flatten_nodes(nodes, *tree);
    lap("flatten");
    return tree;
}

// ---- binary database (tree.rs:146-164): bincode 1.3 default options = little-endian, fixed-width integers, usize and all
// lengths as u64, enum variants as u32, struct fields in declaration order (tree.rs:36-43, 181-194), no framing -------------
struct BinWriter {
    FILE* f;
    bool ok = true;
    void raw(const void* p, size_t n) {
        if (ok && n && fwrite(p, 1, n, f) != n) ok = false;
    }
    void u64v(u64 v) { raw(&v, 8); }
    void u32v(u32 v) { raw(&v, 4); }
    void str(const std::string& x) {
        u64v(x.size());
        raw(x.data(), x.size());
    }
};

// The full Node tree of Tree::new (tree.rs:56-127), every Sequence leaf included, as a pure function of the sorted lineages;
// written depth-first in the field order label, confidence_range, children, node_type.
struct FullNode {
    std::string label;
    u64 lo, hi;
    u32 type;
    std::vector<u32> children;
};
static void full_nodes(const std::vector<std::string>& lineages, std::vector<FullNode>& nodes) {
    nodes.clear();
    nodes.push_back(FullNode{"root", 0, 1, 0, {}});
    u64 ci = 0;
    std::vector<std::string> levels;
    for (const std::string& lineage : lineages) {
        levels.clear();
        for (size_t start = 0;;) {
            const size_t p = lineage.find(',', start);
            if (p == std::string::npos) {
                levels.emplace_back(lineage, start);
                break;
            }
            levels.emplace_back(lineage, start, p - start);
            start = p + 1;
        }
        const size_t last = levels.size() - 1;
        u32 cur = 0;
        for (size_t level = 0; level < levels.size(); ++level) {
            const bool have = !nodes[cur].children.empty();
            if (!have || nodes[nodes[cur].children.back()].label != levels[level]) {
                const u32 id = (u32)nodes.size();
                nodes.push_back(FullNode{levels[level], ci, ci + 1, level == last ? 1u : 0u, {}});
                nodes[cur].children.push_back(id);
            }
            nodes[cur].hi = ci + 1;
            if (level == last) ci += 1;
            cur = nodes[cur].children.back();
        }
        const u32 id = (u32)nodes.size();
        nodes.push_back(FullNode{nodes[cur].label, ci - 1, ci, 2, {}});
        nodes[cur].children.push_back(id);
        nodes[cur].hi = ci;
    }
    nodes[0].hi = ci;
}
static void write_node(BinWriter& w, const std::vector<FullNode>& nodes, u32 id) {
    const FullNode& n = nodes[id];
    w.str(n.label);
    w.u64v(n.lo);
    w.u64v(n.hi);
    w.u64v(n.children.size());
    for (u32 c : n.children) write_node(w, nodes, c);
    w.u32v(n.type);
}

// Tree::save_to_file (tree.rs:146-152)
static void save_bin(const Tree& t, const char* path) {
    FILE* f = fopen(path, "wb");
    if (!f) throw Error(std::string("cannot create ") + path);
    BinWriter w{f};
    {
        std::vector<FullNode> nodes;
        full_nodes(t.lineages, nodes);
        write_node(w, nodes, 0);
    }
    w.u64v(t.lineages.size());
    for (const auto& l : t.lineages) w.str(l);
    {   // sequences: HashMap<Vec<u8>, Vec<u32>> (tree.rs:40), any order; one entry per distinct sequence
        u64 distinct = 0;
        std::vector<std::vector<u32>> groups;
        for (const u32 e : t.ex_head) {
            if (!e) continue;
            std::vector<u32> same;
            for (u32 id = e - 1; id != Tree::kNone; id = t.ex_next[id]) same.push_back(id);  // ascending
            groups.push_back(std::move(same));
            ++distinct;
        }
        w.u64v(distinct);
        for (const auto& g : groups) {
            const u64 o = t.seq_off[g[0]], l = t.seq_off[g[0] + 1] - o;
            w.u64v(l);
            w.raw(t.seq_codes.data() + o, l);
            w.u64v(g.size());
            w.raw(g.data(), g.size() * 4);
        }
    }
    ensure_csr(t);
    w.u64v(65536);
    for (u32 k = 0; k < 65536; ++k) {
        const u64 a = t.csr_off[k], b = t.csr_off[k + 1];
        w.u64v(b - a);
        w.raw(t.csr_ids.data() + a, (b - a) * 4);
    }
    w.u64v(t.num_tips);
    const bool ok = w.ok;
    if (fclose(f) != 0 || !ok) throw Error(std::string("write error on ") + path);
}

struct BinReader {
    const u8* p;
    const u8* end;
    struct Fail {};
    void need(u64 n) const {
        if ((u64)(end - p) < n) throw Fail{};
    }
    u64 u64v() {
        need(8);
        u64 v;
        memcpy(&v, p, 8);
        p += 8;
        return v;
    }
    u32 u32v() {
        need(4);
        u32 v;
        memcpy(&v, p, 4);
        p += 4;
        return v;
    }
    const u8* bytes(u64 n) {
        need(n);
        const u8* r = p;
        p += n;
        return r;
    }
};
// leaf_seq: set when the node is a Sequence node without children in the file -- the implicit leaves Tree::new hangs under every
// taxon (tree.rs:102-106), which tree_new() above never materialises either
static u32 read_node(BinReader& r, std::vector<BNode>& nodes, int depth, bool* leaf_seq) {
    if (depth > 300) throw BinReader::Fail{};
    const u64 ll = r.u64v();
    const u8* lb = r.bytes(ll);
    const u64 lo = r.u64v(), hi = r.u64v();
    const u64 nc = r.u64v();
    if (nc > (u64)(r.end - r.p) / 28) throw BinReader::Fail{};  // a node is at least 28 bytes
    if (lo > 0xFFFFFFFFull || hi > 0xFFFFFFFFull) throw BinReader::Fail{};
    const u32 id = (u32)nodes.size();
    nodes.push_back(BNode{std::string((const char*)lb, (size_t)ll), (u32)lo, (u32)hi, 0, {}, false});
    std::vector<u32> kids;
    for (u64 c = 0; c < nc; ++c) {
        const size_t before = nodes.size();
        bool leaf = false;
        const u32 cid = read_node(r, nodes, depth + 1, &leaf);
        if (leaf) nodes.resize(before);
        else kids.push_back(cid);
    }
    const u32 ty = r.u32v();
    if (ty > 2) throw BinReader::Fail{};
    nodes[id].type = (u8)ty;
    nodes[id].children = std::move(kids);
    *leaf_seq = ty == 2 && nc == 0;
    return id;
}

// Tree::load_from_file (tree.rs:154-164): nullptr when the bytes do not deserialise as a Tree (the caller then parses FASTA,
// parser.rs:37-44).  Databases written with the reference's `huge_db` feature (u64 ids, tree.rs:18-19) do not deserialise here.
static std::unique_ptr<Tree> load_bin(const u8* data, size_t len) {
    try {
        BinReader r{data, data + len};
        auto tree = std::make_unique<Tree>();
        std::vector<BNode> nodes;
        bool root_leaf = false;
        read_node(r, nodes, 0, &root_leaf);
        const u64 n = r.u64v();
        if (n > 0xFFFFFFFFull || n > (u64)(r.end - r.p) / 8) throw BinReader::Fail{};
        tree->lineages.resize(n);
        tree->ref_levels.resize(n);
        for (u64 i = 0; i < n; ++i) {
            const u64 l = r.u64v();
            const u8* b = r.bytes(l);
            tree->lineages[i].assign((const char*)b, (size_t)l);
            const size_t levels = (size_t)std::count(tree->lineages[i].begin(), tree->lineages[i].end(), ',') + 1;
            if (levels > 255) throw BinReader::Fail{};
            tree->ref_levels[i] = (u8)levels;
        }
        // sequences: key -> ids; every reference id must occur exactly once
        const u64 n_keys = r.u64v();
        if (n_keys > n) throw BinReader::Fail{};
        std::vector<const u8*> key_of(n, nullptr);
        std::vector<u64> len_of(n, 0);
        for (u64 k = 0; k < n_keys; ++k) {
            const u64 kl = r.u64v();
            const u8* kb = r.bytes(kl);
            const u64 ni = r.u64v();
            if (ni > n) throw BinReader::Fail{};
            const u8* ib = r.bytes(ni * 4);
            for (u64 j = 0; j < ni; ++j) {
                u32 id;
                memcpy(&id, ib + 4 * j, 4);
                if (id >= n || key_of[id]) throw BinReader::Fail{};
                key_of[id] = kb ? kb : data;
                len_of[id] = kl;
            }
        }
        tree->seq_off.assign(n + 1, 0);
        for (u64 i = 0; i < n; ++i) {
            if (!key_of[i]) throw BinReader::Fail{};
            tree->seq_off[i + 1] = tree->seq_off[i] + len_of[i];
        }
        tree->seq_codes.resize(tree->seq_off[n]);
        for (u64 i = 0; i < n; ++i) {
            if (len_of[i]) memcpy(tree->seq_codes.data() + tree->seq_off[i], key_of[i], len_of[i]);
        }
        tree->build_exact();
        // k_mer_map
        if (r.u64v() != 65536) throw BinReader::Fail{};
        tree->csr_off.assign(65537, 0);
        for (u32 k = 0; k < 65536; ++k) {
            const u64 l = r.u64v();
            if (l > n) throw BinReader::Fail{};
            const u8* b = r.bytes(l * 4);
            const size_t at = tree->csr_ids.size();
            tree->csr_ids.resize(at + l);
            if (l) memcpy(tree->csr_ids.data() + at, b, l * 4);
            u32 prev = 0;
            for (u64 j = 0; j < l; ++j) {  // ascending and unique (tree.rs:134-137)
                const u32 id = tree->csr_ids[at + j];
                if (id >= n || (j && id <= prev)) throw BinReader::Fail{};
                prev = id;
            }
            tree->csr_off[k + 1] = tree->csr_off[k] + l;
        }
        tree->has_csr = true;
        tree->num_tips = r.u64v();
        if (tree->num_tips != n || nodes.empty() || nodes[0].lo != 0 || nodes[0].hi != n) throw BinReader::Fail{};
        flatten_nodes(nodes, *tree);
        for (size_t i = 0; i < tree->node_lo.size(); ++i)
            if (tree->node_lo[i] > tree->node_hi[i] || tree->node_hi[i] > n) throw BinReader::Fail{};
        return tree;
    } catch (const BinReader::Fail&) {
        return nullptr;
    } catch (const Error&) {
        return nullptr;
    }
}

// ---- FASTA parsing (parser.rs:46-154), by blocks and in parallel --------------------------------------------------------------
// The reference reads the whole file into a String and walks its lines on one thread.  Here the text arrives in blocks (a whole
// buffer, or what a gz / plain reader has produced so far), every block is cut at header lines into pieces that are parsed in
// parallel, and the per-record rules of the reference are applied to the pieces' records in file order afterwards:
//   references (parser.rs:46-105): every header contributes a label; a sequence is pushed at the NEXT header only if it is not empty,
//   the last one unconditionally; more labels than sequences is the "does not match" error
//   queries (parser.rs:117-154): a record whose sequence is empty is dropped, label included, unless it is the last one
struct FastaPiece {
    std::vector<std::string> labels;  // lineage (references) or the whole header line after '>' (queries), one per header
    std::vector<u64> lens;            // codes that follow that header inside the piece
    ByteVec codes;
    std::string error;                // what the serial parser would have raised first inside this piece
    bool headless_codes = false;      // sequence lines before the piece's first header (only the very first piece can have them)
};

static void parse_piece(const char* b0, const char* e0, bool reference, FastaPiece& out) {
    LineReader lr(b0, (size_t)(e0 - b0));
    const char *b, *e;
    out.codes.reserve((size_t)(e0 - b0));
    try {
        while (lr.next(&b, &e)) {
            if (*b == '>') {
                if (reference) {
                    std::string lineage;
                    if (!capture_tax(b + 1, e, &lineage)) throw Error("Unexpected taxonomical annotation detected in label " + std::string(b + 1, e));
                    out.labels.push_back(std::move(lineage));
                } else {
                    out.labels.emplace_back(b + 1, e);
                }
                out.lens.push_back(0);
            } else {
                if (out.lens.empty()) {
                    out.headless_codes = true;
                    return;  // "Not a valid FASTA file": decided by the caller (only possible in the first piece)
                }
                const size_t before = out.codes.size();
                append_codes(out.codes, b, e);
                out.lens.back() += out.codes.size() - before;
            }
        }
    } catch (const std::exception& ex) {
        out.error = ex.what();
    }
}

struct FastaAccumulator {
    const bool reference;
    bool any_line = false;
    std::vector<std::string> labels;  // one per header so far
    std::vector<u64> lens;
    ByteVec codes;
    std::vector<FastaPiece> pieces;  // kept between blocks: their buffers are reused instead of being mapped and faulted in again
    explicit FastaAccumulator(bool ref) : reference(ref) {}

    // [b, e) starts at a header line (or at the start of the file) and ends at a record boundary (or at the end of the file)
    void add_block(const char* b, const char* e) {
        if (b >= e) return;
        // cut at "\n>" into pieces of ~4 MB
        std::vector<const char*> cut{b};
        size_t target = 4u << 20;
        if (const char* ev = getenv("RXH_FASTA_PIECE")) target = (size_t)std::max(1, atoi(ev));  // test hook
        const char* p = b;
        while ((size_t)(e - p) > target) {
            const char* q = p + target;
            const char* hit = nullptr;
            while (q < e) {
                const char* nl = (const char*)memchr(q, '\n', (size_t)(e - q));
                if (!nl || nl + 1 >= e) break;
                if (nl[1] == '>') {
                    hit = nl + 1;
                    break;
                }
                q = nl + 1;
            }
            if (!hit) break;
            cut.push_back(hit);
            p = hit;
        }
        cut.push_back(e);
        const size_t n_pieces = cut.size() - 1;
        if (pieces.size() < n_pieces) pieces.resize(n_pieces);
        parallel_for(n_pieces, [&](size_t i) {
            FastaPiece& pc = pieces[i];
            pc.labels.clear();
            pc.lens.clear();
            pc.codes.clear();
            pc.error.clear();
            pc.headless_codes = false;
            parse_piece(cut[i], cut[i + 1], reference, pc);
        });
        std::vector<size_t> at(n_pieces + 1, codes.size());
        for (size_t i = 0; i < n_pieces; ++i) {
            FastaPiece& pc = pieces[i];
            if (pc.headless_codes) {
                if (labels.empty() && i == 0) throw Error("Not a valid FASTA file");
                throw Error("internal: FASTA block does not start at a header");
            }
            if (!pc.error.empty()) throw Error(pc.error);
            if (!pc.labels.empty() || !pc.codes.empty()) any_line = true;
            for (auto& l : pc.labels) labels.push_back(std::move(l));
            lens.insert(lens.end(), pc.lens.begin(), pc.lens.end());
            at[i + 1] = at[i] + pc.codes.size();
        }
        if (codes.capacity() < at.back()) codes.reserve(std::max(at.back(), codes.capacity() * 2));
        codes.resize(at.back());
        parallel_for(n_pieces, [&](size_t i) {
            if (!pieces[i].codes.empty()) memcpy(codes.data() + at[i], pieces[i].codes.data(), pieces[i].codes.size());
        });
    }
};

// whole text in memory
static void accumulate_text(FastaAccumulator& acc, const char* text, size_t len) {
    if (len == 0) throw Error("File is empty");
    acc.add_block(text, text + len);
    if (acc.labels.empty()) throw Error("Not a valid FASTA file");  // no header line at all (the reference panics indexing lines[0])
}

// gz (by content: gzopen reads plain files as they are) or plain file, block by block: the reader thread decompresses the next block
// while the previous one is parsed
static void accumulate_file(FastaAccumulator& acc, const std::string& path) {
    gzFile f = gzopen(path.c_str(), "rb");
    if (!f) throw Error("cannot read file");
    gzbuffer(f, 1u << 20);
    {   // room for the codes up front: the file's size when it is plain text, a guess of 4x when it is compressed
        struct stat st;
        if (stat(path.c_str(), &st) == 0 && st.st_size > 0) acc.codes.reserve((size_t)st.st_size * (gzdirect(f) ? 1 : 4));
    }
    size_t block = 48u << 20;
    if (const char* e = getenv("RXH_FASTA_BLOCK")) block = (size_t)std::max(16, atoi(e));  // test hook: tiny blocks exercise the carry logic
    std::string carry, next;
    bool eof = false, read_err = false;
    auto read_block = [&](std::string& dst) {  // appends up to `block` bytes
        const size_t at = dst.size();
        dst.resize(at + block);
        size_t got = 0;
        while (got < block) {
            const int n = gzread(f, &dst[at + got], (unsigned)std::min<size_t>(block - got, 1u << 30));
            if (n < 0) {
                read_err = true;
                break;
            }
            if (n == 0) {
                eof = true;
                break;
            }
            got += (size_t)n;
        }
        dst.resize(at + got);
    };
    const bool timing = getenv("RXH_TIMING") != nullptr;
    auto tp0 = std::chrono::steady_clock::now();
    double t_parse = 0.0, t_wait = 0.0, t_shift = 0.0;
    read_block(carry);
    bool any = !carry.empty();
    while (true) {
        // parse carry up to its last record boundary; at the end of the file (or after a read error, reported below) all of it
        const bool more = !eof && !read_err;
        size_t split = carry.size();
        if (more) {
            split = 0;
            for (size_t p = carry.size(); p-- > 1;)
                if (carry[p] == '>' && carry[p - 1] == '\n') {
                    split = p;
                    break;
                }
        }
        // the reader thread puts the next block behind the unparsed rest of this one (less than a record, unless the block holds no
        // header at all), so that the text is not shifted a second time
        std::thread reader;
        auto tp0b = std::chrono::steady_clock::now();
        next.clear();
        if (more) {
            next.assign(carry, split, std::string::npos);
            reader = std::thread([&] { read_block(next); });
        }
        std::exception_ptr perr;
        auto tp1 = std::chrono::steady_clock::now();
        t_shift += std::chrono::duration<double>(tp1 - tp0b).count();
        try {
            if (split > 0) acc.add_block(carry.data(), carry.data() + split);
        } catch (...) {
            perr = std::current_exception();
        }
        auto tp2 = std::chrono::steady_clock::now();
        t_parse += std::chrono::duration<double>(tp2 - tp1).count();
        if (reader.joinable()) reader.join();
        auto tp3 = std::chrono::steady_clock::now();
        t_wait += std::chrono::duration<double>(tp3 - tp2).count();
        if (perr) {
            gzclose(f);
            std::rethrow_exception(perr);
        }
        if (!more) break;
        carry.swap(next);
        any = any || !carry.empty();
    }
    gzclose(f);
    if (timing)
        fprintf(stderr, "[rxh fasta] %zu headers, %.1f MB of codes: total %.3f s (parsing blocks %.3f, waiting for the reader %.3f, moving the carry %.3f)\n",
                acc.labels.size(), acc.codes.size() / 1e6, std::chrono::duration<double>(std::chrono::steady_clock::now() - tp0).count(), t_parse, t_wait, t_shift);
    if (read_err) throw Error("cannot read file");
    if (!any) throw Error("File is empty");
    if (acc.labels.empty()) throw Error("Not a valid FASTA file");
}

static std::unique_ptr<Tree> tree_from_accumulator(FastaAccumulator& acc) {
    const size_t H = acc.labels.size();
    std::vector<u64> off{0};
    off.reserve(H + 1);
    u64 pos = 0;
    for (size_t i = 0; i < H; ++i) {
        pos += acc.lens[i];
        if (acc.lens[i] > 0 || i + 1 == H) off.push_back(pos);  // !current_sequence.is_empty() at the next header; the last one always
    }
    if (H != off.size() - 1) throw Error("Number of sequences does not match number of labels");
    return tree_new(std::move(acc.labels), off.data(), acc.codes.data());
}

// parser.rs:46-105
static std::unique_ptr<Tree> parse_reference_fasta_str(const char* text, size_t len) {
    FastaAccumulator acc(true);
    accumulate_text(acc, text, len);
    return tree_from_accumulator(acc);
}

struct Queries {
    std::vector<std::string> labels;
    std::vector<u64> off;
    ByteVec codes;
    size_t size() const { return labels.size(); }
};

static std::unique_ptr<Queries> queries_from_accumulator(FastaAccumulator& acc) {
    auto q = std::make_unique<Queries>();
    const size_t H = acc.labels.size();
    q->off.push_back(0);
    u64 pos = 0;
    for (size_t i = 0; i < H; ++i) {
        pos += acc.lens[i];
        if (acc.lens[i] > 0 || i + 1 == H) {  // empty records are silently merged into the next one (parser.rs:138-141); the last is pushed as is
            q->labels.push_back(std::move(acc.labels[i]));
            q->off.push_back(pos);
        }
    }
    q->codes = std::move(acc.codes);
    return q;
}

// parser.rs:117-154 (queries_to_skip is applied by the caller that owns the checkpoint)
static std::unique_ptr<Queries> parse_query_fasta_str(const char* text, size_t len) {
    FastaAccumulator acc(false);
    accumulate_text(acc, text, len);
    return queries_from_accumulator(acc);
}

// the closing filter of parser.rs:150-153: drop the queries whose label a checkpoint lists as processed
static void skip_queries(Queries& q, const char* blob, size_t blob_len) {
    std::unordered_map<std::string, bool> skip;
    const char* p = blob;
    const char* end = blob + blob_len;
    while (p < end) {  // BufRead::lines of raxtax.ckp (io.rs:213-214)
        const char* nl = (const char*)memchr(p, '\n', (size_t)(end - p));
        const char* e = nl ? nl : end;
        const char* le = (e > p && e[-1] == '\r') ? e - 1 : e;
        skip.emplace(std::string(p, le), true);
        p = nl ? nl + 1 : end;
    }
    Queries out;
    out.off.push_back(0);
    for (size_t i = 0; i < q.size(); ++i) {
        if (skip.count(q.labels[i])) continue;
        out.labels.push_back(std::move(q.labels[i]));
        out.codes.insert(out.codes.end(), q.codes.begin() + (ptrdiff_t)q.off[i], q.codes.begin() + (ptrdiff_t)q.off[i + 1]);
        out.off.push_back(out.codes.size());
    }
    q = std::move(out);
}

// ---- formatting (lineage.rs:17-48, utils.rs:62-89) ------------------------------------------------------------------
static void append_fixed(std::string& s, double v, int prec) {
    char buf[64];
    int n = snprintf(buf, sizeof buf, "%.*f", prec, v);
    s.append(buf, (size_t)n);
}

struct ResultView {
    const std::string* lineage;
    const double* conf;
    u32 n_levels;
    double local, global;
};

static void output_string(std::string& s, const std::string& label, const ResultView& r) {  // lineage.rs:17-30
    s += label;
    s += '\t';
    s += *r.lineage;
    s += '\t';
    for (u32 i = 0; i < r.n_levels; ++i) {
        if (i) s += ',';
        append_fixed(s, r.conf[i], 2);
    }
    s += '\t';
    append_fixed(s, r.local, 5);
    s += '\t';
    append_fixed(s, r.global, 5);
}

static void tsv_string(std::string& s, const std::string& label, const ResultView& r, const std::string& sequence) {  // lineage.rs:32-48
    s += label;
    s += '\t';
    // itertools::interleave(lineage.split(','), confidences): alternate while both last, then drain the rest
    const std::string& lin = *r.lineage;
    size_t start = 0;
    bool lin_done = false;
    u32 ci = 0;
    bool first = true, take_lin = true;
    while (!lin_done || ci < r.n_levels) {
        bool use_lin = take_lin ? !lin_done : !(ci < r.n_levels);
        if (!first) s += '\t';
        first = false;
        if (use_lin) {
            size_t p = lin.find(',', start);
            if (p == std::string::npos) {
                s.append(lin, start, std::string::npos);
                lin_done = true;
            } else {
                s.append(lin, start, p - start);
                start = p + 1;
            }
        } else {
            append_fixed(s, r.conf[ci++], 2);
        }
        take_lin = !take_lin;
    }
    s += '\t';
    append_fixed(s, r.local, 5);
    s += '\t';
    append_fixed(s, r.global, 5);
    s += '\t';
    s += sequence;
}

static std::string decompress_sequence(const u8* seq, size_t len) {  // utils.rs:70-81
    std::string s(len, '-');
    for (size_t i = 0; i < len; ++i) {
        switch (seq[i]) {
            case 1: s[i] = 'A'; break;
            case 2: s[i] = 'C'; break;
            case 4: s[i] = 'G'; break;
            case 8: s[i] = 'T'; break;
            default: break;
        }
    }
    return s;
}

}  // namespace raxtax

// =================================================================================================================
// C ABI
// =================================================================================================================
using namespace raxtax;

struct rxh_tree {
    std::unique_ptr<Tree> t;
};
struct rxh_queries {
    std::unique_ptr<Queries> q;
};

static thread_local std::string g_err;

#define RXH_API extern "C" __attribute__((visibility("default")))

RXH_API const char* rxh_last_error(void) { return g_err.c_str(); }

RXH_API rxh_tree* rxh_tree_from_fasta(const char* text, size_t len) {
    try {
        auto h = new rxh_tree();
        h->t = parse_reference_fasta_str(text, len);
        return h;
    } catch (const std::exception& e) {
        g_err = e.what();
        return nullptr;
    }
}

// parser::parse_reference_fasta_file (parser.rs:37-44): a binary database if the whole file deserialises as one, else FASTA (plain or
// gz).  A bincode image of Tree starts with the root node's label, the string "root" behind its u64 length: only such a file is read
// in one piece and tried as a database; everything else streams through the block parser without ever being held as one string.
RXH_API rxh_tree* rxh_tree_from_file(const char* path, int* was_database) {
    if (was_database) *was_database = 0;
    try {
        FILE* f = fopen(path, "rb");
        if (!f) throw Error("cannot read file");
        unsigned char head[12];
        const size_t got = fread(head, 1, sizeof head, f);
        static const unsigned char kBinHead[12] = {4, 0, 0, 0, 0, 0, 0, 0, 'r', 'o', 'o', 't'};
        if (got == sizeof head && memcmp(head, kBinHead, sizeof head) == 0) {
            std::string raw((const char*)head, got);
            char buf[1 << 16];
            size_t n;
            while ((n = fread(buf, 1, sizeof buf, f)) > 0) raw.append(buf, n);
            fclose(f);
            auto t = load_bin((const u8*)raw.data(), raw.size());
            if (t) {
                if (was_database) *was_database = 1;
                auto h = new rxh_tree();
                h->t = std::move(t);
                return h;
            }
        } else {
            fclose(f);
        }
        FastaAccumulator acc(true);
        accumulate_file(acc, path);
        auto h = new rxh_tree();
        h->t = tree_from_accumulator(acc);
        return h;
    } catch (const std::exception& e) {
        g_err = e.what();
        return nullptr;
    }
}

RXH_API rxh_queries* rxh_queries_from_file(const char* path) {  // parser::parse_query_fasta_file (parser.rs:108-115) minus the skip filter
    try {
        FastaAccumulator acc(false);
        accumulate_file(acc, path);
        auto h = new rxh_queries();
        h->q = queries_from_accumulator(acc);
        return h;
    } catch (const std::exception& e) {
        g_err = e.what();
        return nullptr;
    }
}

RXH_API rxh_tree* rxh_tree_from_bin(const void* data, size_t len) {
    auto t = load_bin((const u8*)data, len);
    if (!t) {
        g_err = "not a raxtax binary database";
        return nullptr;
    }
    auto h = new rxh_tree();
    h->t = std::move(t);
    return h;
}

RXH_API int rxh_tree_save_bin(const rxh_tree* t, const char* path) {
    try {
        save_bin(*t->t, path);
        return 0;
    } catch (const std::exception& e) {
        g_err = e.what();
        return -1;
    }
}

RXH_API int rxh_queries_skip(rxh_queries* q, const char* label_blob, size_t blob_len) {
    try {
        skip_queries(*q->q, label_blob, blob_len);
        return 0;
    } catch (const std::exception& e) {
        g_err = e.what();
        return -1;
    }
}

static std::vector<std::string> split_blob(const char* blob, size_t blob_len, size_t n) {
    std::vector<std::string> out;
    out.reserve(n);
    const char* p = blob;
    const char* end = blob + blob_len;
    for (size_t i = 0; i < n; ++i) {
        const char* nl = p < end ? (const char*)memchr(p, '\n', (size_t)(end - p)) : nullptr;
        const char* e = nl ? nl : end;
        out.emplace_back(p, e);
        p = nl ? nl + 1 : end;
    }
    return out;
}

RXH_API rxh_tree* rxh_tree_new(size_t n, const char* lineage_blob, size_t blob_len, const uint64_t* seq_offsets, const uint8_t* seq_codes) {
    try {
        auto h = new rxh_tree();
        h->t = tree_new(split_blob(lineage_blob, blob_len, n), seq_offsets, seq_codes);
        return h;
    } catch (const std::exception& e) {
        g_err = e.what();
        return nullptr;
    }
}

RXH_API void rxh_tree_free(rxh_tree* t) { delete t; }
RXH_API size_t rxh_tree_num_tips(const rxh_tree* t) { return t->t->num_tips; }
RXH_API const char* rxh_tree_lineage(const rxh_tree* t, size_t i) { return t->t->lineages[i].c_str(); }
RXH_API void rxh_tree_build_kmer_map(const rxh_tree* t) { ensure_csr(*t->t); }
RXH_API int rxh_tree_has_kmer_map(const rxh_tree* t) { return t->t->has_csr ? 1 : 0; }
RXH_API void rxh_tree_csr(const rxh_tree* t, const uint64_t** offsets, const uint32_t** ids) {
    ensure_csr(*t->t);
    *offsets = t->t->csr_off.data();
    *ids = t->t->csr_ids.data();
}
RXH_API size_t rxh_tree_exact(const rxh_tree* t, const uint8_t* seq, size_t len, uint32_t* out, size_t cap) {
    std::vector<u32> v;
    t->t->exact(seq, len, &v);
    for (size_t i = 0; i < v.size() && i < cap; ++i) out[i] = v[i];
    return v.size();
}

RXH_API int rxh_tree_index_desc(const rxh_tree* h, rtx_index_desc* d) {
    const Tree& t = *h->t;
    memset(d, 0, sizeof *d);
    d->n_refs = t.num_tips;
    d->csr_offsets = t.has_csr ? t.csr_off.data() : nullptr;  // without a materialised k_mer_map the device windows the sequences itself
    d->csr_ids = t.has_csr ? t.csr_ids.data() : nullptr;
    d->ref_seq_offsets = t.seq_off.data();
    d->ref_seq_codes = t.seq_codes.data();
    d->n_nodes = (uint32_t)t.node_lo.size();
    d->node_lo = t.node_lo.data();
    d->node_hi = t.node_hi.data();
    d->node_type = t.node_type.data();
    d->child_first = t.child_first.data();
    d->child_count = t.child_count.data();
    d->ref_levels = t.ref_levels.data();
    d->ref_shard_begin = 0;
    d->ref_shard_end = 0;
    return 0;
}

RXH_API int rxh_tree_upload(const rxh_tree* t, rtx_ctx* ctx, uint64_t shard_begin, uint64_t shard_end) {
    rtx_index_desc d;
    rxh_tree_index_desc(t, &d);
    d.ref_shard_begin = shard_begin;
    d.ref_shard_end = shard_end;
    int rc = rtx_index_upload(ctx, &d);
    if (rc) g_err = rtx_last_error(ctx);
    return rc;
}

RXH_API int rxh_tree_upload_sharded(const rxh_tree* t, rtx_ctx* ctx, uint32_t n_shards, uint32_t shard_rank, const uint64_t* shard_cuts) {
    rtx_index_desc d;
    rxh_tree_index_desc(t, &d);
    d.n_shards = n_shards;
    d.shard_rank = shard_rank;
    d.shard_cuts = shard_cuts;
    int rc = rtx_index_upload(ctx, &d);
    if (rc) g_err = rtx_last_error(ctx);
    return rc;
}

RXH_API rxh_queries* rxh_queries_from_fasta(const char* text, size_t len) {
    try {
        auto h = new rxh_queries();
        h->q = parse_query_fasta_str(text, len);
        return h;
    } catch (const std::exception& e) {
        g_err = e.what();
        return nullptr;
    }
}

RXH_API rxh_queries* rxh_queries_new(size_t n, const char* label_blob, size_t blob_len, const uint64_t* seq_offsets, const uint8_t* seq_codes) {
    try {
        auto h = new rxh_queries();
        h->q = std::make_unique<Queries>();
        h->q->labels = split_blob(label_blob, blob_len, n);
        h->q->off.assign(seq_offsets, seq_offsets + n + 1);
        const u64 base = n ? seq_offsets[0] : 0;
        for (auto& o : h->q->off) o -= base;
        h->q->codes.assign(seq_codes + base, seq_codes + base + h->q->off[n]);
        return h;
    } catch (const std::exception& e) {
        g_err = e.what();
        return nullptr;
    }
}
RXH_API void rxh_queries_free(rxh_queries* q) { delete q; }
RXH_API size_t rxh_queries_len(const rxh_queries* q) { return q->q->size(); }
RXH_API const char* rxh_queries_label(const rxh_queries* q, size_t i) { return q->q->labels[i].c_str(); }
RXH_API void rxh_queries_arrays(const rxh_queries* q, const uint64_t** seq_offsets, const uint8_t** seq_codes) {
    *seq_offsets = q->q->off.data();
    *seq_codes = q->q->codes.data();
}

RXH_API uint64_t rxh_exact_batch(const rxh_tree* t, size_t n, const uint64_t* seq_offsets, const uint8_t* seq_codes, uint32_t* exact_offsets,
                                 uint32_t* exact_ids, uint64_t cap) {
    std::vector<u32> v;
    u64 total = 0;
    for (size_t q = 0; q < n; ++q) {
        exact_offsets[q] = (u32)total;
        t->t->exact(seq_codes + seq_offsets[q], (size_t)(seq_offsets[q + 1] - seq_offsets[q]), &v);
        for (u32 id : v) {
            if (total < cap) exact_ids[total] = id;
            ++total;
        }
    }
    exact_offsets[n] = (u32)total;
    return total;
}

// raxtax::raxtax (raxtax.rs:14-97).  The reference fans chunks of queries out over the rayon pool (raxtax.rs:35-39) and a separate
// writer thread drains the channel (main.rs:126-136).  Here every context (= GPU, index replicated) has one DRIVER thread that pulls
// chunks from a shared counter and keeps two batches in flight on its device (the two batch slots of rtx_batch_slot): while the
// kernels of chunk i run, chunk i+1 is de-duplicated, looked up (exact matches), uploaded and queued behind it, and chunk i-1 is
// formatted by the EMITTER -- the calling thread -- with a few helper threads, then handed to the sender one query at a time.
// Between the contexts there is no collective; queries arrive in completion order (in query order with one context), the lines of
// a query contiguous, as in the reference.
namespace {

// ---- "{:.N}" of an f64 (Rust rounds the exact binary value to nearest, ties to even -- what glibc's %.Nf does too) ---------------
// Fast path: scale, round, print two integers.  The scaled value carries a relative error of 2^-53, so whenever it sits closer than
// 1e-6 to a rounding tie -- or is negative, huge or not finite -- the exact (slow) conversion decides.
static inline char* put_uint(char* p, u64 v) {
    char tmp[24];
    int n = 0;
    do {
        tmp[n++] = (char)('0' + v % 10);
        v /= 10;
    } while (v);
    while (n) *p++ = tmp[--n];
    return p;
}
static char* put_fixed(char* p, double v, int prec) {
    static const double pw[] = {1.0, 10.0, 100.0, 1e3, 1e4, 1e5, 1e6};
    if (prec >= 1 && prec <= 6 && v >= 0.0 && v < 1e9 && !std::signbit(v)) {
        const double x = v * pw[prec];
        const double fl = std::floor(x);
        const double frac = x - fl;
        if (std::fabs(frac - 0.5) > 1e-6) {
            const u64 r = (u64)fl + (frac > 0.5 ? 1u : 0u);
            const u64 scale = (u64)pw[prec];
            p = put_uint(p, r / scale);
            *p++ = '.';
            u64 f = r % scale;
            for (int i = prec - 1; i >= 0; --i) {
                p[i] = (char)('0' + f % 10);
                f /= 10;
            }
            return p + prec;
        }
    }
    return p + snprintf(p, 400, "%.*f", prec, v);
}

// growable char buffer the formatters write into with raw pointers
struct CharBuf {
    std::vector<char> v;
    size_t n = 0;
    char* reserve(size_t more) {
        if (n + more > v.size()) v.resize(std::max(v.size() * 2, n + more + 4096));
        return v.data() + n;
    }
    void put(const char* s, size_t len) {
        memcpy(reserve(len), s, len);
        n += len;
    }
    void put(char c) {
        *reserve(1) = c;
        n += 1;
    }
    void fixed(double val, int prec) {
        char* p = reserve(420);
        n += (size_t)(put_fixed(p, val, prec) - p);
    }
};

// --strand both: the complement of a 4-bit code is its bit-reversed nibble (A1 <-> T8, C2 <-> G4, R5 <-> Y10, N15 <-> N15)
static inline u8 complement_code(u8 c) {
    return (u8)(((c & 1u) << 3) | ((c & 2u) << 1) | ((c & 4u) >> 1) | ((c & 8u) >> 3));
}
// decompress_sequence of the reverse complement, from the decompressed text ('-' for every ambiguous code stays '-')
static std::string reverse_complement_text(const std::string& t) {
    std::string r(t.rbegin(), t.rend());
    for (char& c : r) c = c == 'A' ? 'T' : c == 'T' ? 'A' : c == 'C' ? 'G' : c == 'G' ? 'C' : c;
    return r;
}
// the strand column of --strand both: `+` classified as given, `-` as the reverse complement
static inline void strand_column(CharBuf& s, bool minus) {
    s.put('\t');
    s.put(minus ? '-' : '+');
}
static inline void uint_column(CharBuf& s, u64 v) {
    s.put('\t');
    char* p = s.reserve(24);
    s.n += (size_t)(put_uint(p, v) - p);
}

static void output_line(CharBuf& s, const std::string& label, const ResultView& r) {  // lineage.rs:17-30
    s.put(label.data(), label.size());
    s.put('\t');
    s.put(r.lineage->data(), r.lineage->size());
    s.put('\t');
    for (u32 i = 0; i < r.n_levels; ++i) {
        if (i) s.put(',');
        s.fixed(r.conf[i], 2);
    }
    s.put('\t');
    s.fixed(r.local, 5);
    s.put('\t');
    s.fixed(r.global, 5);
}

static void tsv_line(CharBuf& s, const std::string& label, const ResultView& r, const std::string& sequence) {  // lineage.rs:32-48
    s.put(label.data(), label.size());
    s.put('\t');
    // itertools::interleave(lineage.split(','), confidences): alternate while both last, then drain the rest
    const std::string& lin = *r.lineage;
    size_t start = 0;
    bool lin_done = false;
    u32 ci = 0;
    bool first = true, take_lin = true;
    while (!lin_done || ci < r.n_levels) {
        const bool use_lin = take_lin ? !lin_done : !(ci < r.n_levels);
        if (!first) s.put('\t');
        first = false;
        if (use_lin) {
            const size_t p = lin.find(',', start);
            if (p == std::string::npos) {
                s.put(lin.data() + start, lin.size() - start);
                lin_done = true;
            } else {
                s.put(lin.data() + start, p - start);
                start = p + 1;
            }
        } else {
            s.fixed(r.conf[ci++], 2);
        }
        take_lin = !take_lin;
    }
    s.put('\t');
    s.fixed(r.local, 5);
    s.put('\t');
    s.fixed(r.global, 5);
    s.put('\t');
    s.put(sequence.data(), sequence.size());
}

// page-locked array from the device library (results land in it by DMA), grown on demand
template <typename T>
struct PinnedArr {
    T* p = nullptr;
    size_t cap = 0;
    PinnedArr() = default;
    PinnedArr(const PinnedArr&) = delete;
    PinnedArr& operator=(const PinnedArr&) = delete;
    ~PinnedArr() {
        if (p) rtx_host_free(p);
    }
    void ensure(size_t n) {
        if (n <= cap) return;
        rtx_host_free(p);
        p = nullptr;
        cap = 0;
        const size_t want = n + n / 4 + 64;
        void* q = nullptr;
        if (rtx_host_alloc(want * sizeof(T), &q) != RTX_OK) throw Error("rtx_host_alloc failed (page-locked result buffers)");
        p = (T*)q;
        cap = want;
    }
};

// distinct sequences of a chunk: open addressing over (hash, first query with that sequence)
struct FlatDedup {
    std::vector<u64> hash;
    std::vector<u32> slot;  // unique id + 1, 0 = empty
    size_t mask = 0;
    void reset(size_t n) {
        size_t cap = 64;
        while (cap < n * 2) cap <<= 1;
        if (slot.size() != cap) {
            slot.assign(cap, 0);
            hash.assign(cap, 0);
        } else std::fill(slot.begin(), slot.end(), 0u);
        mask = cap - 1;
    }
};

struct ChunkJob {
    size_t c0 = 0, cn = 0, n_uniq = 0;
    bool compact = false;
    int dev_slot = 0;
    std::vector<u32> rep, uniq_first, exact_off, exact_ids;
    std::vector<u64> u_off, uniq_hash;
    std::vector<u8> u_codes;
    std::vector<u8> rc_seq, strand;  // --strand both: a reverse complement being looked up; per distinct sequence, 1 = classified as rc
    std::vector<u32> hit_n, hit_ref;   // best hits (rtx_batch_best_hits) per distinct sequence
    std::vector<u16> hit_count;
    PinnedArr<u16> n_kmers;
    PinnedArr<u32> result_begin, first_ref;
    PinnedArr<double> global, conf, local;
    PinnedArr<u8> n_levels;
    u32 ML = 1;
    std::atomic<bool> busy{false};  // owned by the pipeline (prep .. emitted)
};

// The jobs -- above all their page-locked result arrays -- are kept per context between calls of rxh_raxtax: cudaHostAlloc /
// cudaFreeHost cost milliseconds each and wait for the device, which a caller classifying batch after batch would pay 21 times per
// call.  rxh_release_buffers() (or the end of the process) frees them.
struct JobPool {
    std::mutex mtx;
    std::unordered_map<rtx_ctx*, std::vector<std::unique_ptr<ChunkJob>>> idle;
    std::vector<std::unique_ptr<ChunkJob>> take(rtx_ctx* ctx) {
        std::lock_guard<std::mutex> g(mtx);
        std::vector<std::unique_ptr<ChunkJob>> v;
        auto it = idle.find(ctx);
        if (it != idle.end()) {
            v = std::move(it->second);
            idle.erase(it);
        }
        while (v.size() < 3) v.emplace_back(new ChunkJob());
        for (auto& j : v) j->busy.store(false);  // a run that failed half-way may have left its jobs marked
        return v;
    }
    void give(rtx_ctx* ctx, std::vector<std::unique_ptr<ChunkJob>> v) {
        std::lock_guard<std::mutex> g(mtx);
        idle[ctx] = std::move(v);
    }
    void clear() {
        std::lock_guard<std::mutex> g(mtx);
        idle.clear();
    }
};
static JobPool& job_pool() {
    static JobPool* p = new JobPool();  // leaked on purpose: no cudaFreeHost from a static destructor after the CUDA runtime is gone
    return *p;
}

// The first chunk of a context is prepared (hashed, de-duplicated, looked up) before its device has anything to do, and the last
// one is formatted and sent after the device is through: with eight equal chunks that is a quarter of a chunk's host work on
// either side of the job (12 + 16 ms of a 1.17 s C3 job, profiles/r2y_e2e_probe_c3.txt).  When the chunk size is the library's
// choice (`ramp`) the job starts and ends with chunks of an eighth, a quarter and a half of it -- one set per context.
// -> chunk i = [begin[i], begin[i + 1]), begin.back() == nq
static std::vector<size_t> plan_chunk_begins(size_t nq, size_t n_ctx, size_t chunk_size, bool ramp) {
    std::vector<size_t> begin(1, 0);
    if (nq == 0) return begin;
    chunk_size = std::max<size_t>(1, chunk_size);
    n_ctx = std::max<size_t>(1, n_ctx);
    std::vector<size_t> steps;
    for (size_t c = std::max<size_t>(1024, chunk_size / 8); c < chunk_size; c *= 2) steps.push_back(c);
    size_t edge = 0;
    for (size_t c : steps) edge += c * n_ctx;
    if (!ramp || steps.empty() || nq < 2 * edge + 2 * n_ctx * chunk_size) {
        for (size_t c = chunk_size; c < nq; c += chunk_size) begin.push_back(c);
        begin.push_back(nq);
        return begin;
    }
    size_t pos = 0;
    for (size_t c : steps)
        for (size_t k = 0; k < n_ctx; ++k) begin.push_back(pos += c);
    const size_t mid_end = nq - edge;
    const size_t n_head = begin.size();
    while (pos + chunk_size < mid_end) begin.push_back(pos += chunk_size);
    if (pos < mid_end) {  // the rest of the middle part: a chunk of its own, or -- a full launch sequence for a few queries does not pay -- part of the last one
        if (mid_end - pos < chunk_size / 2 && begin.size() > n_head) begin.back() = mid_end;
        else begin.push_back(mid_end);
        pos = mid_end;
    }
    for (size_t i = steps.size(); i-- > 0;)
        for (size_t k = 0; k < n_ctx; ++k) begin.push_back(pos += steps[i]);
    return begin;
}

struct Worker {
    const Tree& tree;
    const Queries& qs;
    const size_t nq;
    size_t chunk_size;
    const int skip_exact_matches, raw_confidence, tsv;
    rxh_sender sender;
    void* sender_user;
    rxh_logger logger;
    void* logger_user;
    std::atomic<size_t> next_chunk{0};
    std::vector<size_t> chunk_begin{};  // query-partitioned drivers: chunk i = [chunk_begin[i], chunk_begin[i + 1])
    bool ramp = false;                  // the chunk size was left to the library: small chunks at both ends of the job (plan_chunks)
    std::atomic<bool> failed{false}, warned{false};
    std::mutex io_mtx{}, err_mtx{};
    std::string err{};
    // driver -> emitter
    std::mutex q_mtx{};
    std::condition_variable q_cv{}, free_cv{};
    std::deque<ChunkJob*> ready{};
    size_t drivers_running = 0;
    // emitter's helpers
    struct FormatPart {
        CharBuf buf;
        std::vector<size_t> off;  // per query: start of the primary string, of the tsv string and (with best hits) of the hit lines
    };
    std::vector<FormatPart> parts{};
    std::vector<std::thread> helpers{};
    std::mutex h_mtx{};
    std::condition_variable h_cv{}, h_done_cv{};
    ChunkJob* h_job = nullptr;
    u64 h_epoch = 0;
    size_t h_pending = 0;
    bool h_quit = false;
    // stage clocks (seconds), printed to stderr at the end of a run when RXH_TIMING is set
    struct Clock {
        std::atomic<u64> ns{0};
        void add(std::chrono::steady_clock::time_point t0) {
            ns += (u64)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0).count();
        }
        double s() const { return (double)ns.load() * 1e-9; }
    };
    Clock t_prep{}, t_issue{}, t_collect{}, t_acquire{}, t_format{}, t_send{}, t_emit_wait{};
    std::chrono::steady_clock::time_point t_start{}, t_first_issue{}, t_last_collect{};
    std::atomic<bool> first_issued{false};
    bool both = false;  // --strand both (rxh_raxtax_both_strands): RTX_BOTH_STRANDS batches, strand column in both outputs
    u32 best_hits = 0;  // --best-hits (rxh_raxtax_best_hits): RTX_OPT_BEST_HITS of every batch, lines to hits_sender
    rxh_hits_sender hits_sender = nullptr;
    void* hits_user = nullptr;
    static std::chrono::steady_clock::time_point now() { return std::chrono::steady_clock::now(); }

    void fail(const std::string& what) {
        failed.store(true);
        {
            std::lock_guard<std::mutex> g(err_mtx);
            if (err.empty()) err = what;
        }
        std::lock_guard<std::mutex> g(q_mtx);
        q_cv.notify_all();
        free_cv.notify_all();
    }

    // ---- driver side ---------------------------------------------------------------------------------------------------------
    // de-duplication, exact-match lookup (raxtax.rs:42) and the log lines of raxtax.rs:43-53 for queries [c0, c0 + cn)
    void prep(ChunkJob& j, size_t c0, size_t cn, FlatDedup& dd, bool dedup, bool log = true) {
        j.c0 = c0;
        j.cn = cn;
        // Queries with identical sequences (amplicon reads of an abundant taxon) get identical results: the device sees every
        // distinct sequence of the chunk once, the lines are then written per query label as the reference would (RXH_NO_DEDUP=1
        // switches this off).  rep[i] = position of query i's sequence among the distinct ones.
        j.rep.resize(cn);
        j.uniq_first.clear();
        j.uniq_hash.clear();
        if (dedup && cn > 1) {
            dd.reset(cn);
            for (size_t i = 0; i < cn; ++i) {
                const u8* sp = qs.codes.data() + qs.off[c0 + i];
                const size_t sl = (size_t)(qs.off[c0 + i + 1] - qs.off[c0 + i]);
                const u64 h = Tree::hash_bytes(sp, sl);
                size_t at = (size_t)(h ^ (h >> 31)) & dd.mask;
                u32 found = 0xFFFFFFFFu;
                while (dd.slot[at]) {
                    if (dd.hash[at] == h) {
                        const size_t k = j.uniq_first[dd.slot[at] - 1];
                        const size_t kl = (size_t)(qs.off[c0 + k + 1] - qs.off[c0 + k]);
                        if (kl == sl && (sl == 0 || memcmp(qs.codes.data() + qs.off[c0 + k], sp, sl) == 0)) {
                            found = dd.slot[at] - 1;
                            break;
                        }
                    }
                    at = (at + 1) & dd.mask;
                }
                if (found == 0xFFFFFFFFu) {
                    found = (u32)j.uniq_first.size();
                    j.uniq_first.push_back((u32)i);
                    j.uniq_hash.push_back(h);
                    dd.slot[at] = found + 1;
                    dd.hash[at] = h;
                }
                j.rep[i] = found;
            }
            j.n_uniq = j.uniq_first.size();
        } else {
            j.n_uniq = cn;
        }
        j.compact = j.n_uniq < cn;
        if (j.compact) {  // the distinct sequences, contiguous
            j.u_off.assign(1, 0);
            j.u_codes.clear();
            for (size_t u = 0; u < j.n_uniq; ++u) {
                const size_t q = c0 + j.uniq_first[u];
                j.u_codes.insert(j.u_codes.end(), qs.codes.begin() + (ptrdiff_t)qs.off[q], qs.codes.begin() + (ptrdiff_t)qs.off[q + 1]);
                j.u_off.push_back(j.u_codes.size());
            }
        } else {
            for (size_t i = 0; i < cn; ++i) j.rep[i] = (u32)i;
        }
        j.exact_off.assign(j.n_uniq + 1, 0);
        j.exact_ids.clear();
        const bool have_hash = j.uniq_hash.size() == j.n_uniq;
        for (size_t u = 0; u < j.n_uniq; ++u) {  // tree.sequences.get(query_sequence) (raxtax.rs:42), once per distinct sequence
            const size_t q = c0 + (have_hash ? j.uniq_first[u] : u);
            const u8* sp = qs.codes.data() + qs.off[q];
            const size_t sl = (size_t)(qs.off[q + 1] - qs.off[q]);
            for (u32 id = tree.exact_head(sp, sl, have_hash ? j.uniq_hash[u] : Tree::hash_bytes(sp, sl)); id != Tree::kNone; id = tree.ex_next[id])
                j.exact_ids.push_back(id);
            j.exact_off[u + 1] = (u32)j.exact_ids.size();
        }
        if (both) {  // entries [n, 2n): the exact matches of the reverse complements, the orientation the device may choose instead
            j.exact_off.resize(2 * j.n_uniq + 1);
            for (size_t u = 0; u < j.n_uniq; ++u) {
                const size_t q = c0 + (have_hash ? j.uniq_first[u] : u);
                const u8* sp = qs.codes.data() + qs.off[q];
                const size_t sl = (size_t)(qs.off[q + 1] - qs.off[q]);
                j.rc_seq.resize(sl);
                for (size_t k = 0; k < sl; ++k) j.rc_seq[k] = complement_code(sp[sl - 1 - k]);
                const u8* rp = sl ? j.rc_seq.data() : sp;
                for (u32 id = tree.exact_head(rp, sl, Tree::hash_bytes(rp, sl)); id != Tree::kNone; id = tree.ex_next[id]) j.exact_ids.push_back(id);
                j.exact_off[j.n_uniq + u + 1] = (u32)j.exact_ids.size();
            }
            return;  // the log lines are those of the classified orientation: written after collect (log_exact)
        }
        if (log) log_exact(j);
    }

    // the log lines of raxtax.rs:43-53, per query of the job; with --strand both for the orientation each query was classified in
    void log_exact(const ChunkJob& j) {
        if (skip_exact_matches || j.exact_ids.empty()) return;
        std::string msg, first_parent;
        for (size_t i = 0; i < j.cn; ++i) {
            const size_t q = j.c0 + i;
            const size_t s = both && j.strand[j.rep[i]] ? j.n_uniq + j.rep[i] : j.rep[i];
            const u32 e0 = j.exact_off[s], e1 = j.exact_off[s + 1];
            bool all_equal = true;
            for (u32 e = e0; e < e1; ++e) {
                const std::string& l = tree.lineages[j.exact_ids[e]];
                if (logger) {
                    msg = "Exact sequence match for query " + qs.labels[q] + ": " + l;
                    std::lock_guard<std::mutex> g(io_mtx);
                    logger(logger_user, 3, msg.c_str());
                }
                const size_t p = l.rfind(',');
                if (p == std::string::npos) throw Error("called `Option::unwrap()` on a `None` value: lineage without ',' (raxtax.rs:49)");
                if (e == e0) first_parent.assign(l, 0, p);
                else if (l.compare(0, p, first_parent) != 0 || p != first_parent.size()) all_equal = false;
            }
            if (!all_equal) {
                if (logger) {
                    msg = "Exact matches for " + qs.labels[q] + " differ above the leafs of the lineage tree!";
                    std::lock_guard<std::mutex> g(io_mtx);
                    logger(logger_user, 2, msg.c_str());
                }
                warned.store(true);
            }
        }
    }

    static bool is_oom(rtx_ctx* ctx) { return strstr(rtx_last_error(ctx), "out of memory") != nullptr; }

    // H2D + all kernels of the job, queued behind whatever the device is doing; returns false when device memory ran out
    bool issue(rtx_ctx* ctx, ChunkJob& j, int dev_slot) {
        rtx_batch batch{};
        batch.n_queries = (u32)j.n_uniq;
        batch.seq_offsets = j.compact ? j.u_off.data() : qs.off.data() + j.c0;
        batch.seq_codes = j.compact ? j.u_codes.data() : qs.codes.data();
        batch.exact_offsets = j.exact_off.data();
        batch.exact_ids = j.exact_ids.empty() ? nullptr : j.exact_ids.data();
        batch.flags = (skip_exact_matches ? RTX_SKIP_EXACT_MATCHES : 0u) | (raw_confidence ? RTX_RAW_CONFIDENCE : 0u) | (both ? RTX_BOTH_STRANDS : 0u);
        j.dev_slot = dev_slot;
        if (rtx_batch_slot(ctx, dev_slot)) throw Error(std::string("rtx_batch_slot: ") + rtx_last_error(ctx));
        if (best_hits && rtx_ctx_set_option(ctx, RTX_OPT_BEST_HITS, best_hits))
            throw Error(std::string("rtx_ctx_set_option(RTX_OPT_BEST_HITS): ") + rtx_last_error(ctx));
        int rc = rtx_batch_upload(ctx, &batch);
        if (rc == RTX_ERR_CUDA && is_oom(ctx)) return false;
        if (rc) throw Error(std::string("rtx_batch_upload: ") + rtx_last_error(ctx));
        rc = rtx_batch_run(ctx);
        if (rc == RTX_ERR_CUDA && is_oom(ctx)) return false;
        if (rc) throw Error(std::string("rtx_batch_run: ") + rtx_last_error(ctx));
        return true;
    }

    // waits for the job's kernels, D2H into its page-locked arrays.  The result lines stay on the device until they fit: a too
    // small capacity only repeats the copy, never the kernels.
    void collect(rtx_ctx* ctx, ChunkJob& j) {
        if (rtx_batch_slot(ctx, j.dev_slot)) throw Error(std::string("rtx_batch_slot: ") + rtx_last_error(ctx));
        const u32 ML = rtx_index_max_levels(ctx);
        j.ML = ML;
        j.n_kmers.ensure(j.n_uniq);
        j.result_begin.ensure(j.n_uniq + 1);
        j.global.ensure(j.n_uniq);
        size_t cap = std::max<size_t>(j.first_ref.cap, j.n_uniq * 8 + 64);
        while (true) {
            j.first_ref.ensure(cap);
            j.n_levels.ensure(cap);
            j.conf.ensure(cap * ML);
            j.local.ensure(cap);
            cap = std::min(std::min(j.first_ref.cap, j.n_levels.cap), std::min(j.conf.cap / ML, j.local.cap));
            rtx_results res{};
            res.n_kmers = j.n_kmers.p;
            res.result_begin = j.result_begin.p;
            res.global_signal = j.global.p;
            res.result_capacity = cap;
            res.first_ref = j.first_ref.p;
            res.n_levels = j.n_levels.p;
            res.confidence = j.conf.p;
            res.local_signal = j.local.p;
            const int rc = rtx_batch_download(ctx, &res);
            if (rc == RTX_ERR_INVALID && res.n_results > cap) {
                cap = res.n_results + 64;
                continue;
            }
            if (rc) throw Error(std::string("rtx_batch_download: ") + rtx_last_error(ctx));
            break;
        }
        if (both) {
            j.strand.resize(std::max<size_t>(j.n_uniq, 1));
            if (rtx_batch_strands(ctx, j.strand.data())) throw Error(std::string("rtx_batch_strands: ") + rtx_last_error(ctx));
            log_exact(j);
        }
        if (best_hits) {
            j.hit_n.resize(std::max<size_t>(j.n_uniq, 1));
            j.hit_ref.resize(std::max<size_t>(j.n_uniq, 1) * best_hits);
            j.hit_count.resize(std::max<size_t>(j.n_uniq, 1) * best_hits);
            if (rtx_batch_best_hits(ctx, j.hit_n.data(), j.hit_ref.data(), j.hit_count.data()))
                throw Error(std::string("rtx_batch_best_hits: ") + rtx_last_error(ctx));
        }
    }

    void hand_over(ChunkJob* j) {
        std::lock_guard<std::mutex> g(q_mtx);
        ready.push_back(j);
        q_cv.notify_all();
    }

    ChunkJob* acquire(std::vector<std::unique_ptr<ChunkJob>>& jobs) {
        std::unique_lock<std::mutex> g(q_mtx);
        while (true) {
            for (auto& j : jobs)
                if (!j->busy.load()) {
                    j->busy.store(true);
                    return j.get();
                }
            if (failed.load()) return nullptr;
            free_cv.wait(g);
        }
    }

    void drive(rtx_ctx* ctx) {
        try {
            drive_inner(ctx);
        } catch (const std::exception& e) {
            fail(e.what());
        }
        std::lock_guard<std::mutex> g(q_mtx);
        --drivers_running;
        q_cv.notify_all();
    }

    void drive_inner(rtx_ctx* ctx) {
        if (rtx_index_n_refs(ctx) != tree.num_tips) throw Error("the context's index does not belong to this tree");
        const bool dedup = getenv("RXH_NO_DEDUP") == nullptr;
        std::vector<std::unique_ptr<ChunkJob>> jobs = job_pool().take(ctx);
        struct Return {
            rtx_ctx* ctx;
            std::vector<std::unique_ptr<ChunkJob>>& jobs;
            ~Return() { job_pool().give(ctx, std::move(jobs)); }
        } ret{ctx, jobs};
        FlatDedup dd;
        ChunkJob* inflight = nullptr;
        int dev_slot = 0;
        std::vector<std::pair<size_t, size_t>> todo;  // ranges of this thread's current chunk (split further when memory runs out)
        while (true) {
            if (todo.empty()) {
                const size_t ci = next_chunk.fetch_add(1);
                if (ci + 1 >= chunk_begin.size() || failed.load()) break;
                todo.emplace_back(chunk_begin[ci], chunk_begin[ci + 1] - chunk_begin[ci]);
            }
            const std::pair<size_t, size_t> range = todo.back();
            todo.pop_back();
            auto t0 = now();
            ChunkJob* j = acquire(jobs);
            t_acquire.add(t0);
            if (!j) break;
            t0 = now();
            prep(*j, range.first, range.second, dd, dedup);
            t_prep.add(t0);
            t0 = now();
            const bool issued = issue(ctx, *j, dev_slot);
            t_issue.add(t0);
            if (!first_issued.exchange(true)) t_first_issue = now();
            if (!issued) {
                // the batch does not fit the device next to the index: drain, then classify it in two halves
                j->busy.store(false);
                if (inflight) {
                    collect(ctx, *inflight);
                    hand_over(inflight);
                    inflight = nullptr;
                }
                if (range.second <= 1) throw Error(std::string("not even one query fits the device memory: ") + rtx_last_error(ctx));
                const size_t h = range.second / 2;
                todo.emplace_back(range.first + h, range.second - h);
                todo.emplace_back(range.first, h);
                continue;
            }
            dev_slot ^= 1;
            if (inflight) {
                t0 = now();
                collect(ctx, *inflight);
                t_collect.add(t0);
                hand_over(inflight);
            }
            inflight = j;
        }
        if (inflight) {
            auto t0 = now();
            collect(ctx, *inflight);
            t_collect.add(t0);
            t_last_collect = now();
            hand_over(inflight);
        }
        // the jobs (and their page-locked arrays) must outlive the emitter's use of them
        std::unique_lock<std::mutex> g(q_mtx);
        while (true) {
            bool any = false;
            for (auto& j : jobs) any |= j->busy.load();
            if (!any) break;
            free_cv.wait(g);
        }
    }

    // Reference-sharded mode over NCCL: ctx is rank `rank` of `n_ranks` (index uploaded with rxh_tree_upload_sharded, communicator
    // set up).  Every rank walks the same chunks in the same order -- the collectives inside rtx_shard_run / rtx_shard_gather need
    // all of them -- and prepares the same batch; rank 0 gets the merged lines, writes the log lines and feeds the emitter.
    void drive_sharded(rtx_ctx* ctx, int rank) {
        try {
            if (rtx_index_n_refs(ctx) != tree.num_tips) throw Error("a context's index does not belong to this tree");
            const bool dedup = getenv("RXH_NO_DEDUP") == nullptr;
            std::vector<std::unique_ptr<ChunkJob>> jobs = job_pool().take(ctx);
            struct Return {
                rtx_ctx* ctx;
                std::vector<std::unique_ptr<ChunkJob>>& jobs;
                ~Return() { job_pool().give(ctx, std::move(jobs)); }
            } ret{ctx, jobs};
            FlatDedup dd;
            for (size_t c0 = 0; c0 < nq && !failed.load(); c0 += chunk_size) {
                auto t0 = now();
                ChunkJob* j = acquire(jobs);
                t_acquire.add(t0);
                if (!j) break;
                t0 = now();
                prep(*j, c0, std::min(chunk_size, nq - c0), dd, dedup, rank == 0);
                t_prep.add(t0);
                t0 = now();
                rtx_batch batch{};
                batch.n_queries = (u32)j->n_uniq;
                batch.seq_offsets = j->compact ? j->u_off.data() : qs.off.data() + j->c0;
                batch.seq_codes = j->compact ? j->u_codes.data() : qs.codes.data();
                batch.exact_offsets = j->exact_off.data();
                batch.exact_ids = j->exact_ids.empty() ? nullptr : j->exact_ids.data();
                batch.flags = (skip_exact_matches ? RTX_SKIP_EXACT_MATCHES : 0u) | (raw_confidence ? RTX_RAW_CONFIDENCE : 0u);
                j->dev_slot = 0;
                if (rtx_batch_slot(ctx, 0) || rtx_batch_upload(ctx, &batch)) throw Error(std::string("rtx_batch_upload: ") + rtx_last_error(ctx));
                if (rtx_shard_run(ctx)) throw Error(std::string("rtx_shard_run: ") + rtx_last_error(ctx));
                if (rtx_shard_gather(ctx, 0)) throw Error(std::string("rtx_shard_gather: ") + rtx_last_error(ctx));
                t_issue.add(t0);
                if (rank == 0) {
                    t0 = now();
                    collect(ctx, *j);
                    t_collect.add(t0);
                    hand_over(j);
                } else {
                    j->busy.store(false);
                }
            }
            std::unique_lock<std::mutex> g(q_mtx);
            while (true) {
                bool any = false;
                for (auto& j : jobs) any |= j->busy.load();
                if (!any) break;
                free_cv.wait(g);
            }
        } catch (const std::exception& e) {
            fail(e.what());
        }
        std::lock_guard<std::mutex> g(q_mtx);
        --drivers_running;
        q_cv.notify_all();
    }

    // ---- emitter side --------------------------------------------------------------------------------------------------------
    // utils::get_results / get_results_tsv (raxtax.rs:85-87) for the queries [i0, i1) of a job
    void format_range(const ChunkJob& j, size_t i0, size_t i1, FormatPart& out) const {
        out.buf.n = 0;
        out.off.clear();
        const u32 ML = j.ML;
        std::string seq;
        for (size_t i = i0; i < i1; ++i) {
            const size_t q = j.c0 + i;
            const u32 u = j.rep[i];
            const u32 r0 = j.result_begin.p[u], r1 = j.result_begin.p[u + 1];
            const bool minus = both && j.strand[u];
            out.off.push_back(out.buf.n);
            for (u32 r = r0; r < r1; ++r) {
                const ResultView rv{&tree.lineages[j.first_ref.p[r]], j.conf.p + (size_t)r * ML, j.n_levels.p[r], j.local.p[r], j.global.p[u]};
                if (r != r0) out.buf.put('\n');
                output_line(out.buf, qs.labels[q], rv);
                if (both) strand_column(out.buf, minus);
            }
            out.buf.put('\0');
            out.off.push_back(out.buf.n);
            if (tsv) {
                seq = decompress_sequence(qs.codes.data() + qs.off[q], (size_t)(qs.off[q + 1] - qs.off[q]));
                if (minus) seq = reverse_complement_text(seq);  // the sequence in the orientation that was classified
                for (u32 r = r0; r < r1; ++r) {
                    const ResultView rv{&tree.lineages[j.first_ref.p[r]], j.conf.p + (size_t)r * ML, j.n_levels.p[r], j.local.p[r], j.global.p[u]};
                    if (r != r0) out.buf.put('\n');
                    tsv_line(out.buf, qs.labels[q], rv, seq);
                    if (both) strand_column(out.buf, minus);
                }
                out.buf.put('\0');
            }
            if (hits_sender) {  // {label}\t{rank}\t{lineage}\t{shared 8-mers}\t{K}\t{reference id}[\t{strand}]
                out.off.push_back(out.buf.n);
                const std::string& label = qs.labels[q];
                for (u32 k = 0; k < j.hit_n[u]; ++k) {
                    const size_t h = (size_t)u * best_hits + k;
                    const u32 ref = j.hit_ref[h];
                    if (k) out.buf.put('\n');
                    out.buf.put(label.data(), label.size());
                    uint_column(out.buf, k + 1);
                    out.buf.put('\t');
                    out.buf.put(tree.lineages[ref].data(), tree.lineages[ref].size());
                    uint_column(out.buf, j.hit_count[h]);
                    uint_column(out.buf, j.n_kmers.p[u]);
                    uint_column(out.buf, ref);
                    if (both) strand_column(out.buf, minus);
                }
                out.buf.put('\0');
            }
        }
    }
    static void part_range(size_t cn, size_t n_parts, size_t k, size_t* i0, size_t* i1) {
        *i0 = cn * k / n_parts;
        *i1 = cn * (k + 1) / n_parts;
    }
    void helper_main(size_t k) {
        u64 seen = 0;
        while (true) {
            ChunkJob* j;
            {
                std::unique_lock<std::mutex> g(h_mtx);
                h_cv.wait(g, [&] { return h_quit || h_epoch != seen; });
                if (h_quit) return;
                seen = h_epoch;
                j = h_job;
            }
            size_t i0, i1;
            part_range(j->cn, parts.size(), k, &i0, &i1);
            try {
                format_range(*j, i0, i1, parts[k]);
            } catch (const std::exception& e) {
                fail(e.what());
            }
            std::lock_guard<std::mutex> g(h_mtx);
            if (--h_pending == 0) h_done_cv.notify_all();
        }
    }
    void emit(ChunkJob& j) {
        // the helpers are worth their wake-up (two condition-variable round trips, ~0.1 ms) only on chunks of several thousand queries
        const size_t n_parts = j.cn >= 6144 ? parts.size() : 1;
        if (n_parts > 1) {
            std::lock_guard<std::mutex> g(h_mtx);
            h_job = &j;
            h_pending = n_parts - 1;
            ++h_epoch;
            h_cv.notify_all();
        }
        size_t i0, i1;
        auto t0 = now();
        part_range(j.cn, n_parts, 0, &i0, &i1);
        format_range(j, i0, i1, parts[0]);
        if (n_parts > 1) {
            std::unique_lock<std::mutex> g(h_mtx);
            h_done_cv.wait(g, [&] { return h_pending == 0; });
        }
        t_format.add(t0);
        if (!sender || failed.load()) return;
        t0 = now();
        struct SendClock {
            Clock& c;
            std::chrono::steady_clock::time_point t0;
            ~SendClock() { c.add(t0); }
        } sc{t_send, t0};
        std::lock_guard<std::mutex> g(io_mtx);
        for (size_t k = 0; k < n_parts; ++k) {
            part_range(j.cn, n_parts, k, &i0, &i1);
            const FormatPart& fp = parts[k];
            const char* base = fp.buf.v.data();
            const size_t stride = hits_sender ? 3 : 2;
            for (size_t i = i0; i < i1; ++i) {
                const size_t o = (i - i0) * stride;
                const char* label = qs.labels[j.c0 + i].c_str();
                if (hits_sender && hits_sender(hits_user, label, base + fp.off[o + 2]) != 0)
                    throw Error("sending on a disconnected channel (best hits)");
                if (sender(sender_user, label, base + fp.off[o], tsv ? base + fp.off[o + 1] : nullptr) != 0)
                    throw Error("sending on a disconnected channel (raxtax.rs:87)");
            }
        }
    }

    void plan_chunks(size_t n_ctx) { chunk_begin = plan_chunk_begins(nq, n_ctx, chunk_size, ramp); }

    void run(rtx_ctx* const* ctxs, size_t n_ctx, bool sharded = false) {
        t_start = now();
        if (!sharded) plan_chunks(n_ctx);
        t_first_issue = t_last_collect = t_start;
        size_t n_helpers = 0;
        if (const char* e = getenv("RXH_FORMAT_THREADS")) n_helpers = (size_t)std::max(0, atoi(e) - 1);
        else n_helpers = std::min<size_t>(3, std::max<size_t>(1, std::thread::hardware_concurrency() / 8));
        if (nq < 512 || chunk_size < 6144) n_helpers = 0;  // emit() only fans chunks of >= 6144 queries out
        parts.resize(n_helpers + 1);
        for (size_t k = 1; k <= n_helpers; ++k) helpers.emplace_back([this, k] { helper_main(k); });
        drivers_running = n_ctx;
        std::vector<std::thread> drivers;
        for (size_t i = 0; i < n_ctx; ++i) {
            if (sharded) drivers.emplace_back([this, ctx = ctxs[i], i] { drive_sharded(ctx, (int)i); });
            else drivers.emplace_back([this, ctx = ctxs[i]] { drive(ctx); });
        }
        while (true) {  // the calling thread is the writer side of the channel (main.rs:126-136)
            ChunkJob* j = nullptr;
            {
                auto t0 = now();
                std::unique_lock<std::mutex> g(q_mtx);
                q_cv.wait(g, [&] { return !ready.empty() || drivers_running == 0; });
                t_emit_wait.add(t0);
                if (ready.empty()) break;
                j = ready.front();
                ready.pop_front();
            }
            if (!failed.load()) {
                try {
                    emit(*j);
                } catch (const std::exception& e) {
                    fail(e.what());
                }
            }
            std::lock_guard<std::mutex> g(q_mtx);
            j->busy.store(false);
            free_cv.notify_all();
        }
        for (auto& t : drivers) t.join();
        {
            std::lock_guard<std::mutex> g(h_mtx);
            h_quit = true;
            h_cv.notify_all();
        }
        for (auto& t : helpers) t.join();
        if (getenv("RXH_TIMING"))
            fprintf(stderr, "[rxh raxtax] %zu queries, %zu ctx, chunk %zu, %zu format threads | drivers: acquire %.4f prep %.4f issue %.4f collect %.4f | "
                            "emitter: wait %.4f format %.4f send %.4f | wall %.4f (first batch issued after %.4f, last results on the host %.4f before the end) s\n",
                    nq, n_ctx, chunk_size, parts.size(), t_acquire.s(), t_prep.s(), t_issue.s(), t_collect.s(), t_emit_wait.s(), t_format.s(), t_send.s(),
                    std::chrono::duration<double>(now() - t_start).count(), std::chrono::duration<double>(t_first_issue - t_start).count(),
                    std::chrono::duration<double>(now() - t_last_collect).count());
    }
};
}  // namespace

// sender / logger that only count: what a benchmark hands to rxh_raxtax so that formatting, ordering and the per-query hand-off are
// all inside the timed region without a file system or an interpreter behind them
RXH_API int rxh_count_sender(void* user, const char* query_label, const char* primary_results, const char* tsv_results) {
    rxh_counts* c = (rxh_counts*)user;
    if (!c) return 0;
    c->queries += 1;
    c->label_bytes += strlen(query_label);
    const size_t n = strlen(primary_results);
    c->primary_bytes += n;
    uint64_t lines = n ? 1 : 0;
    for (const char* p = primary_results; (p = (const char*)memchr(p, '\n', (size_t)(primary_results + n - p))) != nullptr; ++p) ++lines;
    c->lines += lines;
    c->checksum += Tree::hash_bytes((const u8*)primary_results, n);  // a sum of per-query hashes: independent of the arrival order
    if (tsv_results) c->tsv_bytes += strlen(tsv_results);
    return 0;
}
RXH_API void rxh_release_buffers(void) { job_pool().clear(); }

RXH_API size_t rxh_format_fixed(double value, int precision, char* out, size_t cap) {
    char buf[448];
    if (precision < 0 || precision > 17) return 0;
    const size_t n = (size_t)(put_fixed(buf, value, precision) - buf);
    if (n + 1 > cap) return 0;
    memcpy(out, buf, n);
    out[n] = '\0';
    return n;
}
RXH_API void rxh_count_logger(void* user, int level, const char* message) {
    rxh_counts* c = (rxh_counts*)user;
    if (!c) return;
    c->log_lines += 1;
    c->log_bytes += strlen(message);
    if (level == 2) c->warn_lines += 1;
}

// ~8 chunks per context so that the pipeline (upload | kernels | formatting) has something to overlap and results, the progress file
// with them, appear while the run is going; bounded above so that the per-batch device arrays (~15 KB per 1.5 kb query) stay small
// next to the index, and below so that the index is not re-read from HBM for a handful of queries
static size_t default_chunk_size(size_t nq, size_t n_ctx) {
    return std::min<size_t>(32768, std::max<size_t>(1024, (nq + n_ctx * 8 - 1) / (n_ctx * 8)));
}

RXH_API size_t rxh_plan_chunks(size_t n_queries, size_t n_ctx, size_t chunk_size, size_t* begins, size_t cap) {
    n_ctx = std::max<size_t>(1, n_ctx);
    const bool ramp = chunk_size == 0;
    if (ramp) chunk_size = default_chunk_size(n_queries, n_ctx);
    const std::vector<size_t> b = plan_chunk_begins(n_queries, n_ctx, chunk_size, ramp);
    for (size_t i = 0; i < b.size() && i < cap; ++i) begins[i] = b[i];
    return b.size();
}

static int raxtax_query_partitioned(rtx_ctx* const* ctxs, size_t n_ctx, const rxh_queries* queries, const rxh_tree* tree_h, int skip_exact_matches,
                                    int raw_confidence, size_t chunk_size, rxh_sender sender, void* sender_user, int tsv, rxh_logger logger,
                                    void* logger_user, int* warnings, int both_strands, u32 best_hits, rxh_hits_sender hits_sender,
                                    void* hits_user, const char* who) {
    if (warnings) *warnings = 0;
    if (!ctxs || n_ctx == 0 || !queries || !tree_h) {
        g_err = std::string(who) + ": no context";
        return -1;
    }
    if (best_hits > 64) {
        g_err = std::string(who) + ": best_hits must be in [0, 64]";
        return -1;
    }
    const size_t nq = queries->q->size();
    const bool ramp = chunk_size == 0;
    if (chunk_size == 0) chunk_size = default_chunk_size(nq, n_ctx);
    Worker w{*tree_h->t, *queries->q, nq, chunk_size, skip_exact_matches, raw_confidence, tsv, sender, sender_user, logger, logger_user};
    w.ramp = ramp;
    w.both = both_strands != 0;
    w.best_hits = best_hits;
    w.hits_sender = best_hits ? hits_sender : nullptr;
    w.hits_user = hits_user;
    w.run(ctxs, n_ctx);
    if (best_hits)  // the option outlives the call in the contexts: leave them as they were handed in
        for (size_t i = 0; i < n_ctx; ++i) rtx_ctx_set_option(ctxs[i], RTX_OPT_BEST_HITS, 0);
    if (warnings) *warnings = w.warned.load() ? 1 : 0;
    if (w.failed.load()) {
        g_err = w.err;
        return -1;
    }
    return 0;
}

RXH_API int rxh_raxtax_multi(rtx_ctx* const* ctxs, size_t n_ctx, const rxh_queries* queries, const rxh_tree* tree_h, int skip_exact_matches,
                             int raw_confidence, size_t chunk_size, rxh_sender sender, void* sender_user, int tsv, rxh_logger logger,
                             void* logger_user, int* warnings) {
    return raxtax_query_partitioned(ctxs, n_ctx, queries, tree_h, skip_exact_matches, raw_confidence, chunk_size, sender, sender_user, tsv, logger,
                                    logger_user, warnings, 0, 0, nullptr, nullptr, "rxh_raxtax_multi");
}

RXH_API int rxh_raxtax_both_strands(rtx_ctx* const* ctxs, size_t n_ctx, const rxh_queries* queries, const rxh_tree* tree_h, int skip_exact_matches,
                                    int raw_confidence, size_t chunk_size, rxh_sender sender, void* sender_user, int tsv, rxh_logger logger,
                                    void* logger_user, int* warnings) {
    return raxtax_query_partitioned(ctxs, n_ctx, queries, tree_h, skip_exact_matches, raw_confidence, chunk_size, sender, sender_user, tsv, logger,
                                    logger_user, warnings, 1, 0, nullptr, nullptr, "rxh_raxtax_both_strands");
}

RXH_API int rxh_raxtax_best_hits(rtx_ctx* const* ctxs, size_t n_ctx, const rxh_queries* queries, const rxh_tree* tree_h, int skip_exact_matches,
                                 int raw_confidence, size_t chunk_size, rxh_sender sender, void* sender_user, int tsv, rxh_logger logger,
                                 void* logger_user, int* warnings, int both_strands, uint32_t best_hits, rxh_hits_sender hits_sender,
                                 void* hits_user) {
    return raxtax_query_partitioned(ctxs, n_ctx, queries, tree_h, skip_exact_matches, raw_confidence, chunk_size, sender, sender_user, tsv, logger,
                                    logger_user, warnings, both_strands, best_hits, hits_sender, hits_user, "rxh_raxtax_best_hits");
}

// Reference-sharded mode: the result lines the ranks emitted for one batch, merged per query.  Lines are ordered like
// lineage.rs:93 (confidence vectors descending lexicographically, on an equal prefix the longer vector first; ties in depth-first
// push order == ascending first reference), then the one-exact-match override of raxtax.rs:73-84 is applied -- it needs the best
// line of ALL ranks, which is why the ranks leave it to the merge.
RXH_API int rxh_merge_shard_results(size_t n_ranks, size_t n_queries, uint32_t max_levels, const uint32_t* const* result_begin,
                                    const uint32_t* const* first_ref, const uint8_t* const* n_levels, const double* const* confidence,
                                    const double* const* local_signal, const uint32_t* exact_offsets, const uint32_t* exact_ids,
                                    const uint8_t* ref_levels, int skip_exact_matches, int raw_confidence, uint32_t* out_begin,
                                    uint32_t* out_first, uint8_t* out_nlev, double* out_conf, double* out_local, uint64_t out_capacity,
                                    uint64_t* n_out) {
    try {
        struct Line {
            u32 rank, idx, first;
            u8 n;
        };
        const u32 ML = max_levels;
        std::vector<Line> lines;
        u64 w = 0;
        out_begin[0] = 0;
        for (size_t q = 0; q < n_queries; ++q) {
            lines.clear();
            for (size_t r = 0; r < n_ranks; ++r)
                for (u32 i = result_begin[r][q]; i < result_begin[r][q + 1]; ++i) lines.push_back(Line{(u32)r, i, first_ref[r][i], n_levels[r][i]});
            if (lines.empty()) throw Error("query " + std::to_string(q) + ": empty evaluation result (raxtax.rs:72)");
            auto hundredths = [&](const Line& l, u32 lev) { return (long)std::lround(confidence[l.rank][(size_t)l.idx * ML + lev] * 100.0); };
            std::sort(lines.begin(), lines.end(), [&](const Line& a, const Line& b) {
                for (u32 lev = 0; lev < ML; ++lev) {
                    const bool ha = lev < a.n, hb = lev < b.n;
                    if (!ha && !hb) break;
                    if (ha != hb) return ha;  // equal prefix: the longer vector first
                    const long ka = hundredths(a, lev), kb = hundredths(b, lev);
                    if (ka != kb) return ka > kb;
                }
                return a.first < b.first;
            });
            const u32 ne = exact_offsets ? exact_offsets[q + 1] - exact_offsets[q] : 0u;
            if (!raw_confidence && !skip_exact_matches && ne == 1) {
                if (w + 1 > out_capacity) throw Error("rxh_merge_shard_results: output capacity too small");
                const u32 id = exact_ids[exact_offsets[q]];
                const u32 n = ref_levels[id];
                out_first[w] = id;
                out_nlev[w] = (u8)n;
                for (u32 lev = 0; lev < ML; ++lev) out_conf[w * ML + lev] = lev < n ? 1.0 : 0.0;
                out_local[w] = local_signal[lines[0].rank][lines[0].idx];  // signals of the best computed line
                ++w;
            } else {
                if (w + lines.size() > out_capacity) throw Error("rxh_merge_shard_results: output capacity too small");
                for (const Line& l : lines) {
                    out_first[w] = l.first;
                    out_nlev[w] = l.n;
                    memcpy(out_conf + w * ML, confidence[l.rank] + (size_t)l.idx * ML, (size_t)ML * 8);
                    out_local[w] = local_signal[l.rank][l.idx];
                    ++w;
                }
            }
            out_begin[q + 1] = (u32)w;
        }
        if (n_out) *n_out = w;
        return 0;
    } catch (const std::exception& e) {
        g_err = e.what();
        return -1;
    }
}

// raxtax::raxtax over a reference-sharded index held by ONE process: ctxs[r] is shard r (rxh_tree_upload_sharded).  Per chunk: batch
// to every shard, phase 1, histogram exchange, phase 2, record exchange, phase 3, per-rank downloads, merge, then the same formatting
// and sending as rxh_raxtax, in query order.  (With one process per GPU the same phases run with NCCL in between: raxtax_b200/dist.py.)
RXH_API int rxh_raxtax_sharded(rtx_ctx* const* ctxs, size_t n_ctx, const rxh_queries* queries, const rxh_tree* tree_h, int skip_exact_matches,
                               int raw_confidence, size_t chunk_size, rxh_sender sender, void* sender_user, int tsv, rxh_logger logger,
                               void* logger_user, int* warnings) {
    try {
        if (warnings) *warnings = 0;
        if (!ctxs || n_ctx == 0 || !queries || !tree_h) throw Error("rxh_raxtax_sharded: no context");
        const Tree& tree = *tree_h->t;
        const Queries& qs = *queries->q;
        const size_t nq = qs.size();
        const u32 ML = rtx_index_max_levels(ctxs[0]);
        for (size_t r = 0; r < n_ctx; ++r)
            if (rtx_index_n_refs(ctxs[r]) != tree.num_tips) throw Error("a context's index does not belong to this tree");
        {
            // every shard on its own GPU: the exchanges are NCCL collectives inside the device library (rtx_shard_run / rtx_shard_gather),
            // one driver thread per rank.  Several shards on one GPU (tests, a database too large for the GPUs at hand): NCCL does not
            // take two ranks on one device, the exchanges below are staged through page-locked host memory instead.
            bool distinct = n_ctx > 1;
            for (size_t a = 0; a < n_ctx && distinct; ++a)
                for (size_t b = a + 1; b < n_ctx; ++b) distinct &= rtx_ctx_device(ctxs[a]) != rtx_ctx_device(ctxs[b]);
            if (distinct && getenv("RXH_SHARD_NO_NCCL") == nullptr) {
                unsigned char uid[RTX_COMM_UNIQUE_ID_BYTES];
                if (rtx_comm_unique_id(uid)) throw Error(std::string("rtx_comm_unique_id: ") + rtx_last_error(nullptr));
                std::vector<int> rcs(n_ctx, 0);
                {
                    std::vector<std::thread> th;  // ncclCommInitRank blocks until every rank has joined
                    for (size_t r = 0; r < n_ctx; ++r) th.emplace_back([&, r] { rcs[r] = rtx_comm_init(ctxs[r], uid, (int)r, (int)n_ctx); });
                    for (auto& t : th) t.join();
                }
                for (size_t r = 0; r < n_ctx; ++r)
                    if (rcs[r]) throw Error(std::string("rtx_comm_init: ") + rtx_last_error(ctxs[r]));
                if (chunk_size == 0) chunk_size = std::min<size_t>(32768, std::max<size_t>(2048, (nq + 3) / 4));
                Worker w{tree, qs, nq, chunk_size, skip_exact_matches, raw_confidence, tsv, sender, sender_user, logger, logger_user};
                w.run(ctxs, n_ctx, true);
                for (size_t r = 0; r < n_ctx; ++r) rtx_comm_destroy(ctxs[r]);
                if (warnings) *warnings = w.warned.load() ? 1 : 0;
                if (w.failed.load()) throw Error(w.err);
                return 0;
            }
        }
        if (chunk_size == 0) chunk_size = std::min<size_t>(std::max<size_t>(nq, 1), 8192);
        struct RankOut {
            std::vector<u32> begin, first;
            std::vector<u16> n_kmers;
            std::vector<u8> nlev;
            std::vector<double> conf, local, global;
        };
        std::vector<RankOut> ro(n_ctx);
        std::vector<u32> exact_off, exact_ids, ex, m_begin, m_first;
        std::vector<u8> m_nlev;
        std::vector<double> m_conf, m_local;
        std::string primary, tsv_out, msg;
        bool warned = false;
        auto dev = [&](int rc, rtx_ctx* c, const char* what) {
            if (rc) throw Error(std::string(what) + ": " + rtx_last_error(c));
        };
        for (size_t c0 = 0; c0 < nq;) {
            const size_t cn = std::min(chunk_size, nq - c0);
            exact_off.assign(cn + 1, 0);
            exact_ids.clear();
            for (size_t i = 0; i < cn; ++i) {  // tree.sequences.get(query_sequence) (raxtax.rs:42)
                const size_t q = c0 + i;
                tree.exact(qs.codes.data() + qs.off[q], (size_t)(qs.off[q + 1] - qs.off[q]), &ex);
                exact_ids.insert(exact_ids.end(), ex.begin(), ex.end());
                exact_off[i + 1] = (u32)exact_ids.size();
            }
            rtx_batch batch{};
            batch.n_queries = (u32)cn;
            batch.seq_offsets = qs.off.data() + c0;
            batch.seq_codes = qs.codes.data();
            batch.exact_offsets = exact_off.data();
            batch.exact_ids = exact_ids.empty() ? nullptr : exact_ids.data();
            batch.flags = (skip_exact_matches ? RTX_SKIP_EXACT_MATCHES : 0u) | (raw_confidence ? RTX_RAW_CONFIDENCE : 0u);
            bool too_big = false;
            for (size_t r = 0; r < n_ctx && !too_big; ++r) {
                dev(rtx_batch_upload(ctxs[r], &batch), ctxs[r], "rtx_batch_upload");
                too_big = rtx_batch_sub_batch(ctxs[r]) < cn;  // sharded batches must fit one sub-batch of every shard
            }
            if (too_big) {
                if (chunk_size <= 1) throw Error("rxh_raxtax_sharded: not even one query fits the shards' scratch memory");
                chunk_size = (chunk_size + 1) / 2;
                continue;
            }
            for (size_t r = 0; r < n_ctx; ++r) dev(rtx_shard_phase1(ctxs[r]), ctxs[r], "rtx_shard_phase1");
            dev(rtx_shard_exchange_hist_local(ctxs, (uint32_t)n_ctx), ctxs[0], "rtx_shard_exchange_hist_local");
            for (size_t r = 0; r < n_ctx; ++r) dev(rtx_shard_phase2(ctxs[r]), ctxs[r], "rtx_shard_phase2");
            dev(rtx_shard_exchange_records_local(ctxs, (uint32_t)n_ctx), ctxs[0], "rtx_shard_exchange_records_local");
            for (size_t r = 0; r < n_ctx; ++r) dev(rtx_shard_phase3(ctxs[r]), ctxs[r], "rtx_shard_phase3");
            size_t total = 0;
            for (size_t r = 0; r < n_ctx; ++r) {
                RankOut& o = ro[r];
                o.n_kmers.resize(cn);
                o.begin.resize(cn + 1);
                o.global.resize(cn);
                size_t cap = std::max<size_t>(o.first.size(), cn * 8 + 64);
                while (true) {
                    o.first.resize(cap);
                    o.nlev.resize(cap);
                    o.conf.resize(cap * ML);
                    o.local.resize(cap);
                    rtx_results res{};
                    res.n_kmers = o.n_kmers.data();
                    res.result_begin = o.begin.data();
                    res.global_signal = o.global.data();
                    res.result_capacity = cap;
                    res.first_ref = o.first.data();
                    res.n_levels = o.nlev.data();
                    res.confidence = o.conf.data();
                    res.local_signal = o.local.data();
                    const int rc = rtx_batch_download(ctxs[r], &res);
                    if (rc == RTX_ERR_INVALID && res.n_results > cap) {
                        cap = res.n_results + 64;
                        continue;
                    }
                    dev(rc, ctxs[r], "rtx_batch_download");
                    total += res.n_results;
                    break;
                }
            }
            // merge the shards' lines per query (order of lineage.rs:93, then the override of raxtax.rs:73-84)
            std::vector<const u32*> pb(n_ctx), pf(n_ctx);
            std::vector<const u8*> pn(n_ctx);
            std::vector<const double*> pc(n_ctx), pl(n_ctx);
            for (size_t r = 0; r < n_ctx; ++r) {
                pb[r] = ro[r].begin.data();
                pf[r] = ro[r].first.data();
                pn[r] = ro[r].nlev.data();
                pc[r] = ro[r].conf.data();
                pl[r] = ro[r].local.data();
            }
            const size_t mcap = total + cn;
            m_begin.resize(cn + 1);
            m_first.resize(mcap);
            m_nlev.resize(mcap);
            m_conf.resize(mcap * ML);
            m_local.resize(mcap);
            uint64_t n_out = 0;
            if (rxh_merge_shard_results(n_ctx, cn, ML, pb.data(), pf.data(), pn.data(), pc.data(), pl.data(), exact_off.data(),
                                        exact_ids.empty() ? exact_off.data() : exact_ids.data(), tree.ref_levels.data(), skip_exact_matches,
                                        raw_confidence, m_begin.data(), m_first.data(), m_nlev.data(), m_conf.data(), m_local.data(), mcap, &n_out) != 0)
                throw Error(g_err);
            for (size_t i = 0; i < cn; ++i) {
                const size_t q = c0 + i;
                if (!skip_exact_matches) {  // the log lines of raxtax.rs:43-53
                    bool all_equal = true;
                    std::string first_parent;
                    for (u32 j = exact_off[i]; j < exact_off[i + 1]; ++j) {
                        const std::string& l = tree.lineages[exact_ids[j]];
                        if (logger) {
                            msg = "Exact sequence match for query " + qs.labels[q] + ": " + l;
                            logger(logger_user, 3, msg.c_str());
                        }
                        const size_t p = l.rfind(',');
                        if (p == std::string::npos)
                            throw Error("called `Option::unwrap()` on a `None` value: lineage without ',' (raxtax.rs:49)");
                        if (j == exact_off[i]) first_parent.assign(l, 0, p);
                        else if (l.compare(0, p, first_parent) != 0 || p != first_parent.size()) all_equal = false;
                    }
                    if (!all_equal) {
                        if (logger) {
                            msg = "Exact matches for " + qs.labels[q] + " differ above the leafs of the lineage tree!";
                            logger(logger_user, 2, msg.c_str());
                        }
                        warned = true;
                    }
                }
                primary.clear();
                tsv_out.clear();
                std::string seq;
                if (tsv) seq = decompress_sequence(qs.codes.data() + qs.off[q], (size_t)(qs.off[q + 1] - qs.off[q]));
                for (u32 r = m_begin[i]; r < m_begin[i + 1]; ++r) {
                    ResultView rv{&tree.lineages[m_first[r]], m_conf.data() + (size_t)r * ML, m_nlev[r], m_local[r], ro[0].global[i]};
                    if (r != m_begin[i]) primary += '\n';
                    output_string(primary, qs.labels[q], rv);
                    if (tsv) {
                        if (r != m_begin[i]) tsv_out += '\n';
                        tsv_string(tsv_out, qs.labels[q], rv, seq);
                    }
                }
                if (sender && sender(sender_user, qs.labels[q].c_str(), primary.c_str(), tsv ? tsv_out.c_str() : nullptr) != 0)
                    throw Error("sending on a disconnected channel (raxtax.rs:87)");
            }
            c0 += cn;
        }
        if (warnings) *warnings = warned ? 1 : 0;
        return 0;
    } catch (const std::exception& e) {
        g_err = e.what();
        return -1;
    }
}

RXH_API int rxh_raxtax(rtx_ctx* ctx, const rxh_queries* queries, const rxh_tree* tree_h, int skip_exact_matches, int raw_confidence,
                       size_t chunk_size, rxh_sender sender, void* sender_user, int tsv, rxh_logger logger, void* logger_user, int* warnings) {
    rtx_ctx* one[1] = {ctx};
    return rxh_raxtax_multi(one, 1, queries, tree_h, skip_exact_matches, raw_confidence, chunk_size, sender, sender_user, tsv, logger,
                            logger_user, warnings);
}

