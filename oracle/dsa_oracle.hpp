// TEST INFRASTRUCTURE — NOT PRODUCT CODE.
//
// CPU oracle for the DynamicSparseArrays.jl hot path (PMA / PCSR insert, update,
// delete, find, column gather, SpMV, buffered flush).  It is a literal,
// single-threaded C++17 restatement of the reference's Julia algorithms
// (reference = /root/reference, atoptima/DynamicSparseArrays.jl v0.7.2), with
// 1-based positions and Float64 arithmetic exactly where the reference uses it.
// Every function cites the reference file:line it follows.
//
// Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl
// reference legs may load this code, and only as the checker / baseline.  The
// product (libdsa.so, CUDA) never links or calls it.
//
// Parity pinning: Julia is not installed in the build container, so the
// reference itself cannot be executed here.  The oracle is pinned against every
// known-answer assertion the reference's own test-suite holds for this path
// (test/unit/finds.jl, writes.jl, comparison.jl, views.jl, spmv.jl,
// test/functional/sparsevector.jl, sparsematrix.jl, README.md) — see
// tests/test_oracle_golden.py.  Two points are "parity unpinned" (no reference
// test fixes them; SURVEY.md §8c): explicit zeros in SpMV output, and the fold
// order of >=3 Float64 duplicates in the matrix builder (input-order left fold
// adopted, which is what sortperm's index tie-break yields).
//
// Compile with -ffp-contract=off (no FMA contraction: Julia does not contract).
#pragma once
#include <cstdint>
#include <cstddef>
#include <vector>
#include <string>
#include <optional>
#include <unordered_map>
#include <algorithm>
#include <cmath>

namespace orc {

enum ErrCode : int {
    OK = 0,
    ERR_ARGUMENT = 1,   // Julia ArgumentError
    ERR_BOUNDS = 2,     // Julia BoundsError
    ERR_ERROR = 3,      // Julia ErrorException (error("..."))
    ERR_ASSERT = 4,     // Julia AssertionError (@assert)
};

struct Error {
    int code;
    std::string msg;
};

enum Combine : int { COMB_ADD = 0, COMB_MUL = 1, COMB_LAST = 2, COMB_FIRST = 3, COMB_MIN = 4, COMB_MAX = 5 };

// Base.min / Base.max on IEEE floats: NaN if either argument is NaN (the NaN argument itself, as x86 returns it from the
// `x - y` Base computes), -0.0 orders below 0.0, otherwise the smaller / larger argument
inline double julia_min(double a, double b) {
    if (std::isnan(a)) return a;
    if (std::isnan(b)) return b;
    if (a == b) return std::signbit(a) ? a : b;
    return b < a ? b : a;
}
inline double julia_max(double a, double b) {
    if (std::isnan(a)) return a;
    if (std::isnan(b)) return b;
    if (a == b) return std::signbit(a) ? b : a;
    return b > a ? b : a;
}

inline double combine_apply(int c, double a, double b) {
    switch (c) {
        case COMB_ADD: return a + b;
        case COMB_MUL: return a * b;
        case COMB_LAST: return b;
        case COMB_FIRST: return a;
        case COMB_MIN: return julia_min(a, b);
        case COMB_MAX: return julia_max(a, b);
    }
    return a + b;
}

// Elements{K,T} = Vector{Union{Nothing,Tuple{K,T}}}   (DynamicSparseArrays.jl:18)
// Julia lays an isbits-Union array out as a 16 B payload array + a 1 B type-tag
// array; mirrored here so the CPU baseline has the reference's memory behaviour.
struct KV { int64_t key; double val; };
struct Elements {
    std::vector<KV> kv;
    std::vector<uint8_t> tag;  // 1 = Tuple, 0 = nothing
    Elements() {}
    explicit Elements(size_t n) : kv(n, KV{0, 0.0}), tag(n, 0) {}
    int64_t length() const { return (int64_t)tag.size(); }
    bool empty_at(int64_t pos) const { return tag[pos - 1] == 0; }            // utils.jl:1  _isempty
    const KV& at(int64_t pos) const { return kv[pos - 1]; }
    void set(int64_t pos, int64_t k, double v) { kv[pos - 1] = KV{k, v}; tag[pos - 1] = 1; }
    void set_nothing(int64_t pos) { tag[pos - 1] = 0; }
    void copy_cell(int64_t dst, int64_t src) { kv[dst - 1] = kv[src - 1]; tag[dst - 1] = tag[src - 1]; }
    void resize(int64_t n) { kv.resize(n, KV{0, 0.0}); tag.resize(n, 0); }  // resize! zero-tags new cells (pma.jl:29,149)
};

// semaphores::Vector{Union{Nothing,Int}} — 0 encodes `nothing` (positions are >= 1)
using Semaphores = std::vector<int64_t>;

// ---- utils.jl ----------------------------------------------------------------
int64_t nextemptypos(const Elements& a, int64_t from);          // utils.jl:3
int64_t previousemptypos(const Elements& a, int64_t from);      // utils.jl:21
int64_t nbcells(const Elements& a, int64_t from, int64_t to);   // utils.jl:48
// ---- finds.jl ----------------------------------------------------------------
int64_t find(const Elements& a, int64_t key, int64_t from, int64_t to);  // finds.jl:29 (returns pos; 0 = (0,nothing))
// ---- moves.jl ----------------------------------------------------------------
void movecellstoright(Elements& a, int64_t from, int64_t to, Semaphores* sem);  // moves.jl:7
void movecellstoleft(Elements& a, int64_t from, int64_t to, Semaphores* sem);   // moves.jl:50
void pack(Elements& a, int64_t window_start, int64_t window_end, int64_t m);    // moves.jl:94
void spread4(Elements& a, int64_t window_start, int64_t window_end, int64_t m); // moves.jl:120
void spread5(Elements& a, int64_t window_start, int64_t window_end, int64_t m, Semaphores* sem);  // moves.jl:142
// ---- writes.jl ---------------------------------------------------------------
struct PosFlag { int64_t pos; bool flag; };
PosFlag insert(Elements& a, int64_t key, double value, int64_t from, int64_t to, Semaphores* sem);  // writes.jl:14
PosFlag insert_after(Elements& a, int64_t key, double value, int64_t pos, Semaphores* sem);         // writes.jl:26 _insert!
PosFlag del(Elements& a, int64_t key, int64_t from, int64_t to);  // writes.jl:57
struct PurgeRes { int64_t mid; int64_t nb; };
PurgeRes purge(Elements& a, int64_t from, int64_t to);            // writes.jl:80
bool arrays_equal(const Elements& a1, const Elements& a2);        // pma.jl:236

// ---- pma.jl ------------------------------------------------------------------
struct Pma {   // pma.jl:8-24
    int64_t capacity = 0, segment_capacity = 0, nb_segments = 0, nb_elements = 0, height = 0;
    double t_h = 0.7, t_0 = 0.92, p_h = 0.3, p_0 = 0.08, t_d = 0, p_d = 0;
    Elements array;
};
struct Window { int64_t start, end, nbcells; };
void pma_init(Pma& p, int64_t nb_elements);                          // pma.jl:42 _pma (array already sized/filled)
void pma_build_sorted(Pma& p, const int64_t* keys, const double* vals, int64_t n);  // pma.jl:69 with sort=false
void pma_empty(Pma& p, int64_t expected_nb_elems = 100);              // pma.jl:86
Window look_for_rebalance(Pma& p, int64_t pos);                       // pma.jl:105
void pma_even_rebalance(Pma& p, int64_t ws, int64_t we, int64_t m);   // pma.jl:94
double pma_get(const Pma& p, int64_t key);                            // pma.jl:189
void pma_set(Pma& p, double value, int64_t key);                      // pma.jl:196

// ---- vector.jl ---------------------------------------------------------------
void prepare_keys_vals(std::vector<int64_t>& keys, std::vector<double>& vals, int combine);  // vector.jl:10
struct Vec {   // vector.jl:1-4
    int64_t n = 0;
    Pma pma;
};
void vec_build(Vec& v, std::vector<int64_t> I, std::vector<double> V, int combine, int64_t n, bool n_given);  // vector.jl:38-62
void vec_set(Vec& v, double value, int64_t key);   // vector.jl:76
double vec_get(const Vec& v, int64_t key);         // vector.jl:72

// ---- pcsr.jl -----------------------------------------------------------------
struct Pcsc {   // pcsr.jl:4-9
    int64_t nb_partitions = 0;
    Semaphores semaphores;
    Pma pma;
};
struct ColKeys {   // Vector{Union{Nothing,L}}  (pcsr.jl:17)
    std::vector<int64_t> key;
    std::vector<uint8_t> live;
    int64_t length() const { return (int64_t)key.size(); }
};
struct Mpcsc {   // pcsr.jl:16-19
    ColKeys col_keys;
    Pcsc pcsc;
};
void pcsc_build(Pcsc& m, const std::vector<std::vector<int64_t>>& row_keys,
                const std::vector<std::vector<double>>& values, int combine);   // pcsr.jl:26
void pcsc_empty(Pcsc& m);                                                         // pcsr.jl:65
void pcsc_addpartition_end(Pcsc& m);                                              // pcsr.jl:99
void pcsc_addpartition_after(Pcsc& m, int64_t prev_sem_id);                       // pcsr.jl:114
int64_t pos_of_partition_start(const Pcsc& m, int64_t partition);                 // pcsr.jl:171
int64_t pos_of_partition_end(const Pcsc& m, int64_t partition);                   // pcsr.jl:177
void pcsc_deletepartition(Pcsc& m, int64_t partition);                            // pcsr.jl:188
double pcsc_get(const Pcsc& m, int64_t key, int64_t partition);                   // pcsr.jl:228
void pcsc_set(Pcsc& m, double value, int64_t key, int64_t partition);             // pcsr.jl:294
int64_t colkeys_find(const ColKeys& ck, int64_t col, bool* exact);                // finds.jl:59 on col_keys
int64_t mpcsc_addcolumn(Mpcsc& m, int64_t col, int64_t prev_col_pos);             // pcsr.jl:148
void mpcsc_deletecolumn(Mpcsc& m, int64_t col);                                   // pcsr.jl:206
double mpcsc_get(const Mpcsc& m, int64_t row, int64_t col);                       // pcsr.jl:261
void mpcsc_set(Mpcsc& m, double value, int64_t row, int64_t col);                 // pcsr.jl:341
void mpcsc_build_coo(Mpcsc& m, std::vector<int64_t> I, std::vector<int64_t> J, std::vector<double> V, int combine);  // pcsr.jl:354,433
void mpcsc_column(const Mpcsc& m, int64_t col, std::vector<int64_t>& keys, std::vector<double>& vals);  // pcsr.jl:285 / views.jl:15
void mpcsc_row(const Mpcsc& m, int64_t row, std::vector<int64_t>& keys, std::vector<double>& vals);     // pcsr.jl:269
// operations.jl:62-135   SpMSpV of the column-major structure with a sparse x (ascending keys)
void mpcsc_mul(const Mpcsc& m, const int64_t* xk, const double* xv, int64_t nx,
               std::vector<int64_t>& yk, std::vector<double>& yv);

// ---- buffer.jl / matrix.jl -----------------------------------------------------
struct Buffer {   // buffer.jl:1-4 (Dict row -> (colids, vals)); row order = first insertion
    std::unordered_map<int64_t, size_t> index;
    std::vector<int64_t> rowid;
    std::vector<std::vector<int64_t>> colids;
    std::vector<std::vector<double>> vals;
    int64_t length = 0;
};
struct Matrix {   // matrix.jl:1-8
    int64_t m = 0, n = 0;
    bool fillmode = false;
    Buffer buffer;
    Mpcsc colmajor, rowmajor;
};
void matrix_build(Matrix& A, const std::vector<int64_t>& I, const std::vector<int64_t>& J,
                  const std::vector<double>& V, int64_t m, int64_t n, bool dims_given, int combine = COMB_ADD);  // matrix.jl:15
void matrix_empty(Matrix& A, bool fill_mode);                                  // matrix.jl:31
void matrix_set(Matrix& A, double val, int64_t row, int64_t col);              // matrix.jl:43
double matrix_get(const Matrix& A, int64_t row, int64_t col);                  // matrix.jl:64
void matrix_deletecolumn(Matrix& A, int64_t col);                              // matrix.jl:95
void matrix_deleterow(Matrix& A, int64_t row);                                 // matrix.jl:104
void matrix_addrow(Matrix& A, int64_t row, const std::vector<int64_t>& colids, const std::vector<double>& vals);  // matrix.jl:113
void matrix_closefillmode(Matrix& A);                                          // matrix.jl:126

}  // namespace orc
