/*
 * gnn_oracle.c — CPU restatement of the reference's message-passing hot path.
 *
 * TEST INFRASTRUCTURE, NOT PRODUCT.  Only tests/, __graft_entry__.smoke() and bench.py's CPU legs
 * (`cpu_baseline`, `--impl reference`) may load this; the product path (libgnnb200.so) never does and has
 * no CPU fallback.
 *
 * What it restates (file:line under CarloLucibello/GraphNeuralNetworks.jl @ e46d1b04):
 *   GNNlib/src/msgpass.jl:71-79,117-129,145-149,191-208,215-238   propagate / apply_edges / aggregate_neighbors
 *   GNNGraphs/src/gatherscatter.jl:1-18                            _gather / _scatter -> NNlib.gather / scatter
 *   GNNlib/src/utils.jl:84-97                                      softmax_edge_neighbors
 *   GNNlib/src/layers/conv.jl:14-72,112-167,277-283                gcn_conv / gat_conv / sage_conv (edge parts;
 *                                                                  gat_conv's also in closed-form pullback)
 *   GNNGraphs/src/query.jl:220-231,314-369                         adjacency_matrix / degree
 *   GNNGraphs/src/convert.jl:221-237                               to_sparse (COO -> CSC, duplicates summed)
 * The arithmetic itself lives in a third-party dependency that is NOT in the reference tree:
 * NNlib.jl (compat "0.9", resolved 0.9.21 in the Pluto manifests) `gather`/`scatter`, plus the SparseArrays
 * stdlib dense x CSC product.  Their published semantics are restated here (SURVEY.md §8 a5).
 *
 * PINNING.  Julia is not installed in this image or on the GPU box, so the reference cannot be executed.
 * The oracle is pinned against every known-answer vector the reference's own tests hold for this path
 * (tests/test_oracle_golden.py; list in SURVEY.md §8c).  What those tests do NOT pin is stated there and in
 * DESIGN.md: max/min aggregation through propagate (tie gradients, ∓Inf for isolated targets) is
 * "parity unpinned" — it follows NNlib's documented semantics only.
 *
 * Build: oracle/Makefile -> oracle/liboracle.so   (gcc -O3 -march=native -fopenmp).  There is no oracle/_ref:
 * the reference is pure Julia, nothing in it compiles with gcc (DESIGN.md).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

enum { ORC_SUM = 0, ORC_MEAN = 1, ORC_MAX = 2, ORC_MIN = 3 };
enum { ORC_DIR_OUT = 0, ORC_DIR_IN = 1, ORC_DIR_BOTH = 2 };

#define T float
#define FN(name) name##_f32
#define EXPFN expf
#define SQRTFN sqrtf
#include "gnn_oracle_impl.h"
#undef T
#undef FN
#undef EXPFN
#undef SQRTFN

#define T double
#define FN(name) name##_f64
#define EXPFN exp
#define SQRTFN sqrt
#include "gnn_oracle_impl.h"
#undef T
#undef FN
#undef EXPFN
#undef SQRTFN

int orc_num_threads(void) {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}

/* ---- index arithmetic (bit-exact) ------------------------------------------------------------- */

/* add_self_loops (GNNGraphs/src/transform.jl:12-28): s=[s;1:n], t=[t;1:n]; weights padded with 1 */
void orc_add_self_loops(const int64_t* s, const int64_t* t, int64_t E, int64_t n, int64_t* s2, int64_t* t2) {
    memcpy(s2, s, sizeof(int64_t) * (size_t)E);
    memcpy(t2, t, sizeof(int64_t) * (size_t)E);
    for (int64_t i = 0; i < n; ++i) { s2[E + i] = i + 1; t2[E + i] = i + 1; }
}

/* Stable CSR by `key` (t for the forward plan, s for the transposed one): the index arithmetic our plan must
 * reproduce exactly.  rowptr[n+1], col[E] (= other[perm]), perm[E] 0-based COO positions, all 0-based. */
void orc_csr(const int64_t* key, const int64_t* other, int64_t E, int64_t n, int32_t* rowptr, int32_t* col,
             int32_t* perm) {
    for (int64_t i = 0; i <= n; ++i) rowptr[i] = 0;
    for (int64_t k = 0; k < E; ++k) rowptr[key[k]]++;
    for (int64_t i = 0; i < n; ++i) rowptr[i + 1] += rowptr[i];
    int32_t* pos = (int32_t*)malloc(sizeof(int32_t) * (size_t)(n > 0 ? n : 1));
    for (int64_t i = 0; i < n; ++i) pos[i] = rowptr[i];
    for (int64_t k = 0; k < E; ++k) {
        int32_t p = pos[key[k] - 1]++;
        col[p] = (int32_t)(other[k] - 1);
        perm[p] = (int32_t)k;
    }
    free(pos);
}

/* ---- RMAT generator: bit-identical to gnnb_rmat_edges (csrc/api.cu) ------------------------------ */
static inline uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
void orc_rmat(int64_t N, int64_t E, uint64_t seed, int64_t* src, int64_t* dst) {
    const uint32_t TA = 9563013u, TB = 12750684u, TC = 15938355u;
    int scale = 0;
    while (((int64_t)1 << scale) < N) ++scale;
#pragma omp parallel for schedule(static)
    for (int64_t id = 0; id < E; ++id) {
        uint64_t s = 0, d = 0;
        for (uint64_t retry = 0;; ++retry) {
            uint64_t state = splitmix64(seed ^ splitmix64((uint64_t)id * 0x100000001B3ull + retry));
            s = 0; d = 0;
            for (int l = 0; l < scale; ++l) {
                state = splitmix64(state);
                const uint32_t u = (uint32_t)(state >> 40);
                const uint64_t sb = (u >= TB) ? 1 : 0;
                const uint64_t db = ((u >= TA && u < TB) || (u >= TC)) ? 1 : 0;
                s = (s << 1) | sb;
                d = (d << 1) | db;
            }
            if ((int64_t)s < N && (int64_t)d < N) break;
            if (retry >= 63) { s %= (uint64_t)N; d %= (uint64_t)N; break; }
        }
        src[id] = (int64_t)s + 1;
        dst[id] = (int64_t)d + 1;
    }
}

/* ---- generous all-cores baseline (NOT how the reference runs — it is serial): prebuilt CSR, OpenMP over
 * target rows.  out[i,:] = ct[i] * sum_e w[e] cs[col[e]] x[col[e],:]  with w in CSR order. ---------- */
void orc_spmm_csr_omp(const int32_t* rowptr, const int32_t* col, int64_t n, const float* x, const float* w,
                      const float* cs, const float* ct, int64_t D, float* out) {
#pragma omp parallel for schedule(dynamic, 256)
    for (int64_t i = 0; i < n; ++i) {
        float* o = out + i * D;
        for (int64_t f = 0; f < D; ++f) o[f] = 0.f;
        for (int32_t p = rowptr[i]; p < rowptr[i + 1]; ++p) {
            const float* xr = x + (int64_t)col[p] * D;
            float a = w ? w[p] : 1.f;
            if (cs) a *= cs[col[p]];
            for (int64_t f = 0; f < D; ++f) o[f] += a * xr[f];
        }
        if (ct) for (int64_t f = 0; f < D; ++f) o[f] *= ct[i];
    }
}
