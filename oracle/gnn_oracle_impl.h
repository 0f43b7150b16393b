/* gnn_oracle_impl.h — type-generic body of the oracle; included twice by gnn_oracle.c with
 * T = float (the reference's own fp32 arithmetic, same operation order) and T = double (tight oracle).
 * TEST INFRASTRUCTURE ONLY — see the header comment of gnn_oracle.c. */

/* NNlib.gather: dst[:,k] = src[:, idx[k]]   (call site GNNGraphs/src/gatherscatter.jl:4) */
void FN(orc_gather)(const T* src, const int64_t* idx, int64_t E, int64_t D, T* dst) {
    for (int64_t k = 0; k < E; ++k) memcpy(dst + k * D, src + (idx[k] - 1) * D, sizeof(T) * (size_t)D);
}

/* NNlib.scatter(op, src, idx; dstsize=(D,n))   (call site GNNGraphs/src/gatherscatter.jl:12-18)
 * dst is initialised to the op's neutral element, then dst[:,idx[k]] = op(dst[:,idx[k]], src[:,k]) in k
 * order; mean = sum ./ count with 0 for empty targets (SURVEY.md §8 a5: restated NNlib 0.9 semantics). */
void FN(orc_scatter)(int aggr, const T* src, const int64_t* idx, int64_t E, int64_t D, int64_t n, T* dst) {
    T init = 0;
    if (aggr == ORC_MAX) init = (T)-INFINITY;
    if (aggr == ORC_MIN) init = (T)INFINITY;
    for (int64_t i = 0; i < n * D; ++i) dst[i] = init;
    for (int64_t k = 0; k < E; ++k) {
        T* restrict d = dst + (idx[k] - 1) * D;
        const T* restrict s = src + k * D;
        if (aggr == ORC_SUM || aggr == ORC_MEAN)
            for (int64_t f = 0; f < D; ++f) d[f] = d[f] + s[f];
        else if (aggr == ORC_MAX)
            for (int64_t f = 0; f < D; ++f) d[f] = d[f] > s[f] ? d[f] : s[f];
        else
            for (int64_t f = 0; f < D; ++f) d[f] = d[f] < s[f] ? d[f] : s[f];
    }
    if (aggr == ORC_MEAN) {
        int64_t* cnt = (int64_t*)calloc((size_t)(n > 0 ? n : 1), sizeof(int64_t));
        for (int64_t k = 0; k < E; ++k) cnt[idx[k] - 1]++;
        for (int64_t i = 0; i < n; ++i) {
            T c = (T)(cnt[i] > 0 ? cnt[i] : 1);
            for (int64_t f = 0; f < D; ++f) dst[i * D + f] = dst[i * D + f] / c;
        }
        free(cnt);
    }
}

/* w_mul_xj / e_mul_xj with a vector e: m[:,k] = w[k] * xj[:,k]   (GNNlib/src/msgpass.jl:191-208) */
void FN(orc_w_mul)(const T* w, int64_t E, int64_t D, T* m) {
    for (int64_t k = 0; k < E; ++k)
        for (int64_t f = 0; f < D; ++f) m[k * D + f] = w[k] * m[k * D + f];
}

/* The UNFUSED path every GPU call and every mean/max CPU call takes (GNNlib/src/msgpass.jl:75-79):
 * materialise the (D,E) gather, apply the message, sequential scatter. */
int FN(orc_propagate_unfused)(int aggr, const int64_t* s, const int64_t* t, int64_t E, int64_t n, const T* x,
                              const T* w, int64_t D, T* out) {
    T* m = (T*)malloc(sizeof(T) * (size_t)(E * D > 0 ? E * D : 1));
    if (!m) return 1;
    FN(orc_gather)(x, s, E, D, m);
    if (w) FN(orc_w_mul)(w, E, D, m);
    FN(orc_scatter)(aggr, m, t, E, D, n, out);
    free(m);
    return 0;
}

/* to_sparse(coo): A = sparse(s, t, w, n, n)  (GNNGraphs/src/convert.jl:221-237; called on EVERY fused forward from
 * adjacency_matrix, GNNGraphs/src/query.jl:227).  Duplicates are summed, rows are sorted inside a column.
 * colptr[n+1], rowval/nzval capacity E (0-based).  Returns nnz, or -1 on allocation failure.
 * For unweighted graphs A holds the integer edge counts. */
int64_t FN(orc_csc_build)(const int64_t* s, const int64_t* t, int64_t E, int64_t n, const T* w, int64_t* colptr,
                          int64_t* rowval, T* nzval) {
    /* two stable counting sorts (by row, then by column) = entries ordered by (column, row), duplicates adjacent
     * and in COO order — O(E) like Julia's sparse() */
    int64_t* cnt = (int64_t*)calloc((size_t)n + 2, sizeof(int64_t));
    int64_t* pos = (int64_t*)malloc(sizeof(int64_t) * (size_t)(n + 1));
    int64_t* ord = (int64_t*)malloc(sizeof(int64_t) * (size_t)(E > 0 ? E : 1));
    if (!cnt || !pos || !ord) return -1;
    for (int64_t k = 0; k < E; ++k) cnt[s[k]]++;
    for (int64_t j = 0; j < n; ++j) cnt[j + 1] += cnt[j];
    for (int64_t j = 0; j < n; ++j) pos[j] = cnt[j];
    for (int64_t k = 0; k < E; ++k) ord[pos[s[k] - 1]++] = k;   /* edge ids sorted by row, stable */
    memset(cnt, 0, sizeof(int64_t) * ((size_t)n + 2));
    for (int64_t k = 0; k < E; ++k) cnt[t[k]]++;              /* cnt[j+1] = size of column j */
    for (int64_t j = 0; j < n; ++j) cnt[j + 1] += cnt[j];     /* cnt[j] = start of column j */
    for (int64_t j = 0; j < n; ++j) pos[j] = cnt[j];
    for (int64_t q = 0; q < E; ++q) {                         /* stable counting sort by column */
        const int64_t k = ord[q];
        int64_t p = pos[t[k] - 1]++;
        rowval[p] = s[k] - 1;
        nzval[p] = w ? w[k] : (T)1;
    }
    free(ord);
    int64_t nnz = 0;
    for (int64_t j = 0; j < n; ++j) {
        const int64_t a = cnt[j], b = cnt[j + 1];
        const int64_t newstart = nnz;
        for (int64_t p = a; p < b; ++p) {                     /* sum duplicates (compaction runs behind p) */
            if (nnz > newstart && rowval[nnz - 1] == rowval[p]) nzval[nnz - 1] = nzval[nnz - 1] + nzval[p];
            else { rowval[nnz] = rowval[p]; nzval[nnz] = nzval[p]; ++nnz; }
        }
        colptr[j] = newstart;
    }
    colptr[n] = nnz;
    free(cnt); free(pos);
    return nnz;
}

/* xj * A : the serial SparseArrays dense x CSC product the `+` specialisations dispatch to
 * (GNNlib/src/msgpass.jl:217,227,237):  out[:,j] = sum_{p in col j} x[:,rowval[p]] * nzval[p], row order. */
void FN(orc_dense_times_csc)(const T* x, int64_t n, int64_t D, const int64_t* colptr, const int64_t* rowval,
                             const T* nzval, T* out) {
    for (int64_t j = 0; j < n; ++j) {
        T* restrict o = out + j * D;
        for (int64_t f = 0; f < D; ++f) o[f] = 0;
        for (int64_t p = colptr[j]; p < colptr[j + 1]; ++p) {
            const T* restrict xr = x + rowval[p] * D;
            const T a = nzval[p];
            for (int64_t f = 0; f < D; ++f) o[f] = o[f] + xr[f] * a;   /* @simd loop of SparseArrays' mul! */
        }
    }
}

/* Δ * A' : the pullback of `xj * A` w.r.t. xj (ChainRules rule for dense x sparse), same stored entries:
 * out[:,i] += d[:,j] * A[i,j]  for every stored (i,j), column by column. */
void FN(orc_dense_times_csc_t)(const T* d, int64_t n, int64_t D, const int64_t* colptr, const int64_t* rowval,
                               const T* nzval, T* out) {
    for (int64_t i = 0; i < n * D; ++i) out[i] = 0;
    for (int64_t j = 0; j < n; ++j) {
        const T* restrict dr = d + j * D;
        for (int64_t p = colptr[j]; p < colptr[j + 1]; ++p) {
            T* restrict o = out + rowval[p] * D;
            const T a = nzval[p];
            for (int64_t f = 0; f < D; ++f) o[f] = o[f] + dr[f] * a;
        }
    }
}

/* The FUSED CPU path for `+` (GNNlib/src/msgpass.jl:215-238): CSC rebuilt from COO on every call, then xj * A. */
int FN(orc_propagate_fused)(const int64_t* s, const int64_t* t, int64_t E, int64_t n, const T* x, const T* w,
                            int64_t D, T* out) {
    int64_t* colptr = (int64_t*)malloc(sizeof(int64_t) * (size_t)(n + 1));
    int64_t* rowval = (int64_t*)malloc(sizeof(int64_t) * (size_t)(E > 0 ? E : 1));
    T* nzval = (T*)malloc(sizeof(T) * (size_t)(E > 0 ? E : 1));
    if (!colptr || !rowval || !nzval) return 1;
    if (FN(orc_csc_build)(s, t, E, n, w, colptr, rowval, nzval) < 0) return 1;
    FN(orc_dense_times_csc)(x, n, D, colptr, rowval, nzval, out);
    free(colptr); free(rowval); free(nzval);
    return 0;
}

/* degree(g, T; dir, edge_weight) -> _degree (GNNGraphs/src/query.jl:355-369): zeros .+ scatter(+, w|ones, s|t) */
void FN(orc_degree)(const int64_t* s, const int64_t* t, int64_t E, int64_t n, int dir, const T* w, T* out) {
    T* tmp = (T*)malloc(sizeof(T) * (size_t)(n > 0 ? n : 1));
    T* ones = NULL;
    if (!w) {
        ones = (T*)malloc(sizeof(T) * (size_t)(E > 0 ? E : 1));
        for (int64_t k = 0; k < E; ++k) ones[k] = 1;
        w = ones;
    }
    for (int64_t i = 0; i < n; ++i) out[i] = 0;
    if (dir == ORC_DIR_OUT || dir == ORC_DIR_BOTH) {
        FN(orc_scatter)(ORC_SUM, w, s, E, 1, n, tmp);
        for (int64_t i = 0; i < n; ++i) out[i] = out[i] + tmp[i];
    }
    if (dir == ORC_DIR_IN || dir == ORC_DIR_BOTH) {
        FN(orc_scatter)(ORC_SUM, w, t, E, 1, n, tmp);
        for (int64_t i = 0; i < n; ++i) out[i] = out[i] + tmp[i];
    }
    free(tmp); free(ones);
}

/* softmax_edge_neighbors (GNNlib/src/utils.jl:84-97), the reference's own six-step sequence */
void FN(orc_softmax_edge_neighbors)(const int64_t* t, int64_t E, int64_t n, const T* e, int64_t K, T* out) {
    T* stat = (T*)malloc(sizeof(T) * (size_t)(n * K > 0 ? n * K : 1));
    FN(orc_scatter)(ORC_MAX, e, t, E, K, n, stat);                     /* max_ = scatter(max, e, t) */
    for (int64_t k = 0; k < E; ++k)                                    /* num = exp.(e .- gather(max_, t)) */
        for (int64_t h = 0; h < K; ++h) out[k * K + h] = (T)EXPFN(e[k * K + h] - stat[(t[k] - 1) * K + h]);
    FN(orc_scatter)(ORC_SUM, out, t, E, K, n, stat);                   /* den = scatter(+, num, t) */
    for (int64_t k = 0; k < E; ++k)                                    /* num ./ gather(den, t) */
        for (int64_t h = 0; h < K; ++h) out[k * K + h] = out[k * K + h] / stat[(t[k] - 1) * K + h];
    free(stat);
}

/* The message-passing core of gcn_conv (GNNlib/src/layers/conv.jl:52-67) with the default norm_fn
 * d -> 1 ./ sqrt.(d) (GraphNeuralNetworks/src/layers/conv.jl:99).  (s,t,w) must already contain the self
 * loops when the layer adds them (conv.jl:26-34).  fused != 0 takes the `+` SpMM path (CPU arrays),
 * fused == 0 the gather/scatter path.  c_out (n) optionally receives c. */
int FN(orc_gcn_propagate)(const int64_t* s, const int64_t* t, int64_t E, int64_t n, const T* x, const T* w,
                          int64_t D, int fused, T* out, T* c_out) {
    T* c = (T*)malloc(sizeof(T) * (size_t)(n > 0 ? n : 1));
    T* xs = (T*)malloc(sizeof(T) * (size_t)(n * D > 0 ? n * D : 1));
    if (!c || !xs) return 1;
    FN(orc_degree)(s, t, E, n, ORC_DIR_IN, w, c);
    for (int64_t i = 0; i < n; ++i) c[i] = (T)1 / (T)SQRTFN(c[i]);
    for (int64_t i = 0; i < n; ++i)
        for (int64_t f = 0; f < D; ++f) xs[i * D + f] = x[i * D + f] * c[i];     /* xj .* cout' */
    int rc = fused ? FN(orc_propagate_fused)(s, t, E, n, xs, w, D, out)
                   : FN(orc_propagate_unfused)(ORC_SUM, s, t, E, n, xs, w, D, out);
    for (int64_t i = 0; i < n; ++i)
        for (int64_t f = 0; f < D; ++f) out[i * D + f] = out[i * D + f] * c[i];  /* x .* cin' */
    if (c_out) memcpy(c_out, c, sizeof(T) * (size_t)n);
    free(c); free(xs);
    return rc;
}

/* The edge part of gat_conv + gat_message (GNNlib/src/layers/conv.jl:136-141,152-167), restated step by
 * step: gather Wxi[:,:,t], Wxj[:,:,s]; logα = leakyrelu(sum(a .* vcat(Wxi,Wxj), dims=1)); α = softmax over
 * in-neighbourhoods; out = scatter(+, α .* Wxj, t).  Wx is (C,H,n), a is (2C,H), out (C,H,n), alpha (H,E). */
int FN(orc_gat_aggregate)(const int64_t* s, const int64_t* t, int64_t E, int64_t n, const T* Wx, const T* a,
                          int64_t C, int64_t H, T slope, T* out, T* alpha) {
    T* logit = (T*)malloc(sizeof(T) * (size_t)(E * H > 0 ? E * H : 1));
    T* al = alpha ? alpha : (T*)malloc(sizeof(T) * (size_t)(E * H > 0 ? E * H : 1));
    T* beta = (T*)malloc(sizeof(T) * (size_t)(E * H * C > 0 ? E * H * C : 1));
    if (!logit || !al || !beta) return 1;
    for (int64_t k = 0; k < E; ++k) {
        const T* wi = Wx + (t[k] - 1) * C * H;
        const T* wj = Wx + (s[k] - 1) * C * H;
        for (int64_t h = 0; h < H; ++h) {
            T acc = 0;                                  /* sum over the 2C rows of a .* [Wxi; Wxj], row order */
            for (int64_t c = 0; c < C; ++c) acc = acc + a[h * 2 * C + c] * wi[h * C + c];
            for (int64_t c = 0; c < C; ++c) acc = acc + a[h * 2 * C + C + c] * wj[h * C + c];
            logit[k * H + h] = acc > 0 ? acc : slope * acc;   /* leakyrelu */
        }
    }
    FN(orc_softmax_edge_neighbors)(t, E, n, logit, H, al);
    for (int64_t k = 0; k < E; ++k) {
        const T* wj = Wx + (s[k] - 1) * C * H;
        for (int64_t h = 0; h < H; ++h)
            for (int64_t c = 0; c < C; ++c) beta[(k * H + h) * C + c] = al[k * H + h] * wj[h * C + c];
    }
    FN(orc_scatter)(ORC_SUM, beta, t, E, C * H, n, out);
    free(logit); free(beta);
    if (!alpha) free(al);
    return 0;
}

/* Pullback of the edge part above for an upstream dout (C,H,n), with the logit halves el[h,i] = a[1:C,h]·Wx[:,h,i] and
 * er[h,j] = a[C+1:2C,h]·Wx[:,h,j] as inputs (z_k = el[t_k] + er[s_k]; their chain into a and Wx is linear):
 *     α = softmax over in-neighbourhoods of leakyrelu(z);   dα_k = <dout[:,h,t_k], Wx[:,h,s_k]>
 *     T_i = Σ_{k: t_k=i} α_k dα_k;   dz_k = α_k (dα_k − T_{t_k}) · leakyrelu'(z_k)
 *     del = scatter(+, dz, t);   der = scatter(+, dz, s);   dWx = scatter(+, α .* dout[:,:,t], s)   (edge part only)
 * Every sum runs in COO edge order.  Only (H,E) temporaries: no (C,H,E) tensor.  alpha (H,E) is optional. */
int FN(orc_gat_aggregate_bwd)(const int64_t* s, const int64_t* t, int64_t E, int64_t n, const T* Wx, const T* el,
                              const T* er, int64_t C, int64_t H, T slope, const T* dout, T* dWx, T* del, T* der,
                              T* alpha) {
    const size_t EH = (size_t)(E * H > 0 ? E * H : 1);
    T* u = (T*)malloc(sizeof(T) * EH);
    T* al = alpha ? alpha : (T*)malloc(sizeof(T) * EH);
    T* dz = (T*)malloc(sizeof(T) * EH);                 /* α·dα, then dz */
    T* tn = (T*)malloc(sizeof(T) * (size_t)(n * H > 0 ? n * H : 1));
    if (!u || !al || !dz || !tn) return 1;
    for (int64_t k = 0; k < E; ++k)
        for (int64_t h = 0; h < H; ++h) {
            const T z = el[(t[k] - 1) * H + h] + er[(s[k] - 1) * H + h];
            u[k * H + h] = z > 0 ? z : slope * z;
        }
    FN(orc_softmax_edge_neighbors)(t, E, n, u, H, al);
    for (int64_t k = 0; k < E; ++k) {
        const T* di = dout + (t[k] - 1) * C * H;
        const T* wj = Wx + (s[k] - 1) * C * H;
        for (int64_t h = 0; h < H; ++h) {
            T acc = 0;                                  /* dα = <dout[:,h,t], Wx[:,h,s]>, channel order */
            for (int64_t c = 0; c < C; ++c) acc = acc + di[h * C + c] * wj[h * C + c];
            dz[k * H + h] = acc;
            u[k * H + h] = al[k * H + h] * acc;
        }
    }
    FN(orc_scatter)(ORC_SUM, u, t, E, H, n, tn);        /* T = scatter(+, α .* dα, t) */
    for (int64_t k = 0; k < E; ++k)
        for (int64_t h = 0; h < H; ++h) {
            const T z = el[(t[k] - 1) * H + h] + er[(s[k] - 1) * H + h];
            dz[k * H + h] = al[k * H + h] * (dz[k * H + h] - tn[(t[k] - 1) * H + h]) * (z > 0 ? (T)1 : slope);
        }
    FN(orc_scatter)(ORC_SUM, dz, t, E, H, n, del);
    FN(orc_scatter)(ORC_SUM, dz, s, E, H, n, der);
    for (int64_t i = 0; i < n * C * H; ++i) dWx[i] = 0;
    for (int64_t k = 0; k < E; ++k) {                   /* scatter(+, α .* dout[:,:,t], s) without the (C,H,E) tensor */
        T* dj = dWx + (s[k] - 1) * C * H;
        const T* di = dout + (t[k] - 1) * C * H;
        for (int64_t h = 0; h < H; ++h) {
            const T w = al[k * H + h];
            for (int64_t c = 0; c < C; ++c) dj[h * C + c] = dj[h * C + c] + w * di[h * C + c];
        }
    }
    free(u); free(dz); free(tn);
    if (!alpha) free(al);
    return 0;
}
