// Host-side pieces shared by the batched fold-in drivers (mfrec_fold_in_kmf in sgd.cu,
// mfrec_fold_in_funk in funk.cu): which ratings belong to the listed rows, and the compact copies of
// the rows those ratings name.  Host code only.
#pragma once

#include <stdint.h>

#include <algorithm>
#include <vector>

#include "mfrec_b200.h"

int mfrec_set_error(mfrec_ctx *ctx, int code, const char *fmt, ...);

// The rows a fold-in's ratings name, copied out of the caller's full arrays into compact ones and
// back (KMFRecommender.retrain_user / retrain_item / add_user, kmf.py:120-172, name a handful of
// rows: only those move, so the untouched rest of u / v / the biases stays bit-identical like in the
// reference).  users / items: the distinct ids the ratings name, sorted; idx: ratings_index
// renumbered into them.  Compact factors are [k][m] like the caller's, or [m][k] with row_major.
struct FoldRows {
    int k = 0;
    bool row_major = false;
    std::vector<int32_t> users, items, idx;
    std::vector<double> u, v, ib, ub;

    static std::vector<int32_t> distinct(const int32_t *ratings_index, int64_t nnz, int col)
    {
        std::vector<int32_t> ids(nnz);
        for (int64_t n = 0; n < nnz; ++n) ids[n] = ratings_index[2 * n + col];
        std::sort(ids.begin(), ids.end());
        ids.erase(std::unique(ids.begin(), ids.end()), ids.end());
        return ids;
    }
    size_t at(size_t m, size_t a, int f) const { return row_major ? a * k + f : (size_t)f * m + a; }

    void gather(int k_, bool row_major_, const double *u_, const double *v_, const double *ib_,
                const double *ub_, int32_t ni, int32_t nu, const int32_t *ratings_index, int64_t nnz)
    {
        k = k_;
        row_major = row_major_;
        users = distinct(ratings_index, nnz, 0);
        items = distinct(ratings_index, nnz, 1);
        const size_t mu = users.size(), mi = items.size();
        u.resize((size_t)k * mi);
        v.resize((size_t)k * mu);
        ib.resize(mi);
        ub.resize(mu);
        for (int f = 0; f < k; ++f) {
            for (size_t a = 0; a < mi; ++a) u[at(mi, a, f)] = u_[(size_t)f * ni + items[a]];
            for (size_t a = 0; a < mu; ++a) v[at(mu, a, f)] = v_[(size_t)f * nu + users[a]];
        }
        for (size_t a = 0; a < mi; ++a) ib[a] = ib_[items[a]];
        for (size_t a = 0; a < mu; ++a) ub[a] = ub_[users[a]];
        idx.resize((size_t)2 * nnz);
        for (int64_t n = 0; n < nnz; ++n) {
            idx[2 * n] = (int32_t)(std::lower_bound(users.begin(), users.end(), ratings_index[2 * n]) - users.begin());
            idx[2 * n + 1] = (int32_t)(std::lower_bound(items.begin(), items.end(), ratings_index[2 * n + 1]) - items.begin());
        }
    }
    // writes the compact rows back into every non-null array
    void scatter(double *u_, double *v_, double *ib_, double *ub_, int32_t ni, int32_t nu) const
    {
        const size_t mu = users.size(), mi = items.size();
        for (int f = 0; f < k; ++f) {
            if (u_) for (size_t a = 0; a < mi; ++a) u_[(size_t)f * ni + items[a]] = u[at(mi, a, f)];
            if (v_) for (size_t a = 0; a < mu; ++a) v_[(size_t)f * nu + users[a]] = v[at(mu, a, f)];
        }
        if (ib_) for (size_t a = 0; a < mi; ++a) ib_[items[a]] = ib[a];
        if (ub_) for (size_t a = 0; a < mu; ++a) ub_[users[a]] = ub[a];
    }
};

// The ratings of the rows a batched fold-in lists (side MFREC_FOLD_USERS: rows are users, column 0
// of ratings_index names them; MFREC_FOLD_ITEMS: items, column 1).  count() validates and counts,
// gather() copies: listed row p's ratings end up at [rptr[p], rptr[p + 1]) of idx / r, in input
// order.  Ratings naming no listed row are ignored, whatever their indices.
struct FoldSelection {
    std::vector<int64_t> rptr;   // [n_rows + 1]
    std::vector<int32_t> idx;    // [nsel][2] (user, item)
    std::vector<double> r;       // [nsel]

    int64_t nsel() const { return rptr.back(); }

    // rows outside [0, n) and ratings of a listed row whose other index is out of range:
    // MFREC_ERR_INDEX; a row listed twice: MFREC_ERR_BAD_ARG (fn names the caller in the message)
    int count(mfrec_ctx *ctx, const char *fn, int side, const int32_t *ratings_index, int64_t nnz,
              int32_t ni, int32_t nu, const int32_t *rows, int32_t n_rows)
    {
        const bool by_user = side == MFREC_FOLD_USERS;
        tc_ = by_user ? 0 : 1;   // column of ratings_index naming the trained row; 1 - tc_ the frozen one
        const int32_t n_side = by_user ? nu : ni, n_other = by_user ? ni : nu;
        // list position of every trained-side row (-1: not listed)
        pos_.assign(n_side, -1);
        for (int32_t p = 0; p < n_rows; ++p) {
            const int32_t t = rows[p];
            if (t < 0 || t >= n_side)
                return mfrec_set_error(ctx, MFREC_ERR_INDEX, "%s: rows[%d] = %d outside [0, %d)", fn, p, t, n_side);
            if (pos_[t] >= 0)
                return mfrec_set_error(ctx, MFREC_ERR_BAD_ARG, "%s: row %d is listed twice (%d, %d)", fn, t, pos_[t], p);
            pos_[t] = p;
        }
        // every listed row's ratings in input order: a stable counting sort by list position
        rptr.assign((size_t)n_rows + 1, 0);
        for (int64_t n = 0; n < nnz; ++n) {
            const int32_t p = listed(ratings_index, n);
            if (p < 0) continue;
            const int32_t o = ratings_index[2 * n + 1 - tc_];
            if (o < 0 || o >= n_other)
                return mfrec_set_error(ctx, MFREC_ERR_INDEX, "%s: rating %lld has (user,item)=(%d,%d)", fn,
                                       (long long)n, ratings_index[2 * n], ratings_index[2 * n + 1]);
            ++rptr[p + 1];
        }
        for (int32_t p = 0; p < n_rows; ++p) rptr[p + 1] += rptr[p];
        return MFREC_OK;
    }

    void gather(const int32_t *ratings_index, const double *ratings, int64_t nnz)
    {
        idx.resize((size_t)2 * nsel());
        r.resize(nsel());
        std::vector<int64_t> cur(rptr.begin(), rptr.end() - 1);
        for (int64_t n = 0; n < nnz; ++n) {
            const int32_t p = listed(ratings_index, n);
            if (p < 0) continue;
            const int64_t s = cur[p]++;
            idx[2 * s] = ratings_index[2 * n];
            idx[2 * s + 1] = ratings_index[2 * n + 1];
            r[s] = ratings[n];
        }
    }

  private:
    int tc_ = 0;
    std::vector<int32_t> pos_;

    int32_t listed(const int32_t *ratings_index, int64_t n) const
    {
        const int32_t t = ratings_index[2 * n + tc_];
        return t >= 0 && t < (int32_t)pos_.size() ? pos_[t] : -1;
    }
};
