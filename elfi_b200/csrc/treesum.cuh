// treesum.cuh -- NumPy's pairwise summation for runs longer than one leaf, term by term.
//
// Same result as PairwiseStream (pairwise.cuh) but with the accumulator interface of LeafSum
// (leafsum.cuh): terms arrive one at a time with their index modulo 8 known at compile time, so
// a column group whose 16 terms fall inside the whole-groups range of the current leaf takes the
// branch-free path, and the recursion stack is only touched once per <= 128-term leaf.  The
// row-stream summary kernels use it for rows of 129..7688 terms (see summaries.cu).
//
// NumPy (DOUBLE_pairwise_sum): n <= 128 is a leaf (8 strided accumulators + sequential tail);
// longer runs split at n/2 rounded down to a multiple of 8, left part first.  Every left part is
// a multiple of 8 long, so leaves start at multiples of 8 and only the last leaf has a tail.
// Compiles for the host as well (tests/harness/leaf_harness.cpp).
#pragma once

#include <stdint.h>

#include "leafsum.cuh"

namespace elfi {

template <int MAXD>
struct TreeSum {
    double r[8];
    double res;
    double left_val[MAXD];     // [0] = innermost open split
    int pending_right[MAXD];   // length of the right part still to come, per open split
    uint32_t has_left;         // bit d: split d already holds its left sum
    int depth;
    int first8_end;            // leaf start + 8: terms below it initialise r[]
    int leaf_end;              // one past the last term of the current leaf
    int tail_start;            // first sequential term of the current leaf (== leaf_end: none)
    bool in_tail;

    ELFI_HD void open_split(int right) {
        ELFI_UNROLL
        for (int d = MAXD - 1; d > 0; --d) {
            pending_right[d] = pending_right[d - 1];
            left_val[d] = left_val[d - 1];
        }
        pending_right[0] = right;
        left_val[0] = 0.0;
        has_left <<= 1;
        ++depth;
    }
    ELFI_HD void close_split() {
        ELFI_UNROLL
        for (int d = 0; d < MAXD - 1; ++d) {
            pending_right[d] = pending_right[d + 1];
            left_val[d] = left_val[d + 1];
        }
        has_left >>= 1;
        --depth;
    }
    // descend to the first leaf of the run [start, start + n)
    ELFI_HD void descend(int start, int n) {
        while (n > LEAF_MAX_TERMS) {
            int left = n / 2;
            left -= left % 8;
            open_split(n - left);
            n = left;
        }
        first8_end = start + 8;
        leaf_end = start + n;
        in_tail = n < 8;                       // a short leaf is summed sequentially from 0.0
        tail_start = in_tail ? start : start + (n - n % 8);
        res = 0.0;
    }
    ELFI_HD void begin(int m) {
        depth = 0;
        has_left = 0;
        ELFI_UNROLL
        for (int k = 0; k < 8; ++k) r[k] = 0.0;
        ELFI_UNROLL
        for (int d = 0; d < MAXD; ++d) {
            left_val[d] = 0.0;
            pending_right[d] = 0;
        }
        descend(0, m);
    }
    ELFI_HD double fold() const {
        return leaf_add(leaf_add(leaf_add(r[0], r[1]), leaf_add(r[2], r[3])),
                        leaf_add(leaf_add(r[4], r[5]), leaf_add(r[6], r[7])));
    }
    // the current leaf is complete: hand its value up the open splits and open the next leaf
    ELFI_HD void next_leaf() {
        double v = in_tail ? res : fold();
        const int next = leaf_end;
        while (depth > 0) {
            if (!(has_left & 1u)) {
                left_val[0] = v;
                has_left |= 1u;
                descend(next, pending_right[0]);
                return;
            }
            v = leaf_add(left_val[0], v);
            close_split();
        }
    }
    // term j (K = j % 8); terms must arrive in index order
    template <int K>
    ELFI_HD void push(int j, double v) {
        if (K == 0) {   // leaves and tails start at multiples of 8
            if (j == leaf_end) next_leaf();
            if (!in_tail && j == tail_start) {
                res = fold();
                in_tail = true;
            }
        }
        if (in_tail) {
            res = leaf_add(res, v);
        } else if (j < first8_end) {
            r[K] = v;
        } else {
            r[K] = leaf_add(r[K], v);
        }
    }
    // a term known to lie in the whole-groups range of the current leaf
    template <int K>
    ELFI_HD void push_mid(double v) {
        r[K] = leaf_add(r[K], v);
    }
    ELFI_HD bool all_mid(int j_first, int j_last) const {
        return !in_tail && j_first >= first8_end && j_last < tail_start;
    }
    // 0.0 + total: np.add.reduce starts from the identity (see LeafSum::finish)
    ELFI_HD double finish(int) const {
        double v = in_tail ? res : fold();
        ELFI_UNROLL
        for (int d = 0; d < MAXD; ++d)
            if (d < depth) v = leaf_add(left_val[d], v);
        return leaf_add(0.0, v);
    }
    // longest run that never needs more than MAXD open splits (a right part has up to n/2 + 7
    // terms): 7688 for MAXD = 6
    static constexpr int64_t max_terms() { return (int64_t(120) << MAXD) + 8; }
};

}  // namespace elfi
