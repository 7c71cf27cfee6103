"""Two-segment AIR descriptions for the sharded aux prover (wf_prove_air_aux_sharded), in the flat u64 format of tests/airs.py
and built with its AirBuilder. Each builder also builds any range of its aux columns (`builder.columns`), as a rank of a
sharded proof does."""
import numpy as np

from airs import AirBuilder, P


def perm_rap_lanes(n, lanes=3, seed=5):
    """`lanes` independent copies of perm_rap side by side (lane l: main columns 3l..3l+2, aux columns 3l..3l+2, its own
    permutation, seed + l), sharing the two random elements and the periodic column: a two-segment AIR wide enough to split
    its aux segment unevenly over several ranks. Three lanes is as many as the aux program's 96 registers allow
    (12 lanes + 3 inputs and 13 temporaries per lane). Returns (description, main trace, builder): builder(rand) -> all aux
    columns [3 lanes, n, d]; builder.columns(rand, first_col, num_cols) -> aux columns [first_col, first_col + num_cols) only,
    built from the lanes covering them."""
    from oracle import oracle as O
    k = [1, 2, 3, 4]
    w = 3 * lanes
    tr = np.zeros((w, n), dtype=np.uint64)
    A = AirBuilder(w)
    A.periodic = [k]
    a = b = 1
    for i in range(n):   # the FibSmall pair, the same in every lane
        tr[0, i], tr[1, i] = a, b
        a = (a + b) % P
        b = (b + a) % P
    for l in range(lanes):   # lane l's b: perm_rap's permutation for seed + l
        tr[3 * l: 3 * l + 2] = tr[0:2]
        perm = np.random.default_rng(seed + l).permutation(n - 1)
        tr[3 * l + 2, : n - 1] = tr[0, perm]
        tr[3 * l + 2, n - 1] = 12345
    A.pub = [int(tr[1, n - 1])]
    for l in range(lanes):
        x0, x1 = 3 * l, 3 * l + 1
        A.constraint(A.sub(A.nxt(x0), A.add(A.cur(x0), A.cur(x1))), 1)
        A.constraint(A.sub(A.nxt(x1), A.add(A.cur(x1), A.nxt(x0))), 1)
        A.assert_single(x0, 0, 1)
        A.assert_single(x1, 0, 1)
        A.assert_single(x1, n - 1, int(tr[x1, n - 1]))
    X = A.aux(3 * lanes, 2)
    gamma, alpha = X.rnd(0), X.rnd(1)
    for l in range(lanes):
        x0, x1, bb = 3 * l, 3 * l + 1, 3 * l + 2   # main: the pair and the permuted column
        p, q, c = 3 * l, 3 * l + 1, 3 * l + 2      # aux: running product, running sum, counter
        lhs = X.mul(X.anxt(p), X.add(X.cur(bb), gamma))
        rhs = X.mul(X.acur(p), X.add(X.cur(x0), gamma))
        X.constraint(X.sub(lhs, rhs), 2)
        term = X.mul(X.mul(alpha, X.per(0)), X.mul(X.cur(x1), X.acur(p)))
        X.constraint(X.sub(X.anxt(q), X.add(X.acur(q), term)), 2, [4])
        X.assert_single(p, 0, (1, 0, 0))
        X.assert_single(p, n - 1, (1, 0, 0))
        X.assert_single(q, 0, (0, 0, 0))
        one = X.const(1)
        X.constraint(X.sub(X.anxt(c), X.add(X.acur(c), one)), 1)
        X.assert_sequence(c, 1, n // 4, [(5 + 1 + j * (n // 4), 0, 0) for j in range(4)])

    def columns(rand, first_col, num_cols):
        l0, l1 = first_col // 3, (first_col + num_cols - 1) // 3
        aux = np.concatenate([O.perm_rap_aux(tr[3 * l: 3 * l + 3], rand) for l in range(l0, l1 + 1)])
        return aux[first_col - 3 * l0: first_col - 3 * l0 + num_cols]

    def builder(rand):
        return columns(rand, 0, w)

    builder.columns = columns
    return A.build(), tr, builder



def rap_sums(n, k=8, aw=8):
    """A two-segment AIR whose segments split evenly: main = FibSmall x k (2k columns, as fib_small_x), aux column j a running
    sum s_j' = s_j + gamma * x_j, s_j[0] = 0 (one random element). With k = 8, aw = 8 and a quadratic extension both
    segments have 16 base columns: whole 8-column segments, the same number on each of 2 ranks. Returns (description, main
    trace, builder) with builder(rand) -> [aw, n, d] and builder.columns(rand, first_col, num_cols) as perm_rap_lanes."""
    tr = np.zeros((2 * k, n), dtype=np.uint64)
    res = []
    for j in range(k):
        a = b = j + 1
        for i in range(n):
            tr[2 * j, i], tr[2 * j + 1, i] = a, b
            a = (a + b) % P
            b = (b + a) % P
        res.append(int(tr[2 * j + 1, n - 1]))
    A = AirBuilder(2 * k)
    A.pub = res
    for j in range(k):
        A.constraint(A.sub(A.nxt(2 * j), A.add(A.cur(2 * j), A.cur(2 * j + 1))), 1)
        A.constraint(A.sub(A.nxt(2 * j + 1), A.add(A.cur(2 * j + 1), A.nxt(2 * j))), 1)
        A.assert_single(2 * j, 0, j + 1)
        A.assert_single(2 * j + 1, 0, j + 1)
        A.assert_single(2 * j + 1, n - 1, res[j])
    X = A.aux(aw, 1)
    for j in range(aw):
        X.constraint(X.sub(X.anxt(j), X.add(X.acur(j), X.mul(X.rnd(0), X.cur(j % (2 * k))))), 1)
        X.assert_single(j, 0, (0, 0, 0))
    # s_j[i] = gamma * (x_j[0] + ... + x_j[i-1]): every component of gamma times one base-field prefix sum
    prefix = [np.concatenate([[0], np.cumsum(tr[j % (2 * k)].astype(object))[:-1]]) % P for j in range(aw)]

    def columns(rand, first_col, num_cols):
        d = rand.shape[1]
        out = np.zeros((num_cols, n, d), dtype=np.uint64)
        for t in range(num_cols):
            for q in range(d):
                out[t, :, q] = (prefix[first_col + t] * int(rand[0, q]) % P).astype(np.uint64)
        return out

    def builder(rand):
        return columns(rand, 0, aw)

    builder.columns = columns
    return A.build(), tr, builder
