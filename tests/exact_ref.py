"""Float64 NumPy / SciPy reference of the exact posterior expectations (`pb.expected_sumstats`), and a brute-force
enumeration that checks it on small trees.

Statistic k in the fixed-Q sampler row layout: k < n dwell time in state k, then the changes (i, j), i != j, row-major
with the diagonal skipped.  M[k] = int_0^t P(s) C_k P(t - s) ds with C_k = E_kk (dwell) or Q_ij E_ij (change), the
upper-right block of expm(t [[Q, C], [0, Q]]) (Van Loan 1978); then E[stat_k on branch p -> c | X_p = a, X_c = b] =
M[k][a, b] / P(t)[a, b].
"""
import numpy as np
from scipy.linalg import expm


def stat_pairs(n):
    """(i, j) of every statistic: (i, i) for the dwell in i, then the changes in sampler column order."""
    return [(i, i) for i in range(n)] + [(i, j) for i in range(n) for j in range(n) if i != j]


def van_loan(Q, C, t):
    n = Q.shape[0]
    A = np.zeros((2 * n, 2 * n))
    A[:n, :n] = Q
    A[n:, n:] = Q
    A[:n, n:] = C
    return expm(A * t)[:n, n:]


def branch_integrals(Q, t):
    """[n^2, n, n]: M[k] of one branch of length t."""
    n = Q.shape[0]
    out = []
    for k, (i, j) in enumerate(stat_pairs(n)):
        C = np.zeros((n, n))
        C[i, j] = 1.0 if k < n else Q[i, j]
        out.append(van_loan(Q, C, t))
    return np.array(out)


def tip_vector(state, n, parity):
    """Tip partial of a 1-based observed state: one-hot, or the hidden-rate (1,0,1,0..) / (0,1,0,1..) pattern."""
    if parity:
        return np.array([1.0 if j % 2 == (state - 1) % 2 else 0.0 for j in range(n)])
    v = np.zeros(n)
    v[state - 1] = 1.0
    return v


def _structure(edge):
    edge = np.asarray(edge) - 1
    E = len(edge)
    T = (E + 2) // 2
    kids = {}
    pedge = {}
    for e, (p, c) in enumerate(edge):
        kids.setdefault(int(p), []).append(e)
        pedge[int(c)] = e
    root = [v for v in range(T, 2 * T - 1) if v not in pedge][0]
    order = []  # pre-order
    stack = [root]
    while stack:
        v = stack.pop()
        order.append(v)
        stack.extend(int(edge[e, 1]) for e in kids.get(v, []))
    return edge, T, kids, pedge, root, order


def branch_model(blen, Q):
    """(P(t_e), M_e) of every branch, shared by the sites of a tree."""
    Q = np.asarray(Q, dtype=np.float64)
    return [expm(Q * t) for t in blen], [branch_integrals(Q, t) for t in blen]


def exact(edge, blen, Q, pid, states, parity=False, model=None):
    """Inside / outside recursion for one site.  states: 1-based tip states [T]; model: branch_model(blen, Q) if already
    computed.  Returns (stats [n^2], branch stats [E, n^2], node marginals [2T-1, n], log p(y | Q))."""
    Q = np.asarray(Q, dtype=np.float64)
    n = Q.shape[0]
    edge, T, kids, pedge, root, order = _structure(edge)
    E = len(edge)
    P, M = branch_model(blen, Q) if model is None else model
    alpha = {v: tip_vector(states[v], n, parity) for v in range(T)}
    logscale = 0.0
    for v in reversed(order):
        if v < T:
            continue
        a = np.ones(n)
        for e in kids[v]:
            a = a * (P[e] @ alpha[int(edge[e, 1])])
        s = a.sum()
        logscale += np.log(s)
        alpha[v] = a / s
    loglik = np.log(pid @ alpha[root]) + logscale
    beta = {root: np.asarray(pid, dtype=np.float64)}
    bstats = np.zeros((E, n * n))
    marg = np.zeros((2 * T - 1, n))
    marg[root] = pid * alpha[root] / (pid @ alpha[root])
    for v in order:
        if v < T:
            continue
        es = kids[v]
        ys = [P[e] @ alpha[int(edge[e, 1])] for e in es]
        for i, e in enumerate(es):
            c = int(edge[e, 1])
            u = beta[v].copy()
            for j, y in enumerate(ys):
                if j != i:
                    u = u * y
            Z = u @ ys[i]
            bstats[e] = [u @ M[e][k] @ alpha[c] / Z for k in range(n * n)]
            b = P[e].T @ u
            beta[c] = b / b.sum()
            m = alpha[c] * beta[c]
            marg[c] = m / m.sum()
    return bstats.sum(0), bstats, marg, loglik


def brute_force(edge, blen, Q, pid, states, parity=False):
    """The same quantities by enumerating every joint assignment of node states (tips restricted to their partial's
    support): weight pid[x_root] prod_e P_e[x_p, x_c], conditional statistic of branch e M_e[k][x_p, x_c] / P_e[x_p, x_c]."""
    import itertools
    Q = np.asarray(Q, dtype=np.float64)
    n = Q.shape[0]
    edge, T, kids, pedge, root, order = _structure(edge)
    E = len(edge)
    P, M = branch_model(blen, Q)
    choices = [list(np.flatnonzero(tip_vector(states[v], n, parity))) for v in range(T)] + [list(range(n))] * (T - 1)
    W = 0.0
    bst = np.zeros((E, n * n))
    marg = np.zeros((2 * T - 1, n))
    for x in itertools.product(*choices):
        w = pid[x[root]]
        for e in range(E):
            w *= P[e][x[edge[e, 0]], x[edge[e, 1]]]
        W += w
        for e in range(E):
            a, b = x[edge[e, 0]], x[edge[e, 1]]
            bst[e] += w * M[e][:, a, b] / P[e][a, b]
        for v in range(2 * T - 1):
            marg[v, x[v]] += w
    bst /= W
    return bst.sum(0), bst, marg / W, np.log(W)


def random_q(n, rng, scale=0.5):
    Q = rng.uniform(0.05, 1.0, (n, n)) * scale
    np.fill_diagonal(Q, 0.0)
    np.fill_diagonal(Q, -Q.sum(1))
    return Q
