"""Synthetic problem generators of the BASELINE.json configurations (SURVEY.md §8d), shared by bench.py and
the tests. All PCG64-seeded so that the oracle and the device see the same bytes."""
import numpy as np


def random_sym(rng, n):
    R = rng.uniform(-1.0, 1.0, size=(n, n))
    return 0.5 * (R + R.T)


def random_dense_lmi(n, m, seed):
    """conex/test/test_sdp.cc:170-185 + test_util.cc:19,67-73: A_i = sym(U[-1,1]), C = I."""
    rng = np.random.Generator(np.random.PCG64(seed))
    mats = [random_sym(rng, n) for _ in range(m)]
    return mats, np.eye(n)


def maxcut_lmi(n, seed, p=0.5):
    """MaxCut dual (SURVEY.md §8d C2): A_i = -e_i e_i^T, C = -L/4, b = -1."""
    rng = np.random.Generator(np.random.PCG64(seed))
    upper = np.triu(rng.random((n, n)) < p, 1).astype(np.float64)
    adj = upper + upper.T
    lap = np.diag(adj.sum(axis=1)) - adj
    mats = []
    for i in range(n):
        E = np.zeros((n, n))
        E[i, i] = -1.0
        mats.append(E)
    return mats, -lap / 4.0, -np.ones(n)


def lovasz_theta_lmi(n, num_edges, seed):
    """Lovász-theta dual (SURVEY.md §8d C4): vars (t, y_e); A_0 = -I, A_e = E_ij + E_ji, C = -J,
    maximise -t."""
    rng = np.random.Generator(np.random.PCG64(seed))
    pairs = [(i, j) for i in range(n) for j in range(i + 1, n)]
    idx = rng.choice(len(pairs), size=num_edges, replace=False)
    mats = [-np.eye(n)]
    for k in sorted(idx.tolist()):
        i, j = pairs[k]
        E = np.zeros((n, n))
        E[i, j] = 1.0
        E[j, i] = 1.0
        mats.append(E)
    b = np.zeros(num_edges + 1)
    b[0] = -1.0
    return mats, -np.ones((n, n)), b


def small_multicone_problem(seed, m=40, psd_blocks=3, psd_order=20, soc_cones=2, soc_order=10, lp_rows=40):
    """One program of BASELINE config 3 (SURVEY.md §8d C3): `psd_blocks` dense LMI blocks
    (A_i = sym(U[-1,1]), C = I), `soc_cones` Lorentz cones of order `soc_order` (A uniform,
    c = (1, 0, ...), interfaces/python/test/run_tests.py:23-34) and one LP block (A uniform, c = 1),
    all on the same m variables; b = sum over cones of the feasible objective AW/2 at W = I
    (cone_program.cc:535-545), so both primal and dual are strictly feasible."""
    rng = np.random.Generator(np.random.PCG64(seed))
    cones = []
    b = np.zeros(m)
    for _ in range(psd_blocks):
        mats = [random_sym(rng, psd_order) for _ in range(m)]
        cones.append(("psd", mats, np.eye(psd_order)))
        b += 0.5 * np.array([np.trace(M) for M in mats])
    for _ in range(soc_cones):
        A = rng.uniform(-1.0, 1.0, size=(soc_order + 1, m))
        c = np.zeros(soc_order + 1)
        c[0] = 1.0
        cones.append(("soc", A, c))
        b += 0.5 * 2.0 * A[0, :]
    if lp_rows:
        A = rng.uniform(-1.0, 1.0, size=(lp_rows, m))
        cones.append(("lp", A, np.ones(lp_rows)))
        b += 0.5 * A.sum(axis=0)
    return cones, b


def small_multicone_equality_problem(seed, equalities=((8, None, None),), y0_scale=0.02, **shape):
    """small_multicone_problem with equality blocks A_eq y[variables] = b_eq added. `equalities`: one
    (rows, variables, position) per block; variables None = all m variables in order, position None = after the
    cones, else the block's index in the constraint list. Both sides stay strictly feasible: b_eq = A_eq y0[variables]
    for a small y0 at which every cone slack is interior, and A_eq^T lambda0 is added to b (the cone part of the
    primal point is unchanged, the multipliers are free). Equality entries of the returned list are
    ("eq", A_eq, (b_eq, variables))."""
    cones, b = small_multicone_problem(seed, **shape)
    m = b.size
    rng = np.random.Generator(np.random.PCG64(10 ** 6 + seed))
    y0 = y0_scale * rng.uniform(-1.0, 1.0, size=m)
    for kind, A, c in cones:  # the slacks at y0 are interior
        if kind == "psd":
            assert np.linalg.eigvalsh(c - sum(yi * Ai for yi, Ai in zip(y0, A))).min() > 0.1
        elif kind == "soc":
            s = c - A @ y0
            assert s[0] - np.linalg.norm(s[1:]) > 0.1
        else:
            assert (c - A @ y0).min() > 0.1
    out = list(cones)
    blocks = []
    for rows, variables, position in equalities:
        v = list(range(m)) if variables is None else list(variables)
        A_eq = rng.uniform(-1.0, 1.0, size=(rows, len(v)))
        b_eq = A_eq @ y0[v]
        lam0 = rng.uniform(-1.0, 1.0, size=rows)
        np.add.at(b, v, A_eq.T @ lam0)
        blocks.append((position, ("eq", A_eq, (b_eq, None if variables is None else v))))
    for position, entry in blocks:
        if position is None:
            out.append(entry)
        else:
            out.insert(position, entry)
    return out, b


def add_cones(P, cones):
    """Adds the constraints of a generator's list to P. A cone entry may carry a fourth element, the list of
    variables its columns act on (dense LMIs through CONEX_AddSparseLMIConstraint, LP and second-order cones through
    CONEXB200_AddSparseLinearConstraint / CONEXB200_AddSparseSocConstraint); without one it acts on all variables."""
    for entry in cones:
        kind, A, c = entry[:3]
        variables = entry[3] if len(entry) > 3 else None
        if kind == "eq":
            P.add_equality(A, c[0], c[1])
        elif variables is not None:
            if kind == "psd":
                P.add_dense_lmi(A, c, variables)
            elif kind == "soc":
                P.add_soc(A, c, variables=variables)
            else:
                P.add_linear(A, c, variables=variables)
        elif kind == "psd":
            P.add_dense_lmi(A, c)
        elif kind == "soc":
            P.add_soc(A, c)
        else:
            P.add_linear(A, c)


def pad_cones(cones, m):
    """The same constraints with every cone on all m variables in order: zero columns (LMIs: zero matrices) for the
    variables a cone does not act on. Equality blocks are kept as they are."""
    out = []
    for entry in cones:
        kind, A, c = entry[:3]
        variables = entry[3] if len(entry) > 3 else None
        if kind == "eq" or variables is None:
            out.append((kind, A, c))
        elif kind == "psd":
            mats = [np.zeros_like(c, dtype=np.float64) for _ in range(m)]
            for j, v in enumerate(variables):
                mats[v] = A[j]
            out.append((kind, mats, c))
        else:
            Ap = np.zeros((A.shape[0], m))
            Ap[:, list(variables)] = A
            out.append((kind, Ap, c))
    return out


def mpc_problem(seed, stages=8, stage_vars=6, lp_rows=12, soc_order=6, lmi_order=8, eq_rows=4, y0_scale=0.02):
    """A program shaped like a model-predictive-control horizon: `stages` stages of `stage_vars` variables
    (m = stages * stage_vars). Per stage, an LP block of `lp_rows` rows (A uniform, c = 1) and a Lorentz cone of
    order `soc_order` (A uniform, c = e_0) on the stage's variables; per pair of adjacent stages, a dense LMI of order
    `lmi_order` (A_i = sym(U[-1,1]), C = I) and an equality block of `eq_rows` rows on the two stages' variables
    (none with eq_rows = 0; the equality blocks are drawn last, so the cones do not depend on eq_rows).
    Constraint order: stage s's LP and SOC, then (s > 0) the LMI and the equality block coupling s - 1 and s.
    Strictly feasible by construction, like small_multicone_equality_problem: b = sum over cones of AW/2 at W = I plus
    A_eq^T lambda0, and b_eq = A_eq y0[variables] for a y0 at which every cone slack is interior.
    Returns (cones, padded, b): the list in the add_cones format with a variable list per cone, the same program
    with every cone on all m variables (pad_cones), and b."""
    rng = np.random.Generator(np.random.PCG64(seed))
    m = stages * stage_vars
    b = np.zeros(m)
    cones = []
    couplings = []
    for s in range(stages):
        v = list(range(s * stage_vars, (s + 1) * stage_vars))
        A = rng.uniform(-1.0, 1.0, size=(lp_rows, stage_vars))
        cones.append(("lp", A, np.ones(lp_rows), v))
        np.add.at(b, v, 0.5 * A.sum(axis=0))
        A = rng.uniform(-1.0, 1.0, size=(soc_order + 1, stage_vars))
        c = np.zeros(soc_order + 1)
        c[0] = 1.0
        cones.append(("soc", A, c, v))
        np.add.at(b, v, A[0, :])
        if s > 0:
            w = list(range((s - 1) * stage_vars, (s + 1) * stage_vars))
            mats = [random_sym(rng, lmi_order) for _ in w]
            cones.append(("psd", mats, np.eye(lmi_order), w))
            np.add.at(b, w, 0.5 * np.array([np.trace(M) for M in mats]))
            couplings.append((len(cones), w))
    # an interior y0: halved until every cone slack is interior with a margin
    y0 = y0_scale * rng.uniform(-1.0, 1.0, size=m)

    def margin(y):
        out = np.inf
        for kind, A, c, v in cones:
            if kind == "psd":
                out = min(out, np.linalg.eigvalsh(c - sum(yi * Ai for yi, Ai in zip(y[v], A))).min())
            elif kind == "soc":
                sl = c - A @ y[v]
                out = min(out, sl[0] - np.linalg.norm(sl[1:]))
            else:
                out = min(out, (c - A @ y[v]).min())
        return out

    while margin(y0) <= 0.1:
        y0 *= 0.5
    # after each LMI; reversed: earlier positions stay valid
    for position, w in reversed(couplings if eq_rows > 0 else []):
        A_eq = rng.uniform(-1.0, 1.0, size=(eq_rows, len(w)))
        lam0 = rng.uniform(-1.0, 1.0, size=eq_rows)
        np.add.at(b, w, A_eq.T @ lam0)
        cones.insert(position, ("eq", A_eq, (A_eq @ y0[w], w)))
    return cones, pad_cones(cones, m), b


def block_arrow_program(blocks, private, shared, order, seed):
    """`blocks` LMI cones of order `order`, cone k on its own `private` variables plus the same
    `shared` variables: H is block-arrow."""
    rng = np.random.default_rng(seed)
    m = blocks * private + shared
    cones = []
    for k in range(blocks):
        variables = list(range(k * private, (k + 1) * private)) + list(range(blocks * private, m))
        mats = [random_sym(rng, order) for _ in variables]
        cones.append((mats, np.eye(order), variables))
    return m, cones


# ----------------------------------------------------------------------------------------------
# Device-resident generators for operators that do not fit the host (C2: 64 GB, C5: 160 GB); torch
# only owns / indexes device memory here.
# ----------------------------------------------------------------------------------------------
def lovasz_edges(n, num_edges, seed=4):
    rng = np.random.Generator(np.random.PCG64(seed))
    idx = np.sort(rng.choice(n * (n - 1) // 2, size=num_edges, replace=False))
    # unrank the pair (i < j) from its index in row-major order of the strict upper triangle
    i = (n - 2 - np.floor(np.sqrt(-8.0 * idx + 4.0 * n * (n - 1) - 7) / 2.0 - 0.5)).astype(np.int64)
    j = (idx + i + 1 - n * (n - 1) // 2 + (n - i) * ((n - i) - 1) // 2).astype(np.int64)
    return i, j


class _Raw:
    def __init__(self, ptr, count):
        self.__cuda_array_interface__ = {"shape": (count,), "typestr": "<f8", "data": (ptr, False),
                                         "version": 2}


def device_view(ptr, count):
    """torch view (no copy) of `count` doubles of library-owned device memory."""
    import torch
    return torch.as_tensor(_Raw(ptr, count), device="cuda")


def maxcut_affine_term_device(n):
    """C = -L/4 of the C2 graph G(n, 0.5) drawn on the device (torch CUDA generator, seed 2): n x n tensor."""
    import torch
    g = torch.Generator(device="cuda")
    g.manual_seed(2)
    upper = torch.triu((torch.rand((n, n), generator=g, device="cuda") < 0.5).double(), 1)
    adj = upper + upper.T
    return -(torch.diag(adj.sum(1)) - adj) / 4.0


def fill_workload(kind, n, m, row_begin, row_count, A, Cm):
    """Writes this rank's constraint matrices (global indices row_begin .. row_begin+row_count-1) into
    A (row_count x n*n view, column-major n x n blocks) and the affine term into Cm (n x n), in place
    on the device; returns the local slice of the cost vector b. Same bytes for any sharding."""
    import torch
    idx = torch.arange(row_count, device="cuda")
    gi = idx + row_begin
    if kind == "maxcut":  # A_i = -e_i e_i^T, C = -L/4, b = -1 (SURVEY.md 8d, C2)
        Cm.copy_(maxcut_affine_term_device(n))
        A.zero_()
        A[idx, gi * n + gi] = -1.0
        return -np.ones(row_count)
    if kind == "random":  # A_i = sym(U[-1,1]), C = I, b = tr(A_i)/2 (test_util.cc:19,67-73; C1/C5)
        Cm.copy_(torch.eye(n, dtype=torch.float64, device="cuda"))
        b = torch.empty(row_count, dtype=torch.float64, device="cuda")
        blk = 32
        A3 = A.view(row_count, n, n)
        for g0 in range((row_begin // blk) * blk, row_begin + row_count, blk):
            g = torch.Generator(device="cuda")
            g.manual_seed(1000003 + g0)
            R = torch.rand((blk, n, n), generator=g, device="cuda", dtype=torch.float64) * 2.0 - 1.0
            R = 0.5 * (R + R.transpose(1, 2))
            lo, hi = max(g0, row_begin), min(g0 + blk, row_begin + row_count)
            A3[lo - row_begin:hi - row_begin] = R[lo - g0:hi - g0]
            b[lo - row_begin:hi - row_begin] = 0.5 * R[lo - g0:hi - g0].diagonal(dim1=1, dim2=2).sum(-1)
        return b.cpu().numpy()
    if kind == "lovasz":  # vars (t, y_e): A_0 = -I, A_e = E_ij + E_ji, C = -J, maximise -t (C4)
        Cm.fill_(-1.0)
        A.zero_()
        ei, ej = lovasz_edges(n, m - 1)
        ei = torch.from_numpy(ei).cuda()
        ej = torch.from_numpy(ej).cuda()
        is0 = gi == 0
        if bool(is0.any()):
            d = torch.arange(n, device="cuda")
            A[0, d * n + d] = -1.0
        e = gi[~is0] - 1
        rows = idx[~is0]
        A[rows, ej[e] * n + ei[e]] = 1.0
        A[rows, ei[e] * n + ej[e]] = 1.0
        b = np.zeros(row_count)
        if row_begin == 0:
            b[0] = -1.0
        return b
    raise ValueError(kind)


def structured_problem(w):
    """Entry-sparse form of the MaxCut / Lovasz-theta operators for the incremental API:
    (list of (var, r, c, val) lower-triangle entries, dense C, b). w: dict(kind, n, m)."""
    n, m = w["n"], w["m"]
    if w["kind"] == "maxcut_entries":
        rng = np.random.Generator(np.random.PCG64(2))
        upper = np.triu(rng.random((n, n)) < 0.5, 1).astype(np.float64)
        adj = upper + upper.T
        Cm = -(np.diag(adj.sum(axis=1)) - adj) / 4.0
        entries = [(i, i, i, -1.0) for i in range(n)]
        return entries, Cm, -np.ones(n)
    ei, ej = lovasz_edges(n, m - 1)
    entries = [(0, d, d, -1.0) for d in range(n)]
    entries += [(e + 1, int(max(ei[e], ej[e])), int(min(ei[e], ej[e])), 1.0) for e in range(m - 1)]
    b = np.zeros(m)
    b[0] = -1.0
    return entries, -np.ones((n, n)), b
