"""Host-side input provider: problem matrices, AMG hierarchy, smoothed transfers, RHS,
thread-group (-> CTA-group) partition.  Mirrors what the reference's SMEM_Setup hands to
the solve phase (/root/reference/src/SMEM_Setup.cpp:55-180, 182-276, 590-1036, 1038-1171).

hypre-BoomerAMG is absent from this image; `libamg_host.so` (host/amg_host.cpp) supplies a
classical AMG hierarchy of the same shape (diag-first CSR A_l, P_l).  All of this runs on
the CPU and is NOT the accelerated path.
"""
import ctypes as C
import os
import numpy as np

from . import build as _build

# enums shared with the reference (src/Main.hpp:47-75) ------------------------------------
JACOBI = 0
HYBRID_JACOBI_GAUSS_SEIDEL = 2
SEMI_ASYNC_GAUSS_SEIDEL = 4
ASYNC_GAUSS_SEIDEL = 5
L1_JACOBI = 6
L1_HYBRID_JACOBI_GAUSS_SEIDEL = 12      # Parfor smoother only (BPX): hybrid JGS divided by the l1 norms
MULT, AFACX, MULTADD, BPX = 0, 1, 2, 3
ASYNC_AFACX, ASYNC_MULTADD = 5, 6
PAR_BPX = 17                        # `-solver par_bpx` (src/Main.hpp:77): see par_bpx_equivalent
IMPLICIT_EXTENDED_SYSTEM_BPX = 16   # `-solver iebpx` (src/Main.hpp:76, src/SMEM_ExtendedSystem.cpp)


def par_bpx_equivalent(smoother, smooth_weight):
    """`-solver par_bpx` (SMEM_Sync_Parfor_BPXcycle's PAR_BPX branch, src/SMEM_Sync_AMG.cpp:183-236) is BPX on the concatenated level
    vectors with ONE Jacobi loop over all levels, xx = w * rr / A_diag_ext.  A_diag_ext already holds a_ii / w
    (src/SMEM_Setup.cpp:451-460), so the weight is applied twice: the cycle equals BPX with weighted Jacobi and weight w^2
    (confirmed against the reference's object code by the CPU test suite).  With the L1 smoother the step is w / l1 -- a
    weighted L1 Jacobi that no other solver of the reference has; it is not offered on the device.
    -> (solver, smoother, smooth_weight) to hand to Solver / amgb_options."""
    if smoother in (L1_JACOBI,):
        raise ValueError("par_bpx with the L1 smoother (step w / l1, src/SMEM_Sync_AMG.cpp:207-212) has no device equivalent")
    return BPX, JACOBI, smooth_weight * smooth_weight


class _CSR(C.Structure):
    _fields_ = [("nrows", C.c_int), ("ncols", C.c_int), ("nnz", C.c_int),
                ("i", C.POINTER(C.c_int)), ("j", C.POINTER(C.c_int)), ("data", C.POINTER(C.c_double))]


_lib = None


def host_lib():
    global _lib
    if _lib is None:
        path = _build.HOST_LIB
        if not os.path.exists(path):
            _build.build_host()
        L = C.CDLL(path)
        L.amgh_setup.restype = C.c_void_p
        L.amgh_setup.argtypes = [C.POINTER(_CSR), C.c_double, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
        L.amgh_level_A.restype = C.POINTER(_CSR)
        L.amgh_level_A.argtypes = [C.c_void_p, C.c_int]
        L.amgh_level_P.restype = C.POINTER(_CSR)
        L.amgh_level_P.argtypes = [C.c_void_p, C.c_int]
        L.amgh_num_levels.argtypes = [C.c_void_p]
        L.amgh_destroy.argtypes = [C.c_void_p]
        L.amgh_level_cpts.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.amgh_level_cpts.restype = None
        L.amgh_rand_fill.argtypes = [C.c_void_p, C.c_long, C.c_double, C.c_double, C.c_uint]
        L.amgh_rand_fill.restype = None
        L.amgh_csr_free.argtypes = [C.POINTER(_CSR)]
        L.amgh_csr_free.restype = None
        L.amgh_smooth_transfer.argtypes = [C.POINTER(_CSR), C.POINTER(_CSR), C.c_int, C.c_double,
                                           C.c_int, C.c_int, C.POINTER(_CSR), C.POINTER(_CSR)]
        L.amgh_setup_systems.restype = C.c_void_p
        L.amgh_setup_systems.argtypes = [C.POINTER(_CSR), C.c_int, C.c_double, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
        L.amgh_elasticity_beam.argtypes = [C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double,
                                           C.c_double, C.POINTER(_CSR), C.c_void_p]
        L.amgh_build_extended_matrix.argtypes = [C.c_int, C.POINTER(_CSR), C.POINTER(_CSR), C.POINTER(_CSR), C.POINTER(_CSR),
                                                 C.POINTER(C.c_int)]
        L.amgh_difconv_7pt.argtypes = [C.c_int] * 3 + [C.c_double] * 6 + [C.c_int, C.POINTER(_CSR)]
        L.amgh_permute.argtypes = [C.POINTER(_CSR), C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_int, C.POINTER(_CSR)]
        L.amgh_read_binary_triplets.argtypes = [C.c_char_p, C.c_int, C.POINTER(_CSR)]
        L.amgh_write_binary_triplets.argtypes = [C.POINTER(_CSR), C.c_char_p, C.c_int]
        _lib = L
    return _lib


class CSR:
    """Plain CSR triple (int32 indices, fp64 values) -- the layout of hypre_CSRMatrix
    {i, j, data} the reference kernels index (src/SMEM_MatVec.cpp:311-322)."""

    def __init__(self, nrows, ncols, indptr, indices, data):
        self.nrows, self.ncols = int(nrows), int(ncols)
        self.indptr = np.ascontiguousarray(indptr, dtype=np.int32)
        self.indices = np.ascontiguousarray(indices, dtype=np.int32)
        self.data = np.ascontiguousarray(data, dtype=np.float64)
        self.nnz = int(self.indptr[-1])

    @property
    def shape(self):
        return (self.nrows, self.ncols)

    def to_scipy(self):
        import scipy.sparse as sp
        return sp.csr_matrix((self.data, self.indices, self.indptr), shape=self.shape)

    @staticmethod
    def from_scipy(m, diag_first=False):
        m = m.tocsr()
        m.sort_indices()
        c = CSR(m.shape[0], m.shape[1], m.indptr, m.indices, m.data)
        if diag_first:
            c.make_diag_first()
        return c

    def make_diag_first(self):
        ip, ix, dv = self.indptr, self.indices, self.data
        rows = np.repeat(np.arange(self.nrows, dtype=np.int64), np.diff(ip))
        isd = ix == rows
        pos = np.nonzero(isd)[0]
        for p in pos:  # small matrices only (tests); the C++ path does the big ones
            r = rows[p]
            s = ip[r]
            if p != s:
                ix[s + 1:p + 1], ix[s] = ix[s:p].copy(), ix[p]
                dv[s + 1:p + 1], dv[s] = dv[s:p].copy(), dv[p]

    def diagonal(self):
        return self.data[self.indptr[:-1]].copy()

    def _as_c(self):
        s = _CSR()
        s.nrows, s.ncols, s.nnz = self.nrows, self.ncols, self.nnz
        s.i = self.indptr.ctypes.data_as(C.POINTER(C.c_int))
        s.j = self.indices.ctypes.data_as(C.POINTER(C.c_int))
        s.data = self.data.ctypes.data_as(C.POINTER(C.c_double))
        return s


def _take(cs, free=True):
    """copy a C-side amgh_csr into numpy-owned arrays"""
    n, nnz = cs.nrows, cs.nnz
    ip = np.ctypeslib.as_array(cs.i, shape=(n + 1,)).copy()
    ix = np.ctypeslib.as_array(cs.j, shape=(max(nnz, 1),))[:nnz].copy()
    dv = np.ctypeslib.as_array(cs.data, shape=(max(nnz, 1),))[:nnz].copy()
    out = CSR(n, cs.ncols, ip, ix, dv)
    if free:
        host_lib().amgh_csr_free(C.byref(cs))
    return out


def set_host_threads(n):
    """OpenMP threads of the host input provider (torchrun exports OMP_NUM_THREADS=1)"""
    host_lib().amgh_set_num_threads(C.c_int(int(n)))


def laplacian(problem, nx, ny=None, nz=None):
    """'5pt' (n x n), '7pt', '27pt' (nx x ny x nz); diag-first CSR, natural ordering."""
    L = host_lib()
    out = _CSR()
    ny = nx if ny is None else ny
    nz = nx if nz is None else nz
    if problem == "5pt":
        rc = L.amgh_laplacian_5pt(C.c_int(nx), C.byref(out))
    elif problem == "7pt":
        rc = L.amgh_laplacian_7pt(C.c_int(nx), C.c_int(ny), C.c_int(nz), C.byref(out))
    elif problem == "27pt":
        rc = L.amgh_laplacian_27pt(C.c_int(nx), C.c_int(ny), C.c_int(nz), C.byref(out))
    else:
        raise ValueError("unknown problem %r" % problem)
    if rc != 0:
        raise ValueError("problem too large for int32 CSR")
    return _take(out)


def difconv(nx, ny=None, nz=None, c=(1.0, 1.0, 1.0), a=(1.0, 1.0, 1.0), atype=-1):
    """`-problem difconv`: 3-D 7-point convection-diffusion stencil (src/BuildHypreMatrix.cpp:104-245; reference defaults
    c = a = 1, atype = -1 = centred, src/SMEM_Main.cpp:47-53).  Nonsymmetric; diag-first CSR, natural ordering."""
    ny = nx if ny is None else ny
    nz = nx if nz is None else nz
    out = _CSR()
    rc = host_lib().amgh_difconv_7pt(nx, ny, nz, c[0], c[1], c[2], a[0], a[1], a[2], int(atype), C.byref(out))
    if rc != 0:
        raise ValueError("problem too large for int32 CSR")
    return _take(out)


def elasticity_beam(ex, ey=None, ez=None, h=None, lam=(50.0, 1.0), mu=(50.0, 1.0)):
    """Stand-in for the reference's MFEM elasticity problem (DMEM_BuildMfemMatrix, src/DMEM_BuildMatrix.cpp:442-719;
    BASELINE.json configs[3]): Q1 hexahedra on an ex x ey x ez beam (default 8:1:1 like beam-hex.mesh), two materials,
    face x = 0 clamped, traction on x = L.  Returns (A, b): 3 unknowns per node, interleaved; use
    amg_setup(A, num_functions=3)."""
    ey = max(1, ex // 8) if ey is None else ey
    ez = ey if ez is None else ez
    h = 8.0 / ex if h is None else h
    out = _CSR()
    n = 3 * (ex + 1) * (ey + 1) * (ez + 1)
    b = np.zeros(n, dtype=np.float64)
    rc = host_lib().amgh_elasticity_beam(ex, ey, ez, h, lam[0], mu[0], lam[1], mu[1], C.byref(out), b.ctypes.data_as(C.c_void_p))
    if rc != 0:
        raise ValueError("elasticity problem too large for int32 CSR" if rc == 1 else "bad beam dimensions")
    return _take(out), b


def extended_system(h, f=None):
    """Explicit extended system of `-solver eebpx` (BuildExtendedMatrix + the bb assembly of InitAlgebra,
    src/SMEM_Setup.cpp:1426-1521,505-541) for a hierarchy whose transfers are the plain ones of BPX: returns (AA, disp[, bb])
    with AA the (sum_l n_l)-square matrix of blocks A_k P^{k<-l} / R^{l<-k} A_k^T (diag-first rows), disp[l] the first row
    of block l, and bb = (f, R_0 f, R_1 R_0 f, ...)."""
    L = h.num_levels
    As = (_CSR * L)(*[a._as_c() for a in h.A])
    Ps = (_CSR * max(L - 1, 1))(*[p._as_c() for p in h.P])
    Rs = (_CSR * max(L - 1, 1))(*[r._as_c() for r in h.R])
    out = _CSR()
    disp = np.zeros(L + 1, dtype=np.int32)
    rc = host_lib().amgh_build_extended_matrix(L, As, Ps, Rs, C.byref(out), disp.ctypes.data_as(C.POINTER(C.c_int)))
    if rc != 0:
        raise ValueError("extended matrix too large for int32 CSR")
    AA = _take(out)
    if f is None:
        return AA, disp
    parts = [np.asarray(f, dtype=np.float64)]
    for l in range(L - 1):
        parts.append(h.R[l].to_scipy() @ parts[-1])
    return AA, disp, np.concatenate(parts)


def extended_solution(h, disp, xx):
    """x = sum_l P_0 ... P_{l-1} x_l from the blocks of an extended-system iterate (src/SMEM_ExtendedSystem.cpp:736-759)"""
    L = h.num_levels
    v = np.array(xx[disp[L - 1]:disp[L]], dtype=np.float64)
    for l in range(L - 2, -1, -1):
        v = xx[disp[l]:disp[l + 1]] + h.P[l].to_scipy() @ v
    return v


def read_matrix(path, symm_flag=1):
    """`-problem file`: the reference's binary triplet format (ReadBinary_fread_HypreParCSR, src/Misc.cpp:800-915;
    SMEM_Setup calls it with symm_flag = 1, src/SMEM_Setup.cpp:1646-1650).  Diag-first CSR."""
    out = _CSR()
    rc = host_lib().amgh_read_binary_triplets(os.fsencode(path), C.c_int(int(symm_flag)), C.byref(out))
    if rc != 0:
        raise IOError({1: "cannot open matrix file %r", 2: "matrix file %r is not in the 16-byte triplet format",
                       3: "matrix file %r has an index outside 1..num_rows"}.get(rc, "cannot read %r") % path)
    return _take(out)


def write_matrix(m, path, lower_only=True):
    """the matching writer (PrintCSRMatrix, bin_file = 1, src/Misc.cpp:752-798); lower_only: one triangle, the
    form the SMEM reader mirrors"""
    cs = m._as_c()
    if host_lib().amgh_write_binary_triplets(C.byref(cs), os.fsencode(path), C.c_int(1 if lower_only else 0)) != 0:
        raise IOError("cannot write %r" % path)


def rand_rhs(n, lo=-1.0, hi=1.0, seed=0):
    """SMEM RHS: srand(0); b_i = RandDouble(-1,1) (src/SMEM_Setup.cpp:1729-1742)."""
    b = np.empty(n, dtype=np.float64)
    host_lib().amgh_rand_fill(b.ctypes.data_as(C.c_void_p), C.c_long(n), lo, hi, C.c_uint(seed))
    return b


def reference_processor_grid(num_procs, nx, ny, nz):
    """(P, Q, R) the reference's search picks for `num_procs` ranks (src/DMEM_BuildMatrix.cpp:169-240 = src/BuildHypreMatrix.cpp:36-76):
    1 rank -> (1,1,1); a prime count -> (1, num_procs, 1), y-slabs; otherwise the first (x, y, z) with x*y*z = num_procs when the
    divisors are tried in ascending order with z fastest -- (1, 1, num_procs), z-slabs, whenever num_procs <= nz.  The partitioned
    path here uses z-slabs for every count (DESIGN.md section 6)."""
    if num_procs == 1:
        return 1, 1, 1
    divs = [d for d in range(1, num_procs + 1) if num_procs % d == 0]
    if len(divs) == 2:
        return 1, num_procs, 1
    x = y = z = 1
    done = False
    for di in divs:
        for dj in divs:
            for dk in divs:
                if dk > nz or done:
                    break
                x, y, z = di, dj, dk
                if x * y * z == num_procs:
                    done = True
            if dj > ny or done:
                break
        if di > nx or done:
            break
    return x, y, z


def rand_rhs_dmem(row_starts):
    """DMEM RHS (SURVEY.md 5.9j): EVERY rank seeds srand(0) and draws its local rows from RandDouble(-.5, .5)
    (src/DMEM_Setup.cpp:1293,1351), so the global b is the same glibc sequence repeated per rank and depends on the number of
    ranks.  row_starts: the P + 1 row offsets of the partition."""
    parts = [rand_rhs(int(row_starts[p + 1] - row_starts[p]), -0.5, 0.5, 0) for p in range(len(row_starts) - 1)]
    return np.concatenate(parts) if parts else np.empty(0)


def max_eig_estimate_cg(A, iters=20, seed=1):
    """Largest / smallest eigenvalue estimate of D^-1/2 A D^-1/2 (= those of D^-1 A) from `iters` CG steps: the Lanczos
    tridiagonal of the CG coefficients, as hypre_ParCSRMaxEigEstimateCG(A, scale = 1, max_iter, ...) computes them (hypre
    par_relax_more.c; hypre is un-vendored, so this follows the published algorithm: right-hand side 0, random start vector,
    T_jj = 1/alpha_j + beta_{j-1}/alpha_{j-1}, T_j,j+1 = sqrt(beta_j)/alpha_j).  The start vector comes from a
    Park-Miller generator like hypre_Rand's; PARITY UNPINNED -- the estimate depends on it in the third digit.
    -> (max_eig, min_eig)"""
    S = A.to_scipy().tocsr()
    n = S.shape[0]
    d = np.asarray(A.diagonal(), dtype=np.float64)
    ds = 1.0 / np.sqrt(np.abs(d))
    x = np.empty(n)
    st = int(seed) % 2147483647 or 1
    for i in range(n):                       # minimal-standard LCG: a = 16807, m = 2^31 - 1, value 2 s / m - 1
        st = (16807 * st) % 2147483647
        x[i] = 2.0 * st / 2147483647.0 - 1.0
    r = -(ds * (S @ (ds * x)))                # r = 0 - B x
    p = r.copy()
    gamma = float(r @ r)
    diag, off = [], []
    alpha_old, beta = 1.0, 0.0
    for j in range(iters):
        if gamma == 0.0:
            break
        s_ = ds * (S @ (ds * p))
        sdotp = float(s_ @ p)
        if sdotp == 0.0:
            break
        alpha = gamma / sdotp
        diag.append(1.0 / alpha + (beta / alpha_old if j > 0 else 0.0))
        x += alpha * p
        r -= alpha * s_
        gamma_old, gamma = gamma, float(r @ r)
        beta = gamma / gamma_old
        off.append(np.sqrt(beta) / alpha)
        p = r + beta * p
        alpha_old = alpha
    k = len(diag)
    T = np.diag(diag) + np.diag(off[:k - 1], 1) + np.diag(off[:k - 1], -1)
    ev = np.linalg.eigvalsh(T)
    return float(ev[-1]), float(ev[0])


def dmem_default_smooth_weight(A, iters=20):
    """DMEM's default Jacobi weight (SURVEY.md 5.9k): 1 / lambda_max(D^-1 A) from 20 CG steps (src/DMEM_Setup.cpp:77-87,
    -eig_CG_max_iters; off when -smooth_weight is given, src/DMEM_Main.cpp:443-447)"""
    return 1.0 / max_eig_estimate_cg(A, iters)[0]


class Hierarchy:
    """Per-level A (diag-first), P (plain), and the transfer operators the selected cycle
    uses: for MULTADD P̄ = G P and R̄ = Pᵀ GT (SMEM_Setup.cpp:244-260,1173-1254); for
    AFACX / BPX plain P and R = Pᵀ (SMEM_Setup.cpp:262-274)."""

    def __init__(self, A, P):
        self.A = A
        self.P_plain = P
        self.num_levels = len(A)
        self.n = [a.nrows for a in A]
        self.P = None
        self.R = None
        self.R_plain = [None] * (len(A) - 1)     # P_l^T, built on demand (plain_restriction)
        self.smooth_weight = None
        self.l1 = None
        self.cpts = None      # cpts[l][j]: level-l index of coarse point j of level l+1 (row partitions follow it)

    def build_transfers(self, solver=MULTADD, smooth_weight=1.0, smooth_interp_type=JACOBI,
                        num_pre=1, num_post=1, factor_level0=False):
        """factor_level0: leave P_0 / R_0 plain (amgb_options.factor_level0 applies the smoothing factors on the fly)"""
        L = host_lib()
        self.P, self.R = [], []
        self.smooth_weight = smooth_weight
        for l in range(self.num_levels - 1):
            a_c, p_c = self.A[l]._as_c(), self.P_plain[l]._as_c()
            if solver in (MULTADD, ASYNC_MULTADD) and (num_pre > 0 or num_post > 0) and not (factor_level0 and l == 0):
                pb, rb = _CSR(), _CSR()
                kind = 0 if smooth_interp_type in (JACOBI, HYBRID_JACOBI_GAUSS_SEIDEL) else 1
                L.amgh_smooth_transfer(C.byref(a_c), C.byref(p_c), kind, smooth_weight,
                                       int(num_post > 0), int(num_pre > 0), C.byref(pb), C.byref(rb))
                self.P.append(_take(pb) if num_post > 0 else self.P_plain[l])
                if num_pre > 0:
                    self.R.append(_take(rb))
                else:
                    self.R.append(self._transpose(self.P_plain[l]))
            else:
                self.P.append(self.P_plain[l])
                self.R.append(self._transpose(self.P_plain[l]))
        return self

    def plain_restriction(self, l):
        """P_l^T from the plain interpolation, built once and kept: what amgb_options.factor_restriction uploads as R_l for
        l >= 1 (the explicit products in self.R stay for the other solvers)"""
        if self.R_plain[l] is None:
            self.R_plain[l] = self._transpose(self.P_plain[l])
        return self.R_plain[l]

    @staticmethod
    def _transpose(p):
        L = host_lib()
        out = _CSR()
        pc = p._as_c()
        L.amgh_restriction_from_P(C.byref(pc), C.byref(out))
        return _take(out)

    def l1_norms(self):
        if self.l1 is None:
            self.l1 = []
            for a in self.A:
                rows = np.repeat(np.arange(a.nrows), np.diff(a.indptr))
                self.l1.append(np.bincount(rows, weights=np.abs(a.data), minlength=a.nrows))
        return self.l1

    def operator_complexity(self):
        return sum(a.nnz for a in self.A) / self.A[0].nnz


def amg_setup(A, theta=0.25, max_levels=25, max_coarse=9, pmax=4, jacobi_interp_steps=1, verbose=False, num_functions=1):
    """Classical AMG hierarchy (stand-in for HYPRE_BoomerAMGSetup, SMEM_Setup.cpp:65).  num_functions > 1: systems of
    PDEs with interleaved unknowns, unknown-based coarsening (HYPRE_BoomerAMGSetNumFunctions; the reference sets
    num_functions = dim for elasticity, src/DMEM_BuildMatrix.cpp:470)."""
    L = host_lib()
    a_c = A._as_c()
    h = L.amgh_setup_systems(C.byref(a_c), int(num_functions), theta, max_levels, max_coarse, pmax, jacobi_interp_steps,
                             int(verbose))
    nl = L.amgh_num_levels(h)
    As = [_take(L.amgh_level_A(h, l).contents, free=False) for l in range(nl)]
    Ps = [_take(L.amgh_level_P(h, l).contents, free=False) for l in range(nl - 1)]
    cpts = []
    for l in range(nl - 1):
        c = np.empty(As[l + 1].nrows, dtype=np.int32)
        L.amgh_level_cpts(h, l, c.ctypes.data_as(C.c_void_p))
        cpts.append(c)
    L.amgh_destroy(h)
    hh = Hierarchy(As, Ps)
    hh.cpts = cpts
    return hh


# ---------------------------------------------------------------------------------------------
# data-layout experiment: tiled ordering of the unknowns (fewer distinct cache lines per x gather of the Galerkin /
# transfer operators, profiles/README.md section 3).  The hierarchy is built in the reference's natural ordering and then
# permuted consistently on every level, so it is the SAME hierarchy: same cycle counts, same history up to summation order.
# ---------------------------------------------------------------------------------------------
def tiled_permutation(nx, ny, nz, tile):
    """new_of_old for a structured nx x ny x nz grid in natural ordering: unknowns numbered tile by tile (tile^3 blocks in
    x-fastest order, x-fastest inside a tile)"""
    ix, iy, iz = np.meshgrid(np.arange(nx), np.arange(ny), np.arange(nz), indexing="ij")
    ix, iy, iz = (a.transpose(2, 1, 0).ravel() for a in (ix, iy, iz))          # natural order: x fastest
    tx, ty, tz = ix // tile, iy // tile, iz // tile
    ntx, nty = -(-nx // tile), -(-ny // tile)
    key = (((tz * nty + ty) * ntx + tx).astype(np.int64) * tile ** 3 +
           ((iz % tile) * tile + (iy % tile)) * tile + (ix % tile))
    order = np.argsort(key, kind="stable")            # order[new] = old
    new_of_old = np.empty(order.size, dtype=np.int32)
    new_of_old[order] = np.arange(order.size, dtype=np.int32)
    return new_of_old


def _permute(m, new_row, new_col, diag_first):
    out = _CSR()
    mc = m._as_c()
    nr = np.ascontiguousarray(new_row, dtype=np.int32)
    ncl = np.ascontiguousarray(new_col, dtype=np.int32)
    rc = host_lib().amgh_permute(C.byref(mc), nr.ctypes.data_as(C.POINTER(C.c_int)), ncl.ctypes.data_as(C.POINTER(C.c_int)),
                                 int(diag_first), C.byref(out))
    if rc != 0:
        raise ValueError("not a permutation")
    return _take(out)


def reorder_hierarchy(h, new_of_old0):
    """(hierarchy with every level renumbered, [new_of_old per level]): level 0 by `new_of_old0`, every coarser level by the
    new index of its points' fine parents (so coarse points keep following their fine points, as cpts requires)"""
    if h.cpts is None:
        raise ValueError("hierarchy has no coarse-point map")
    perms = [np.ascontiguousarray(new_of_old0, dtype=np.int32)]
    for l in range(h.num_levels - 1):
        parent_new = perms[l][h.cpts[l]]
        order = np.argsort(parent_new, kind="stable")
        p = np.empty(order.size, dtype=np.int32)
        p[order] = np.arange(order.size, dtype=np.int32)
        perms.append(p)
    A = [_permute(h.A[l], perms[l], perms[l], True) for l in range(h.num_levels)]
    P = [_permute(h.P_plain[l], perms[l], perms[l + 1], False) for l in range(h.num_levels - 1)]
    out = Hierarchy(A, P)
    out.cpts = []
    for l in range(h.num_levels - 1):
        c = np.empty(h.n[l + 1], dtype=np.int32)
        c[perms[l + 1]] = perms[l][h.cpts[l]]
        out.cpts.append(c)
    return out, perms


# ---------------------------------------------------------------------------------------------
# work model and group partition (src/SMEM_Setup.cpp:1038-1171, 770-854, 870-893, 945-979)
# ---------------------------------------------------------------------------------------------
def compute_work(h, solver=MULTADD, num_pre=1, num_post=1, fine_sweeps=1, coarse_sweeps=1):
    """level_work / frac_level_work for res_compute_type == LOCAL."""
    L = h.num_levels
    work = [0] * L
    multadd = solver in (MULTADD, ASYNC_MULTADD)
    for level in range(L):
        w = h.A[0].nnz + h.A[0].nrows
        coarsest = level if multadd else level + 1
        for inner in range(coarsest):
            if inner >= L - 1:
                continue
            if multadd:
                w += h.R[inner].nnz
            elif level < L - 1:
                w += inner * h.R[inner].nnz
        if level == L - 1:
            w += h.A[level].nnz
        elif multadd:
            if num_post > 0 and num_pre > 0:
                w += fine_sweeps * (h.A[level].nnz + h.A[level].nrows)
            else:
                w += h.A[level].nrows
        else:
            w += ((coarse_sweeps - 1) * h.A[level + 1].nnz + h.P[level].nnz + h.A[level].nnz
                  + (fine_sweeps - 1) * h.A[level].nnz)
        for inner in range(level):
            w += h.P[inner].nnz
        work[level] = w
    tot = float(sum(work))
    return work, [x / tot for x in work]


def balanced_threads(frac, num_threads):
    """BALANCED_THREADS distribution of src/SMEM_Setup.cpp:770-854: deal threads round-robin,
    then move one thread at a time from the most over- to the most under-provisioned level."""
    L = len(frac)
    tpl = [0] * L
    lvl = 0
    for _ in range(num_threads):
        tpl[lvl] += 1
        lvl = lvl + 1 if lvl < L - 1 else 0
    prev = float("inf")
    while True:
        max_diff, k_max = 0.0, 0
        for k in range(L):
            diff = frac[k] - tpl[k] / num_threads
            if abs(diff) > abs(max_diff):
                if max_diff < 0.0 and tpl[k] == 1:
                    pass
                else:
                    max_diff, k_max = diff, k
        min_diff, k_min, not_found = float("inf"), 0, True
        for k in range(L):
            if k == k_max:
                continue
            diff = frac[k] - tpl[k] / num_threads
            if max_diff > 0.0:
                if diff < 0.0 and tpl[k] > 1 and abs(diff) < abs(min_diff):
                    min_diff, k_min, not_found = diff, k, False
            else:
                if diff > 0.0 and abs(diff) < abs(min_diff):
                    min_diff, k_min, not_found = diff, k, False
        if abs(max_diff) >= abs(prev) or not_found:
            break
        prev = max_diff
        if max_diff > 0.0:
            tpl[k_min] -= 1
            tpl[k_max] += 1
        else:
            tpl[k_min] += 1
            tpl[k_max] -= 1
    return tpl


def nnz_balanced_bounds(indptr, nparts):
    """[ns,ne) per part from the nnz-balanced split (hypre_LowerBound on the row pointer),
    src/SMEM_Setup.cpp:870-893."""
    n = len(indptr) - 1
    nnz = int(indptr[-1])
    per = (nnz + nparts - 1) // nparts
    b = [0]
    for t in range(1, nparts):
        b.append(int(np.searchsorted(indptr[:n], per * t, side="left")))
    b.append(n)
    return np.asarray(b, dtype=np.int32)


def uniform_blocks(n, block_rows):
    """hybrid-JGS block list used on the GPU: contiguous blocks of `block_rows` rows."""
    b = np.arange(0, n + block_rows, block_rows, dtype=np.int64)
    b[-1] = n
    if len(b) >= 2 and b[-2] >= n:
        b = b[:-1]
        b[-1] = n
    return b.astype(np.int32)


# ---------------------------------------------------------------------------------------------
# algorithmic byte model (SURVEY.md 8d / BASELINE.md 3)
# ---------------------------------------------------------------------------------------------
def bytes_spmv(m, with_b):
    return 12 * m.nnz + 4 * (m.nrows + 1) + 8 * m.ncols + 8 * m.nrows + (8 * m.nrows if with_b else 0)


def bytes_sync_multadd_cycle(h, symmetric=True):
    L = h.num_levels
    tot = bytes_spmv(h.A[0], True)
    for l in range(L - 1):
        tot += bytes_spmv(h.R[l], False)
        tot += (bytes_spmv(h.A[l], False) + 8 * h.n[l]) if symmetric else 24 * h.n[l]
        tot += bytes_spmv(h.P[l], True)
    tot += 8 * h.n[0]
    return tot


def bytes_plain_restriction(p):
    """bytes_spmv(P^T, False) from the interpolation P itself, without forming the transpose"""
    return 12 * p.nnz + 4 * (p.ncols + 1) + 8 * p.nrows + 8 * p.ncols


def bytes_sync_multadd_cycle_factored(h, factor_restriction=True):
    """the same cycle with the level-0 transfers in factorised form (amgb_options.factor_level0; h.P[0] / h.R[0] plain):
    residual on A_0, t_0 pass on A_0 (reads r_0, writes t_0), R_0, P_0, final pass on A_0 (reads v, r_0, t_0, w/d, u; writes u).
    factor_restriction (amgb_options.factor_restriction, the single-GPU default): on the levels l >= 1 the plain P_l^T
    replaces Rbar_l and the smoother's pass over A_l also stores t_l (8 n_l); False: the explicit h.R[l] (the partitioned
    multi-GPU cycle).  As in bytes_sync_multadd_cycle, every level below the coarsest counts one restriction."""
    L = h.num_levels
    n0 = h.n[0]
    tot = bytes_spmv(h.A[0], True)                                  # r = f - A u
    tot += bytes_spmv(h.A[0], True)                                 # t_0 = r_0 - A_0 diag(w/d) r_0
    tot += bytes_spmv(h.R[0], False) + bytes_spmv(h.P[0], False)    # plain transfers
    tot += bytes_spmv(h.A[0], True) + 3 * 8 * n0                    # u += v + (w/d) o (r_0 + t_0 - A_0 v): extra reads t_0, w/d, u
    for l in range(1, L - 1):                                       # coarser levels as in bytes_sync_multadd_cycle
        rb = bytes_plain_restriction(h.P_plain[l]) + 8 * h.n[l] if factor_restriction else bytes_spmv(h.R[l], False)
        tot += rb + bytes_spmv(h.A[l], False) + 8 * h.n[l] + bytes_spmv(h.P[l], True)
    return tot


def bytes_async_chain(h, k, symmetric=True, fact0=False):
    """algorithmic bytes of ONE correction of level k's group (SURVEY.md 8d).  fact0: h.P[0] / h.R[0] are the plain transfers
    and the smoothing factors are applied on the fly (two extra passes over A_0 for every group below level 0)"""
    tot = 0
    for l in range(min(k, h.num_levels - 1)):
        tot += bytes_spmv(h.R[l], False) + bytes_spmv(h.P[l], False)
        if fact0 and l == 0:
            tot += 2 * bytes_spmv(h.A[0], True)
    if k < h.num_levels - 1:
        tot += (bytes_spmv(h.A[k], False) + 8 * h.n[k]) if symmetric else 24 * h.n[k]
    tot += bytes_spmv(h.A[0], True) + 32 * h.n[0]
    return tot
