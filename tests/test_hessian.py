"""Hessians of scalar functions: finite_difference_hessian! (src/hessians.jl:202-292).

CPU: the Hessian oracle (oracle_hessian/) against the reference's own known answers and, bit for bit, against an
independent Python transcription of hessians.jl:202-292 written below; the step-size helpers of the C ABI; the mirror's
constructor rules.  GPU (through the C ABI and the Python mirror): H bit-identical to the oracle for several n and batch
sizes, symmetry, untouched padding, the call sequence, the closed-form synthetic Hessian, the known answers, error paths.
"""
import ctypes as C
import functools
import math

import numpy as np
import pytest

torch = pytest.importorskip("torch")

RELSTEP_H = 2.0 ** -13      # eps(Float64)^(1/4)  epsilons.jl:134-144


@pytest.fixture(scope="module")
def horc():
    from oracle_hessian import hessian_oracle
    hessian_oracle.build()
    hessian_oracle.lib()
    return hessian_oracle


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__  # noqa: F401  (puts the repository root on sys.path)
    import _bootstrap
    p = _bootstrap.load_package()
    p._lib.lib()
    return p


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def err_func(a, b):
    # test/finitedifftests.jl:20
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b))))


def jl_isapprox(a, b):
    # Base.isapprox for arrays: norm(a - b) <= sqrt(eps) * max(norm(a), norm(b))
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.linalg.norm(a - b) <= math.sqrt(np.finfo(float).eps) * max(np.linalg.norm(a), np.linalg.norm(b))


def jl_sum_abs2(x):
    # sum(abs2, x) for length < 16: sequential left-to-right reduction
    s = x[0] * x[0]
    for k in range(1, len(x)):
        s = s + x[k] * x[k]
    return s


# ------------------------------------------------------------------------------------------ independent transcription
def _jl_max(a, b):
    # Base.max(::Float64, ::Float64)
    if math.isnan(a) or math.isnan(b):
        return a + b
    if b > a or (math.copysign(1.0, a) < 0 < math.copysign(1.0, b)):
        return b
    return a


def transcribed_hessian(f, x, relstep=None, absstep=None, cache=None):
    """hessians.jl:202-292, in-place branch, line by line in Python floats (IEEE double, no contraction).
    Returns (H as list of lists, eps per component, calls, points evaluated in call order)."""
    x = [float(v) for v in x]
    n = len(x)
    relstep = RELSTEP_H if relstep is None else relstep                         # :204
    absstep = relstep if absstep is None else absstep                           # :205
    pts = []

    def call(v):
        pts.append(list(v))
        return f(np.array(v))

    H = [[0.0] * n for _ in range(n)]
    if cache is None:
        xpp, xpm, xmp, xmm = list(x), list(x), list(x), list(x)                  # HessianCache(x) :85-88
    else:
        xpp, xpm, xmp, xmm = [list(map(float, c)) for c in cache]
    fx = call(x)                                                                # :209
    xpp[:], xpm[:], xmp[:], xmm[:] = list(x), list(x), list(x), list(x)         # :213-216
    steps = []
    for i in range(n):                                                          # :221
        xi = x[i]
        epsilon = _jl_max(relstep * abs(xi), absstep)                           # :223
        steps.append(epsilon)
        xpp[i] = xi + epsilon                                                   # :226
        xmm[i] = xi - epsilon                                                   # :227
        a = call(xpp)
        b = call(xmm)
        H[i][i] = (a - 2 * fx + b) / (epsilon * epsilon)                        # :233 (epsilon^2 is literal_pow: e*e)
        epsiloni = _jl_max(relstep * abs(xi), absstep)                          # :234
        xp = xi + epsiloni
        xm = xi - epsiloni
        xpp[i] = xp; xpm[i] = xp; xmp[i] = xm; xmm[i] = xm                      # :239-242
        for j in range(i + 1, n):                                               # :250
            xj = x[j]
            epsilonj = _jl_max(relstep * abs(xj), absstep)                      # :252
            xp = xj + epsilonj
            xm = xj - epsilonj
            xpp[j] = xp; xpm[j] = xm; xmp[j] = xp; xmm[j] = xm                  # :257-260
            f1 = call(xpp); f2 = call(xpm); f3 = call(xmp); f4 = call(xmm)
            H[i][j] = (f1 - f2 - f3 + f4) / (4 * epsiloni * epsilonj)           # :268-269
            xpp[j] = xj; xpm[j] = xj; xmp[j] = xj; xmm[j] = xj                  # :272-275
        xpp[i] = xi; xpm[i] = xi; xmp[i] = xi; xmm[i] = xi                      # :285-288
    for i in range(n):                                                          # copytri!(H, 'U') :291
        for j in range(i):
            H[i][j] = H[j][i]
    return np.array(H, dtype=np.float64).reshape(n, n), np.array(steps), len(pts), pts


def layout_points(x, eps):
    """The call order the library lays out (include/fdjac_b200.h): p = 0 is x; row i at R(i) = 1 + 2i(2n-i) holds
    x_i+e_i, x_i-e_i, then for j > i the (+,+), (+,-), (-,+), (-,-) moves of (i, j)."""
    n = len(x)
    out = [list(x)]
    for i in range(n):
        assert len(out) == 1 + 2 * i * (2 * n - i)
        for s in (1, -1):
            v = list(x)
            v[i] = x[i] + eps[i] if s > 0 else x[i] - eps[i]
            out.append(v)
        for j in range(i + 1, n):
            for si, sj in ((1, 1), (1, -1), (-1, 1), (-1, -1)):
                v = list(x)
                v[i] = x[i] + eps[i] if si > 0 else x[i] - eps[i]
                v[j] = x[j] + eps[j] if sj > 0 else x[j] - eps[j]
                out.append(v)
    assert len(out) == 2 * n * n + 1
    return out


def random_scalar_fn(rng, n):
    a = rng.uniform(-2, 2, n)
    c = rng.uniform(-1, 1, n)

    def f(v):
        s = 0.0
        for k in range(len(v)):
            s = s + math.sin(a[k] * v[k]) + c[k] * v[k] * v[k] * v[k]
        for k in range(len(v) - 1):
            s = s + v[k] * v[k + 1]
        return s
    return f


def hess_poly_closed_form(x, w):
    n = len(x)
    H = np.full((n, n), 1.0 / n)
    H[np.arange(n), np.arange(n)] = 6 * w * x + 1.0 / n
    idx = np.arange(n - 1)
    H[idx, idx + 1] = 1 + 1.0 / n
    H[idx + 1, idx] = 1 + 1.0 / n
    return H


def hess_poly_tolerance(x, w, eps):
    """Rounding bound for the synthetic f's Hessian (its truncation error is 0: f is a cubic).  Each of the four values
    of an entry carries at most (n/32 + 8) roundings of a sum whose magnitude is T; the entry divides their
    combination by 4 e_i e_j >= 4 min(e)^2 (2 min(e)^2 on the diagonal, with f(x) counted twice)."""
    n = len(x)
    T = float(np.sum(np.abs(w * x ** 3)) + np.sum(np.abs(x[:-1] * x[1:])) + np.sum(np.abs(x)) ** 2 / (2 * n))
    return 4 * (n / 32 + 8) * 2.0 ** -53 * T / min(eps) ** 2


# ------------------------------------------------------------------------------------------ CPU: oracle known answers
X_SINCOS = np.array([0.3, 0.7])


def test_oracle_kat_sin_cos(horc):
    # test/finitedifftests.jl:561-576 (x = rand(2) there; a fixed point here)
    f = lambda v: math.sin(v[0]) + math.cos(v[1])
    x = X_SINCOS
    H_ref = np.array([[-math.sin(x[0]), 0.0], [0.0, -math.cos(x[1])]])
    cached = horc.hessian(f, x, cache=tuple(x.copy() for _ in range(4)))
    cacheless = horc.hessian(f, x)
    assert err_func(cached["H"], H_ref) < 1e-4
    assert err_func(cacheless["H"], H_ref) < 1e-4
    assert np.array_equal(bits(cached["H"]), bits(cacheless["H"]))          # the immutable / in-place branches agree
    assert cached["fcalls"] == 9


def test_oracle_kat_half_sum_abs2(horc):
    # finitedifftests.jl:593-598: sum(abs2, t)/2 at ones(2) ≈ I
    r = horc.hessian(lambda v: jl_sum_abs2(v) / 2, np.ones(2))
    assert jl_isapprox(r["H"], np.eye(2))


def test_oracle_kat_cache_from_other_x_is_exact(horc):
    # finitedifftests.jl:608-614 (issue #185): sum(abs2) at 1:4 with the cache built from 1:4 and from 5:8 == Diagonal(2)
    x1, x2 = np.arange(1.0, 5.0), np.arange(5.0, 9.0)
    for src in (x1, x2):
        r = horc.hessian(jl_sum_abs2, x1, cache=tuple(src.copy() for _ in range(4)))
        assert np.array_equal(r["H"], np.diag(np.full(4, 2.0)))


def test_oracle_kat_poisoned_cache(horc):
    # cache_reuse_tests.jl:130-139
    h = lambda v: v[0] * v[0] + 2 * (v[1] * v[1])
    cache = tuple(np.full(2, 1e10) for _ in range(4))
    r = horc.hessian(h, np.array([1.0, 2.0]), cache=cache)
    assert np.allclose(r["H"], [[2.0, 0.0], [0.0, 4.0]], rtol=0, atol=1e-3)
    # the restores leave the cache arrays equal to x (hessians.jl:272-275, 285-288)
    for c in cache:
        assert np.array_equal(c, [1.0, 2.0])


def test_default_relstep_and_epsilon(pkg, horc):
    lib = pkg._lib.lib()
    assert horc.default_relstep() == RELSTEP_H
    assert lib.fdb_default_relstep(pkg._lib.FDB_HCENTRAL) == RELSTEP_H
    assert pkg.default_relstep("hcentral") == RELSTEP_H
    for xv in (-4.0, 0.0, 1e-30, 3.5e10, -0.0):
        for rs, ab in ((1e-3, 1e-8), (0.0, 1e-5), (1e-4, 0.0), (RELSTEP_H, RELSTEP_H)):
            for d in (1.0, -1.0):   # no dir for hcentral
                got = lib.fdb_compute_epsilon(pkg._lib.FDB_HCENTRAL, xv, rs, ab, d)
                assert got == horc.compute_epsilon(xv, rs, ab) == _jl_max(rs * abs(xv), ab)
    # the forward / central helpers are unchanged
    assert pkg.default_relstep("forward") == 1.4901161193847656e-08
    assert pkg.default_relstep("central") == 6.0554544523933395e-06


def _random_problem(rng, k):
    n = int(rng.integers(0, 13))
    x = rng.uniform(-3, 3, n)
    x[np.abs(x) < 1e-3] = 0.5
    mode = k % 4
    if mode == 0:
        relstep = absstep = None
    elif mode == 1:
        relstep, absstep = 0.0, float(rng.uniform(1e-6, 1e-3))                  # pure absolute step
    elif mode == 2:
        relstep, absstep = float(rng.uniform(1e-6, 1e-3)), 0.0                  # pure relative step
    else:
        relstep, absstep = float(rng.uniform(1e-6, 1e-3)), float(rng.uniform(1e-6, 1e-3))
    return n, x, relstep, absstep


def test_oracle_equals_transcription(horc):
    """>= 100 random small problems: H, steps, call count 2n^2+1 and the exact sequence of evaluated points, bit for bit."""
    rng = np.random.default_rng(20261017)
    for k in range(120):
        n, x, relstep, absstep = _random_problem(rng, k)
        f = random_scalar_fn(rng, n)
        seen = []

        def fo(v, f=f):
            seen.append(np.array(v, dtype=np.float64))
            return f(v)
        r = horc.hessian(fo, x, relstep=relstep, absstep=absstep)
        H, steps, calls, pts = transcribed_hessian(f, x, relstep, absstep)
        assert calls == r["fcalls"] == 2 * n * n + 1 == len(seen), (k, n)
        assert np.array_equal(bits(r["H"]), bits(H)), (k, n)
        assert np.array_equal(bits(r["eps"]), bits(steps)), (k, n)
        assert all(np.array_equal(bits(a), bits(np.array(b))) for a, b in zip(seen, pts)), (k, n)
        # and the layout the library evaluates in is this same sequence
        lay = layout_points(list(x), list(steps))
        assert all(np.array_equal(bits(np.array(a)), bits(np.array(b))) for a, b in zip(lay, pts)), (k, n)


def test_oracle_synthetic_closed_form(horc):
    rng = np.random.default_rng(7)
    for n in (1, 2, 5, 40, 97):
        x = rng.uniform(0.5, 1.5, n)
        w = rng.uniform(-1, 1, n)
        r = horc.hess_poly(x, w)
        assert r["fcalls"] == 2 * n * n + 1
        assert np.max(np.abs(r["H"] - hess_poly_closed_form(x, w))) <= hess_poly_tolerance(x, w, r["eps"]), n


def test_four_array_cache_without_inplace_raises(pkg):
    t = [torch.zeros(2, dtype=torch.float64) for _ in range(4)]
    with pytest.raises(TypeError, match="inplace"):
        pkg.HessianCache(*t, "hcentral")
    with pytest.raises(TypeError, match="inplace"):
        pkg.HessianCache(*t)


def test_plan_create_checks_without_gpu(pkg):
    L = pkg._lib
    h = C.c_void_p()
    o = L.PlanOpts(fdtype=L.FDB_CENTRAL)
    assert L.lib().fdb_hessian_plan_create(C.byref(h), 3, C.byref(o)) == L.FDB_ERR_UNSUPPORTED   # hessians.jl:206
    assert L.lib().fdb_hessian_plan_create(C.byref(h), 3, None) == L.FDB_ERR_UNSUPPORTED
    o = L.PlanOpts(fdtype=L.FDB_HCENTRAL, world=2)
    assert L.lib().fdb_hessian_plan_create(C.byref(h), 3, C.byref(o)) == L.FDB_ERR_UNSUPPORTED
    o = L.PlanOpts(fdtype=L.FDB_HCENTRAL, use_graph=1)
    assert L.lib().fdb_hessian_plan_create(C.byref(h), 3, C.byref(o)) == L.FDB_ERR_UNSUPPORTED
    if L.lib().fdb_device_count() == 0:
        o = L.PlanOpts(fdtype=L.FDB_HCENTRAL)
        assert L.lib().fdb_hessian_plan_create(C.byref(h), 3, C.byref(o)) == L.FDB_ERR_NO_DEVICE
        assert h.value is None


# ------------------------------------------------------------------------------------------ GPU, through the C ABI
def _hess_plan(L, n, max_batch=0, scratch_bytes=0):
    h = C.c_void_p()
    o = L.PlanOpts(fdtype=L.FDB_HCENTRAL, device=0, max_batch=max_batch, scratch_bytes=scratch_bytes)
    L.check(L.lib().fdb_hessian_plan_create(C.byref(h), n, C.byref(o)))
    return h


def _poly_inputs(n, seed):
    rng = np.random.default_rng(seed)
    return rng.uniform(0.5, 1.5, n), rng.uniform(-1.0, 1.0, n)


@functools.lru_cache(maxsize=None)
def _poly_oracle(n, seed):
    from oracle_hessian import hessian_oracle
    x, w = _poly_inputs(n, seed)
    return hessian_oracle.hess_poly(x, w)


def _gpu_hessian(pkg, n, seed, max_batch, ldH=None, fill=0.0, relstep=None, absstep=None):
    L = pkg._lib
    dev = torch.device("cuda:0")
    x, w = _poly_inputs(n, seed)
    dx = torch.from_numpy(x).to(dev)
    dw = torch.from_numpy(w).to(dev)
    ld = n if ldH is None else ldH
    Hbuf = torch.full((max(n, 1) * max(ld, 1),), fill, dtype=torch.float64, device=dev)
    ctx = L.HessPolyCtx(n, dw.data_ptr(), 0)
    plan = _hess_plan(L, n, max_batch)
    try:
        x_before = dx.clone()
        st = L.lib().fdb_hessian(plan, C.cast(L.synth().fdbs_hess_poly, C.c_void_p), C.cast(C.pointer(ctx), C.c_void_p),
                                 dx.data_ptr(), Hbuf.data_ptr(), ld,
                                 L.STEP_DEFAULT if relstep is None else relstep,
                                 L.STEP_DEFAULT if absstep is None else absstep, None)
        L.check(st)
        torch.cuda.synchronize()
        eps = np.zeros(max(n, 1))
        L.check(L.lib().fdb_plan_get_eps(plan, eps.ctypes.data_as(C.POINTER(C.c_double)), len(eps), None))
        info, cnt = L.PlanInfo(), L.Counters()
        L.check(L.lib().fdb_plan_info(plan, C.byref(info)))
        L.check(L.lib().fdb_plan_counters(plan, C.byref(cnt)))
        assert torch.equal(dx.view(torch.int64), x_before.view(torch.int64)), "x was written"
    finally:
        L.lib().fdb_plan_destroy(plan)
    Hfull = Hbuf.cpu().numpy().reshape(max(n, 1), max(ld, 1)).T          # column-major (ld, n)
    return Hfull, eps[:n], info.as_dict(), cnt.as_dict(), ctx.calls


PARITY_CASES = [(n, b) for n in (0, 1, 2, 3, 31) for b in (1, 3, 4, 7, 0, 2 * n * n + 2)] + \
               [(257, b) for b in (1, 7, 0, 4096, 2 * 257 * 257 + 2)] + [(1024, 1000), (1024, 65536)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,max_batch", PARITY_CASES)
def test_gpu_bit_identical_to_oracle(pkg, n, max_batch):
    Hfull, eps, info, cnt, calls = _gpu_hessian(pkg, n, 11, max_batch)
    total = 2 * n * n + 1
    assert calls == total == info["fcalls_per_jacobian"] == cnt["f_points"]
    B = min(max(max_batch, 1), total)
    assert cnt["f_invocations"] == -(-total // B)
    if n == 0:
        return
    H = Hfull[:n, :n]
    ref = _poly_oracle(n, 11)
    assert np.array_equal(bits(eps), bits(ref["eps"]))
    assert np.array_equal(bits(H), bits(ref["H"])), f"n={n} B={max_batch}: H differs from the oracle"
    assert np.array_equal(bits(H), bits(H.T)), "H is not symmetric bit for bit"
    assert cnt["scatter_launches"] == 1


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 5, 33, 70])
def test_gpu_padding_rows_untouched(pkg, n):
    sentinel = -12345.678
    Hfull, eps, *_ = _gpu_hessian(pkg, n, 5, 16, ldH=n + 3, fill=sentinel)
    assert np.all(Hfull[n:, :] == sentinel)
    assert np.array_equal(bits(Hfull[:n, :n]), bits(_poly_oracle(n, 5)["H"]))


@pytest.mark.gpu
def test_gpu_steps_and_relstep_absstep(pkg, horc):
    n = 9
    for rs, ab in ((0.0, 1e-4), (1e-3, 0.0), (2e-4, 3e-5)):
        Hfull, eps, *_ = _gpu_hessian(pkg, n, 3, 5, relstep=rs, absstep=ab)
        x, w = _poly_inputs(n, 3)
        ref = horc.hess_poly(x, w, relstep=rs, absstep=ab)
        assert np.array_equal(bits(eps), bits(ref["eps"]))
        assert np.array_equal(bits(Hfull[:n, :n]), bits(ref["H"]))


@pytest.mark.gpu
def test_gpu_closed_form_synthetic(pkg):
    n = 257
    Hfull, eps, *_ = _gpu_hessian(pkg, n, 21, 8192)
    x, w = _poly_inputs(n, 21)
    assert np.max(np.abs(Hfull[:n, :n] - hess_poly_closed_form(x, w))) <= hess_poly_tolerance(x, w, eps)


@pytest.mark.gpu
def test_gpu_recorded_call_sequence(pkg):
    """A recording Python callback at n = 4 sees the reference's point sequence (hessians.jl:209-269)."""
    dev = torch.device("cuda:0")
    x = torch.tensor([0.7, -1.3, 2.0, 0.25], dtype=torch.float64, device=dev)
    f = random_scalar_fn(np.random.default_rng(3), 4)
    for batch in (1, 3, 64):
        seen = []

        def fr(v):
            seen.append(v.cpu().numpy().copy())
            return f(v.cpu().numpy())
        cache = pkg.HessianCache(x, max_batch=batch)
        H = pkg.finite_difference_hessian(fr, x, cache)
        Ht, steps, calls, pts = transcribed_hessian(f, x.cpu().numpy())
        assert len(seen) == calls == 33
        assert all(np.array_equal(bits(a), bits(np.array(b))) for a, b in zip(seen, pts))
        assert np.array_equal(bits(H.cpu().numpy()), bits(Ht))
        assert np.array_equal(bits(cache._last_plan.eps()), bits(steps))


def _kat_fns():
    def sincos(v):
        return torch.sin(v[0]) + torch.cos(v[1])
    sincos_b = lambda X: torch.sin(X[:, 0]) + torch.cos(X[:, 1])
    sincos_b.batched = True

    def sum_abs2(v):
        s = v[0] * v[0]
        for k in range(1, v.shape[-1]):
            s = s + v[k] * v[k]
        return s

    def sum_abs2_b(X):
        s = X[:, 0] * X[:, 0]
        for k in range(1, X.shape[1]):
            s = s + X[:, k] * X[:, k]
        return s
    sum_abs2_b.batched = True
    return (sincos, sincos_b), (sum_abs2, sum_abs2_b)


@pytest.mark.gpu
def test_gpu_known_answers_through_mirror(pkg):
    dev = torch.device("cuda:0")
    (sc, sc_b), (sa, sa_b) = _kat_fns()
    # finitedifftests.jl:561-576: cache-less, cached, immutable-branch cache, in-place and out-of-place forms
    x = torch.tensor(X_SINCOS, device=dev)
    H_ref = np.array([[-math.sin(X_SINCOS[0]), 0.0], [0.0, -math.cos(X_SINCOS[1])]])
    for f in (sc, sc_b):
        outs = [pkg.finite_difference_hessian(f, x), pkg.finite_difference_hessian(f, x, pkg.HessianCache(x)),
                pkg.finite_difference_hessian(f, x, pkg.HessianCache(x, "hcentral", False))]
        for cache in (None, pkg.HessianCache(x)):
            H = torch.empty(2, 2, dtype=torch.float64, device=dev)
            pkg.finite_difference_hessian_(H, f, x, cache)
            outs.append(H)
        for H in outs:
            assert err_func(H.cpu().numpy(), H_ref) < 1e-4
    # :593-598: sum(abs2)/2 at ones(2) ≈ I
    for f in (lambda v: sa(v) / 2, ):
        assert jl_isapprox(pkg.finite_difference_hessian(f, torch.ones(2, dtype=torch.float64, device=dev)).cpu(), np.eye(2))
    half_b = lambda X: sa_b(X) / 2
    half_b.batched = True
    assert jl_isapprox(pkg.finite_difference_hessian(half_b, torch.ones(2, dtype=torch.float64, device=dev)).cpu(), np.eye(2))
    # :608-614 (issue #185): exact, with the cache built from the same x and from another one
    x1 = torch.arange(1.0, 5.0, dtype=torch.float64, device=dev)
    x2 = torch.arange(5.0, 9.0, dtype=torch.float64, device=dev)
    for f in (sa, sa_b):
        for src in (x1, x2):
            H = pkg.finite_difference_hessian(f, x1, pkg.HessianCache(src))
            assert torch.equal(H.cpu(), torch.diag(torch.full((4,), 2.0, dtype=torch.float64)))
    # cache_reuse_tests.jl:130-139: a poisoned four-array cache
    h = lambda v: v[0] * v[0] + 2 * (v[1] * v[1])
    cache = pkg.HessianCache(*[torch.full((2,), 1e10, dtype=torch.float64, device=dev) for _ in range(4)], "hcentral", True)
    H = torch.zeros(2, 2, dtype=torch.float64, device=dev)
    pkg.finite_difference_hessian_(H, h, torch.tensor([1.0, 2.0], dtype=torch.float64, device=dev), cache)
    assert np.allclose(H.cpu().numpy(), [[2.0, 0.0], [0.0, 4.0]], rtol=0, atol=1e-3)
    # a row-major view is filled as well (H is symmetric bit for bit)
    xr = torch.tensor([0.3, -0.8, 1.1], dtype=torch.float64, device=dev)
    Hc = pkg.zeros_colmajor(3, 3)
    Hr = torch.zeros(3, 3, dtype=torch.float64, device=dev)
    f3 = lambda X: torch.sin(X[:, 0] * X[:, 1]) + X[:, 2] * X[:, 2] * X[:, 0]
    f3.batched = True
    pkg.finite_difference_hessian_(Hc, f3, xr)
    pkg.finite_difference_hessian_(Hr, f3, xr)
    assert torch.equal(Hc.contiguous().view(torch.int64), Hr.view(torch.int64))


@pytest.mark.gpu
def test_gpu_native_fn_through_mirror(pkg):
    L = pkg._lib
    n = 31
    x, w = _poly_inputs(n, 11)
    dev = torch.device("cuda:0")
    dx, dw = torch.from_numpy(x).to(dev), torch.from_numpy(w).to(dev)
    ctx = L.HessPolyCtx(n, dw.data_ptr(), 0)
    f = pkg.NativeFn(C.cast(L.synth().fdbs_hess_poly, C.c_void_p).value, ctx, max_batch=100)
    H = pkg.finite_difference_hessian(f, dx)
    torch.cuda.synchronize()
    assert np.array_equal(bits(H.cpu().numpy()), bits(_poly_oracle(n, 11)["H"]))
    assert ctx.calls == 2 * n * n + 1


@pytest.mark.gpu
def test_gpu_error_paths(pkg):
    L = pkg._lib
    lib = L.lib()
    dev = torch.device("cuda:0")
    n = 4
    x = torch.ones(n, dtype=torch.float64, device=dev)
    H = torch.zeros(n * n, dtype=torch.float64, device=dev)
    h = C.c_void_p()
    for fd in (L.FDB_FORWARD, L.FDB_CENTRAL, L.FDB_COMPLEX, 7):
        o = L.PlanOpts(fdtype=fd)
        assert lib.fdb_hessian_plan_create(C.byref(h), n, C.byref(o)) == L.FDB_ERR_UNSUPPORTED
    assert lib.fdb_hessian_plan_create(C.byref(h), n, C.byref(L.PlanOpts(fdtype=L.FDB_HCENTRAL, world=2))) == L.FDB_ERR_UNSUPPORTED
    assert lib.fdb_hessian_plan_create(C.byref(h), n, C.byref(L.PlanOpts(fdtype=L.FDB_HCENTRAL, use_graph=1))) == L.FDB_ERR_UNSUPPORTED
    # the Hessian plan kind and the others do not mix
    hp = _hess_plan(L, n, 8)
    dp = C.c_void_p()
    L.check(lib.fdb_plan_create_dense(C.byref(dp), n, n, n, C.byref(L.PlanOpts(fdtype=L.FDB_CENTRAL))))
    jp = C.c_void_p()
    L.check(lib.fdb_jvp_plan_create(C.byref(jp), n, n, C.byref(L.PlanOpts())))
    try:
        tctx = L.TridiagCtx(n, 0)
        ctx = C.cast(C.pointer(tctx), C.c_void_p)
        tri = C.cast(L.synth().fdbs_tridiag, C.c_void_p)
        fail = C.cast(L.synth().fdbs_fail, C.c_void_p)
        nan = L.STEP_DEFAULT
        assert lib.fdb_jacobian(hp, tri, ctx, x.data_ptr(), H.data_ptr(), None, None, nan, nan, 1.0, None) == L.FDB_ERR_INVALID
        assert b"fdb_hessian" in lib.fdb_last_error()
        assert lib.fdb_jvp(hp, tri, ctx, H.data_ptr(), x.data_ptr(), x.data_ptr(), None, None, None, nan, nan, 1.0, None) == L.FDB_ERR_INVALID
        assert lib.fdb_color_eps(hp, x.data_ptr(), nan, nan, 1.0, None, None) == L.FDB_ERR_INVALID
        assert lib.fdb_plan_set_external_eps(hp, x.data_ptr()) == L.FDB_ERR_INVALID
        for other in (dp, jp):
            assert lib.fdb_hessian(other, fail, None, x.data_ptr(), H.data_ptr(), n, nan, nan, None) == L.FDB_ERR_INVALID
        assert lib.fdb_hessian(hp, fail, None, x.data_ptr(), H.data_ptr(), n - 1, nan, nan, None) == L.FDB_ERR_INVALID
        assert lib.fdb_hessian(hp, fail, None, x.data_ptr(), H.data_ptr(), n, nan, nan, None) == L.FDB_ERR_CALLBACK
        # timing covers the combine launch
        L.check(lib.fdb_plan_enable_timing(hp, 1))
        wd = torch.zeros(n, dtype=torch.float64, device=dev)
        pctx = L.HessPolyCtx(n, wd.data_ptr(), 0)
        L.check(lib.fdb_hessian(hp, C.cast(L.synth().fdbs_hess_poly, C.c_void_p), C.cast(C.pointer(pctx), C.c_void_p),
                                x.data_ptr(), H.data_ptr(), n, nan, nan, None))
        ms, cnt = C.c_double(), C.c_int64()
        L.check(lib.fdb_plan_read_timing(hp, C.byref(ms), C.byref(cnt)))
        assert cnt.value == 1 and ms.value >= 0.0
        info = L.PlanInfo()
        L.check(lib.fdb_plan_info(hp, C.byref(info)))
        assert info.fcalls_per_jacobian == 2 * n * n + 1 and info.n_colors == n and info.m == 1
        assert info.moved_bytes_scatter == 8 * (2 * n * n + 1) + 8 * n + 8 * n * n
    finally:
        for p in (hp, dp, jp):
            lib.fdb_plan_destroy(p)
    # a Python exception in f propagates through the mirror
    def boom(v):
        raise KeyError("from f")
    with pytest.raises(KeyError, match="from f"):
        pkg.finite_difference_hessian(boom, x)
    with pytest.raises(AssertionError):
        pkg.finite_difference_hessian(lambda v: v.sum(), x, pkg.HessianCache(x, "central"))
