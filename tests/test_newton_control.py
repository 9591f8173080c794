"""The per-program control of the interior-point loop that NewtonDriver::Run and BatchProgram::Maximize share
(NewtonControl, conex_b200/csrc/host/newton_control.cc), compiled for the host with a C shim
(tests/emul/emul_newton_control.cc). Scripted inputs drive it and `Model`, a Python restatement of the reference's
Solve() (cone_program.cc:166-214, 312-530), side by side; every state the control reports must match bit for bit.
The scripts reach the branches the GPU workloads rarely reach: each step of the mu fallback chain, the clamp, both
warm-start aborts, the infeasibility flags at their thresholds and max_iters_reached.
"""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRCS = [os.path.join(ROOT, "tests", "emul", "emul_newton_control.cc"),
        os.path.join(ROOT, "conex_b200", "csrc", "host", "newton_control.cc"),
        os.path.join(ROOT, "conex_b200", "csrc", "host", "divergence.cc")]
SO = os.path.join(ROOT, "tests", "emul", "_build", "libemul_newton_control.so")
INCLUDE = os.path.join(ROOT, "include", "conex_b200")
CUDA_INCLUDE = "/usr/local/cuda/include"  # cuda_runtime_api.h, for the declarations cone_program.h pulls in
D, I = C.c_double, C.c_int
DP = C.POINTER(C.c_double)


@pytest.fixture(scope="module")
def lib():
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    headers = [os.path.join(INCLUDE, f) for f in os.listdir(INCLUDE)]
    newest = max(os.path.getmtime(f) for f in SRCS + headers)
    if not os.path.exists(SO) or os.path.getmtime(SO) < newest:
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-I", INCLUDE, "-I", CUDA_INCLUDE,
                               "-o", SO] + SRCS)
    L = C.CDLL(SO)
    L.nc_fields.restype = C.c_char_p
    L.nc_create.restype = C.c_void_p
    L.nc_create.argtypes = [DP, I, DP, I, D, D]
    L.nc_begin.argtypes = [C.c_void_p, I]
    L.nc_rescale.argtypes = [C.c_void_p, D]
    L.nc_choose_k.argtypes = [C.c_void_p, I, DP]
    L.nc_step.argtypes = [C.c_void_p, D, D, DP]
    L.nc_end.argtypes = [C.c_void_p, D, D, D, D]
    L.nc_finish.argtypes = [C.c_void_p, DP, I, C.POINTER(I)]
    L.nc_state.argtypes = [C.c_void_p, DP, C.POINTER(I)]
    for name in ["nc_destroy", "nc_needs_aqc_norm", "nc_restart_on_factorization_failure", "nc_update_mu",
                 "nc_needs_eigenvalues"]:
        getattr(L, name).argtypes = [C.c_void_p]
    L.nc_scale_dual_variable.argtypes = [I, I, D, D, DP, I]
    L.nc_divergence_upper_bound_inverse.argtypes = [D] * 6
    L.nc_divergence_upper_bound_inverse.restype = D
    return L


def darr(x):
    return np.ascontiguousarray(x, dtype=np.float64)


def ptr(a):
    return a.ctypes.data_as(DP)


def default_config(L):
    fields = L.nc_fields().decode().rstrip(",").split(",")
    v = darr(np.zeros(len(fields)))
    L.nc_default_config(ptr(v))
    return dict(zip(fields, v.tolist()))


class Model:
    """The reference's per-program loop control, line by line."""

    def __init__(self, cfg, rank, b, b_scaling, c_scaling, div_inverse):
        self.cfg, self.rank, self.div_inverse = cfg, rank, div_inverse
        self.warm = cfg["initialization_mode"] != 0
        self.initial_centering_steps = int(cfg["initial_centering_steps_warmstart" if self.warm
                                               else "initial_centering_steps_coldstart"])
        self.k, self.kmax, self.cx, self.by, self.kkt_error = 0.0, cfg["inv_sqrt_mu_max"], 1.0, -1.0, 0.0
        self.b_scaling, self.c_scaling, self.d_2, self.d_inf = b_scaling, c_scaling, 0.0, 0.0
        self.b_norm = 0.0
        for v in b:
            self.b_norm += v * v
        self.b_norm = math.sqrt(self.b_norm)
        self.centering_steps = self.num_iter = 0
        self.done = self.failed = self.restarted = self.warmstart_aborted = False
        self.max_iters_reached = True
        self.i = -1
        self.branch = None  # the step of the mu rule the last new k came from

    def begin(self, i):  # cone_program.cc:312-336
        if self.done:
            return False
        c = self.cfg
        self.i, self.restarted = i, False
        self.initial_centering = i < self.initial_centering_steps
        self.final_centering = (self.k >= self.kmax or self.kkt_error > c["kkt_error_tolerance"]
                                or i >= c["max_iterations"] - c["final_centering_steps"])
        self.update_mu = i == 0 or not (self.initial_centering or self.final_centering) or self.warmstart_aborted
        self.warmstart_aborted = False
        if self.final_centering and self.centering_steps >= c["final_centering_steps"]:
            self.max_iters_reached = i >= c["max_iterations"] - 1
            self.done = True
            return False
        return True

    def rescale(self, aqc2):  # cone_program.cc:343-357
        if self.i != 0 or not self.cfg["enable_rescaling"]:
            return
        if not self.warm:
            self.b_scaling = 1.0 / (1 + self.b_norm)
            self.c_scaling = 1.0 / (1 + math.sqrt(aqc2))
        mu_target = (1.0 / (self.kmax * self.kmax)) * (self.b_scaling * self.c_scaling)
        self.kmax = 1.0 / math.sqrt(mu_target)

    def factorization_failed(self):  # cone_program.cc:360-371
        if self.i == 0 and self.warm:
            self.restarted = self.warmstart_aborted = True
            return True
        self.done = self.failed = True
        return False

    def mu_from_eigenvalues(self, lmin, lmax, frob, trace):  # cone_program.cc:166-214
        r = self.rank
        k = self.div_inverse(self.cfg["divergence_upper_bound"] * r, lmin, lmax, frob, trace, float(r))
        self.branch = "divergence bound"
        if k == -1:
            k = 2.0 / (lmin + lmax) if lmin > 0 else -1
            self.branch = "lambda_min > 0"
        if k < 0 and trace > 1e-12:
            kstar = trace / frob
            norm_bound = 1.5 * (frob * kstar * kstar - 2 * trace * kstar + r)
            norm_bound = min(norm_bound, r * .7)
            qa, qb, qc = frob, -2 * trace, r - norm_bound
            disc = qb * qb - 4 * qa * qc
            k = kstar if disc < 0 else (-qb + math.sqrt(disc)) / (2 * qa)
            self.branch = "quadratic, disc < 0" if disc < 0 else "quadratic, disc >= 0"
        return k

    def choose_k(self, cones):  # cone_program.cc:373-399
        if self.update_mu:
            cand = self.k if self.cfg["enable_line_search"] else -1
            if cand < 0:
                lmin = min([30000.0] + [c[0] for c in cones])
                lmax = max([-30000.0] + [c[1] for c in cones])
                frob = trace = 0.0
                for c in cones:
                    frob += c[2]
                    trace += c[3]
                cand = self.mu_from_eigenvalues(lmin, lmax, frob, trace)
            if cand > 0:
                self.k = cand
            else:
                self.k, self.branch = 0.5 * self.k, "halving"
        elif not self.initial_centering:
            self.centering_steps += 1
        self.k = max(min(self.k, self.kmax), math.sqrt(1.0 / (1e-15 + self.cfg["maximum_mu"])))

    def step(self, ninf, nsq):  # cone_program.cc:418-436
        self.d_2, self.d_inf = math.sqrt(abs(nsq)), abs(ninf)
        step_size = min(1.0, 2.0 / (ninf * ninf))
        if self.i == 0 and self.warm and ninf >= self.cfg["warmstart_abort_threshold"]:
            self.warmstart_aborted = True
            return False, step_size
        return True, step_size

    def end(self, b_dot_y, aqc_dot_y, w_dot_c, c_dot_qc):  # cone_program.cc:441-478
        k = self.k
        self.by = b_dot_y / (k * self.c_scaling)
        self.cx = (2 * w_dot_c + aqc_dot_y - k * c_dot_qc * self.c_scaling) / (k * self.b_scaling)
        mu = (1.0 / k) * (1.0 / k)
        s_dot_x = mu * (self.rank - self.d_2 * self.d_2) / (self.b_scaling * self.c_scaling)
        self.kkt_error = abs(self.cx - self.by - s_dot_x) / s_dot_x
        self.num_iter = self.i + 1
        if (self.final_centering or k >= self.kmax) and self.d_inf <= self.cfg["final_centering_tolerance"]:
            self.max_iters_reached, self.done = False, True
            return True
        return False

    def finish(self, y):  # cone_program.cc:486-530
        status = dict(solved=0, num_iterations=self.num_iter, primal_infeasible=0, dual_infeasible=0)
        if self.failed:
            return status, y
        if (1.0 / self.k) * (1.0 / self.k) > self.cfg["infeasibility_threshold"]:
            status["primal_infeasible"] = int(self.cx * self.k <= -.5)
            status["dual_infeasible"] = int(self.by * self.k >= .5)
        else:
            status["solved"] = 1
        if status["solved"]:
            y = [v / self.k / self.c_scaling for v in y]
            if self.max_iters_reached:
                status["solved"] = 0
        return status, y


class Pair:
    """One NewtonControl and one Model, driven by the same calls; every call compares their states."""

    def __init__(self, L, rank=10, b=(0.3, -1.2, 2.0), b_scaling=1.0, c_scaling=1.0, **overrides):
        self.L = L
        self.cfg = default_config(L)
        for key, v in overrides.items():
            assert key in self.cfg, key
            self.cfg[key] = float(v)
        v = darr(list(self.cfg.values()))
        bb = darr(b)
        self.h = L.nc_create(ptr(v), rank, ptr(bb), len(b), b_scaling, c_scaling)
        self.m = Model(self.cfg, rank, list(b), b_scaling, c_scaling, L.nc_divergence_upper_bound_inverse)

    def __del__(self):
        self.L.nc_destroy(self.h)

    def state(self):
        d, f = darr(np.zeros(9)), (I * 3)()
        self.L.nc_state(self.h, ptr(d), f)
        return d, list(f)

    def check(self):
        d, f = self.state()
        m = self.m
        mu = (1.0 / m.k) * (1.0 / m.k) / (m.c_scaling * m.b_scaling) if m.k else None  # what the log shows
        want = [m.k, mu, m.b_scaling, m.c_scaling, m.by, m.cx, m.kkt_error, m.d_2, m.d_inf]
        for j, (got, w) in enumerate(zip(d.tolist(), want)):
            if w is not None:
                assert got == w, (j, got, w)
        assert f == [m.num_iter, int(not m.done and not m.restarted), int(m.failed)]

    def begin(self, i):
        got = bool(self.L.nc_begin(self.h, i))
        assert got == self.m.begin(i)
        if got:
            assert bool(self.L.nc_update_mu(self.h)) == self.m.update_mu
        self.check()
        return got

    def rescale(self, aqc2=4.0):
        assert bool(self.L.nc_needs_aqc_norm(self.h)) == (self.m.i == 0 and bool(self.cfg["enable_rescaling"])
                                                          and not self.m.warm)
        self.L.nc_rescale(self.h, aqc2)
        self.m.rescale(aqc2)
        self.check()

    def factorization_failed(self):
        got = bool(self.L.nc_restart_on_factorization_failure(self.h))
        assert got == self.m.factorization_failed()
        self.check()
        return got

    def choose_k(self, cones):
        cones = [tuple(float(x) for x in c) for c in cones]
        needs = self.m.update_mu and (self.m.k if self.cfg["enable_line_search"] else -1) < 0
        assert bool(self.L.nc_needs_eigenvalues(self.h)) == needs
        a = darr(np.array(cones).reshape(-1))
        self.m.branch = None
        self.L.nc_choose_k(self.h, len(cones), ptr(a))
        self.m.choose_k(cones)
        self.check()
        return self.m.branch

    def step(self, ninf, nsq=0.25):
        s = darr([0.0])
        got = bool(self.L.nc_step(self.h, ninf, nsq, ptr(s)))
        take, size = self.m.step(ninf, nsq)
        assert got == take and s[0] == size
        self.check()
        return got

    def end(self, dots=(0.4, 0.3, 0.2, 0.1)):
        got = bool(self.L.nc_end(self.h, *dots))
        assert got == self.m.end(*dots)
        self.check()
        return got

    def finish(self, y=(1.0, -2.0, 3.5)):
        a, st = darr(y), (I * 4)()
        self.L.nc_finish(self.h, ptr(a), len(y), st)
        want, wy = self.m.finish(list(y))
        assert list(st) == [want["solved"], want["num_iterations"], want["primal_infeasible"],
                            want["dual_infeasible"]]
        assert a.tolist() == wy
        return want, a.tolist()

    def iteration(self, i, cones, ninf=0.5, dots=(0.4, 0.3, 0.2, 0.1)):
        """One Newton step that factors; returns whether the loop stopped (at Begin or converged)."""
        if not self.begin(i):
            return True
        self.rescale()
        self.choose_k(cones)
        self.step(ninf)
        return self.end(dots)


# per-cone summaries {lambda_min, lambda_max, |.|_F^2, trace} near the central path
CENTRAL = [(0.8, 1.3, 4.1, 4.0), (0.9, 1.1, 2.0, 2.0), (0.95, 1.05, 4.0, 4.0)]


def test_mu_rule_each_fallback(lib):
    """Random summaries until every step of the chain has been taken: the divergence bound, 2 / (lambda_min +
    lambda_max), the norm-bound quadratic with a negative and with a non-negative discriminant, and the halving of k
    (second iteration, so that k > 0 is halved)."""
    rng = np.random.default_rng(5)
    seen = {}
    for trial in range(4000):
        if len(seen) == 5:
            break
        rank = int(rng.integers(1, 40))
        p = Pair(lib, rank=rank, enable_rescaling=0, inv_sqrt_mu_max=1e6, maximum_mu=1e12,
                 divergence_upper_bound=float(rng.choice([1.0, 1e-3, 1e-9])))
        assert p.iteration(0, CENTRAL, ninf=5.0) is False
        assert p.begin(1) and p.m.update_mu
        p.rescale()
        n = int(rng.integers(1, 5))
        lam = rng.uniform(-2.0, 3.0, (n, 2))
        lam.sort(axis=1)
        scale = rng.choice([1.0, 0.0])  # zero traces and norms leave only the halving
        frob = rng.uniform(0, 5, n) * scale
        trace = rng.uniform(-3, 5, n) * scale
        if rng.random() < 0.3:  # negative traces: the quadratic is skipped (trace <= 1e-12)
            trace = -np.abs(trace)
        cones = [(lam[j, 0], lam[j, 1], frob[j], trace[j]) for j in range(n)]
        branch = p.choose_k(cones)
        seen.setdefault(branch, trial)
    assert set(seen) == {"divergence bound", "lambda_min > 0", "quadratic, disc < 0", "quadratic, disc >= 0",
                         "halving"}, seen


def test_clamp_to_kmax_and_to_maximum_mu(lib):
    """k is clamped to [sqrt(1 / (1e-15 + maximum_mu)), kmax]; kmax is the rescaled inv_sqrt_mu_max."""
    p = Pair(lib, inv_sqrt_mu_max=0.5, enable_rescaling=0)
    p.begin(0)
    p.choose_k(CENTRAL)
    assert p.m.k == 0.5
    p = Pair(lib, maximum_mu=1e-4)
    p.begin(0)
    p.rescale(9.0)
    p.choose_k([(-1.0, 1.0, 0.0, 0.0)])  # halving of k = 0
    assert p.m.k == math.sqrt(1.0 / (1e-15 + 1e-4))
    p = Pair(lib, inv_sqrt_mu_max=0.3)
    p.begin(0)
    p.rescale(9.0)
    assert p.m.kmax != 0.3 and p.m.b_scaling == 1.0 / (1 + p.m.b_norm) and p.m.c_scaling == 0.25
    p.choose_k(CENTRAL)
    assert p.m.k == p.m.kmax


@pytest.mark.parametrize("warm", [False, True])
def test_factorization_failure_restarts_only_a_warm_start(lib, warm):
    """The first factorisation of a warm start may fail: the iteration counts neither an iteration nor a centering
    step and the next one chooses a new mu. Any other failure ends the solve unsolved with y untouched."""
    p = Pair(lib, rank=6, initialization_mode=int(warm), b_scaling=0.25, c_scaling=0.5, kkt_error_tolerance=-1,
             final_centering_steps=1, max_iterations=10)
    assert p.begin(0)
    p.rescale()
    assert p.m.b_scaling == (0.25 if warm else 1.0 / (1 + p.m.b_norm))
    assert p.factorization_failed() is warm
    if not warm:
        assert not p.begin(1)
        status, y = p.finish()
        assert status["solved"] == 0 and status["num_iterations"] == 0 and y == [1.0, -2.0, 3.5]
        return
    assert p.m.num_iter == 0 and p.m.centering_steps == 0
    # final centering throughout (kkt_error > -1): iteration 1 updates mu because of the restart, iteration 2 is
    # the one centering step, after which Begin stops
    assert p.begin(1) and p.m.update_mu
    p.choose_k(CENTRAL)
    p.step(5.0)
    p.end()
    assert p.m.centering_steps == 0
    assert p.iteration(2, CENTRAL, ninf=5.0) is False and p.m.centering_steps == 1
    assert not p.begin(3)
    status, _ = p.finish()
    assert status["num_iterations"] == 3  # the index of the last completed iteration + 1, as in the reference


def test_warm_start_first_step_too_large(lib):
    """d_inf >= warmstart_abort_threshold on the first step of a warm start: the cones are reset instead of stepped,
    the iteration is still counted, and the next iteration chooses a new mu. Later steps are never aborted."""
    for ninf, aborts in [(2.0, True), (np.nextafter(2.0, 0), False)]:
        p = Pair(lib, initialization_mode=1, initial_centering_steps_warmstart=3, c_scaling=0.5)
        assert p.begin(0)
        p.rescale()
        p.choose_k(CENTRAL)
        assert p.step(ninf) is (not aborts)
        p.end()
        assert p.m.num_iter == 1
        assert p.begin(1) and p.m.update_mu is aborts  # initial centering otherwise
        p.rescale()
        p.choose_k(CENTRAL)
        assert p.step(100.0)


@pytest.mark.parametrize("threshold", [1.0, 4.0])
def test_infeasibility_flags_at_their_thresholds(lib, threshold):
    """k = 1/2, scalings 1: mu_final = 4, cx k and by k exact. mu_final > infeasibility_threshold reports the
    flags cx k <= -.5 and by k >= .5, otherwise the program is solved."""
    below = np.nextafter(0.5, 0)
    for aqc, bdy in [(-0.5, 0.5), (-below, below), (-0.5, below), (-below, 0.5)]:
        p = Pair(lib, inv_sqrt_mu_max=0.5, enable_rescaling=0, infeasibility_threshold=threshold)
        p.iteration(0, CENTRAL, ninf=0.001, dots=(bdy, aqc, 0.0, 0.0))
        assert p.m.k == 0.5 and p.m.done
        status, y = p.finish()
        if threshold == 4.0:
            assert status["solved"] == 1 and status["primal_infeasible"] == status["dual_infeasible"] == 0
            assert y == [2.0, -4.0, 7.0]
        else:
            assert status["solved"] == 0 and y == [1.0, -2.0, 3.5]
            assert status["primal_infeasible"] == int(aqc == -0.5)
            assert status["dual_infeasible"] == int(bdy == 0.5)


def test_max_iterations_reached_is_unsolved(lib):
    """A solve that reaches max_iterations without converging is unsolved although y is rescaled; one that stops at
    Begin on its last iteration too; one that converges is solved."""
    for max_iterations, ninf, solved in [(3, 0.5, 0), (3, 0.001, 1)]:
        p = Pair(lib, max_iterations=max_iterations, final_centering_steps=1)
        stopped = False
        for i in range(max_iterations):
            if p.iteration(i, CENTRAL, ninf=ninf):
                stopped = True
                break
        assert stopped is bool(solved)
        status, y = p.finish()
        assert status["solved"] == solved and y != [1.0, -2.0, 3.5]
    # the final centering step is used up before the last iteration: Begin stops at i = max_iterations - 1
    p = Pair(lib, max_iterations=3, final_centering_steps=1, kkt_error_tolerance=-1)
    assert not p.iteration(0, CENTRAL) and not p.iteration(1, CENTRAL)
    assert not p.begin(2) and p.m.max_iters_reached
    assert p.finish()[0]["solved"] == 0


def test_dual_variable_scale(lib):
    """W / (k b_scaling) after a solve with iterations that is not primal infeasible; W otherwise."""
    for n_iter, infeasible, scaled in [(3, 0, True), (0, 0, False), (3, 1, False)]:
        w = darr([1.0, -3.0, 0.7])
        lib.nc_scale_dual_variable(n_iter, infeasible, 0.3, 7.0, ptr(w), 3)
        scale = 0.3 * 7.0
        assert w.tolist() == ([1.0 / scale, -3.0 / scale, 0.7 / scale] if scaled else [1.0, -3.0, 0.7])
