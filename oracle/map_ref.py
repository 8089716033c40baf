"""CPU restatement of the synthesis-setting MAP problem the samplers' drift is the gradient flow of, and of FISTA (Beck &
Teboulle, SIAM J. Imaging Sci. 2009) on it.  TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

    F(x) = 1/2 (Phi Psi x - d)^dagger IC (Phi Psi x - d) + mu sum_i w_i |x_i|

with gradg(x) = Psi^dagger Phi^dagger IC (Phi Psi x - d) (``pxmcmc_ref.ForwardOperator.calc_gradg`` of the
predictions) and the prox of t mu sum w |x| the soft threshold at (t / lmda) T, T = lmda mu w (``pxmcmc_ref.L1``).
Kept apart from ``pxmcmc_ref``, which stays pinned to the reference's fixtures.
"""
import copy

import numpy as np

from .pxmcmc_ref import myula_step, soft


def gradg(fwd, X):
    return fwd.calc_gradg(fwd.forward(X))


def objective(fwd, prior, mu, X):
    """F(x): 1/2 the reference's L2 (vdot(d, IC d), real for a real positive IC) + mu prior(x)"""
    diff = fwd.data - fwd.forward(X)
    return 0.5 * np.vdot(diff, fwd.invcov * diff).real + mu * prior.prior(X)


def dense_operator(fwd):
    """the matrix of Psi^dagger Phi^dagger IC Phi Psi (the linear part of gradg), assembled column by column from the
    operator with its data set to zero"""
    op = copy.copy(fwd)
    op.data = np.zeros_like(np.asarray(fwd.data))
    n = fwd.nparams
    M = np.empty((n, n), dtype=complex)
    e = np.zeros(n, dtype=complex)
    for i in range(n):
        e[i] = 1.0
        M[:, i] = gradg(op, e)
        e[i] = 0.0
    return M


def fista(fwd, prior, lmda, t, X0, niter):
    """the iterates x_1 .. x_niter of FISTA from x_0 = y_0 = X0 with step t and threshold (t / lmda) T:
    x_{k+1} = soft(y_k - t gradg(y_k), (t / lmda) T), y_{k+1} = x_{k+1} + (tau_k - 1)/tau_{k+1} (x_{k+1} - x_k),
    tau_0 = 1, tau_{k+1} = (1 + sqrt(1 + 4 tau_k^2)) / 2"""
    x = np.asarray(X0, dtype=complex)
    y, tau, out = x.copy(), 1.0, []
    T = (t / lmda) * np.asarray(prior.T)
    for _ in range(niter):
        xn = soft(y - t * gradg(fwd, y), T)
        tau_n = (1.0 + np.sqrt(1.0 + 4.0 * tau * tau)) / 2.0
        y = xn + ((tau - 1.0) / tau_n) * (xn - x)
        x, tau = xn, tau_n
        out.append(x)
    return out


def ista(fwd, prior, lmda, t, X0, niter):
    """niter plain proximal-gradient steps x <- soft(x - t gradg(x), (t / lmda) T)"""
    x = np.asarray(X0, dtype=complex)
    T = (t / lmda) * np.asarray(prior.T)
    for _ in range(niter):
        x = soft(x - t * gradg(fwd, x), T)
    return x


def fixed_point_residual(fwd, prior, lmda, t, X):
    """|x - soft(x - t gradg(x), (t / lmda) T)| / |x|: zero exactly at a minimiser of F"""
    r = X - soft(X - t * gradg(fwd, X), (t / lmda) * np.asarray(prior.T))
    return np.linalg.norm(r) / np.linalg.norm(X)


def myula_factor(a, lmda, delta, T=1e300):
    """R of one MYULA step (``pxmcmc_ref.myula_step``, no noise) on the scalar target with gradg(x) = a x and the prior
    prox soft(x, T): x' = R x.  Where the threshold zeroes x (the default T) the Moreau-Yosida term is x / lmda and
    R = 1 - delta (a + 1 / lmda); with T = 0 it vanishes and R = 1 - delta a"""
    x = 1.0
    return myula_step(x, soft(np.array([x]), T)[0], a * x, delta, lmda, 0.0) / x
