"""Golden vectors of the reference's C routine _grad_X (GPy/kern/src/stationary_utils.c), for
tests/test_oracle.py::test_grad_X_matches_reference_C_routine.

    python tests/golden/make_golden_grad_x.py        (writes tests/golden/grad_x_stationary_utils.npz)

The routine is grad[n, d] = sum_m tmp[n, m] * (X[n, d] - X2[m, d]), summed in m order from 0.0, one product and one
add per term (built with gcc -O3 for baseline x86-64: no FMA contraction).  With the reference's sources at hand,
`make -C oracle` builds the routine itself and the test checks it against these vectors too.
"""
import os

import numpy as np


def grad_x_c_order(X, X2, tmp):
    N, D = X.shape
    M = X2.shape[0]
    grad = np.zeros((N, D))
    for d in range(D):
        for n in range(N):
            acc = 0.0
            for m in range(M):
                acc += float(tmp[n, m]) * (float(X[n, d]) - float(X2[m, d]))
            grad[n, d] = acc
    return grad


if __name__ == "__main__":
    rng = np.random.default_rng(2)
    N, D, M = 13, 5, 21
    X, X2, tmp = rng.standard_normal((N, D)), rng.standard_normal((M, D)), rng.standard_normal((N, M))
    out = os.path.join(os.path.dirname(os.path.abspath(__file__)), "grad_x_stationary_utils.npz")
    np.savez(out, X=X, X2=X2, tmp=tmp, grad=grad_x_c_order(X, X2, tmp))
    print(out)
