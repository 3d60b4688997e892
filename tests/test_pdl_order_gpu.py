"""Results under overlapped launches. Consecutive knot-kernel launches on one stream may overlap (programmatic
dependent launch): the warp-specialised kernel loads and computes its first tiles before the previous launch has
completed, and waits only before its first global store. Every output of a sequence of launches enqueued back to back
must be bit-identical to the same launch made alone between two device synchronisations.

What these tests can see: a store that is missing (outputs are set to NaN in stream order first), and inputs read
too early when a copy or a torch kernel changes them inside the stream between two launches. Through the public API
two launches that write the same output array also compute the same values, so a store issued before the previous
launch has completed (a write-after-write race) would leave the same bits and is not observable here.
Cartpole stages its outputs in two buffers per compute warp, acrobot (larger tiles) in one."""
import numpy as np
import pytest

import dto_b200 as D
from dto_b200.evaluator import A_C, A_G, A_H, A_J, A_Z, K_CONSTRAINT, K_GRADIENT, K_JAC_HESS
from examples import models as M
from util import make_inputs

pytestmark = pytest.mark.gpu

B = 4096


def _batches(name, kw, config, count, stream):
    """`count` batches of one shape with distinct seeded inputs, all enqueueing on `stream`"""
    model = M.BUILDERS[name](D, **kw)
    n0 = D.solver_from(model, batch=B, devices=[0]).nlp
    nl = [n0] + [n0.new_batch() for _ in range(count - 1)]
    for i, n in enumerate(nl):
        z, lam, sigma, w = make_inputs(name, model, n.num_variables, n.num_constraint, n.num_parameter, B, config, i)
        if n.num_parameter:
            n.set_parameters(w)
        n.set_x(z)
        n.set_duals(sigma, lam)
        n.set_stream(stream.cuda_stream)
    return nl


def _view(n, array, width):
    import torch
    from dto_b200 import sqp
    return torch.as_tensor(sqp._CudaArray(n.device_pointer(array, 0), (n.batch, width)), device=torch.device("cuda", 0))


def _outputs(n, kernel_id):
    return {K_GRADIENT: [(A_G, n.num_variables)], K_CONSTRAINT: [(A_C, n.num_constraint)],
            K_JAC_HESS: [(A_J, n.num_jacobian), (A_H, n.num_hessian)]}[kernel_id]


def _alone(n, kernel_id):
    """the outputs of one launch with nothing else on the device before or after it"""
    import torch
    torch.cuda.synchronize()
    n.launch(kernel_id)
    torch.cuda.synchronize()
    return [_view(n, a, w).clone() for a, w in _outputs(n, kernel_id)]


def _poison(n, kernel_id, stream):
    """NaN into the launch's outputs, in stream order: a store that does not happen shows"""
    import torch
    with torch.cuda.stream(stream):
        for a, w in _outputs(n, kernel_id):
            _view(n, a, w).fill_(float("nan"))


def _same_bits(got, ref, what):
    import torch
    for g, r in zip(got, ref):
        assert torch.equal(g.view(torch.int64), r.view(torch.int64)), what


def _close(nl):
    for n in nl:
        n.close()


@pytest.mark.parametrize("name,kw,config", [("cartpole", dict(T=101), 2), ("acrobot", dict(T=101), 3)], ids=["cartpole", "acrobot"])
def test_back_to_back_rotating_sets(name, kw, config):
    """the benchmark's pattern: 33 fused Jacobian+Hessian launches over 3 rotating batches, no synchronisation between"""
    import torch
    st = torch.cuda.Stream()
    nl = _batches(name, kw, config, 3, st)
    ref = [_alone(n, K_JAC_HESS) for n in nl]
    for n in nl:
        _poison(n, K_JAC_HESS, st)
    with torch.cuda.stream(st):
        for i in range(33):
            nl[i % 3].launch(K_JAC_HESS)
    torch.cuda.synchronize()
    for i, n in enumerate(nl):
        _same_bits([_view(n, a, w) for a, w in _outputs(n, K_JAC_HESS)], ref[i], f"{name} set {i}")
    _close(nl)


def test_inputs_changed_in_stream_between_launches():
    """a torch kernel rewrites z in place between two launches on the same stream; then set_x between two launches"""
    import torch
    st = torch.cuda.Stream()
    (n,) = _batches("cartpole", dict(T=101), 2, 1, st)
    z = _view(n, A_Z, n.num_variables)
    dz = torch.as_tensor(np.random.default_rng(5).normal(0, 0.1, (B, n.num_variables)), device=z.device)
    with torch.cuda.stream(st):
        n.launch(K_JAC_HESS)
        first = [_view(n, a, w).clone() for a, w in _outputs(n, K_JAC_HESS)]
        z.add_(dz)
        n.launch(K_JAC_HESS)
        second = [_view(n, a, w).clone() for a, w in _outputs(n, K_JAC_HESS)]
    torch.cuda.synchronize()
    assert not torch.equal(first[0], second[0])
    _poison(n, K_JAC_HESS, st)
    _same_bits(second, _alone(n, K_JAC_HESS), "after the in-stream change of z")

    z2 = make_inputs("cartpole", M.BUILDERS["cartpole"](D, T=101), n.num_variables, n.num_constraint, n.num_parameter, B, 2, 7)[0]
    with torch.cuda.stream(st):
        n.launch(K_JAC_HESS)
    n.set_x(z2)
    with torch.cuda.stream(st):
        n.launch(K_JAC_HESS)
        got = [_view(n, a, w).clone() for a, w in _outputs(n, K_JAC_HESS)]
    torch.cuda.synchronize()
    assert not torch.equal(got[0], second[0])
    _poison(n, K_JAC_HESS, st)
    _same_bits(got, _alone(n, K_JAC_HESS), "after set_x")
    _close([n])


def test_mixed_passes_back_to_back():
    """gradient, constraint and fused Jacobian+Hessian on one batch, then the fused pass on a second batch"""
    import torch
    st = torch.cuda.Stream()
    nl = _batches("cartpole", dict(T=101), 2, 2, st)
    seq = [(nl[0], K_GRADIENT), (nl[0], K_CONSTRAINT), (nl[0], K_JAC_HESS), (nl[1], K_JAC_HESS)]
    ref = [_alone(n, k) for n, k in seq]
    for n, k in seq:
        _poison(n, k, st)
    with torch.cuda.stream(st):
        for n, k in seq:
            n.launch(k)
    torch.cuda.synchronize()
    for (n, k), r in zip(seq, ref):
        _same_bits([_view(n, a, w) for a, w in _outputs(n, k)], r, f"kernel {k}")
    _close(nl)
