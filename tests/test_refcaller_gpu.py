"""GPU: the reference's OWN search driver — /root/reference/core/mcts.py:7-57, unmodified, byte-compiled into
oracle/_ref/refpy/ by oracle/Makefile — run twice on the same model outputs:
  (a) against the reference's own Cython `cytree` built with the rand() == 0 shim (oracle/_ref/det), and
  (b) against the drop-in `core.ctree.cytree` that dropin/ puts on the import path (hanabizero_b200.cytree -> C ABI ->
      sm_100a kernels).
Lists in, lists out, host gathers, .tolist() marshalling: exactly what the reference's callers do.  Visit counts,
trajectories and selected actions must be identical; root values within 1e-5 relative (asserted bit-exact)."""
import os
import sys

import numpy as np
import pytest
import torch

from helpers import CONST, ROOT, bits_equal, tree_inputs

pytestmark = pytest.mark.gpu


class _Out:
    pass


class _FakeModel:
    """recurrent_inference with the reference's NetworkOutput contract (numpy fields, core/model.py:74-84):
    a fixed random projection of (hidden, action) evaluated on the GPU, so both runs see identical numbers."""

    def __init__(self, F, A, seed):
        g = torch.Generator(device="cuda").manual_seed(seed)
        self.w_h = torch.randn(F, F, device="cuda", generator=g) / F ** 0.5
        self.w_a = torch.randn(A, F, device="cuda", generator=g)
        self.w_p = torch.randn(F, A, device="cuda", generator=g)
        self.w_v = torch.randn(F, 2, device="cuda", generator=g)
        self.calls = 0

    def eval(self):
        return self

    def recurrent_inference(self, hidden_states, last_actions):
        assert hidden_states.is_cuda and last_actions.dtype == torch.int64 and last_actions.shape[1] == 1
        self.calls += 1
        h = torch.tanh(hidden_states.float() @ self.w_h + self.w_a[last_actions.view(-1)])
        o = _Out()
        o.hidden_state = h.cpu().numpy()
        vr = (h @ self.w_v).cpu().numpy()
        o.value, o.reward = vr[:, :1].copy(), vr[:, 1:].copy()
        o.policy_logits = (h @ self.w_p).cpu().numpy()
        if self.calls == 3:
            o.policy_logits[0, 2] = np.nan      # core/mcts.py:48-49 zeroes NaN logits on the host
        return o


class _Cfg:
    pb_c_base, pb_c_init, discount, value_delta_max = CONST["pb_c_base"], CONST["pb_c_init"], CONST["discount"], CONST["delta"]
    amp_type = "none"

    def __init__(self, sims):
        self.num_simulations = sims


@pytest.mark.parametrize("N,A,S,seed", [(16, 11, 50, 1), (64, 20, 50, 2), (256, 20, 30, 3)])
def test_unmodified_reference_mcts_drives_the_dropin(N, A, S, seed):
    from oracle import refpy
    if not refpy.available():
        pytest.skip("oracle/_ref/refpy not built (no reference sources at build time)")
    sys.path.insert(0, os.path.join(ROOT, "dropin"))
    try:
        for k in [k for k in sys.modules if k == "core" or k.startswith("core.")]:
            del sys.modules[k]
        import core.ctree.cytree as dropin_cytree          # resolves to dropin/core/ctree/cytree.py
    finally:
        sys.path.remove(os.path.join(ROOT, "dropin"))
    assert dropin_cytree.Roots.__module__ == "hanabizero_b200.cytree"
    ref_cytree = refpy.load_ref_cytree(deterministic=True)
    F = 64
    d = tree_inputs(N, A, S, seed)
    hidden_roots = np.random.default_rng(seed).standard_normal((N, F)).astype(np.float32)
    legal = [row.astype(np.float64) for row in d["mask"]]       # core/selfplay_worker.py:268 passes float 0/1 arrays
    results = []
    for tree in (ref_cytree, dropin_cytree):
        MCTS = refpy.load_mcts_class(tree)
        roots = tree.Roots(N, A, S)
        roots.prepare(CONST["frac"], d["noise"].tolist(), d["reward"].tolist(), d["logits"].tolist(), legal)
        model = _FakeModel(F, A, seed)
        MCTS(_Cfg(S)).run_multi(roots, model, hidden_roots)
        assert model.calls == S - 1                              # core/mcts.py:25-26 skips the last iteration
        results.append((roots.get_distributions(), roots.get_values(), roots.get_trajectories()))
    (dist_ref, val_ref, traj_ref), (dist, val, traj) = results
    assert dist == dist_ref, "root visit counts"
    assert [int(np.argmax(r)) for r in dist] == [int(np.argmax(r)) for r in dist_ref], "selected actions"
    assert traj == traj_ref, "best-action trajectories"
    np.testing.assert_allclose(val, val_ref, rtol=1e-5, atol=0)
    assert bits_equal(np.asarray(val, np.float32), np.asarray(val_ref, np.float32))
    assert all(sum(r) == S - 1 for r in dist)
