"""Batched user models, CPU checks: a 2-D `params` makes a model of many datasets (UserModel.batched, n_datasets,
dataset(g)), its fingerprint covers the whole table, its plugin methods refuse to run, glabc_user_model_t's batched fields
match the header, and the batched kernels (-DGLABC_BATCHED) compile for sm_100a at theta_dim 1..8 with every proposal kind."""
import ctypes as C
import os
import subprocess

import pytest
import torch

from helpers import abi
from test_user_model_eval import GENERIC_SRC
from test_user_model_proposals import GAUSS_SRC, KINDS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _g():
    import glabc_b200 as g
    return g


def _batched(G=3, d=2):
    table = torch.arange(G * (2 + d), dtype=torch.float32).reshape(G, 2 + d) / 7.0
    return _g().UserModel(GAUSS_SRC, theta_dim=d, y_dim=d, n_noise=d, epsilon=0.3, params=table), table


def test_two_dimensional_params_make_a_batched_model():
    g = _g()
    um, table = _batched()
    assert um.batched and um.n_datasets == 3 and um.n_params == 4 and um.params is None
    for gi in range(3):
        one = um.dataset(gi)
        assert isinstance(one, g.UserModel) and not one.batched and one.n_datasets == 1
        assert torch.equal(torch.tensor(one.params, dtype=torch.float32), table[gi])
        assert (one.source, one.theta_dim, one.y_dim, one.n_noise, one.epsilon) == (um.source, 2, 2, 2, 0.3)
    with pytest.raises(IndexError):
        um.dataset(3)
    # lists of rows and numpy arrays are tables too; a 1-D params is the one-dataset model, as before
    assert g.UserModel(GAUSS_SRC, 2, 2, 2, 0.3, params=table.tolist()).batched
    assert g.UserModel(GAUSS_SRC, 2, 2, 2, 0.3, params=table.numpy()).n_datasets == 3
    flat = g.UserModel(GAUSS_SRC, 2, 2, 2, 0.3, params=table[0].tolist())
    assert not flat.batched and flat.n_datasets == 1 and flat.dataset(0) is flat and flat.params == table[0].tolist()
    with pytest.raises(ValueError, match="at most"):
        g.UserModel(GAUSS_SRC, 2, 2, 2, 0.3, params=torch.zeros(2, abi.USER_MAX_PARAMS + 1))
    with pytest.raises(ValueError, match="at least one dataset"):
        g.UserModel(GAUSS_SRC, 2, 2, 2, 0.3, params=torch.zeros(0, 4))


def test_fingerprint_covers_the_table():
    g = _g()
    um, table = _batched()
    assert um.fingerprint() == _batched()[0].fingerprint()
    assert um.fingerprint() != um.dataset(0).fingerprint()
    changed = table.clone()
    changed[2, 3] += 1e-3
    assert g.UserModel(GAUSS_SRC, 2, 2, 2, 0.3, params=changed).fingerprint() != um.fingerprint()
    assert g.UserModel(GAUSS_SRC, 2, 2, 2, 0.3, params=table[:2]).fingerprint() != um.fingerprint()
    # the one-dataset fingerprint is unchanged by the batched fields
    flat = g.UserModel(GAUSS_SRC, 2, 2, 2, 0.3, params=[1.0, 2.0])
    assert flat.fingerprint() == g.UserModel(GAUSS_SRC, 2, 2, 2, 0.3, params=(1.0, 2.0)).fingerprint()


def test_plugin_methods_of_a_batched_model_refuse():
    um, _ = _batched()
    x = torch.zeros(4, 2)
    for call in (lambda: um.generate_samples(x), lambda: um.prior_log_prob(x), lambda: um.discrepancy(x),
                 lambda: um.calculate_log_kernel(x)):
        with pytest.raises(ValueError, match=r"dataset\(g\)"):
            call()


def test_pod_of_a_batched_model():
    um, _ = _batched()
    pod = um.user_pod(chains_per_dataset=5)            # no device: the table stays on the host (a compile check needs none)
    assert (pod.n_datasets, pod.chains_per_dataset, pod.dataset_params, pod.n_params) == (3, 5, None, 4)
    flat = um.dataset(1).user_pod()
    assert (flat.n_datasets, flat.chains_per_dataset, flat.dataset_params) == (0, 0, None)


def test_user_model_layout_matches_the_header(tmp_path):
    prog = tmp_path / "layout.c"
    prog.write_text(r'''
#include <stdio.h>
#include <stddef.h>
#include "glabc.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu\n", sizeof(glabc_user_model_t), offsetof(glabc_user_model_t, epsilon),
         offsetof(glabc_user_model_t, dataset_params), offsetof(glabc_user_model_t, n_datasets),
         offsetof(glabc_user_model_t, chains_per_dataset));
  return 0;
}''')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(prog), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    U = abi.UserModelPOD
    assert got == [C.sizeof(U), U.epsilon.offset, U.dataset_params.offset, U.n_datasets.offset, U.chains_per_dataset.offset]


def _check(um, local_kind, far_kind):
    log = C.create_string_buffer(8192)
    pod = um.user_pod(chains_per_dataset=1)
    st = abi.load().glabc_user_model_check_proposals(C.byref(pod), local_kind, far_kind, 100, log, len(log))
    return st, log.value.decode(errors="replace")


# every kind in each slot over the eight dimensions, with 0, 1 and 32 simulator normals and y_dim 16
CASES = [(d, (0, 1, 32)[d % 3], KINDS[(d - 1) % 4], KINDS[(d + 1) % 4]) for d in range(1, 9)]


@pytest.mark.parametrize("d,nn,local_kind,far_kind", CASES)
def test_batched_kernels_compile(d, nn, local_kind, far_kind):
    um = _g().UserModel(GENERIC_SRC, theta_dim=d, y_dim=16, n_noise=nn, epsilon=0.1, params=torch.ones(5, 2))
    st, log = _check(um, local_kind, far_kind)
    assert st == abi.OK, log


def test_check_refuses_a_negative_dataset_count():
    um, _ = _batched()
    pod = um.user_pod()
    pod.n_datasets = -1
    log = C.create_string_buffer(256)
    st = abi.load().glabc_user_model_check_proposals(C.byref(pod), abi.DIST_DIAG_GAUSSIAN, abi.DIST_DIAG_GAUSSIAN, 100, log, len(log))
    assert st == abi.ERR_INVALID
    assert um.check()
