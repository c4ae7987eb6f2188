"""CPU: the heterogeneous-batch ABI (hmz_multi_t) — struct layout against gcc, argument errors reported before any CUDA
call, and the WeightSets blob layout."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from oracle import port


def test_multi_desc_matches_the_header_as_compiled_by_gcc(tmp_path):
    from muzero_hanoi_b200 import _lib

    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "hmz.h"', "int main(void) {",
             '  printf(". %zu\\n", sizeof(hmz_multi_t));']
    lines += [f'  printf("{f} %zu\\n", offsetof(hmz_multi_t, {f}));' for f, *_ in _lib.MultiDesc._fields_]
    lines.append("  return 0;\n}")
    (tmp_path / "m.c").write_text("\n".join(lines))
    subprocess.run(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(tmp_path / "m.c"), "-o", str(tmp_path / "m")], check=True)
    rows = subprocess.run([str(tmp_path / "m")], check=True, capture_output=True, text=True).stdout.split()
    got = dict(zip(rows[::2], map(int, rows[1::2])))
    assert got.pop(".") == ctypes.sizeof(_lib.MultiDesc) == 40
    assert got == {f: getattr(_lib.MultiDesc, f).offset for f in got} and len(got) == 6
    assert ctypes.sizeof(_lib.SearchDesc) == 80


def _args(lib, mode=0, n=512, n_records=101, budgets=(100, 50), n_sets=2, stride=None, schedule=0):
    from muzero_hanoi_b200 import _lib

    hbb = np.ascontiguousarray(budgets, dtype=np.int32)
    need = lib.hmz_weights_packed_bytes(3, mode)
    md = _lib.MultiDesc(block_set=16, budget=16, host_block_budget=hbb.ctypes.data,
                        weight_stride=(need + 255) // 256 * 256 if stride is None else stride, n_sets=n_sets, n_disks=3)
    sd = _lib.SearchDesc(nodes=None, latents=None, root_prior=None, root_W=None, minmax=None, workspace=None, capture=None,
                         n_searches=n, n_records=n_records, latent_dtype=0, root_prior_is_f64=0, schedule=schedule)
    return md, sd, hbb, need


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_multi_argument_errors_without_gpu(lib, mode):
    from muzero_hanoi_b200 import _lib

    def run(**kw):
        md, sd, hbb, _ = _args(lib, mode, **kw)
        return lib.hmz_search_run_multi(ctypes.byref(sd), ctypes.byref(md), 16, mode, 16, 0.8, None)

    def policy(**kw):
        md, sd, hbb, _ = _args(lib, mode, **kw)
        return lib.hmz_search_root_policy_multi(ctypes.byref(sd), ctypes.byref(md), 1.0, 1, None, None, None, None, None, None, None)

    need = lib.hmz_weights_packed_bytes(3, mode)
    for fn in (run, policy):
        assert fn(n=300, budgets=(100, 50)) == _lib.ERR_INVALID and b"multiple of 256" in lib.hmz_last_error()
        assert fn(budgets=(50, 100)) == _lib.ERR_INVALID and b"must not increase" in lib.hmz_last_error()
        assert fn(budgets=(101, 50)) == _lib.ERR_INVALID and b"n_records" in lib.hmz_last_error()
        assert fn(budgets=(100, 0)) == _lib.ERR_INVALID
        assert fn(n_sets=0) == _lib.ERR_INVALID and b"n_sets" in lib.hmz_last_error()
    assert run(stride=(need + 255) // 256 * 256 - 256) == _lib.ERR_INVALID and b"weight_stride" in lib.hmz_last_error()
    assert run(stride=(need + 255) // 256 * 256 + 16) == _lib.ERR_INVALID and b"weight_stride" in lib.hmz_last_error()
    for schedule in (_lib.SCHEDULE_PERSISTENT, _lib.SCHEDULE_SERVER, _lib.SCHEDULE_SERVER | 2):
        assert run(schedule=schedule) == _lib.ERR_UNSUPPORTED
    assert run(schedule=17) == _lib.ERR_INVALID
    md, sd, hbb, _ = _args(lib, mode)
    rc = lib.hmz_net_initial_multi(16, ctypes.byref(md), mode, 16, 16, 101, 0, 16, 16, 300, None)
    assert rc == _lib.ERR_INVALID and b"multiple of 256" in lib.hmz_last_error()
    md.weight_stride = need - 1
    assert lib.hmz_net_initial_multi(16, ctypes.byref(md), mode, 16, 16, 101, 0, 16, 16, 256, None) == _lib.ERR_INVALID
    assert lib.hmz_search_run_multi(ctypes.byref(sd), None, 16, mode, 16, 0.8, None) == _lib.ERR_INVALID
    assert lib.hmz_rng_uniform_keyed(None, 4, 0, None, 0, None, None) == _lib.ERR_INVALID


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_weight_sets_blob_layout(lib, mode):
    from muzero_hanoi_b200.engine import WeightSets, pack_host

    sds = [port.make_weights(4, 3), port.lesion_weights(port.make_weights(4, 3), ["policy_net"], seed=1),
           port.lesion_weights(port.make_weights(4, 5), ["value_net", "rwd_net"], seed=2)]
    ws = WeightSets(sds, 4, mode, device="cpu")
    need = lib.hmz_weights_packed_bytes(4, mode)
    assert ws.stride % 256 == 0 and need <= ws.stride < need + 256 and ws.set_bytes == need
    blob = ws.blob.numpy()
    assert blob.size == 3 * ws.stride
    for k, sd in enumerate(sds):
        assert np.array_equal(blob[k * ws.stride: k * ws.stride + need], pack_host(sd, 4, mode))
        assert not blob[k * ws.stride + need: (k + 1) * ws.stride].any()
    assert not np.array_equal(blob[:need], blob[ws.stride: ws.stride + need])


def test_dirichlet_counter_domain_without_gpu(lib):
    """The Dirichlet streams keep the draw's block in the low 8 bits of Philox counter word 3, above counter bits 32-55:
    hmz_rng_dirichlet and hmz_selfplay_move reject counters from 2^56 on, before any CUDA call."""
    from muzero_hanoi_b200 import _lib

    for counter in (1 << 56, (1 << 64) - 1):
        assert lib.hmz_rng_dirichlet(None, 0, 0.25, 0, counter, 0, None) == _lib.ERR_INVALID and b"2^56" in lib.hmz_last_error()
        assert lib.hmz_selfplay_move(ctypes.byref(_lib.SelfPlayDesc()), counter, None) == _lib.ERR_INVALID
        assert b"2^56" in lib.hmz_last_error()
    assert lib.hmz_rng_dirichlet(None, 4, 0.25, 0, (1 << 56) - 1, 0, None) == _lib.ERR_INVALID
    assert b"bad arguments" in lib.hmz_last_error()  # the largest counter allowed passes the domain check
    sp = _lib.SelfPlayDesc()
    sp.search.n_searches = 4
    assert lib.hmz_selfplay_move(ctypes.byref(sp), (1 << 56) - 1, None) == _lib.ERR_INVALID
    assert b"null buffer" in lib.hmz_last_error()
