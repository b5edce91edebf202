"""Host-side checks of bench.py's workloads (no GPU): the synthetic inputs of the BASELINE.json configurations,
the product-side weight containers and the oracle stand-ins share state-dict keys, and the coalition rows follow
the reference's row family."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


@pytest.mark.parametrize("name", ["tiny", "c4_small"])
def test_workload_models_share_state_dict_keys(name):
    wl = bench.Workload(name)
    arch = wl.make_model()
    om = wl.oracle_model(arch)  # load_state_dict(strict) inside: raises on any key / shape mismatch
    for k, v in arch.state_dict().items():
        assert torch.equal(om.state_dict()[k], v)
    assert wl.x.shape == (wl.n, wl.f) and wl.ei.shape == (2, wl.e)
    assert int(wl.ei.min()) >= 0 and int(wl.ei.max()) < wl.n
    assert wl.com_of.shape == (wl.n,) and int(wl.com_of.max()) == wl.c - 1


def test_hetero_workload_is_type_consistent():
    wl = bench.Workload("c4_small")
    ptr = wl.type_ptr
    assert ptr[0] == 0 and ptr[-1] == wl.n and len(ptr) == 6
    assert len(wl.edge_type_names) == 20
    same = sum(1 for (a, _, b) in wl.edge_type_names if a == b)
    assert same >= 4  # SURVEY.md 8d: at least 4 same-type relations
    names = wl.node_type_names
    for r, (a, _, b) in enumerate(wl.edge_type_names):
        sel = wl.edge_type == r
        src, dst = wl.ei[0][sel], wl.ei[1][sel]
        ia, ib = names.index(a), names.index(b)
        assert int(src.min()) >= ptr[ia] and int(src.max()) < ptr[ia + 1]
        assert int(dst.min()) >= ptr[ib] and int(dst.max()) < ptr[ib + 1]
    # type-pure communities (reference README.md:218)
    node_type = wl.node_type.to(torch.int64)
    for c in range(wl.c):
        assert len(torch.unique(node_type[wl.com_of == c])) == 1


def test_mask_rows_follow_the_reference_row_family():
    """Row i: internal community i mod C with iid node bits, every other community switched as a block,
    external halves antithetic (masks.py:138-194)."""
    wl = bench.Workload("tiny")
    rows = 2 * wl.c
    m = bench.make_masks(rows, wl.n, wl.c, wl.com_of, 5).bool()
    half = (rows + 1) // 2
    for i in (0, 3, half + 3):
        own = i % wl.c
        for c in range(wl.c):
            vals = m[i][wl.com_of == c]
            if c != own:
                assert bool(vals.all()) or not bool(vals.any())
    i, j = 3, half + 3  # antithetic pair: every community that is internal to neither row is complementary
    for c in range(wl.c):
        if c in (i % wl.c, j % wl.c):
            continue
        sel = wl.com_of == c
        assert bool(m[i][sel][0]) != bool(m[j][sel][0])


def test_rmat_generator_is_skewed_and_in_range():
    g = torch.Generator().manual_seed(0)
    ei = bench.rmat_edges(1 << 12, 60000, g)
    assert int(ei.min()) >= 0 and int(ei.max()) < (1 << 12)
    indeg = torch.bincount(ei[1], minlength=1 << 12)
    assert int(indeg.max()) > 20 * float(indeg.float().mean())  # hub rows


def test_reference_arm_prints_one_contract_line(tmp_path):
    """`bench.py --impl reference` (the unmodified reference's kernel_output where the reference tree or its staged copy
    exists, else the oracle port) prints ONE JSON line with the contract keys and writes the predictions of its last step
    with --dump-outputs; it must work without a GPU."""
    import json
    import subprocess

    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny", "--steps", "1",
                          "--warmup", "0", "--ref-coalitions", "2", "--no-query-leg", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, env=env, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "coalition evals/s" and d["unit"] == "coalition evals/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["config"]["workload"] == "tiny"
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    y = np.load(tmp_path / "predictions.npy")
    assert y.shape == (2, 1) and y.dtype == np.float32 and np.isfinite(y).all()


def test_reference_and_port_agree_on_the_bench_workload():
    """The two CPU arms of bench.py -- the unmodified reference's kernel_output and the oracle port -- give the same
    predictions on a bench workload (skipped where neither /root/reference nor oracle/_ref exists)."""
    ref = bench._reference_modules()
    if ref is None:
        pytest.skip("reference tree not present")
    wl = bench.Workload("tiny")
    om = wl.oracle_model(wl.make_model())
    m = bench.make_masks(3, wl.n, wl.c, wl.com_of, 5).bool().numpy()
    y_ref, kind = bench.host_eval(wl, om, m, ref)
    y_port, kind2 = bench.host_eval(wl, om, m, None)
    assert (kind, kind2) == ("reference", "port")
    np.testing.assert_allclose(y_ref, y_port, rtol=1e-5, atol=1e-7)


def test_strong_scaling_split_covers_the_job():
    class A:
        coalitions, coalitions_per_gpu = 4096, 0
    for world in (1, 2, 3, 4, 8):
        rows = bench.per_rank_rows(A, world)
        assert sum(rows) == 4096 and all(r % 32 == 0 for r in rows[:-1]) and max(rows) - min(rows) <= 32
    A.coalitions = 1000
    assert sum(bench.per_rank_rows(A, 8)) == 1000
    A.coalitions_per_gpu = 512
    assert bench.per_rank_rows(A, 4) == [512] * 4 and bench.scaling_of(A) == "weak"
