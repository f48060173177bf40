"""CPU: the host side of the deterministic training mode -- mode resolution, the slot ranges and finalize job tables
of determinism.DetPlan, and train.py's switch.  No GPU: the launches are recorded instead of run."""
import ctypes
import os
import subprocess
import sys

import pytest
import torch

import __graft_entry__ as entry
from xmm_superres_denoise_b200 import _lib, determinism, ops


@pytest.fixture
def torch_flag():
    before = torch.are_deterministic_algorithms_enabled()
    yield
    torch.use_deterministic_algorithms(before)


def test_mode_resolution(monkeypatch, torch_flag):
    monkeypatch.delenv("XMM_DETERMINISTIC", raising=False)
    torch.use_deterministic_algorithms(False)
    assert not determinism.enabled()
    torch.use_deterministic_algorithms(True)
    assert determinism.enabled()  # Lightning's Trainer(deterministic=True) sets this flag
    monkeypatch.setenv("XMM_DETERMINISTIC", "0")
    assert not determinism.enabled()  # the variable wins over the flag
    torch.use_deterministic_algorithms(False)
    monkeypatch.setenv("XMM_DETERMINISTIC", "1")
    assert determinism.enabled()
    monkeypatch.setenv("XMM_DETERMINISTIC", "")
    assert not determinism.enabled()
    monkeypatch.setenv("XMM_DETERMINISTIC", "yes")
    with pytest.raises(ValueError):
        determinism.enabled()


SLOTS = {_lib.DET_CONV3X3: 148 * 8, _lib.DET_COLSUM: 100, _lib.DET_EDGE_WGRAD: 7}


@pytest.fixture
def recorded(monkeypatch):
    calls = []
    monkeypatch.setattr(ops, "colsum_multi_det", lambda inp, segs, ws: calls.append(("colsum", segs, ws.data_ptr(),
                                                                                     ws.numel())))
    monkeypatch.setattr(ops, "edge_wgrad", lambda *a, **kw: calls.append(("edge", kw["ws"].data_ptr(), kw["ws"].numel())))
    monkeypatch.setattr(ops, "det_finalize", lambda table, njobs, max_n, base: calls.append(
        ("finalize", table, njobs, max_n, base.data_ptr())))
    return calls


def _plan():
    return determinism.DetPlan(torch.device("cpu"), slot_count=lambda site, b, h, w, c: SLOTS[site])


def _jobs(table):
    arr = (_lib.DetJob * (table.numel() // ctypes.sizeof(_lib.DetJob)))()
    ctypes.memmove(arr, table.numpy().ctypes.data, table.numel())
    return [(j.slots, j.count, j.stride, j.dst, j.n, j.scale, j.accumulate) for j in arr]


def _one_rrdb(plan, flat):
    """The shape of one RRDB group of TrainEngine.backward at F = 32: fused bias gradients of conv1..conv5 of three
    dense blocks (15 conv3x3 launches), then the flush before the RRDB's all-reduce hook."""
    kws = [plan.conv_kwargs(2, 16, 16, flat[32 * k:32 * (k + 1)], 0.2 if k % 5 == 4 else 1.0) for k in range(15)]
    plan.flush()
    return kws


def test_plan_slot_ranges_and_job_tables_per_rrdb(recorded):
    plan = _plan()
    flat = torch.zeros(15 * 32 + 1000)
    ptrs = []
    for call in range(2):  # the second backward of the shape reuses ranges and tables
        plan.begin(flat)
        kws = [_one_rrdb(plan, flat) for _ in range(2)]  # two RRDBs
        ptrs.append([kw["colsum_ws"].data_ptr() for group in kws for kw in group])
        for group in kws:
            for k, kw in enumerate(group):
                assert kw["colsum"].data_ptr() == flat[32 * k:].data_ptr()
                assert kw["colsum_ws"].numel() == SLOTS[_lib.DET_CONV3X3] * 32
    assert ptrs[0] == ptrs[1] and len(set(ptrs[0])) == 30  # one range per launch, the same ones every call
    fins = [c for c in recorded if c[0] == "finalize"]
    assert len(fins) == 4  # one per RRDB and call, never one per conv
    assert fins[0][1] is fins[2][1] and fins[1][1] is fins[3][1]  # tables built once
    jobs = _jobs(fins[0][1])
    assert fins[0][2] == 15 and fins[0][3] == 32
    for k, (slots, count, stride, dst, n, scale, acc) in enumerate(jobs):
        assert (slots, count, stride, dst, n, acc) == (ptrs[0][k], 148 * 8, 32, 32 * k, 32, 1)
        assert scale == pytest.approx(0.2 if k % 5 == 4 else 1.0)


def test_plan_colsum_and_edge_jobs(recorded):
    plan = _plan()
    flat = torch.zeros(4096)
    d_fea = torch.zeros(2, 16, 16, 32, dtype=torch.bfloat16)
    plan.begin(flat)
    # conv_first's bias: two integrands, one job over both inputs' slots (d_fea's, then d_trunk's)
    plan.colsum([d_fea, d_fea], [(0, 32, flat[100:132], 1.0, False)])
    # a dense block's five bias gradients (F = 64 generators): one pass, one job per segment
    plan.colsum([d_fea], [(64 * k, 64, flat[200 + 64 * k:264 + 64 * k], 0.2 if k == 4 else 1.0, True) for k in range(5)])
    s = torch.zeros(2, 1, 16, 16)
    plan.edge_wgrad(s, d_fea, 0, 32, flat[1000:1288].view(1, 32, 9), ssum=flat[1300:1301], gate=s)
    posted = []
    plan.after(lambda: posted.append(len([c for c in recorded if c[0] == "finalize"])))
    plan.flush()
    assert posted == [1]  # host steps run after the finalize they depend on
    c1, c2, c3, e, fin = recorded
    assert c1[0] == c2[0] == c3[0] == "colsum" and c1[3] == c2[3] == 100 * 32
    assert c2[2] == c1[2] + 100 * 32 * 4  # the second input's half of the range
    assert c3[1] == [(64 * k, 64, 0.2 if k == 4 else 1.0) for k in range(5)] and c3[3] == 100 * 5 * 64
    jobs = _jobs(fin[1])
    base = c1[2]
    assert jobs[0][:5] == (base, 200, 32, 100, 32) and jobs[0][6] == 0
    row = 5 * 64
    for k in range(5):
        assert jobs[1 + k][1:5] == (100, row, 200 + 64 * k, 64)
        assert jobs[1 + k][0] == jobs[1][0] + 4 * 64 * k
    er = 32 * 9 + 1
    assert e[2] == 7 * er
    assert jobs[6][1:5] == (7, er, 1000, 32 * 9) and jobs[7][1:5] == (7, er, 1300, 1)
    assert jobs[7][0] == jobs[6][0] + 4 * 32 * 9
    assert fin[2] == 8 and fin[3] == 32 * 9


def test_plan_rejects_shared_or_foreign_destinations(recorded):
    plan = _plan()
    flat = torch.zeros(1024)
    plan.begin(flat)
    plan.conv_kwargs(1, 8, 8, flat[0:32], 1.0)
    with pytest.raises(RuntimeError, match="same gradient"):  # jobs of one finalize run concurrently
        plan.conv_kwargs(1, 8, 8, flat[16:48], 1.0)
    with pytest.raises(RuntimeError, match="outside"):
        plan.conv_kwargs(1, 8, 8, torch.zeros(32), 1.0)
    plan.flush()
    plan.begin(flat)
    plan.slots(SLOTS[_lib.DET_CONV3X3], 32)
    with pytest.raises(RuntimeError, match="slot layout"):
        plan.slots(3, 32)


def test_det_job_mirrors_the_header():
    hdr = open(os.path.join(entry.ROOT, "include", "xmm_b200.h")).read()
    assert "xmm_det_job" in hdr and _lib.EXTRA_STRUCTS["xmm_det_job"] is _lib.DetJob
    for name in ("XMM_DET_CONV3X3 0", "XMM_DET_COLSUM 1", "XMM_DET_EDGE_WGRAD 2"):
        assert f"#define {name}" in hdr


def test_train_py_flag_and_config_key(tmp_path, torch_flag):
    sys.path.insert(0, entry.ROOT)
    import train

    torch.use_deterministic_algorithms(False)
    cfg = train.load_run_config(None)
    assert cfg["trainer"]["deterministic"] is False
    assert train.configure_determinism(cfg, False) is False
    assert not torch.are_deterministic_algorithms_enabled()
    run = tmp_path / "run.toml"
    run.write_text("[trainer]\ndeterministic = true\n")
    cfg = train.load_run_config(str(run))
    assert cfg["trainer"]["deterministic"] is True and cfg["trainer"]["epochs"] == 1
    assert train.configure_determinism(cfg, False) is True
    assert torch.are_deterministic_algorithms_enabled() and determinism.enabled()
    a = torch.rand(4)
    torch.use_deterministic_algorithms(False)
    assert train.configure_determinism(train.load_run_config(None), True) is True  # --deterministic
    assert torch.equal(torch.rand(4), a)  # seeded the same way both times
    out = subprocess.run([sys.executable, os.path.join(entry.ROOT, "train.py"), "--help"], capture_output=True,
                         text=True, check=True).stdout
    assert "--deterministic" in out
