"""Training and validation from a device-resident feature store: the gathering input prologue (dvgr_prep_features_gather)
against the dense one on the torch-gathered batch, loader.DeviceFeatureStore / DeviceBatchLoader, DualVGR.forward_from_store
in both precisions, and the train / eval engines fed by video rows."""
import numpy as np
import pytest
import torch

import dualvgr_oracle as orc

pytestmark = pytest.mark.gpu

BF16, F32 = torch.bfloat16, torch.float32


def _err():
    return torch.zeros(1, dtype=torch.int32, device="cuda")


def _gather(store, rows):
    return store[rows.long()].contiguous()


@pytest.mark.parametrize("store_dtype", [F32, BF16])
@pytest.mark.parametrize("out_dtype", [BF16, F32])
@pytest.mark.parametrize("shape", ["appearance", "motion"])
@pytest.mark.parametrize("p", [0.0, 0.15])
def test_gathered_prologue_is_bit_identical_to_dense(store_dtype, out_dtype, shape, p):
    import dualvgr_videoqa_b200.ops as ops
    g = torch.Generator().manual_seed(3)
    V, N, T, C = 11, 5, 16, 2048
    full = (V, N, T, C) if shape == "appearance" else (V, N, C)
    T = T if shape == "appearance" else 1
    tanh = shape == "appearance"
    store = torch.randn(full, generator=g).to(store_dtype).cuda()
    rows = torch.tensor([7, 2, 2, 10, 0, 5, 7, 3, 9, 1, 4, 10, 6], dtype=torch.int32, device="cuda")   # B = 13, repeats
    err = _err()
    got = ops.prep_features_gather(store, rows, T, tanh, tanh, p, 1234, 5, err, out_dtype=out_dtype)
    ref = ops.prep_features(_gather(store, rows).view(-1, C), T, tanh, tanh, p, 1234, 5, out_dtype=out_dtype)
    assert got.dtype == out_dtype and got.shape == ref.shape
    assert torch.equal(got.view(torch.int16 if out_dtype == BF16 else torch.int32),
                       ref.view(torch.int16 if out_dtype == BF16 else torch.int32))
    assert int(err) == 0
    if p > 0:   # the mask really applies
        assert not torch.equal(got, ops.prep_features_gather(store, rows, T, tanh, tanh, 0.0, 1234, 5, err, out_dtype=out_dtype))


def test_gathered_prologue_offsets_past_2_pow_31_elements():
    """A ~4.6 GB bf16 store: rows whose first element lies beyond element 2^31 (64-bit source offsets)."""
    import dualvgr_videoqa_b200.ops as ops
    V, N, T, C = 3500, 20, 16, 2048
    assert 3277 * N * T * C > 2 ** 31
    store = torch.empty((V, N, T, C), dtype=BF16, device="cuda")
    rows_l = [3499, 5, 3300, 3277, 3300, 3400, 17]
    g = torch.Generator(device="cuda").manual_seed(9)
    for r in set(rows_l):
        store[r] = torch.randn((N, T, C), generator=g, device="cuda").to(BF16)
    rows = torch.tensor(rows_l, dtype=torch.int32, device="cuda")
    err = _err()
    got = ops.prep_features_gather(store, rows, T, True, True, 0.15, 77, 1, err)
    ref = ops.prep_features(_gather(store, rows).view(-1, C), T, True, True, 0.15, 77, 1)
    assert torch.equal(got.view(torch.int16), ref.view(torch.int16)) and int(err) == 0
    del store
    torch.cuda.empty_cache()


def test_out_of_range_rows_read_nothing_and_set_the_error_word():
    import dualvgr_videoqa_b200.ops as ops
    from dualvgr_videoqa_b200.loader import DeviceBatchLoader
    V, N, T, C = 6, 4, 16, 256
    # the store is a view inside a larger allocation: a missing guard would read the neighbouring (valid, non-zero) videos
    big = torch.rand((V + 2, N, T, C), device="cuda") + 1.0
    store = big[1:V + 1]
    rows = torch.tensor([2, V, 0, -1, 5], dtype=torch.int32, device="cuda")
    err = _err()
    out = ops.prep_features_gather(store, rows, T, True, True, 0.0, 0, 0, err).view(T, 5, N, C)
    assert int(err) == 1
    assert float(out[:, 1].abs().max()) == 0.0 and float(out[:, 3].abs().max()) == 0.0
    good = torch.tensor([0, 2, 4], device="cuda")
    ref = ops.prep_features(_gather(store, rows[good]).view(-1, C), T, True, True).view(T, 3, N, C)
    assert torch.equal(out[:, good], ref)
    # motion shape, sticky word: stays set
    mot = big[1:V + 1, :, 0].contiguous()
    out_m = ops.prep_features_gather(mot, rows, 1, False, False, err=err).view(5, N, C)
    assert int(err) == 1 and float(out_m[1].abs().max()) == 0.0 and float(out_m[3].abs().max()) == 0.0

    # host side: the batch loader rejects such rows before anything is launched
    class Store:
        pass
    ds = Store()
    ds.V, ds.row = V, {i: i for i in range(V)}
    samples = {"question": np.zeros((3, 4), np.int64), "question_len": np.full(3, 4), "answer": np.zeros(3, np.int64)}
    for bad in (V, -1):
        with pytest.raises(ValueError, match="outside"):
            DeviceBatchLoader(ds, dict(samples, video_idx=np.array([0, bad, 1])), 2, "cuda")
    with pytest.raises(ValueError, match="not in the store"):
        DeviceBatchLoader(ds, dict(samples, video_id=np.array([0, 99, 1])), 2, "cuda")


def _npy_stores(tmp_path, V=7, N=4, F=16, Dv=2048, seed=0):
    from dualvgr_videoqa_b200.loader import FeatureStore
    g = np.random.default_rng(seed)
    app = np.abs(g.standard_normal((V, N, F, Dv), dtype=np.float32))
    mot = np.abs(g.standard_normal((V, N, Dv), dtype=np.float32))
    np.save(tmp_path / "app.npy", app); np.save(tmp_path / "mot.npy", mot)
    np.save(tmp_path / "app16.npy", FeatureStore.to_bf16_bits(app)); np.save(tmp_path / "mot16.npy", FeatureStore.to_bf16_bits(mot))
    return app, mot


def test_device_store_equals_the_host_store(tmp_path):
    from dualvgr_videoqa_b200.loader import DeviceFeatureStore, FeatureStore
    app, mot = _npy_stores(tmp_path)
    per_video = 4 * 16 * 2048 * 4
    for name, bf16, bits in (("app.npy", False, False), ("app16.npy", False, True), ("app.npy", True, True)):
        host = FeatureStore.open(str(tmp_path / name), str(tmp_path / name.replace("app", "mot")))
        # chunks of 3 videos over V = 7: several chunks and a short last one
        ds = DeviceFeatureStore(host, "cuda", bf16=bf16, chunk_bytes=3 * per_video + 100)
        assert ds.V == 7 and ds.app.shape == app.shape and ds.mot.shape == mot.shape and int(ds.err) == 0
        if bits:    # bf16: stored bits, or the device cast of fp32 features, equal FeatureStore.to_bf16_bits
            assert ds.app.dtype == BF16
            assert np.array_equal(ds.app.view(torch.int16).cpu().numpy().view(np.uint16), FeatureStore.to_bf16_bits(app))
            assert np.array_equal(ds.mot.view(torch.int16).cpu().numpy().view(np.uint16), FeatureStore.to_bf16_bits(mot))
        else:
            assert ds.app.dtype == F32
            assert np.array_equal(ds.app.cpu().numpy(), app) and np.array_equal(ds.mot.cpu().numpy(), mot)
        ds.err.fill_(1)
        assert ds.read_error(clear=True) == 1 and ds.read_error() == 0


def test_device_store_capacity_check_raises_before_allocating(tmp_path, monkeypatch):
    from dualvgr_videoqa_b200.loader import DeviceFeatureStore, FeatureStore
    _npy_stores(tmp_path)
    host = FeatureStore.open(str(tmp_path / "app.npy"), str(tmp_path / "mot.npy"))
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda *a, **k: (5 << 30, 180 << 30))
    need = 7 * 4 * 2048 * 17 * 4
    with pytest.raises(MemoryError, match=rf"needs {need} bytes of device memory, 1000 are available"):
        DeviceFeatureStore(host, "cuda", reserve_bytes=(5 << 30) - 1000)
    assert torch.cuda.memory_allocated() == before


def _model(cfg):
    import dualvgr_videoqa_b200.model.models as M
    B, N, L, A, V, U = cfg
    m = M.DualVGR(vocab=orc.make_vocab(V, A), num_of_nodes=N, graph_module="GAT", graph_layers=1, unit_layers=U)
    m.load_state_dict(orc.make_state_dict(U, A, V), strict=True)
    return m.cuda()


def _store(Vd, N, dtype, seed=5):
    """A DeviceFeatureStore built from in-memory host arrays."""
    from dualvgr_videoqa_b200.loader import DeviceFeatureStore, FeatureStore
    g = np.random.default_rng(seed)
    app = np.abs(g.standard_normal((Vd, N, 16, 2048), dtype=np.float32))
    mot = np.abs(g.standard_normal((Vd, N, 2048), dtype=np.float32))
    if dtype == BF16:
        app, mot = FeatureStore.to_bf16_bits(app), FeatureStore.to_bf16_bits(mot)
    return DeviceFeatureStore(FeatureStore(app, mot), "cuda")


def _flat_grad(model):
    return torch.cat([p.grad.reshape(-1) for p in model.parameters() if p.grad is not None])


def _same(a, b):
    if isinstance(a, (list, tuple)):
        return len(a) == len(b) and all(_same(x, y) for x, y in zip(a, b))
    return a.dtype == b.dtype and a.shape == b.shape and torch.equal(a, b)


@pytest.mark.parametrize("precision,store_dtype", [("bf16", F32), ("bf16", BF16), ("fp32", F32)])
def test_forward_from_store_matches_forward_on_the_gathered_batch(precision, store_dtype):
    import dualvgr_videoqa_b200.autograd as ag
    cfg = (6, 8, 6, 10, 30, 2) if precision == "bf16" else (4, 8, 6, 10, 30, 1)
    B, N, L, A, V, U = cfg
    model = _model(cfg)
    ds = _store(9, N, store_dtype)
    _, _, q, qlen, ans = [t.cuda() for t in orc.make_inputs(*cfg[:5])]
    rows = torch.tensor([3, 0, 8, 3, 5, 1][:B], dtype=torch.int32, device="cuda")
    app, mot = _gather(ds.app, rows), _gather(ds.mot, rows)
    model.set_precision(precision)
    try:
        with torch.no_grad():
            model.eval()
            assert _same(model.forward_from_store(ds, rows, q, qlen), model(app, mot, q, qlen))
        model.train()
        outs, grads = [], []
        saved = dict(ag._rng)
        for run in range(2):
            ag._rng.clear(); ag._rng.update(saved)           # the same dropout seed for both runs
            for p in model.parameters():
                p.grad = None
            out = model.forward_from_store(ds, rows, q, qlen) if run == 0 else model(app, mot, q, qlen)
            torch.nn.functional.cross_entropy(out[0], ans).backward()
            outs.append(out[0].detach())
            grads.append(_flat_grad(model))
        assert torch.equal(outs[0], outs[1])
        rel = float((grads[0] - grads[1]).norm() / grads[1].norm())
        assert rel <= 1e-3, rel          # the backward's atomic sums differ from run to run
        assert ds.read_error() == 0
    finally:
        model.set_precision("bf16")


def test_captured_train_step_from_store_over_shuffled_epochs():
    import dualvgr_videoqa_b200.autograd as ag
    from dualvgr_videoqa_b200.engine import TrainEngine
    from dualvgr_videoqa_b200.loader import DeviceBatchLoader
    B, N, L, A, Vq, U = 5, 8, 6, 10, 30, 1
    ds = _store(10, N, F32)
    g = np.random.default_rng(1)
    S = 23
    qlen = g.integers(2, L + 1, S)
    samples = {"video_idx": g.integers(0, 10, S), "question": g.integers(2, Vq, (S, L)) * (np.arange(L)[None] < qlen[:, None]),
               "question_len": qlen, "answer": g.integers(0, A, S)}
    loader = DeviceBatchLoader(ds, samples, batch_size=B, device="cuda", shuffle=True, seed=4)
    assert len(loader) == 4
    saved = dict(ag._rng)
    # lr 0: the warm-up step leaves the weights as they are, so the first replay starts from the saved initial state
    eng = TrainEngine(_model((B, N, L, A, Vq, U)), lr=0.0)
    losses, first = [], None
    for epoch in range(2):
        seen = []
        for rows, q, ql, ans in loader:
            if eng.graph is None:
                first = [t.clone() for t in (rows, q, ql, ans)]
                eng.capture_from_store(ds, rows, q, ql, ans, warmup=1)
            eng.load_rows(rows, q, ql, ans)
            losses.append(float(eng.replay()))
            seen += rows.tolist()
        assert len(seen) == 20 and set(seen) <= set(samples["video_idx"].tolist())
    assert len(losses) == 8 and all(np.isfinite(losses)), losses
    assert eng.dependency_poll_timeouts() == 0 and ds.read_error() == 0
    eng.close()
    # the dense path on the torch-gathered first batch, same initial state and dropout seeds
    ag._rng.clear(); ag._rng.update(saved)
    ref = TrainEngine(_model((B, N, L, A, Vq, U)), lr=0.0)
    rows, q, ql, ans = first
    ref.capture(_gather(ds.app, rows), _gather(ds.mot, rows), q, ql, ans, warmup=1)
    ref.load_batch(_gather(ds.app, rows), _gather(ds.mot, rows), q, ql, ans)
    assert float(ref.replay()) == losses[0]
    ref.close()


def test_bad_row_turns_the_step_loss_into_nan():
    from dualvgr_videoqa_b200.engine import TrainEngine
    B, N, L, A, Vq, U = 4, 8, 6, 10, 30, 1
    ds = _store(5, N, BF16)
    _, _, q, qlen, ans = [t.cuda() for t in orc.make_inputs(B, N, L, A, Vq)]
    eng = TrainEngine(_model((B, N, L, A, Vq, U)), lr=0.0)
    ok = torch.tensor([0, 1, 2, 3], dtype=torch.int32, device="cuda")
    assert np.isfinite(float(eng.train_step_from_store(ds, ok, q, qlen, ans))) and eng.dependency_poll_timeouts() == 0
    bad = torch.tensor([0, 1, 5, 3], dtype=torch.int32, device="cuda")
    assert np.isnan(float(eng.train_step_from_store(ds, bad, q, qlen, ans))) and eng.dependency_poll_timeouts() == 1
    assert ds.read_error(clear=True) == 1
    assert np.isfinite(float(eng.train_step_from_store(ds, ok, q, qlen, ans)))
    eng.close()


def test_eval_engine_from_store_counts_like_dense_batches():
    from dualvgr_videoqa_b200.evaluate import EvalEngine, SVQA_CATEGORIES
    from dualvgr_videoqa_b200.loader import DeviceBatchLoader
    B, N, L, A, Vq, U = 5, 8, 6, 10, 30, 2
    model = _model((B, N, L, A, Vq, U))
    ds = _store(10, N, BF16)
    g = np.random.default_rng(2)
    S = 23
    qlen = g.integers(2, L + 1, S)
    samples = {"video_idx": g.integers(0, 10, S), "question": g.integers(2, Vq, (S, L)) * (np.arange(L)[None] < qlen[:, None]),
               "question_len": qlen, "answer": g.integers(0, A, S), "category": g.integers(0, 15, S)}
    loader = DeviceBatchLoader(ds, samples, batch_size=B, device="cuda", drop_last=False)
    assert len(loader) == 5
    ev, ref = EvalEngine(model, SVQA_CATEGORIES), EvalEngine(model, SVQA_CATEGORIES)
    seen = 0
    for rows, q, ql, ans, cat in loader:
        n = rows.shape[0]
        idx = np.arange(seen, seen + n)
        assert np.array_equal(rows.cpu().numpy(), samples["video_idx"][idx]) and rows.dtype == torch.int32
        assert np.array_equal(q.cpu().numpy(), samples["question"][idx]) and np.array_equal(cat.cpu().numpy(), samples["category"][idx])
        if n == B:
            if ev.graph is None:
                ev.capture_from_store(ds, rows, q, ql, ans, cat)
            ev.load_rows(rows, q, ql, ans, cat)
            ev.replay()
        else:
            ev.step_from_store(ds, rows, q, ql, ans, cat)                # the partial last batch runs eagerly
        ref.step(_gather(ds.app, rows), _gather(ds.mot, rows), q, ql, ans, cat)
        seen += n
    assert seen == S
    r, r_ref = ev.result(), ref.result()
    assert r["counts"] == r_ref["counts"] and r["counts"]["all"][1] == S
    assert ds.read_error() == 0
