"""Parameter-server / worker / trainer semantics on the CPU oracle (SURVEY 2.6, 4)."""
import socket
import threading

import numpy as np
import pytest
import torch

from distkeras_b200 import networking
from distkeras_b200.data import Dataset
from distkeras_b200.models import Dense, Sequential
from distkeras_b200.ops.flat_optim import FlatOptimizer
from distkeras_b200.parameter_servers import (ADAGParameterServer, DeltaParameterServer, DynSGDParameterServer,
                                              ExperimentalParameterServer)
from distkeras_b200.schemes import Emperor
from distkeras_b200.trainers import (ADAG, AEASGD, DOWNPOUR, EAMSGD, AveragingTrainer, DynSGD, EnsembleTrainer,
                                     Experimental, SingleTrainer)
from distkeras_b200.workers import AEASGDWorker


def tiny_model(seed=0):
    return Sequential([Dense(16, activation="relu", input_shape=(8,)), Dense(3, activation="softmax")], seed=seed)


def tiny_data(n=512, seed=0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, 8, generator=g)
    w = torch.randn(8, 3, generator=g)
    return Dataset({"features": x, "label": (x @ w).argmax(1).to(torch.int32)})


def test_wire_protocol_roundtrip():
    srv = socket.socket()
    srv.bind(("127.0.0.1", 0))
    srv.listen(1)
    port = srv.getsockname()[1]
    payload = {"worker_id": 3, "delta": np.arange(1000, dtype=np.float32), "nested": [np.ones((2, 3)), "x", 7]}
    got = {}

    def server():
        conn, _ = srv.accept()
        got["data"] = networking.recv_data(conn)
        networking.send_data(conn, {"ok": True, "echo": got["data"]["delta"][:5]})
        conn.close()

    t = threading.Thread(target=server)
    t.start()
    c = networking.connect("127.0.0.1", port)
    networking.send_data(c, payload)
    reply = networking.recv_data(c)
    t.join()
    c.close()
    srv.close()
    assert got["data"]["worker_id"] == 3 and np.array_equal(got["data"]["delta"], payload["delta"])
    assert np.array_equal(got["data"]["nested"][0], np.ones((2, 3))) and got["data"]["nested"][1:] == ["x", 7]
    assert reply["ok"] and np.array_equal(reply["echo"], np.arange(5, dtype=np.float32))
    assert networking.determine_host_address()


def test_delta_and_adag_server_accumulate():
    m = tiny_model()
    for cls, key in ((DeltaParameterServer, "delta"), (ADAGParameterServer, "residual")):
        ps = cls(m, None)
        ps.initialize_inproc()
        c0 = ps.center_variable.clone()
        total = torch.zeros_like(c0)
        for i in range(5):
            d = torch.randn_like(c0) * 0.01
            total += d
            ps.apply_commit({"worker_id": i % 2, key: d.numpy()})
        assert torch.allclose(ps.center_variable, c0 + total, atol=1e-6)
        assert ps.get_num_updates() == 6  # counter starts at 1 (parameter_servers.py:37)
        ps.finalize()
        assert torch.allclose(ps.get_model().get_flat_weights(), c0 + total, atol=1e-6)


def test_dynsgd_staleness_scaling():
    ps = DynSGDParameterServer(tiny_model(), None)
    ps.initialize_inproc()
    c0 = ps.center_variable.clone()
    r = torch.ones_like(c0)
    pull = ps.make_pull_payload()
    assert pull["update"] == 1
    ps.apply_commit({"worker_id": 0, "residual": r.numpy(), "last_update": 1})   # staleness 1
    ps.apply_commit({"worker_id": 1, "residual": r.numpy(), "last_update": 1})   # staleness 2
    ps.apply_commit({"worker_id": 1, "residual": r.numpy(), "last_update": 1})   # staleness 3
    assert torch.allclose(ps.center_variable, c0 + (1 + 0.5 + 1 / 3.0), atol=1e-6)


def test_experimental_damping():
    ps = ExperimentalParameterServer(tiny_model(), None, learning_rate=0.5)
    ps.initialize_inproc()
    c0 = ps.center_variable.clone()
    stale = c0 - 0.3
    r = torch.full_like(c0, 0.2)
    ps.apply_commit({"worker_id": 0, "residual": r.numpy(), "stale_center_variable": stale.numpy()})
    d = 1.0 / (2.0 * 0.3 ** 2 + 1.0)
    assert torch.allclose(ps.center_variable, c0 + d * 0.2, atol=1e-6)


def test_elastic_step_conserves_w_plus_c():
    m = tiny_model()
    ps = DeltaParameterServer(m, None)
    ps.initialize_inproc()
    w = AEASGDWorker(m, "sgd", "categorical_crossentropy", communication_window=4, rho=2.0, learning_rate=0.1)
    w.prepare_model()
    w.attach(ps)
    w.connect()
    with torch.no_grad():
        w.replica.W.data.add_(torch.randn_like(w.replica.W.data) * 0.1)
    before = w.replica.W.data.clone() + ps.center_variable
    w.elastic_step()
    assert torch.allclose(w.replica.W.data + ps.center_variable, before, atol=1e-6)


@pytest.mark.parametrize("cls,kw", [
    (ADAG, dict(communication_window=4)), (DOWNPOUR, dict(communication_window=3)),
    (AEASGD, dict(communication_window=4, rho=1.0, learning_rate=0.1)),
    (EAMSGD, dict(communication_window=4, rho=0.1, learning_rate=1.0, momentum=0.5)),
    (DynSGD, dict(communication_window=3)), (Experimental, dict(communication_window=3)),
])
def test_async_trainers_learn(cls, kw):
    ds = tiny_data(1024)
    opt = {"class_name": "adam", "config": {"lr": 0.02}}
    t = cls(tiny_model(0), opt, "categorical_crossentropy", num_workers=2, batch_size=16, num_epoch=2, **kw)
    t.backend = "thread"
    model = t.train(ds)
    model.compile("categorical_crossentropy")
    loss, acc = model.evaluate(ds["features"], ds["label"])
    assert acc > 0.55, (cls.__name__, loss, acc)
    h = t.get_history()
    assert {r["worker_id"] for r in h} == {0, 1} and len(h) == 2 * (512 // 16) * 2
    assert t.get_training_time() > 0 and t.num_updates() > 1
    assert len(t.get_averaged_history()) == (512 // 16) * 2
    assert len(t.get_executor_history(1)) == (512 // 16) * 2


def test_adag_center_equals_sum_of_residuals_single_worker():
    """One worker, deterministic: center == W0 + sum of committed residuals == replaying the loop."""
    ds = tiny_data(256)
    t = ADAG(tiny_model(0), "sgd", "categorical_crossentropy", num_workers=1, batch_size=16, communication_window=4)
    t.backend = "thread"
    model = t.train(ds)
    # oracle: plain loop with the same rule
    ref = tiny_model(0)
    ref.compile("categorical_crossentropy", "sgd")
    center = ref.get_flat_weights().clone()
    w1 = center.clone()
    x, y = ds["features"], ds["label"]
    for it in range(1, 17):
        ref.train_on_batch(x[(it - 1) * 16:it * 16], y[(it - 1) * 16:it * 16])
        if it % 4 == 0:
            center += (ref.get_flat_weights() - w1) / 4.0
            ref.set_flat_weights(center)
            w1 = center.clone()
    assert torch.allclose(model.get_flat_weights(), center, atol=1e-5)


def test_socket_backend_matches_thread_backend():
    ds = tiny_data(256)
    outs = []
    for backend in ("thread", "socket"):
        t = ADAG(tiny_model(0), "sgd", "categorical_crossentropy", num_workers=1, batch_size=16,
                 communication_window=4, master_port=0)
        t.backend = backend
        outs.append(t.train(ds).get_flat_weights())
    assert torch.allclose(outs[0], outs[1], atol=1e-6)


def test_single_averaging_ensemble():
    ds = tiny_data(512)
    adam = {"class_name": "adam", "config": {"lr": 0.02}}
    s = SingleTrainer(tiny_model(0), adam, "categorical_crossentropy", batch_size=16, num_epoch=2)
    s.backend = "thread"
    m = s.train(ds)
    assert len(s.get_history()) == 64
    m.compile("categorical_crossentropy")
    assert m.evaluate(ds["features"], ds["label"])[1] > 0.7
    a = AveragingTrainer(tiny_model(0), adam, "categorical_crossentropy", batch_size=16, num_epoch=2, num_workers=2)
    a.backend = "thread"
    ma = a.train(ds)
    ma.compile("categorical_crossentropy")
    assert ma.evaluate(ds["features"], ds["label"])[1] > 0.5
    e = EnsembleTrainer(tiny_model(0), adam, "categorical_crossentropy", batch_size=16, num_ensembles=3)
    e.backend = "thread"
    models = e.train(ds)
    assert len(models) == 3 and not torch.equal(models[0].get_flat_weights(), models[1].get_flat_weights())


def test_average_models_is_mean():
    a = AveragingTrainer(tiny_model(0), "sgd", "categorical_crossentropy")
    ms = [tiny_model(i) for i in range(3)]
    for m in ms:
        m.build()
    avg = a.average_models(ms)
    want = torch.stack([m.get_flat_weights() for m in ms]).mean(0)
    assert torch.allclose(avg.get_flat_weights(), want)
    avg2 = a.average_models(ms)  # buffer re-zeroed: same answer twice (reference bug, SURVEY 2.7)
    assert torch.allclose(avg2.get_flat_weights(), want)


def test_parallelism_factor_and_shuffle():
    ds = tiny_data(512)
    t = ADAG(tiny_model(0), "adam", "categorical_crossentropy", num_workers=2, batch_size=16, communication_window=2)
    t.backend = "thread"
    t.set_parallelism_factor(3)
    assert t.get_parallelism_factor() == 3
    t.train(ds, shuffle=True)
    assert len({h["worker_id"] for h in t.get_history()}) == 6  # 6 partitions over 2 worker threads


def test_emperor_scheme_decays_learning_rate():
    ds = tiny_data(256)
    t = AEASGD(tiny_model(0), "sgd", "categorical_crossentropy", num_workers=1, batch_size=16, communication_window=4,
               rho=1.0, learning_rate=0.1)
    t.backend = "thread"

    def evaluate_loss(model, val):
        return 1.0  # constant -> plateau from the second round on

    e = Emperor(t, evaluate_loss, num_epoch=2, evaluation_frequency=1, loss_threshold=0.005)
    e.optimize(ds, ds)
    assert t.get_learning_rate() < 0.1 and t.get_num_epoch() == 1


def test_nadam_is_adam_with_a_nesterov_look_ahead():
    """Nadam with a constant beta_1 (Dozat 2016, algorithm 8 without the momentum-decay schedule), float64 oracle."""
    torch.manual_seed(1)
    n, lr, b1, b2, eps = 101, 0.02, 0.9, 0.999, 1e-7
    w0 = torch.randn(n)
    grads = [torch.randn(n) for _ in range(6)]
    opt = FlatOptimizer({"class_name": "nadam", "config": {"lr": lr}}, n, "cpu")
    w = w0.clone()
    for g in grads:
        opt.step(w, g)
    x, m, v = w0.double(), torch.zeros(n, dtype=torch.float64), torch.zeros(n, dtype=torch.float64)
    for t, g in enumerate(grads, 1):
        g = g.double()
        m = b1 * m + (1 - b1) * g
        v = b2 * v + (1 - b2) * g * g
        look_ahead = b1 * m / (1 - b1 ** (t + 1)) + (1 - b1) * g / (1 - b1 ** t)
        x = x - lr * look_ahead / ((v / (1 - b2 ** t)).sqrt() + eps)
    assert torch.allclose(w.double(), x, atol=1e-5)
    # and it differs from plain Adam on the same gradients
    adam = FlatOptimizer({"class_name": "adam", "config": {"lr": lr}}, n, "cpu")
    wa = w0.clone()
    for g in grads:
        adam.step(wa, g)
    assert (wa - w).abs().max() > 1e-3


@pytest.mark.parametrize("name", ["sgd", "adagrad", "rmsprop", "adam", "adadelta", "adamax"])
def test_flat_optimizer_matches_torch(name):
    torch.manual_seed(0)
    n = 257
    w0 = torch.randn(n)
    grads = [torch.randn(n) for _ in range(5)]
    opt = FlatOptimizer({"class_name": name, "config": {"lr": 0.05} if name != "adadelta" else {}}, n, "cpu")
    w = w0.clone()
    for g in grads:
        opt.step(w, g)
    p = torch.nn.Parameter(w0.clone())
    eps = 1e-7
    ref = {"sgd": lambda: torch.optim.SGD([p], lr=0.05),
           "adagrad": lambda: torch.optim.Adagrad([p], lr=0.05, eps=eps),
           "rmsprop": lambda: torch.optim.RMSprop([p], lr=0.05, alpha=0.9, eps=eps),
           "adam": lambda: torch.optim.Adam([p], lr=0.05, eps=eps),
           "adadelta": lambda: torch.optim.Adadelta([p], lr=1.0, rho=0.95, eps=eps),
           "adamax": lambda: torch.optim.Adamax([p], lr=0.05, eps=eps)}[name]()
    for g in grads:
        p.grad = g.clone()
        ref.step()
    tol = 2e-3 if name in ("adam", "adamax") else 1e-5  # Keras vs torch epsilon placement differs slightly
    assert torch.allclose(w, p.data, atol=tol), (name, float((w - p.data).abs().max()))


def test_multiple_feature_columns_are_concatenated():
    g = torch.Generator().manual_seed(0)
    a, b = torch.randn(256, 5, generator=g), torch.randn(256, 3, generator=g)
    w = torch.randn(8, 3, generator=g)
    ds = Dataset({"fa": a, "fb": b, "label": (torch.cat([a, b], 1) @ w).argmax(1).to(torch.int32)})
    t = SingleTrainer(tiny_model(0), {"class_name": "adam", "config": {"lr": 0.02}}, "categorical_crossentropy",
                      features_col=["fa", "fb"], batch_size=16, num_epoch=3)
    t.backend = "thread"
    m = t.train(ds)
    m.compile("categorical_crossentropy")
    assert m.evaluate(torch.cat([a, b], 1), ds["label"])[1] > 0.6


def test_synchronous_easgd_lockstep():
    """Synchronous EASGD: every window all workers read the SAME center (two rendezvous per round), so the
    center moves by exactly sum_i alpha (W_i - C_old); 2 workers x (32 batches / window 4) = 16 commits."""
    from distkeras_b200.trainers import EASGD, SynchronousDistributedTrainer

    ds = tiny_data(1024)
    t = EASGD(tiny_model(0), {"class_name": "adam", "config": {"lr": 0.02}}, "categorical_crossentropy", num_workers=2,
              batch_size=16, num_epoch=1, communication_window=4, rho=1.0, learning_rate=0.25)
    assert isinstance(t, SynchronousDistributedTrainer)
    t.backend = "thread"
    model = t.train(ds)
    assert t.num_updates() == 1 + 2 * (32 // 4)
    model.compile("categorical_crossentropy")
    assert model.evaluate(ds["features"], ds["label"])[1] > 0.6
    # the commits of one round are interleaved pairwise: worker ids alternate in blocks of two
    order = [wid for wid, _ in sorted(((h["worker_id"], h["iteration"]) for h in t.get_history()), key=lambda p: p[1])]
    assert set(order) == {0, 1}


def _oracle_run(rule, n_batches=16, tau=4, **hp):
    """Replay one worker's loop by hand (SURVEY 2.6 A-F) and return the final center."""
    ds = tiny_data(16 * n_batches)
    ref = tiny_model(0)
    ref.compile("categorical_crossentropy", "sgd")
    C = ref.get_flat_weights().clone()   # center
    W1 = C.clone()
    x, y = ds["features"], ds["label"]
    r = torch.zeros_like(C)
    updates = 1  # the PS counter starts at 1
    last_update = 1  # value returned by the initial pull
    for it in range(1, n_batches + 1):
        batch = (x[(it - 1) * 16:it * 16], y[(it - 1) * 16:it * 16])
        if rule in ("downpour", "aeasgd", "eamsgd") and it % tau == 0:  # check BEFORE the batch
            W = ref.get_flat_weights()
            if rule == "downpour":
                C = C + (W - W1)
                ref.set_flat_weights(C)
                W1 = C.clone()
            else:
                E = hp["rho"] * hp["lr"] * (W - C)
                ref.set_flat_weights(W - E)
                C = C + E
        if rule == "eamsgd":
            W = ref.get_flat_weights()
            r_t = hp["momentum"] * r
            W_copy = W.clone()
            ref.set_flat_weights(W + r_t)
            before = ref.get_flat_weights().clone()
            ref.train_on_batch(*batch)
            g = ref.get_flat_weights() - before
            r = r_t - hp["lr"] * g
            ref.set_flat_weights(W_copy - r)
        else:
            ref.train_on_batch(*batch)
        if rule in ("dynsgd", "experimental") and it % tau == 0:  # check AFTER the batch
            W = ref.get_flat_weights()
            if rule == "dynsgd":
                staleness = (updates - last_update) + 1
                C = C + (W - W1) / staleness
                updates += 1
                last_update = updates
            else:
                res = (W - W1) / tau
                d = 1.0 / ((1.0 / hp["lr"]) * (C - W1) ** 2 + 1.0)  # C_stale == W1 for a single worker
                C = C + d * res
            ref.set_flat_weights(C)
            W1 = C.clone()
    return ds, C


@pytest.mark.parametrize("rule,cls,kw,hp", [
    ("downpour", DOWNPOUR, dict(communication_window=4), {}),
    ("aeasgd", AEASGD, dict(communication_window=4, rho=2.0, learning_rate=0.1), dict(rho=2.0, lr=0.1)),
    ("eamsgd", EAMSGD, dict(communication_window=4, rho=2.0, learning_rate=0.1, momentum=0.5),
     dict(rho=2.0, lr=0.1, momentum=0.5)),
    ("dynsgd", DynSGD, dict(communication_window=4), {}),
    ("experimental", Experimental, dict(communication_window=4, learning_rate=0.5), dict(lr=0.5)),
])
def test_single_worker_center_matches_hand_replay(rule, cls, kw, hp):
    """One worker, plain SGD, deterministic: the trainer's final center equals the algorithm replayed by
    hand from the formulas of SURVEY 2.6 (reference ``workers.py`` / ``parameter_servers.py``)."""
    ds, want = _oracle_run(rule, **hp)
    t = cls(tiny_model(0), "sgd", "categorical_crossentropy", num_workers=1, batch_size=16, **kw)
    t.backend = "thread"
    got = t.train(ds).get_flat_weights()
    assert torch.allclose(got, want, atol=2e-5), (rule, float((got - want).abs().max()))


@pytest.mark.parametrize("cls,kw", [(ADAG, dict(communication_window=4)),
                                    (AEASGD, dict(communication_window=4, rho=1.0, learning_rate=0.1)),
                                    (EAMSGD, dict(communication_window=4, rho=0.1, learning_rate=1.0, momentum=0.5))])
def test_library_collectives_baseline_backend(cls, kw, monkeypatch):
    """backend="nccl" (gloo on a CPU host): two spawned ranks, bulk-synchronous all-reduce every window."""
    # the CPU host path on any machine: on a GPU host the backend runs one rank per GPU, so a one-GPU host
    # would train a single worker
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")       # the spawned ranks
    monkeypatch.setattr(torch.cuda, "device_count", lambda: 0)   # the launcher (CUDA may be initialised here)
    ds = tiny_data(1024)
    t = cls(tiny_model(0), {"class_name": "adam", "config": {"lr": 0.02}}, "categorical_crossentropy", num_workers=2,
            batch_size=16, num_epoch=2, **kw)
    t.backend = "nccl"
    model = t.train(ds)
    h = t.get_history()
    assert len(h) == 2 * 2 * (512 // 16) and {r["worker_id"] for r in h} == {0, 1}
    assert t.num_updates() == 1 + 2 * (2 * (512 // 16) // 4)
    model.compile("categorical_crossentropy")
    assert model.evaluate(ds["features"], ds["label"])[1] > 0.6
