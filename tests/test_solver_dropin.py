"""A real Flashy solver on the ``flashy_b200`` path.

The UNMODIFIED reference package (``oracle/_ref/flashy``, installed by ``oracle/install_ref.py``:
``BaseSolver`` / ``run_stage`` / ``commit`` / ``restore`` of ``flashy/solver.py:30-211``, ``StateManager``,
``AdversarialLoss`` of ``flashy/adversarial.py:22-89``, the logger stack) is imported with
``flashy.distrib`` aliased to ``flashy_b200.distrib`` exactly as INTEGRATION.md section 1 shows; ``dora``
and ``colorlog`` are the test-only stand-ins of ``tests/shims``.  The solvers below restate the
reference's own example solvers (``examples/basic/train.py:12-41``, ``examples/cifar/solver.py:11-63``,
``tests/dummy/train.py:40-107``) so that the tests read like the reference's ``tests/test_integ.py``.

CPU part (W = 1): BASELINE configs[0] -- stages, metric history, checkpoints, restore.
GPU part: the CIFAR-style step and ``AdversarialLoss.train_adv`` on 4 virtual ranks, compared with
the oracle (per-rank gradients averaged by ``oracle/numeric.py``, then the same optimizer step).
"""
import sys
from argparse import Namespace
from pathlib import Path

import pytest
import torch
from torch import nn
from torch.nn import functional as F

ROOT = Path(__file__).resolve().parent.parent
REF = ROOT / "oracle" / "_ref"
SHIMS = ROOT / "tests" / "shims"


@pytest.fixture(scope="module")
def flashy():
    if not (REF / "flashy" / "solver.py").exists():
        pytest.skip("upstream Flashy is not installed in oracle/_ref (build() installs it from an upstream checkout)")
    if str(SHIMS) not in sys.path:
        sys.path.insert(0, str(SHIMS))
    if str(REF) not in sys.path:
        sys.path.append(str(REF))
    import flashy_b200.distrib
    sys.modules["flashy.distrib"] = flashy_b200.distrib          # INTEGRATION.md section 1
    import flashy as pkg
    assert pkg.distrib is flashy_b200.distrib
    assert Path(pkg.__file__).resolve().is_relative_to(REF.resolve())
    import flashy.adversarial
    assert flashy.adversarial.distrib is flashy_b200.distrib
    return pkg


# ------------------------------------------------------------------------------------------ solvers
def basic_solver(flashy, cfg):
    """examples/basic/train.py:12-41."""
    class Solver(flashy.BaseSolver):
        def __init__(self, cfg):
            super().__init__()
            self.cfg = cfg
            self.model = torch.nn.Linear(32, 1)
            self.optim = torch.optim.Adam(self.model.parameters(), lr=cfg.lr)
            self.best_state = {}
            self.register_stateful('model', 'optim', 'best_state')

        def run(self):
            self.restore()
            for epoch in range(self.epoch, self.cfg.epochs + 1):
                self.run_stage('train', self.train)
                self.commit(save_checkpoint=epoch % 2 == 1)
                if epoch == self.cfg.stop_at:
                    return

        def train(self):
            x = torch.randn(4, 32)
            loss = self.model(x).abs().mean()
            loss.backward()
            self.optim.step()
            self.optim.zero_grad()
            return {'loss': loss.item()}
    return Solver(cfg)


class SmallNet(nn.Module):
    """A few convolution / batch-norm / linear layers: 10 parameter tensors + BN buffers."""

    def __init__(self):
        super().__init__()
        self.conv1 = nn.Conv2d(3, 8, 3, padding=1)
        self.bn1 = nn.BatchNorm2d(8)
        self.conv2 = nn.Conv2d(8, 16, 3, padding=1, stride=2)
        self.bn2 = nn.BatchNorm2d(16)
        self.fc = nn.Linear(16 * 4 * 4, 10)

    def forward(self, x):
        x = F.relu(self.bn1(self.conv1(x)))
        x = F.relu(self.bn2(self.conv2(x)))
        return self.fc(F.adaptive_avg_pool2d(x, 4).flatten(1))


def cifar_solver(flashy, cfg, model, batches, optim):
    """examples/cifar/solver.py:11-63 (the loader is a list of batches already on the device)."""
    class Solver(flashy.BaseSolver):
        def __init__(self):
            super().__init__()
            self.h = cfg
            self.model = model
            self.optim = optim
            self.register_stateful('model', 'optim')

        def run(self):
            self.restore()
            for epoch in range(self.epoch, self.h.epochs + 1):
                self.run_stage("train", self.do_train_valid, train=True)
                self.commit()

        def get_formatter(self, stage_name):
            return flashy.Formatter({'acc': '.1%', 'loss': '.5f'})

        def do_train_valid(self, train=True):
            lp = self.log_progress(self.current_stage, batches, total=len(batches), updates=self.h.log_updates)
            average = flashy.averager()
            for idx, (img, label) in enumerate(lp):
                est = self.model(img)
                loss = F.cross_entropy(est, label)
                acc = (est.argmax(dim=-1).float() == label).float().mean()
                if train:
                    loss.backward()
                    flashy.distrib.sync_model(self.model)
                    self.optim.step()
                    self.optim.zero_grad()
                metrics = average({'acc': acc, 'loss': loss})
                lp.update(**metrics)
            return flashy.distrib.average_metrics(metrics, len(batches))
    return Solver()


class Network(nn.Module):
    """tests/dummy/train.py:16-25."""

    def __init__(self, dim=8):
        super().__init__()
        self.model = nn.Sequential(nn.Linear(dim, dim), nn.ReLU(), nn.Linear(dim, dim))

    def forward(self, x):
        return self.model(x)


def gan_solver(flashy, cfg, device):
    """tests/dummy/train.py:40-107: teacher / student / adversary, two optimizers."""
    distrib = flashy.distrib

    class NoiseDataset:
        def __init__(self, size, dim):
            self.size, self.dim = size, dim

        def __len__(self):
            return self.size

        def __getitem__(self, index):
            return torch.randn(self.dim)

    class Solver(flashy.BaseSolver):
        def __init__(self):
            super().__init__()
            self.h = cfg
            self.teacher = Network(cfg.dim).to(device)
            distrib.broadcast_model(self.teacher)
            self.model = Network(cfg.dim).to(device)
            distrib.broadcast_model(self.model)
            self.optim = torch.optim.Adam(self.model.parameters())
            adv_model = Network(cfg.dim).to(device)
            adv_opt = torch.optim.Adam(adv_model.parameters())
            self.adv = flashy.adversarial.AdversarialLoss(adv_model, adv_opt)
            self.loader = distrib.loader(NoiseDataset(cfg.dset_size, cfg.dim), shuffle=True, batch_size=cfg.batch_size)
            self.register_stateful('teacher', 'model', 'optim', 'adv')

        def run(self):
            self.restore()
            for epoch in range(self.epoch, self.h.epochs + 1):
                self.run_stage("train", self.do_train_valid, train=True)
                self.run_stage("valid", self.do_train_valid, train=False)
                self.commit()
                if epoch == self.h.stop_at:
                    return

        def do_train_valid(self, train=True):
            label = "train" if train else "valid"
            lp = self.log_progress(label, self.loader, updates=self.h.log_updates)
            average = flashy.averager()
            for noise in lp:
                noise = noise.to(device)
                estimate = self.model(noise)
                gt = self.teacher(noise)
                mse = F.mse_loss(estimate, gt)
                adv_disc = self.adv.train_adv(estimate, gt)
                adv_gen = self.adv(estimate)
                loss = mse + adv_gen
                if train:
                    self.optim.zero_grad()
                    loss.backward()
                    distrib.sync_model(self.model)
                    self.optim.step()
                metrics = average({'loss': loss, 'mse': mse, 'adv_disc': adv_disc, 'adv_gen': adv_gen})
                lp.update(**metrics)
            return distrib.average_metrics(metrics, len(self.loader))
    return Solver()


# ------------------------------------------------------------------------------------------ W = 1 (CPU)
def test_basic_solver_stages_commit_restore(flashy, tmp_path):
    """BASELINE configs[0] and the reference's checkpoint/resume test (tests/test_integ.py:18-27)."""
    import dora
    cfg = Namespace(lr=0.1, epochs=4, stop_at=2)
    dora.use_xp(dora.XP(tmp_path, cfg))
    try:
        flashy.setup_logging()
        flashy.distrib.init()                                   # no-op: single process
        torch.manual_seed(0)
        solver = basic_solver(flashy, cfg)
        solver.run()
        assert len(solver.history) == 2 and solver.epoch == 3
        assert all(set(h) == {'train'} and {'loss', 'duration'} <= set(h['train']) for h in solver.history)
        assert solver.checkpoint_path.exists()                  # written at epoch 1 (odd epochs only)
        assert dora.get_xp().link.updates == 2                  # rank zero reported both epochs
        first = [dict(h['train']) for h in solver.history]

        dora.use_xp(dora.XP(tmp_path, cfg))                     # a fresh process would start like this
        cfg.stop_at = None
        again = basic_solver(flashy, cfg)
        again.run()
        # the checkpoint of epoch 1 is restored (epoch 2 was not saved), then epochs 2..4 run
        assert len(again.history) == 4
        assert again.history[0]['train'] == first[0]
        state = torch.load(again.checkpoint_path, 'cpu')
        assert set(state) == {'history', 'xp.cfg', 'xp.sig', 'model', 'optim', 'best_state'}
        assert len(state['history']) == 3                       # saved at epoch 3

        with pytest.raises(RuntimeError):
            again.log_metrics('train', {})                      # outside a stage without a formatter
        assert flashy.distrib.average_metrics({'a': 1.0}, 3) == {'a': 1.0}      # W = 1: input returned
    finally:
        dora.use_xp(None)


# ------------------------------------------------------------------------------------------ GPU
def _numeric():
    from oracle import numeric
    return numeric


def _per_rank_batches(world, steps, seed=7):
    gens = [torch.Generator().manual_seed(seed + r) for r in range(world)]
    return [[(torch.randn(8, 3, 16, 16, generator=gens[r]), torch.randint(0, 10, (8,), generator=gens[r]))
             for _ in range(steps)] for r in range(world)]


@pytest.mark.gpu
def test_cifar_solver_step_on_four_virtual_ranks(flashy, tmp_path):
    """examples/cifar: loss.backward(); flashy.distrib.sync_model(model); optim.step() inside run_stage,
    against per-rank gradients averaged by the oracle and the same SGD step."""
    import dora
    from flashy_b200 import VirtualWorld
    numeric = _numeric()
    world, steps, lr = 4, 2, 0.05
    torch.backends.cudnn.deterministic = True
    dev = torch.device("cuda", 0)
    data = _per_rank_batches(world, steps)
    torch.manual_seed(1234)
    init = SmallNet().to(dev)

    # ---- oracle: every step, each rank's gradients and BN statistics from identical weights
    replicas = []
    for r in range(world):
        m = SmallNet().to(dev)
        m.load_state_dict(init.state_dict())
        replicas.append(m)
    for s in range(steps):
        grads, bufs = [], []
        for r, m in enumerate(replicas):
            img, label = (t.to(dev) for t in data[r][s])
            m.zero_grad()
            F.cross_entropy(m(img), label).backward()
            grads.append([p.grad.detach().cpu() for p in m.parameters()])
            bufs.append([b.detach().cpu() for b in m.buffers() if b.dtype.is_floating_point])
        mean_g = numeric.average_tensors(grads)[0]
        mean_b = numeric.average_tensors(bufs)[0]
        for m in replicas:
            with torch.no_grad():
                for p, g in zip(m.parameters(), mean_g):
                    p.add_(g.to(dev), alpha=-lr)
                for b, v in zip([b for b in m.buffers() if b.dtype.is_floating_point], mean_b):
                    b.copy_(v.to(dev))
    want = [p.detach().cpu() for p in replicas[0].parameters()]
    want_buf = [b.detach().cpu() for b in replicas[0].buffers()]

    vw = VirtualWorld(world, device=0, arena_mb=64)
    cfg = Namespace(epochs=1, log_updates=1, device="cuda")
    try:
        def body(rank, w):
            dora.use_xp(dora.XP(tmp_path / f"rank{rank}", cfg))
            model = SmallNet().to(dev)
            model.load_state_dict(init.state_dict())
            optim = torch.optim.SGD(model.parameters(), lr=lr)
            batches = [(img.to(dev), label.to(dev)) for img, label in data[rank]]
            solver = cifar_solver(flashy, cfg, model, batches, optim)
            solver.run()
            torch.cuda.synchronize()
            assert len(solver.history) == 1 and {'acc', 'loss', 'duration'} <= set(solver.history[0]['train'])
            assert solver.checkpoint_path.exists() == (rank == 0)          # commit writes on rank zero only
            return ([p.detach().cpu() for p in model.parameters()], [b.detach().cpu() for b in model.buffers()],
                    solver.history[0]['train'])
        got = vw.run(body)
    finally:
        vw.close()
    for r in range(world):
        for g, w_ in zip(got[r][0], want):
            assert torch.allclose(g, w_, rtol=0, atol=2e-6), (g - w_).abs().max()
        for g, w_ in zip(got[r][1], want_buf):
            assert torch.allclose(g.float(), w_.float(), rtol=0, atol=2e-6)
        for g0, g in zip(got[0][0], got[r][0]):
            assert torch.equal(g0, g)                                       # replicas stay bit-identical
        assert got[r][2]['loss'] == got[0][2]['loss'] and got[r][2]['acc'] == got[0][2]['acc']


@pytest.mark.gpu
def test_adversarial_loss_train_adv_on_four_virtual_ranks(flashy):
    """flashy/adversarial.py:49 (broadcast_model at construction) and :64-80 (train_adv: backward inside
    distrib.eager_sync_model, then the adversary's optimizer steps) against the oracle."""
    from flashy_b200 import VirtualWorld
    numeric = _numeric()
    world, dim, lr = 4, 8, 0.1
    dev = torch.device("cuda", 0)
    gens = [torch.Generator().manual_seed(50 + r) for r in range(world)]
    fakes = [torch.randn(16, dim, generator=g) for g in gens]
    reals = [torch.randn(16, dim, generator=g) for g in gens]
    torch.manual_seed(99)
    src = Network(dim)                                                    # rank 0's adversary: what everyone gets

    grads = []
    for r in range(world):
        adv = Network(dim).to(dev)
        adv.load_state_dict(src.state_dict())
        lf, lr_ = adv(fakes[r].to(dev)), adv(reals[r].to(dev))
        loss = F.binary_cross_entropy_with_logits(lf, torch.ones_like(lf)) + F.binary_cross_entropy_with_logits(lr_, torch.zeros_like(lr_))
        loss.backward()
        grads.append([p.grad.detach().cpu() for p in adv.parameters()])
    mean_g = numeric.average_tensors(grads)[0]
    ref = Network(dim).to(dev)
    ref.load_state_dict(src.state_dict())
    opt = torch.optim.SGD(ref.parameters(), lr=lr)
    for p, g in zip(ref.parameters(), mean_g):
        p.grad = g.to(dev)
    opt.step()
    want = [p.detach().cpu() for p in ref.parameters()]

    vw = VirtualWorld(world, device=0, arena_mb=64)
    try:
        def body(rank, w):
            torch.manual_seed(1000 + rank)                                # different initial weights per rank ...
            adversary = Network(dim).to(dev)
            if rank == 0:
                adversary.load_state_dict(src.state_dict())
            optimizer = torch.optim.SGD(adversary.parameters(), lr=lr)
            adv_loss = flashy.adversarial.AdversarialLoss(adversary, optimizer)     # ... until broadcast_model
            for p, q in zip(adversary.parameters(), src.parameters()):
                assert torch.equal(p.detach().cpu(), q.detach())
            loss = adv_loss.train_adv(fakes[rank].to(dev), reals[rank].to(dev))
            gen = adv_loss(fakes[rank].to(dev))
            torch.cuda.synchronize()
            assert loss.dim() == 0 and gen.dim() == 0
            state = adv_loss.state_dict()
            assert 'optimizer' in state                                   # adversarial.py:53-57
            return [p.detach().cpu() for p in adversary.parameters()]
        got = vw.run(body)
    finally:
        vw.close()
    for r in range(world):
        for g, w_ in zip(got[r], want):
            assert torch.allclose(g, w_, rtol=0, atol=1e-6), (g - w_).abs().max()
    for r in range(1, world):
        for a, b in zip(got[0], got[r]):
            assert torch.equal(a, b)


@pytest.mark.gpu
def test_gan_solver_two_optimizers_runs_and_resumes(flashy, tmp_path):
    """BASELINE configs[3] / tests/test_integ.py:18-29 on the CUDA path: the dummy GAN solver (sync_model
    for the generator, eager_sync_model inside AdversarialLoss) on 2 virtual ranks, stop at epoch 2,
    resume to 4; replicas must stay identical and the history must survive the restart."""
    import dora
    from flashy_b200 import VirtualWorld
    dev = torch.device("cuda", 0)
    world = 2
    cfg = Namespace(dim=4, dset_size=16, batch_size=4, epochs=4, stop_at=2, log_updates=1, device="cuda")

    def run_once(stop_at):
        vw = VirtualWorld(world, device=0, arena_mb=64)
        try:
            def body(rank, w):
                dora.use_xp(dora.XP(tmp_path / f"rank{rank}", cfg))
                torch.manual_seed(1234)
                cfg_r = Namespace(**{**vars(cfg), "stop_at": stop_at})
                solver = gan_solver(flashy, cfg_r, dev)
                if rank != 0 and stop_at is None:
                    # only rank 0 wrote checkpoint.th (solver.py:153): give the others the same file, as a
                    # shared experiment folder would
                    import shutil
                    shutil.copy(tmp_path / "rank0" / "checkpoint.th", tmp_path / f"rank{rank}" / "checkpoint.th")
                solver.run()
                torch.cuda.synchronize()
                params = [p.detach().cpu() for m in (solver.model, solver.adv.adversary) for p in m.parameters()]
                return len(solver.history), [dict(h) for h in solver.history], params
            return vw.run(body)
        finally:
            vw.close()

    first = run_once(2)
    assert [f[0] for f in first] == [2, 2]
    for a, b in zip(first[0][2], first[1][2]):
        assert torch.equal(a, b)
    for stage in ("train", "valid"):
        assert first[0][1][0][stage]['loss'] == first[1][1][0][stage]['loss']       # average_metrics agrees
    second = run_once(None)
    assert [s[0] for s in second] == [4, 4]
    assert second[0][1][:2] == first[0][1]                                          # first two epochs unchanged
    for a, b in zip(second[0][2], second[1][2]):
        assert torch.equal(a, b)
