"""Host logic of the training-step harness (ffc_b200/train.py, SURVEY 8(f) rank 4) on CPU with a stand-in module: batch composition
(main.py:49-60), the AMP step sequence (main.py:53-71), id-loader restart (main.py:43-47), label hand-over one step ahead, and the
snapshot dict (main.py:84-85)."""
import os

import torch
import torch.nn as nn

from ffc_b200 import train as T


def test_compose_batch_is_main_py_49_60():
    B = 8
    images1, images2 = torch.randn(B // 2, 3, 4, 4), torch.randn(B // 2, 3, 4, 4)
    ids = torch.tensor([7, 3, 9, 1])
    ins, lab = torch.randn(B, 3, 4, 4), torch.arange(100, 100 + B)
    x, y, xl, yl = T.compose_batch(images1, images2, ids, ins, lab)
    # the reference, verbatim shapes: chunk the instance batch in two, id half first
    assert torch.equal(x, torch.cat([images1, ins[:4]])) and torch.equal(y, torch.cat([images2, ins[4:]]))
    assert xl.tolist() == [7, 3, 9, 1, 100, 101, 102, 103] and yl.tolist() == [7, 3, 9, 1, 104, 105, 106, 107]
    assert xl.dtype == torch.int64 and not xl.is_cuda


def test_synthetic_source_shapes_and_determinism():
    src = T.SyntheticSource(num_class=50, batch_size=8, image_size=6, batches_per_epoch=3, seed=4)
    a = list(src.instance_loader(epoch=1))
    b = list(src.instance_loader(epoch=1))
    assert len(a) == len(src) == 3 and all(torch.equal(u[0], v[0]) and torch.equal(u[1], v[1]) for u, v in zip(a, b))
    img, lab, extra = a[0]
    assert img.shape == (8, 3, 6, 6) and lab.shape == (8,) and lab.dtype == torch.int64 and extra == -1
    it = src.id_loader()
    v1, v2, ids = next(it)
    assert v1.shape == v2.shape == (4, 3, 6, 6) and ids.shape == (4,) and len(set(ids.tolist())) == 4 and int(ids.max()) < 50
    seen = ids.tolist()
    for _ in range(11):                     # 12 batches of 4 = one pass over 48 of the 50 identities: no identity twice
        seen += next(it)[2].tolist()
    assert len(set(seen)) == 48


class _FakeFFC(nn.Module):
    """differentiable stand-in with the FFC call signature; records what it is given and when"""

    def __init__(self):
        super().__init__()
        self.w = nn.Parameter(torch.ones(1))
        self.calls, self.prefetched = [], []

    def forward(self, x, y, x_label, y_label):
        self.calls.append((x.shape[0], x_label.clone(), y_label.clone(), torch.is_autocast_enabled('cpu')))
        return (self.w * (x.mean() + y.mean())) ** 2 + self.w

    def prefetch_labels(self, x_label, y_label):
        self.prefetched.append((len(self.calls), x_label, y_label))

    def checkpoint(self):
        return {'state_dict': self.state_dict(), 'lru': [(1, 0)], 'fc': torch.zeros(2, 4, 2), 'qp': {0: 1}}


def test_train_one_epoch_sequence(tmp_path):
    src = T.SyntheticSource(num_class=9, batch_size=8, image_size=4, batches_per_epoch=5, seed=1)
    net = _FakeFFC()
    opt = torch.optim.SGD(net.parameters(), lr=0.1)
    scaler = torch.amp.GradScaler('cpu', enabled=False)
    w0 = float(net.w)
    logs = []

    def short_id_loader():                  # 2 batches, then exhausted: main.py:43-47 restarts it
        it = src.id_loader()
        for _ in range(2):
            yield next(it)

    class Restartable:
        def __iter__(self):
            return short_id_loader()

    n = T.train_one_epoch(Restartable(), src.instance_loader(), net, opt, scaler, cur_epoch=1, saved_dir=str(tmp_path), real_iter=0,
                          save_every=2, device='cpu', autocast_dtype=torch.bfloat16, log=logs.append)
    assert n == 5 and len(net.calls) == 5 and float(net.w) != w0
    assert all(c[0] == 8 and c[3] for c in net.calls)                     # full batches, under autocast
    # the id half is the same in x and y, the instance halves differ (main.py:58-60)
    for _, xl, yl, _ in net.calls:
        assert torch.equal(xl[:4], yl[:4]) and len(set(xl[:4].tolist())) == 4
    # labels of step k+1 were handed over right after step k was issued, and are the objects step k+1 then receives
    assert [p[0] for p in net.prefetched] == [1, 2, 3, 4]
    for (k, xl, yl), call in zip(net.prefetched, net.calls[1:]):
        assert torch.equal(xl, call[1]) and torch.equal(yl, call[2])
    # snapshots every 2 iterations in the reference's wire format (main.py:84-85)
    assert sorted(os.listdir(tmp_path)) == ['1.pt', '2.pt'] and [l['iter'] for l in logs] == [2, 4]
    ck = torch.load(os.path.join(tmp_path, '1.pt'), weights_only=False)
    assert set(ck) == {'state_dict', 'lru', 'fc', 'qp'}


def test_ir100_is_registered_for_c4(tmp_path, monkeypatch):
    """C4 names ResNet-100: the reference defines iresnet100 (resnet_arcface.py:177) but its create_net does not list it, so create_net
    takes it from model.resnet_arcface.  Checked against a stand-in `model` package with the reference's layout; without any backbone
    package on sys.path the name is a ValueError."""
    import sys
    import pytest
    from ffc_b200 import ffc as F_
    for name in ('model', 'model.resnet_arcface'):
        monkeypatch.delitem(sys.modules, name, raising=False)
    with pytest.raises(ValueError):
        F_.create_net('ir100', feat_dim=512)
    pkg = tmp_path / 'model'
    pkg.mkdir()
    (pkg / '__init__.py').write_text('def create_net(net_type, **kwargs):\n    return ("create_net", net_type, kwargs)\n')
    (pkg / 'resnet_arcface.py').write_text('def iresnet100(**kwargs):\n    return ("iresnet100", kwargs)\n')
    monkeypatch.syspath_prepend(str(tmp_path))
    try:
        assert F_.create_net('ir100', feat_dim=512, fp16=False) == ('iresnet100', {'feat_dim': 512, 'fp16': False})
        assert F_.create_net('ir50', feat_dim=512) == ('create_net', 'ir50', {'feat_dim': 512})      # the others: the package's create_net
    finally:
        for name in ('model', 'model.resnet_arcface'):
            sys.modules.pop(name, None)
