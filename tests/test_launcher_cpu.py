"""CPU: the launcher swaps the class inside the UNMODIFIED reference's define_G (needs the original DAHiTra sources:
$DAHITRA_REFERENCE, else the copy baseline/install_reference.py places under baseline/_ref/ref), and the world_size-2
gloo path of the pair sharding used by bench.py."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("DAHITRA_REFERENCE", os.path.join(ROOT, "baseline", "_ref", "ref"))
NO_REF = f"original DAHiTra sources not found at {REF} (set DAHITRA_REFERENCE or run baseline/install_reference.py)"


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "models")), reason=NO_REF)
def test_reference_define_G_builds_the_native_class():
    code = (
        "import torch\n"
        "from dahitra_b200.launch import install\n"
        f"nets = install({REF!r}, stub_missing=True)\n"
        "class A: net_G = 'newUNetTrans'\n"
        "torch.manual_seed(0)\n"
        "net = nets.define_G(A(), gpu_ids=[])\n"      # the reference's own factory, init_net and init_weights
        "assert type(net).__module__ == 'dahitra_b200.networks', type(net)\n"
        "sd = net.state_dict()\n"
        "assert len(sd) == 425\n"
        "print('OK', float(sd['classifier.weight'].double().sum()))\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "OK" in r.stdout


@pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "models")), reason=NO_REF)
def test_pretrained_trunk_path_equals_the_reference(tmp_path):
    """The reference's define_G with its pretrained=True trunk left ON (models/networks.py:1096; load_state_dict_from_url served
    from a local file instead of the network) against dahitra_b200's define_G reading the same file: all 425 tensors bit-identical
    under the same seed, ImageNet BatchNorm running statistics included."""
    code = (
        "import sys, torch\n"
        "from dahitra_b200 import modules as M\n"
        "torch.manual_seed(99)\n"
        "donor = M.Trunk()\n"
        "for m in donor.modules():\n"
        "    if isinstance(m, torch.nn.BatchNorm2d):\n"
        "        m.running_mean.normal_(); m.running_var.uniform_(0.5, 2.0)\n"
        "ckpt = {k: v for k, v in donor.state_dict().items() if not k.endswith('num_batches_tracked')}\n"
        f"path = {str(tmp_path / 'resnet18-5c106cde.pth')!r}\n"
        "torch.save(ckpt, path)\n"
        "from dahitra_b200.launch import install\n"
        f"nets = install({REF!r}, stub_missing=True, rebind=False)\n"      # the reference's own class, trunk NOT patched
        "import models.resnet as R\n"
        "R.load_state_dict_from_url = lambda url, progress=True: torch.load(path)\n"
        "class A: net_G = 'newUNetTrans'\n"
        "torch.manual_seed(0)\n"
        "ref = nets.define_G(A(), gpu_ids=[])\n"
        "assert type(ref).__module__ == 'models.networks', type(ref)\n"
        "import os; os.environ['DAHITRA_RESNET18_CKPT'] = path\n"
        "from dahitra_b200.networks import define_G\n"
        "torch.manual_seed(0)\n"
        "net = define_G(A(), gpu_ids=[])\n"
        "a, b = ref.state_dict(), net.state_dict()\n"
        "assert list(a) == list(b) and len(a) == 425\n"
        "bad = [k for k in a if not torch.equal(a[k], b[k])]\n"
        "assert not bad, bad[:5]\n"
        "assert torch.equal(b['resnet.bn1.running_mean'], ckpt['bn1.running_mean'])\n"
        "print('OK')\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "OK" in r.stdout


SHARD_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, os.environ["DAHITRA_ROOT"])
from dahitra_b200.sharding import shard_pairs, gather_max_ms
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%s" % os.environ["PORT"],
                        rank=int(os.environ["RANK"]), world_size=2)
r = dist.get_rank()
lo, hi = shard_pairs(11, r, 2)
assert (lo, hi) == ((0, 6) if r == 0 else (6, 11)), (lo, hi)
lo, hi = shard_pairs(64, r, 2)
assert hi - lo == 32
ms = gather_max_ms(10.0 + 5.0 * r, device="cpu")
assert ms == 15.0, ms
dist.destroy_process_group()
print("rank", r, "ok")
"""


def test_pair_sharding_world_size_2_gloo(tmp_path):
    script = tmp_path / "w.py"
    script.write_text(SHARD_WORKER)
    procs = []
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), PORT="29641", DAHITRA_ROOT=ROOT)
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    for p in procs:
        out, err = p.communicate(timeout=300)
        assert p.returncode == 0, err[-2000:]
        assert "ok" in out


TRAIN_WORKER = r"""
import copy, os, sys, torch, torch.distributed as dist
sys.path.insert(0, os.environ["DAHITRA_ROOT"])
from dahitra_b200.train_graph import GraphedTrainStep
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%s" % os.environ["PORT"],
                        rank=int(os.environ["RANK"]), world_size=2)
r = dist.get_rank()
torch.manual_seed(0)                                       # same initial weights on both ranks


class Net(torch.nn.Module):                                # stand-in with the network's traits: BatchNorm, a conv, dead parameters
    def __init__(self):
        super().__init__()
        self.c1 = torch.nn.Conv2d(3, 8, 3, padding=1)
        self.bn = torch.nn.BatchNorm2d(8)
        self.c2 = torch.nn.Conv2d(8, 2, 1)
        self.dead = torch.nn.Linear(4, 4)

    def forward(self, x):
        return self.c2(torch.relu(self.bn(self.c1(x))))


net = Net().to(memory_format=torch.channels_last)
ref = copy.deepcopy(net)
lf = torch.nn.functional.cross_entropy
g = torch.Generator().manual_seed(10 + r)                  # different data per rank
x = torch.randn(4, 3, 8, 8, generator=g)
y = torch.randint(0, 2, (4, 8, 8), generator=g)
ts = GraphedTrainStep(net, lf, (x, y), lambda ps: torch.optim.AdamW(ps, lr=1e-2, weight_decay=0.01), use_graph=False)
assert len(ts.frozen) == 2 and ts.world == 2
opt = torch.optim.AdamW(ref.parameters(), lr=1e-2, weight_decay=0.01)
for i in range(3):
    xi = torch.randn(4, 3, 8, 8, generator=g)
    ts.step(xi, y)
    # reference: plain loop + explicit per-parameter all-reduce (mean) of the gradients
    opt.zero_grad(set_to_none=True)
    lf(ref.train()(xi), y).backward()
    for p in ref.parameters():
        if p.grad is not None:
            dist.all_reduce(p.grad)
            p.grad /= 2
    opt.step()
for (n, a), b in zip(net.state_dict().items(), ref.state_dict().values()):
    if "running" in n or "num_batches" in n:
        continue                                           # BatchNorm statistics are per rank in both
    assert torch.allclose(a.double(), b.double(), rtol=1e-6, atol=1e-7), n
    w = a.clone().contiguous()
    dist.broadcast(w, 0)
    assert torch.equal(w, a.contiguous()), "replicas differ: " + n
dist.destroy_process_group()
print("rank", r, "ok")
"""


def test_graphed_train_step_flat_allreduce_world_size_2_gloo(tmp_path):
    """dahitra_b200.train_graph.GraphedTrainStep (eager form): one flat gradient buffer + ONE all-reduce gives exactly the
    weights of the plain loop with per-parameter gradient averaging; replicas stay identical; dead parameters are frozen."""
    script = tmp_path / "t.py"
    script.write_text(TRAIN_WORKER)
    procs = []
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), PORT="29643", DAHITRA_ROOT=ROOT)
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    for p in procs:
        out, err = p.communicate(timeout=300)
        assert p.returncode == 0, err[-2000:]
        assert "ok" in out
