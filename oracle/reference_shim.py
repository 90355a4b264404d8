"""Import the REAL reference (TimZaman/dotaclient) in place from /root/reference.

TEST INFRASTRUCTURE ONLY.  Works only where ``/root/reference`` exists (the build
container); the GPU box never has it, so nothing in ``-m gpu`` tests, ``smoke()``
or ``bench.py`` may call this.  It is used by

* ``tests/golden/make_golden.py``  -- records reference outputs as the fixtures
  that ``tests/test_oracle.py`` pins the restatement in ``oracle/`` against

The reference's ``optimizer.py`` imports four packages that are not installed
here (``optimizer.py:16-17,19,25``); they are irrelevant to the arithmetic, so we
inject empty stub modules before importing.  Nothing is copied out of the
reference tree.
"""
import importlib
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("DOTACLIENT_REFERENCE", "/root/reference")


def available():
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "optimizer.py"))


def _stub(name, **attrs):
    mod = types.ModuleType(name)
    mod.__dict__.update(attrs)
    sys.modules[name] = mod
    return mod


def load():
    """Returns (reference optimizer module, reference policy module, reference distributed module)."""
    if not available():
        raise RuntimeError("reference tree not present at %s" % REFERENCE_ROOT)
    if "google.cloud.storage" not in sys.modules:
        g = _stub("google")
        gc = _stub("google.cloud")
        st = _stub("google.cloud.storage", Client=object)
        g.cloud = gc
        gc.storage = st
    if "tensorboardX" not in sys.modules:
        _stub("tensorboardX", SummaryWriter=object)
    if "pika" not in sys.modules:
        pk = _stub("pika", ConnectionParameters=lambda **k: None, BlockingConnection=None,
                   BasicProperties=None)
        pk.exceptions = types.SimpleNamespace(ConnectionClosed=Exception, ChannelClosed=Exception)
    if "dotaservice.protos.DotaService_pb2" not in sys.modules:
        _stub("dotaservice")
        _stub("dotaservice.protos")
        _stub("dotaservice.protos.DotaService_pb2", TEAM_DIRE=3, TEAM_RADIANT=2)
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    # The reference's module names are generic ('optimizer', 'policy', 'distributed'); import them
    # under those names (they import each other that way) and hand the module objects back.
    ref_policy = importlib.import_module("policy")
    ref_distributed = importlib.import_module("distributed")
    ref_optimizer = importlib.import_module("optimizer")
    for m in (ref_policy, ref_distributed, ref_optimizer):
        assert os.path.dirname(os.path.abspath(m.__file__)) == os.path.abspath(REFERENCE_ROOT), m.__file__
    return ref_optimizer, ref_policy, ref_distributed


def make_reference_optimizer(seq_len, entropy_coef=5e-4, vf_coef=0.5, learning_rate=5e-5, state_dict=None):
    """Builds a reference ``DotaOptimizer`` without its RMQ/GCS side effects (``optimizer.py:231-284``)."""
    import torch
    O, P, _ = load()
    opt = O.DotaOptimizer.__new__(O.DotaOptimizer)
    torch.manual_seed(7)  # optimizer.py:34
    opt.policy_base = P.Policy()
    if state_dict is not None:
        opt.policy_base.load_state_dict(state_dict)
    opt.policy = opt.policy_base
    opt.seq_len = seq_len
    opt.e_clip = 0.1  # optimizer.py:229
    opt.entropy_coef = entropy_coef
    opt.vf_coef = vf_coef
    opt.optimizer = torch.optim.Adam(opt.policy.parameters(), lr=learning_rate)  # optimizer.py:275
    return opt
