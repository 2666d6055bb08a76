"""The original project's own CUDA extensions, as stored digests of what they returned.

The parity tests compare against the reference's compiled kernels (render_utils_cuda, ub360_utils_cuda,
total_variation_cuda, adam_upd_cuda; oracle/build_ref.py builds them from the original sources, which a
checkout of this repository does not have).  tests/golden/ref_calls.json holds, for every call a test made
into them, a digest of the call's inputs and one of its results (return value and every tensor argument
after the call, so in-place updates count).  A test module's fixture makes ``RefCalls.for_test(request)``,
hands the test ``.ops()`` (the interface of oracle.ops.RefExtOps) or ``.module(name)`` in place of the
extension, and calls ``.finish()`` after it.

Replay (the default): each call runs k4nerf's drop-in module of the same name and fails unless its results
are bit-identical to the reference's for that call, so the test goes on with exactly the reference's values.
With K4_RECORD_REF=1, on a GPU with oracle/_ref built, the reference itself runs and the digests of the
test are rewritten.
"""
import hashlib
import importlib
import json
import os

import torch

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'ref_calls.json')
RECORD = os.environ.get('K4_RECORD_REF') == '1'
_STORED = None


def _stored():
    global _STORED
    if _STORED is None:
        with open(PATH) as f:
            _STORED = json.load(f)
    return _STORED


def digest(x):
    """sha256 (12 hex digits) over dtypes, shapes and bytes of every tensor in x, and the repr of other values."""
    h = hashlib.sha256()

    def walk(v):
        if isinstance(v, torch.Tensor):
            t = v.detach().contiguous().cpu()
            h.update(f'{t.dtype}{tuple(t.shape)}'.encode())
            h.update(t.view(-1).view(torch.uint8).numpy().tobytes() if t.numel() else b'')
        elif isinstance(v, (list, tuple)):
            h.update(b'[')
            for e in v:
                walk(e)
            h.update(b']')
        else:
            h.update(repr(v).encode())
    walk(x)
    return h.hexdigest()[:12]


def _reference(name):
    from oracle import ops
    return ops.load_ref_ext(name)


class RefCalls:
    """The calls of one test into the reference extensions, in order."""

    def __init__(self, key):
        self.key = key
        if RECORD:
            self.calls = []
        else:
            stored = _stored()
            assert key in stored, f'{key}: no stored reference calls in {PATH} (record them with K4_RECORD_REF=1)'
            self.calls = stored[key]
        self.n = 0

    @classmethod
    def for_test(cls, request):
        return cls(f'{request.node.module.__name__}::{request.node.name}')

    def call(self, module, fn, *args):
        d_in = digest(args)
        if RECORD:
            out = getattr(_reference(module), fn)(*args)
            torch.cuda.synchronize()
            self.calls.append(f'{fn} {d_in} {digest((out, args))}')
            return out
        assert self.n < len(self.calls), f'{self.key}: call {self.n} ({fn}) was not made by the recorded run'
        want_fn, want_in, want_out = self.calls[self.n].split()
        assert fn == want_fn, f'{self.key}: call {self.n} is {fn}, the recorded run called {want_fn}'
        out = getattr(importlib.import_module('k4nerf.' + module), fn)(*args)
        torch.cuda.synchronize()
        got = digest((out, args))
        assert got == want_out, (f'{self.key}: call {self.n} ({module}.{fn}) differs from the reference kernel' +
                                 ('' if d_in == want_in else ' (its inputs differ from the recorded run too)'))
        self.n += 1
        return out

    def module(self, name):
        """Stand-in for the reference extension `name`."""
        calls = self

        class _Module:
            def __getattr__(self, fn):
                return lambda *args: calls.call(name, fn, *args)
        return _Module()

    def ops(self):
        """Stand-in for oracle.ops.RefExtOps: render_utils_cuda, with cumdist_thres from ub360_utils_cuda."""
        calls = self

        class _Ops:
            device = 'cuda'

            def cumdist_thres(self, dist, thres):
                return calls.call('ub360_utils_cuda', 'cumdist_thres', dist, thres)

            def __getattr__(self, fn):
                return lambda *args: calls.call('render_utils_cuda', fn, *args)
        return _Ops()

    def finish(self):
        if RECORD:
            stored = json.load(open(PATH)) if os.path.exists(PATH) else {}
            stored[self.key] = self.calls
            with open(PATH, 'w') as f:
                json.dump(stored, f, indent=0, sort_keys=True)
                f.write('\n')
        else:
            assert self.n == len(self.calls), f'{self.key}: {self.n} of the {len(self.calls)} recorded calls made'
