import math

import numpy as _np

from .. import core as mx
from . import losses  # noqa: F401


class Module:
    def __init__(self, params=None):
        if isinstance(params, dict):
            for k, v in params.items():
                setattr(self, k, v)

    def __call__(self, *a, **k):
        return self.forward(*a, **k) if hasattr(self, "forward") else None

    def _children(self):
        out = {}
        for k, v in self.__dict__.items():
            if isinstance(v, (mx.array, Module)):
                out[k] = v
            elif isinstance(v, (list, tuple)) and v and all(isinstance(x, Module) for x in v):
                out[k] = list(v)
        return out

    def parameters(self):
        out = {}
        for k, v in self._children().items():
            if isinstance(v, mx.array):
                out[k] = v
            elif isinstance(v, Module):
                sub = v.parameters()
                if sub:
                    out[k] = sub
            else:
                out[k] = [m.parameters() for m in v]
        return out

    trainable_parameters = parameters

    def update(self, params):
        for k, v in params.items():
            cur = getattr(self, k, None)
            if isinstance(cur, Module):
                cur.update(v)
            elif isinstance(cur, list):
                for m, pv in zip(cur, v):
                    m.update(pv)
            else:
                setattr(self, k, v)
        return self


class Linear(Module):
    def __init__(self, input_dims, output_dims, bias=True):
        super().__init__()
        s = 1.0 / math.sqrt(input_dims)
        # tests/test_oracle_golden.py::attn_proj_weights replays this draw (order, bound, dtype) instead of storing
        # the golden FlashAttention weights: change both together and regenerate tests/golden/reference_vectors.npz
        self.weight = mx.array(_np.random.uniform(-s, s, (output_dims, input_dims)).astype(_np.float32))
        if bias:
            self.bias = mx.array(_np.random.uniform(-s, s, (output_dims,)).astype(_np.float32))

    def __call__(self, x):
        y = mx.matmul(x, self.weight.T)
        return y + self.bias if "bias" in self.__dict__ else y


class Embedding(Module):
    def __init__(self, num_embeddings, dims):
        super().__init__()
        self.weight = mx.array((_np.random.standard_normal((num_embeddings, dims)) * dims ** -0.5).astype(_np.float32))

    def __call__(self, idx):
        return self.weight[_np.asarray(idx)].view(mx.array)


def value_and_grad(model, fn):
    raise NotImplementedError("autograd is not part of the shim")
