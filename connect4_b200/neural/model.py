"""`ModelWrapper`: the evaluator-side surface of oinkoink/neural/pytorch/model.py:137-282 on the CUDA network kernel.

  model(Board)        -> (value ndarray (1,), prior ndarray (7,))      float32   (model.py:252-267)
  model([Board, ...]) -> (values ndarray (N,), priors ndarray (N,7))   float32   (model.py:269-282)
  anything else       -> TypeError                                               (model.py:176-178)

Networks the library compiles (32 or 64 filters, 1..16 residual blocks) run on its CUDA tower (`backend == "cuda"`); any
other geometry is served by a torch restatement of the reference's Net through `TorchModel` (`backend == "torch"`,
neural/torch_model.py): the search and self-play stay on the device engine, the network is called once per pass.

`kernel="layers"` runs any network with a multiple of 16 filters in 16..256 and 1..40 residual blocks on the library's
layer-by-layer tcgen05 kernels instead (`backend == "cuda"`, one launch per conv layer, DESIGN.md 4.3).  The default
route (`kernel="auto"`) does not use them yet: it still sends every geometry the fused tower cannot compile to TorchNet.
Whether the auto route should switch is a separate decision, to be made on the measurements of DESIGN.md 4.0.

Training (model.py:199-240) is outside this path and raises NotImplementedError.  Checkpoints use the reference's
format (`net_state_dict` / `optimiser_state_dict` / `scheduler_state_dict`, model.py:242-250).
"""
import ctypes as C
from typing import List, Optional, Union

import numpy as np

from .. import _lib
from ..board import Board
from .config import ModelConfig, NetConfig
from .weights import fold_state_dict, net_shape


def _init_state_dict(nc: NetConfig):
    """Freshly initialised parameters with the reference's module construction order (model.py:120-128), so that
    torch.manual_seed(s) gives the same network as `Net(config)` does in the reference."""
    import torch.nn as nn
    import torch

    class Res(nn.Module):
        def __init__(s, f):
            super().__init__()
            s.conv1 = nn.Conv2d(f, f, 3, padding=1, bias=False)
            s.conv2 = nn.Conv2d(f, f, 3, padding=1, bias=False)
            s.batch_norm1 = nn.BatchNorm2d(f)
            s.batch_norm2 = nn.BatchNorm2d(f)

    class VH(nn.Module):
        def __init__(s, f, n):
            super().__init__()
            s.conv1 = nn.Conv2d(f, 1, 1)
            s.batch_norm = nn.BatchNorm2d(1)
            s.fcN = nn.Sequential(*[nn.Linear(42, 42) for _ in range(n)])
            s.fc1 = nn.Linear(42, 1)
            s.w1 = nn.Parameter(torch.tensor(1.0), requires_grad=False)
            s.w2 = nn.Parameter(torch.tensor(0.5), requires_grad=False)

    class PH(nn.Module):
        def __init__(s, f):
            super().__init__()
            s.conv1 = nn.Conv2d(f, 2, 1)
            s.batch_norm = nn.BatchNorm2d(2)
            s.fc1 = nn.Linear(84, 7)

    class Params(nn.Module):
        def __init__(s):
            super().__init__()
            s.body = nn.Sequential(
                nn.Sequential(nn.Conv2d(nc.channels, nc.filters, 3, padding=1, bias=False),
                              nn.BatchNorm2d(nc.filters)),
                nn.Sequential(*[Res(nc.filters) for _ in range(nc.n_residuals)]))
            s.value_head = VH(nc.filters, nc.n_fc_layers)
            s.policy_head = PH(nc.filters)

    return {k: v.detach().clone() for k, v in Params().state_dict().items()}


def compiled_geometry(filters: int, n_residuals: int, kernel: str = "auto") -> bool:
    """True where c4_net_create accepts the network's shape (include/c4b200.h): the CUDA tower runs it.  `kernel` other than
    "auto" asks for a particular CUDA kernel, so such a network always goes to c4_net_create (and fails there if it must)."""
    return kernel != "auto" or (filters in (32, 64) and 1 <= n_residuals <= 16)


def flops_per_position(filters: int, n_residuals: int, n_fc: int) -> float:
    """FLOPs (2*MAC, convs + linears) per position of a network of this shape (c4_net_flops_per_position)"""
    F, R = filters, n_residuals
    return 2.0 * (42.0 * 27 * F + 2.0 * R * 42 * 9 * F * F + 42.0 * F + n_fc * 42 * 42 + 42 + 42.0 * F * 2 + 84.0 * 7)


class NetEvaluator():
    """The reference's evaluator protocol and evaluation passes on top of a c4_net handle (`self.c4_net`, `self.device`):
    shared by ModelWrapper and TorchModel, whatever serves the network."""

    def __call__(self, input_: Union[Board, List[Board]]):
        if isinstance(input_, Board):
            v, p = self._call_list([input_])
            return v.reshape(-1), p.reshape(-1)
        elif isinstance(input_, list):
            return self._call_list(input_)
        raise TypeError('{} called with {}. It accepts either a Board nor a list(Board)'.format(type(self).__name__,
                                                                                              type(input_)))

    def _call_list(self, board_list: List[Board]):
        c0 = np.array([int(b.color[0]) for b in board_list], np.uint64)
        c1 = np.array([int(b.color[1]) for b in board_list], np.uint64)
        values, priors = self.evaluate_bitboards(c0, c1)
        values, priors = values.cpu().numpy(), priors.cpu().numpy()
        assert not np.isnan(values).any()
        assert not np.isnan(priors).any()
        return values, priors

    def evaluate_bitboards(self, c0, c1):
        """uint64 bitboards (numpy or CUDA int64 tensors) -> (values f32 [n], priors f32 [n,7]) CUDA tensors."""
        import torch
        from ..engine import _u64_tensor
        t0, t1 = _u64_tensor(c0, self.device.index), _u64_tensor(c1, self.device.index)
        n = int(t0.numel())
        out = torch.empty((n, 8), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().c4_net_forward(self.c4_net, _lib.ptr(t0), _lib.ptr(t1), n, None, _lib.ptr(out),
                                                  _lib.stream_ptr()))
        return out[:, 7].contiguous(), out[:, :7].contiguous()

    # ---- evaluation pass over a labelled set (model.py:180-198,307-342; TrainingLoop._evaluate, training.py:156-171)
    def _eval_batches(self, data, batch_size, shuffle):
        """yields (value_out, prior_out, value_label, prior_label-or-None) CUDA tensors per mini-batch; the positions
        go plane tensor -> bitboards (c4_board_from_planes) -> the network, nothing is evaluated on the host."""
        import torch
        from ..board import BoardBatch
        n = len(data)
        order = torch.randperm(n) if shuffle else torch.arange(n)
        for i in range(0, n, batch_size):
            idx = order[i:i + batch_size]
            planes = data.boards[idx].cuda()
            bb = BoardBatch.from_planes(planes[:, -2], planes[:, -1])        # channels: [to-move,] o, x
            v, p = self.evaluate_bitboards(bb.c0, bb.c1)
            assert not torch.isnan(v).any() and not torch.isnan(p).any()
            yield v, p, data.values[idx].cuda(), (None if data.priors is None else data.priors[idx].cuda())

    def evaluate(self, data, batch_size: int = 4096, shuffle: bool = True):
        """value MSE + policy BCE and the accuracy tallies of CombinedStats (model.py:307-328)"""
        import torch.nn.functional as F
        from .stats import CombinedStats
        stats = CombinedStats()
        for v, p, yv, yp in self._eval_batches(data, batch_size, shuffle):
            assert v.shape == yv.shape and p.shape == yp.shape
            stats.update(v.cpu().numpy(), yv.cpu().numpy(), F.mse_loss(v, yv).item(),
                         p.cpu().numpy(), yp.cpu().numpy(), F.binary_cross_entropy(p, yp).item())
        return stats

    def evaluate_value_only(self, data):
        """ValueStats over a value-labelled set such as the 8-ply positions (model.py:330-342)"""
        import torch.nn.functional as F
        from .stats import ValueStats
        stats = ValueStats()
        for v, _, yv, _ in self._eval_batches(data, 4096, True):
            assert v.shape == yv.shape
            stats.update(v.cpu().numpy(), yv.cpu().numpy(), F.mse_loss(v, yv).item())
        return stats


class ModelWrapper(NetEvaluator):
    def __init__(self, config: Optional[ModelConfig] = None, file_name: Optional[str] = None, state_dict=None,
                 device: Optional[int] = None, operand_dtype: str = "fp16", kernel: str = "auto"):
        import torch
        _lib.require_gpu()
        self.backend = None
        self.config = config if config is not None else ModelConfig()
        self._extra = {}
        if state_dict is not None:
            sd = state_dict
        elif file_name is not None:
            checkpoint = torch.load(file_name, map_location="cpu", weights_only=False)
            sd = checkpoint['net_state_dict']
            self._extra = {k: v for k, v in checkpoint.items() if k != 'net_state_dict'}
        else:
            sd = _init_state_dict(self.config.net_config)
        self.state_dict = {k: (v if torch.is_tensor(v) else torch.as_tensor(np.asarray(v))) for k, v in sd.items()}
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else device)
        self.operand_dtype = operand_dtype
        self.kernel = kernel
        F, R, _ = net_shape(self.state_dict)
        if compiled_geometry(F, R, kernel):
            blob = fold_state_dict(self.state_dict, operand_dtype, kernel)
            h = C.c_void_p()
            _lib.check(_lib.load().c4_net_create(self.device.index, blob.ctypes.data_as(C.c_void_p), blob.size, C.byref(h)))
            self.c4_net = h
            self.backend = "cuda"
        else:
            from .torch_model import TorchModel, TorchNet
            dt = {"fp16": torch.float16, "bf16": torch.bfloat16}[operand_dtype]
            self._served = TorchModel(TorchNet(self.state_dict, dt).to(self.device), self.device, dt)
            self.c4_net = self._served.c4_net
            self.backend = "torch"
        self.n_parameters = sum(int(v.numel()) for k, v in self.state_dict.items()
                                if "running_" not in k and "num_batches" not in k and not k.endswith((".w1", ".w2")))
        print("Constructed NN with {} parameters".format(self.n_parameters))

    def __del__(self):
        try:
            if self.backend == "cuda" and getattr(self, "c4_net", None):     # (a TorchModel owns its own handle)
                _lib.load().c4_net_destroy(self.c4_net)
                self.c4_net = None
        except Exception:
            pass

    @property
    def flops_per_position(self):
        if self.backend == "cuda":
            return float(_lib.load().c4_net_flops_per_position(self.c4_net))
        return flops_per_position(*net_shape(self.state_dict))

    @property
    def trunk_scale_log2(self):
        """k of the power-of-two trunk scale 2^-k chosen at creation so that fp16 operands cannot overflow (0 for
        networks in the usual activation range; see c4_net_get in include/c4b200.h)"""
        return int(_lib.load().c4_net_get(self.c4_net, 3))

    # ---- checkpoints (reference format)
    def save(self, folder_path: str):
        import torch
        d = {'net_state_dict': self.state_dict, 'optimiser_state_dict': self._extra.get('optimiser_state_dict', {}),
             'scheduler_state_dict': self._extra.get('scheduler_state_dict', {})}
        torch.save(d, folder_path + '/net.pth')

    def train(self, *a, **k):
        raise NotImplementedError("training is outside the self-play hot path this package accelerates")
