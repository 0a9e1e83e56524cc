"""Networks the CUDA tower does not compile, served by the caller: `TorchModel` hands any PyTorch network to the device
engine through c4_net_create_external (include/c4b200.h).  The engine keeps the tree passes, the evaluation memo, the
de-duplication of evaluations in flight, the Philox noise and the records; once per lock-step pass it calls back with the
compacted leaf batch, which is turned into input planes on the device (c4_board_to_planes, in the model's input dtype),
run through the module on the engine's stream and written back as the {prior[7], value} rows the tower would write.
Nothing is copied to the host.

`TorchNet` is the reference's Net (oinkoink/neural/pytorch/model.py:20-134) in eval mode on a reference-layout state dict,
for every filters / residual blocks / fc layers setting; ModelWrapper serves it through TorchModel for the geometries the
CUDA tower does not compile.
"""
import ctypes as C

import torch
import torch.nn.functional as F

from .. import _lib
from ..board import PLANE_DTYPES
from .model import NetEvaluator
from .weights import net_shape

LEAKY = 0.01     # nn.LeakyReLU() default slope (model.py:31,43,68,104)
BN_EPS = 1e-5    # nn.BatchNorm2d default eps


class TorchNet():
    """Net.forward (model.py:130-134) in eval mode.  input planes [n, 3, 6, 7] -> (value [n], prior [n, 7]) float32.
    With `operand_dtype` (torch.float16 / torch.bfloat16) the convolutions and linear layers run with operands of that
    type under torch.autocast (their weights are stored in it); batch-norm statistics and the outputs stay float32."""

    def __init__(self, state_dict, operand_dtype=None):
        self.operand_dtype = operand_dtype
        self.filters, self.n_residuals, self.n_fc = net_shape(state_dict)
        self.p = {}
        for k, v in state_dict.items():
            if "num_batches" in k:
                continue
            t = (v if torch.is_tensor(v) else torch.as_tensor(v)).detach().to(torch.float32).clone()
            gemm = ("conv" in k or ".fc" in k or k == "body.0.0.weight") and "batch_norm" not in k
            self.p[k] = t.to(operand_dtype) if operand_dtype is not None and gemm else t

    def to(self, device):
        self.p = {k: v.to(device) for k, v in self.p.items()}
        return self

    def _bn(self, x, prefix):
        p = self.p
        return F.batch_norm(x, p[prefix + ".running_mean"], p[prefix + ".running_var"], p[prefix + ".weight"],
                            p[prefix + ".bias"], training=False, eps=BN_EPS)

    def _forward(self, x):
        p, lk = self.p, (lambda t: F.leaky_relu(t, LEAKY))
        h = lk(self._bn(F.conv2d(x, p["body.0.0.weight"], padding=1), "body.0.1"))          # model.py:20-31
        for i in range(self.n_residuals):                                                     # model.py:45-55
            r = "body.1.%d." % i
            o = lk(self._bn(F.conv2d(h, p[r + "conv1.weight"], padding=1), r + "batch_norm1"))
            o = self._bn(F.conv2d(o, p[r + "conv2.weight"], padding=1), r + "batch_norm2")
            h = lk(o + h)
        # value head (model.py:77-91): 1x1 conv, BN, LeakyReLU, n_fc x Linear(42, 42) without activation in between,
        # LeakyReLU, Linear(42, 1), tanh, (x + w1) * w2
        v = lk(self._bn(F.conv2d(h, p["value_head.conv1.weight"], p["value_head.conv1.bias"]), "value_head.batch_norm"))
        v = v.reshape(v.shape[0], -1)
        for j in range(self.n_fc):
            v = F.linear(v, p["value_head.fcN.%d.weight" % j], p["value_head.fcN.%d.bias" % j])
        v = F.linear(lk(v), p["value_head.fc1.weight"], p["value_head.fc1.bias"]).float()
        v = ((torch.tanh(v) + p["value_head.w1"]) * p["value_head.w2"]).reshape(-1)
        # policy head (model.py:107-117): 1x1 conv (2 channels), BN, LeakyReLU, flatten channel-major, Linear(84, 7), softmax
        q = lk(self._bn(F.conv2d(h, p["policy_head.conv1.weight"], p["policy_head.conv1.bias"]), "policy_head.batch_norm"))
        q = F.linear(q.reshape(q.shape[0], -1), p["policy_head.fc1.weight"], p["policy_head.fc1.bias"]).float()
        return v, torch.softmax(q, dim=1)

    def __call__(self, x):
        if self.operand_dtype is None:
            return self._forward(x.float())
        with torch.autocast(x.device.type, dtype=self.operand_dtype):
            return self._forward(x.to(self.operand_dtype))


class _DeviceArray():
    """a raw device pointer seen through __cuda_array_interface__ (torch.as_tensor makes a tensor over it, no copy)"""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"data": (ptr, False), "shape": shape, "typestr": typestr, "strides": None,
                                         "version": 2}


def _serve(module, device, dtype):
    """the c4_eval_fn of a TorchModel.  It holds no reference to the TorchModel itself, so the model (and with it the
    network handle) is freed as soon as its last user lets go of it."""
    lib = _lib.load()
    code = PLANE_DTYPES[str(dtype).replace("torch.", "")]
    streams = {}

    def serve(user, c0, c1, n, out, stream):
        try:
            if stream not in streams:
                streams[stream] = torch.cuda.ExternalStream(stream, device=device) if stream else \
                    torch.cuda.default_stream(device)
            with torch.inference_mode(), torch.cuda.device(device), torch.cuda.stream(streams[stream]):
                planes = torch.empty((n, 3, 6, 7), dtype=dtype, device=device)
                _lib.check(lib.c4_board_to_planes(c0, c1, _lib.ptr(planes), code, n, stream))
                value, prior = module(planes)
                if tuple(prior.shape) != (n, 7) or tuple(value.shape) not in ((n,), (n, 1)):
                    raise ValueError("the module returned value %s and prior %s for %d positions; expected value [n] or "
                                     "[n, 1] and prior [n, 7]" % (tuple(value.shape), tuple(prior.shape), n))
                rows = torch.as_tensor(_DeviceArray(out, (n, 8), "<f4"), device=device)
                rows[:, :7] = prior
                rows[:, 7] = value.reshape(n)
            return 0
        except BaseException as e:      # the engine call fails and re-raises it (_lib.check)
            _lib.set_callback_error(e)
            return 1
    return serve


class TorchModel(NetEvaluator):
    """Any PyTorch network as the engine's evaluator.

    module: callable with the signature of the reference's Net.forward (model.py:130-134): planes [n, 3, 6, 7] of `dtype`
    (Board.to_array layout: row 0 = top, channel 0 = side to move) -> (value [n] or [n, 1], prior [n, 7]), on `device`.
    It runs under torch.inference_mode() on the engine's CUDA stream.

    The handle `c4_net` makes it a network for every route that takes a ModelWrapper: Engine.set_net, SelfPlayPool /
    game_pool, search_batch / MCTS (a bare model or Evaluator(partial(evaluate_nn, model=...))), Match.play_batched and
    dist.generate_sharded.  These run on the lock-step pass engine with one host synchronise and one module call per pass.
    If the module raises, the engine call raises C4Error with the module's exception as its cause.
    """

    def __init__(self, module, device=None, dtype=torch.float32):
        _lib.require_gpu()
        self.module = module
        if device is None:
            device = torch.cuda.current_device()
        self.device = torch.device("cuda", device.index if isinstance(device, torch.device) else int(device))
        self.dtype = dtype
        self._fn = _lib.EVAL_FN(_serve(module, self.device, self.dtype))     # lives exactly as long as the handle
        h = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().c4_net_create_external(self.device.index, self._fn, None, C.byref(h)))
        self.c4_net = h

    def close(self):
        if getattr(self, "c4_net", None):
            _lib.load().c4_net_destroy(self.c4_net)
            self.c4_net = None
        self._fn = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
