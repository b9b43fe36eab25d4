"""Policy/value network API of the reference, kept verbatim at the call surface:

  Model.predict(states) -> (list[dict[Action, float]], list[list[float]])   models/base/model.py:54-74
  Model.forward(x)      -> (logits[B,7], value[B,2])                        models/base/model.py:51
  Model.get_inference_clone(), state_dict()/load_state_dict()               models/base/model.py:92-96
  Model.training_step / configure_optimizers / format_dataset               models/base/model.py:27-48,76-82

`lightning` is not required: `Model` is a plain `nn.Module` exposing the hooks a Lightning trainer calls.
Parameter names match the reference classes, so their checkpoints' `state_dict`s load unchanged.

What runs where: plane encoding (`_states_to_tensor`) and the legal-only softmax of `predict` are CUDA kernels of
libaz_engine.so (`az_encode_states`, `az_masked_softmax`).  On the search hot path `InferenceNet` picks the evaluator:
`BasicNN` in bf16 -> `TensorCoreMLP` (csrc/az_mlp.cu) and 64-channel `ResNet`s in bf16 -> `TensorCoreTrunk`
(csrc/az_conv.cu), both hand-written tcgen05/TMEM kernels with the leaf gather fused in; every other model runs its
conv / linear layers as library GEMMs (cuBLAS / cuDNN through torch) with BatchNorm folded, bf16 channels-last, so that
only the conv/GEMM layers touch the tensor cores; softmax / tanh epilogues stay in fp32.
"""
from __future__ import annotations

import copy

import numpy as np
import torch
import torch.nn.functional as F
from torch import Tensor, nn

from .engine import LAYOUT_GRID_F32, LAYOUT_PLANES_BF16, LAYOUT_PLANES_F32
from .game import State, rules_engine

ActionPolicy = dict
Value = list


class Model(nn.Module):
    """Abstract policy/value model (reference: `Model(ABC, L.LightningModule)`, models/base/model.py:15)."""

    input_layout: int = LAYOUT_PLANES_F32  # which az_gather_leaves layout `forward` consumes

    def __init__(self, learning_rate: float = 1e-3):
        super().__init__()
        self.learning_rate = learning_rate
        self.model_name = self.__class__.__name__
        self.hparams = {"learning_rate": learning_rate, "model_name": self.model_name}

    # Lightning hooks (no-ops without a trainer)
    def save_hyperparameters(self, *args, **kwargs):
        return None

    def log(self, *args, **kwargs):
        return None

    @property
    def device(self) -> torch.device:
        return next(self.parameters()).device

    def training_step(self, batch: tuple[Tensor, Tensor, Tensor], batch_idx: int = 0) -> Tensor:
        x, policy_target, value_target = batch
        policy_logits, value_logits = self(x)
        policy_loss = F.cross_entropy(policy_logits, policy_target)  # soft targets (visit distribution)
        value_loss = F.mse_loss(value_logits, value_target)
        total = policy_loss + value_loss
        self.log("train_loss", total)
        self.log("policy_loss", policy_loss)
        self.log("value_loss", value_loss)
        return total

    def configure_optimizers(self):
        return torch.optim.Adam(self.parameters(), lr=self.learning_rate, weight_decay=1e-4)

    def forward(self, x: Tensor) -> tuple[Tensor, Tensor]:  # pragma: no cover - abstract
        raise NotImplementedError

    def predict(self, states: list[State]) -> tuple[list[ActionPolicy], list[Value]]:  # pragma: no cover
        raise NotImplementedError

    def format_dataset(self, states, policies, values):
        from torch.utils.data import TensorDataset

        return TensorDataset(self._states_to_tensor(states).cpu(), self._policies_to_tensor(policies),
                             torch.tensor(values, dtype=torch.float32))

    def get_inference_clone(self):
        clone = copy.deepcopy(self)
        clone.eval()
        return clone

    # -- checkpoints in the reference's (Lightning) file shape -----------------------------------------------------------
    def save_checkpoint(self, path: str, epoch: int = 0, global_step: int = 0) -> None:
        """What Lightning's `ModelCheckpoint` writes for the reference (core/training/trainer.py:66-70): the weights under
        `state_dict`, the constructor arguments under `hyper_parameters`."""
        torch.save({"state_dict": {k: v.detach().cpu() for k, v in self.state_dict().items()}, "hyper_parameters": dict(self.hparams),
                    "epoch": int(epoch), "global_step": int(global_step), "pytorch-lightning_version": "2.0.0"}, path)

    @classmethod
    def load_from_checkpoint(cls, checkpoint_path: str, map_location=None, strict: bool = True, **kwargs):
        """`CNNModel.load_from_checkpoint(path)` as scripts/play.py:19-25 calls it: accepts a Lightning checkpoint (weights under
        `state_dict`, constructor arguments under `hyper_parameters`) or a bare `state_dict` file."""
        import inspect

        ckpt = torch.load(checkpoint_path, map_location=map_location or "cpu", weights_only=False)
        if isinstance(ckpt, dict) and "state_dict" in ckpt and isinstance(ckpt["state_dict"], dict):
            sd, hp = ckpt["state_dict"], dict(ckpt.get("hyper_parameters") or {})
        else:
            sd, hp = ckpt, {}
        hp.update(kwargs)
        accepted = set(inspect.signature(cls.__init__).parameters) - {"self"}
        model = cls(**{k: v for k, v in hp.items() if k in accepted})
        model.load_state_dict(sd, strict=strict)
        return model.eval()


def _state_arrays(states: list[State]):
    return (np.array([s.bb0 for s in states], np.uint64), np.array([s.bb1 for s in states], np.uint64),
            np.array([s.player for s in states], np.uint8))


class Connect4Model(Model):
    """`predict` generalised for all Connect4 nets (models/games/connect4/model.py:8-51)."""

    def __init__(self):
        super().__init__()
        self.board_height = 6
        self.board_width = 7

    def _states_to_tensor(self, states: list[State]) -> Tensor:
        bb0, bb1, pl = _state_arrays(states)
        return rules_engine().encode_states(bb0, bb1, pl, self.input_layout)

    @torch.no_grad()
    def predict(self, states: list[State]) -> tuple[list[ActionPolicy], list[Value]]:
        eng = rules_engine()
        x = self._states_to_tensor(states)
        policy_logits, values_tensor = self.forward(x)
        legal = np.array([s.legal_mask for s in states], np.uint8)
        priors = eng.masked_softmax(policy_logits.float(), legal).cpu().numpy()  # legal-only softmax, fp32
        policies: list[ActionPolicy] = []
        for i, state in enumerate(states):
            policies.append({a: float(priors[i, a.column]) for a in state.actions})
        values: list[Value] = values_tensor.detach().float().cpu().tolist()
        return policies, values

    def _policies_to_tensor(self, policies: list[ActionPolicy]) -> Tensor:
        t = torch.zeros((len(policies), self.board_width))
        for i, policy in enumerate(policies):
            for action, prob in policy.items():
                t[i, action.column] = prob
        return t


class BasicNN(Connect4Model):
    """42 -> 512 -> 512 -> {7, 2 (tanh)} on the raw grid (-1 / 0 / 1, absolute) (basic.py:8-47)."""

    input_layout = LAYOUT_GRID_F32

    def __init__(self):
        super().__init__()
        self.flatten = nn.Flatten()
        self.shared_layers = nn.Sequential(
            nn.Linear(self.board_height * self.board_width, 512), nn.ReLU(), nn.Linear(512, 512), nn.ReLU())
        self.policy_head = nn.Linear(512, self.board_width)
        self.value_head = nn.Sequential(nn.Linear(512, 2), nn.Tanh())

    def forward(self, x: Tensor) -> tuple[Tensor, Tensor]:
        x = x.to(self.shared_layers[0].weight.device)
        h = self.shared_layers(self.flatten(x))
        return self.policy_head(h), self.value_head(h)


class CNNModel(Connect4Model):
    """3 x (conv3x3 + BN + ReLU) 3->64->128->256, FC 10752->512, heads 7 / tanh(1) -> [v, -v] (cnn.py:8-100)."""

    input_layout = LAYOUT_PLANES_F32

    def __init__(self):
        super().__init__()
        self.channels = [3, 64, 128, 256]
        self.conv_layers = nn.Sequential(
            nn.Conv2d(3, 64, kernel_size=3, padding=1), nn.BatchNorm2d(64), nn.ReLU(),
            nn.Conv2d(64, 128, kernel_size=3, padding=1), nn.BatchNorm2d(128), nn.ReLU(),
            nn.Conv2d(128, 256, kernel_size=3, padding=1), nn.BatchNorm2d(256), nn.ReLU(),
        )
        self.conv_output_size = 256 * self.board_height * self.board_width
        self.shared_layers = nn.Sequential(nn.Linear(self.conv_output_size, 512), nn.ReLU(), nn.Dropout(0.3))
        self.policy_head = nn.Linear(512, self.board_width)
        self.value_head = nn.Sequential(nn.Linear(512, 1), nn.Tanh())
        self.learning_rate = 1e-3

    def forward(self, x: Tensor) -> tuple[Tensor, Tensor]:
        x = x.to(next(self.parameters()).device)
        x = self.conv_layers(x)
        h = self.shared_layers(x.reshape(x.size(0), -1))
        value = self.value_head(h)
        return self.policy_head(h), torch.cat([value, -value], dim=1)


class ResBlock(nn.Module):
    def __init__(self, num_channels: int):
        super().__init__()
        self.conv1 = nn.Conv2d(num_channels, num_channels, kernel_size=3, padding=1)
        self.bn1 = nn.BatchNorm2d(num_channels)
        self.conv2 = nn.Conv2d(num_channels, num_channels, kernel_size=3, padding=1)
        self.bn2 = nn.BatchNorm2d(num_channels)

    def forward(self, x):
        r = x
        x = F.relu(self.bn1(self.conv1(x)))
        x = self.bn2(self.conv2(x))
        return F.relu(x + r)


class ResNet(Connect4Model):
    """The reference's own ResNet-style net (src/alphazero_simple/resnet.py:30-72: stem conv3x3+BN+ReLU,
    n x ResBlock, policy head conv1x1->32+BN+ReLU+FC, value head conv3x3->3+BN+ReLU+FC->1) behind the main
    package's `Model` API: side-relative planes (cnn.py:93-95), tanh value returned as [v, -v] (cnn.py:73)."""

    input_layout = LAYOUT_PLANES_F32

    def __init__(self, num_res_blocks: int = 9, num_channels: int = 128):
        super().__init__()
        self.num_res_blocks, self.num_channels = num_res_blocks, num_channels
        self.hparams.update(num_res_blocks=num_res_blocks, num_channels=num_channels)
        rows, cols = self.board_height, self.board_width
        self.input_conv = nn.Sequential(nn.Conv2d(3, num_channels, kernel_size=3, padding=1), nn.BatchNorm2d(num_channels), nn.ReLU())
        self.residual_blocks = nn.ModuleList([ResBlock(num_channels) for _ in range(num_res_blocks)])
        self.policy_head = nn.Sequential(nn.Conv2d(num_channels, 32, kernel_size=1), nn.BatchNorm2d(32), nn.ReLU(), nn.Flatten(),
                                         nn.Linear(32 * rows * cols, self.board_width))
        self.value_head = nn.Sequential(nn.Conv2d(num_channels, 3, kernel_size=3, padding=1), nn.BatchNorm2d(3), nn.ReLU(),
                                        nn.Flatten(), nn.Linear(3 * rows * cols, 1))

    def forward(self, x: Tensor) -> tuple[Tensor, Tensor]:
        x = x.to(next(self.parameters()).device)
        x = self.input_conv(x)
        for block in self.residual_blocks:
            x = block(x)
        v = torch.tanh(self.value_head(x))
        return self.policy_head(x), torch.cat([v, -v], dim=1)

    def flops_per_position(self) -> int:
        """2 x MACs of the conv / linear layers for one 6x7 position."""
        c, hw = self.num_channels, 42
        f = 2 * hw * 9 * 3 * c + self.num_res_blocks * 2 * (2 * hw * 9 * c * c)
        f += 2 * hw * c * 32 + 2 * 32 * hw * 7 + 2 * hw * 9 * c * 3 + 2 * 3 * hw
        return f


# ------------------------------------------------------------------------------------------------
def _fold_bn(conv: nn.Conv2d, bn: nn.BatchNorm2d):
    """eval-mode BatchNorm folded into the preceding convolution (fp32 arithmetic)."""
    w = conv.weight.detach().float()
    b = conv.bias.detach().float() if conv.bias is not None else torch.zeros(w.shape[0], device=w.device)
    scale = bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps)
    return w * scale.view(-1, 1, 1, 1), (b - bn.running_mean.detach().float()) * scale + bn.bias.detach().float()


class TensorCoreMLP:
    """BasicNN.forward as one tcgen05 kernel (csrc/az_mlp.cu): bf16 operands, fp32 accumulation in tensor memory."""

    def __init__(self, model: "BasicNN", device: torch.device, dtype: torch.dtype = torch.bfloat16):
        import ctypes as C

        from . import _lib

        self.lib = _lib.load()
        self.device = torch.device(device)
        self.dtype = dtype
        h = C.c_void_p()
        rc = self.lib.az_mlp_create(self.device.index or 0, C.byref(h))
        if rc != 0:
            raise RuntimeError(f"az_mlp_create failed ({rc}): needs an sm_100 device")
        self.h = h
        rc = self.lib.az_mlp_set_operand_format(self.h, _operand_format(dtype))
        if rc != 0:
            raise RuntimeError(f"az_mlp_set_operand_format failed ({rc})")
        self._out: dict[int, tuple[Tensor, Tensor]] = {}
        self.set_weights(model)

    def set_weights(self, model: "BasicNN"):
        f = lambda t: t.detach().to(self.device, torch.float32).contiguous()
        ws = [f(model.shared_layers[0].weight), f(model.shared_layers[0].bias), f(model.shared_layers[2].weight),
              f(model.shared_layers[2].bias), f(model.policy_head.weight), f(model.policy_head.bias),
              f(model.value_head[0].weight), f(model.value_head[0].bias)]
        rc = self.lib.az_mlp_set_weights(self.h, *[w.data_ptr() for w in ws], torch.cuda.current_stream(self.device).cuda_stream)
        if rc != 0:
            raise RuntimeError(f"az_mlp_set_weights failed ({rc}): {self.lib.az_mlp_last_error(self.h).decode()}")
        torch.cuda.current_stream(self.device).synchronize()  # `ws` may be temporaries

    def __call__(self, x: Tensor) -> tuple[Tensor, Tensor]:
        assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous() and x[0].numel() == 42
        n = x.shape[0]
        if n not in self._out:
            self._out[n] = (torch.empty((n, 7), device=x.device), torch.empty((n, 2), device=x.device))
        logits, values = self._out[n]
        rc = self.lib.az_mlp_forward(self.h, x.data_ptr(), n, logits.data_ptr(), values.data_ptr(),
                                     torch.cuda.current_stream(x.device).cuda_stream)
        if rc != 0:
            raise RuntimeError(f"az_mlp_forward failed ({rc}): {self.lib.az_mlp_last_error(self.h).decode()}")
        return logits, values

    def forward_leaves(self, engine) -> tuple[Tensor, Tensor]:
        """Evaluate the leaves chosen by `engine.select_leaves()` directly from the engine's leaf bitboards (the gather is
        fused into the kernel); row i = slot i."""
        n = engine.n_active
        if n not in self._out:
            self._out[n] = (torch.zeros((n, 7), device=self.device), torch.zeros((n, 2), device=self.device))  # rows of slots without an evaluation stay zero
        logits, values = self._out[n]
        rc = self.lib.az_mlp_forward_leaves(self.h, engine.h, logits.data_ptr(), values.data_ptr(),
                                            torch.cuda.current_stream(self.device).cuda_stream)
        if rc != 0:
            raise RuntimeError(f"az_mlp_forward_leaves failed ({rc}): {self.lib.az_mlp_last_error(self.h).decode()}")
        return logits, values

    @property
    def launch_count(self) -> int:
        return int(self.lib.az_mlp_launch_count(self.h))

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.lib.az_mlp_destroy(self.h)
                self.h = None
        except Exception:
            pass


def _operand_format(dtype: torch.dtype) -> int:
    """torch dtype -> AZ_FMT_* of the tensor-core evaluators (include/az_engine.h)."""
    from ._lib import FMT_BF16, FMT_F16

    if dtype == torch.bfloat16:
        return FMT_BF16
    if dtype == torch.float16:
        return FMT_F16
    raise ValueError(f"the tensor-core evaluators take bf16 or fp16 operands, not {dtype}")


def _canonical_kmajor(w: Tensor, dtype: torch.dtype = torch.bfloat16) -> Tensor:
    """[N][K] -> 16-bit operands in the MMA's K-major no-swizzle core-matrix order: [N/8][K/8][8 rows][8 k]."""
    n, k = w.shape
    return w.reshape(n // 8, 8, k // 8, 8).permute(0, 2, 1, 3).contiguous().to(dtype).reshape(-1)


def pack_trunk_weights(model: "ResNet", device, dtype: torch.dtype = torch.bfloat16) -> tuple[Tensor, Tensor]:
    """BatchNorm-folded stem + residual-block convolutions of a 64-channel ResNet as operands of csrc/az_conv.cu:
    per layer 9 taps (tap = 3*ky + kx) of [64 out][K in] bf16 (K = 16 for the stem, zero padded), and fp32 biases."""
    assert model.num_channels == 64, "the tensor-core trunk kernel is built for 64 channels"
    m = copy.deepcopy(model).eval().float().to(device)
    convs = [_fold_bn(m.input_conv[0], m.input_conv[1])]
    for blk in m.residual_blocks:
        convs.append(_fold_bn(blk.conv1, blk.bn1))
        convs.append(_fold_bn(blk.conv2, blk.bn2))
    parts, biases = [], []
    for li, (w, b) in enumerate(convs):
        if li == 0:
            w = torch.cat([w, torch.zeros(64, 13, 3, 3, device=w.device)], dim=1)  # 3 -> 16 input channels
        for ky in range(3):
            for kx in range(3):
                parts.append(_canonical_kmajor(w[:, :, ky, kx], dtype))
        biases.append(b)
    return torch.cat(parts).contiguous(), torch.stack(biases).contiguous().float()


def pack_trunk_weights_pipe(model: "ResNet", device, dtype: torch.dtype = torch.bfloat16, pair: bool = False) -> tuple[Tensor, Tensor]:
    """The same convolutions for the layer-pipelined kernel (csrc/az_resnet_pipe.cu): per layer the pieces [9 taps][C out][16 in]
    in the order the kernel consumes them, K-chunk-major: for ks (16 input channels) for tap (3*ky + kx); the stem has one
    K chunk (3 -> 16).  `pair`: every piece as two halves [half][9 taps][C/2 out][16 in] - what each CTA of a pair stages."""
    C = model.num_channels
    assert C in (64, 128)
    m = copy.deepcopy(model).eval().float().to(device)
    convs = [_fold_bn(m.input_conv[0], m.input_conv[1])]
    for blk in m.residual_blocks:
        convs.append(_fold_bn(blk.conv1, blk.bn1))
        convs.append(_fold_bn(blk.conv2, blk.bn2))
    parts, biases = [], []
    for li, (w, b) in enumerate(convs):
        if li == 0:
            w = torch.cat([w, torch.zeros(C, 13, 3, 3, device=w.device)], dim=1)
        parts += _pieces(w, dtype, pair)
        biases.append(b)
    return torch.cat(parts).contiguous(), torch.stack(biases).contiguous().float()


def _pieces(w: Tensor, dtype: torch.dtype, pair: bool) -> list[Tensor]:
    """[out][in][3][3] -> the (K chunk, [half,] tap) pieces of the layer-pipelined kernels, each [rows][16] in canonical order."""
    n, out = w.shape[0], []
    halves = [(0, n // 2), (n // 2, n)] if pair else [(0, n)]
    for ks in range(w.shape[1] // 16):
        for lo, hi in halves:
            for ky in range(3):
                for kx in range(3):
                    out.append(_canonical_kmajor(w[lo:hi, 16 * ks:16 * ks + 16, ky, kx], dtype))
    return out


def pack_head_weights(model: "ResNet", device, dtype: torch.dtype = torch.bfloat16, pipe: bool = True, pair: bool = False, wide: bool = False):
    """Policy conv1x1 (-> 32) and value conv3x3 (-> 3), BatchNorm folded, as ONE 48-output 3x3 conv for csrc/az_conv.cu
    (the 1x1 weights occupy the centre tap), plus the two fully connected layers in fp32.
    `wide` (csrc/az_resnet_wide.cu): per K chunk the pieces [3 filter rows][64][16] - rows 0..31 the policy channels (centre row
    only), row 32 + 8 kx + v = value channel v, filter column kx; the kernel adds the three columns of a value channel."""
    m = copy.deepcopy(model).eval().float().to(device)
    wp, bp = _fold_bn(m.policy_head[0], m.policy_head[1])  # [32, C, 1, 1]
    wv, bv = _fold_bn(m.value_head[0], m.value_head[1])    # [3, C, 3, 3]
    w = torch.zeros(48, model.num_channels, 3, 3, device=device)
    w[:32, :, 1, 1] = wp[:, :, 0, 0]
    w[32:35] = wv
    b = torch.zeros(48, device=device)
    b[:32], b[32:35] = bp, bv
    if wide:
        rows = torch.zeros(3, 64, model.num_channels, device=device)  # [ky][row][in]
        rows[1, :32] = wp[:, :, 0, 0]
        for kx in range(3):
            rows[:, 32 + 8 * kx:35 + 8 * kx] = wv[:, :, :, kx].permute(2, 0, 1)
        conv = torch.cat([_canonical_kmajor(rows[ky, :, 16 * ks:16 * ks + 16], dtype)
                          for ks in range(model.num_channels // 16) for ky in range(3)]).contiguous()
    elif pipe:  # pieces [48][16] in (ks, tap) order, like the trunk's
        conv = torch.cat(_pieces(w, dtype, pair)).contiguous()
    else:
        conv = torch.cat([_canonical_kmajor(w[:, :, ky, kx], dtype) for ky in range(3) for kx in range(3)]).contiguous()
    f = lambda t: t.detach().float().contiguous()
    return conv, b.contiguous(), f(m.policy_head[4].weight), f(m.policy_head[4].bias), f(m.value_head[4].weight).reshape(-1), f(m.value_head[4].bias)


class TensorCoreTrunk:
    """A ResNet (64 or 128 channels) as one tcgen05 kernel on the engine's leaves (csrc/az_conv.cu, csrc/az_conv128.cu)."""

    def __init__(self, model: "ResNet", device: torch.device, dtype: torch.dtype = torch.bfloat16, variant: int = 0):
        """variant 0: the layer-pipelined kernel (64 or 128 channels); 1: the ping-pong kernel of csrc/az_conv.cu (64 channels);
        2: the layer-pipelined kernel with two 4-position CTAs per SM (64 channels, at most 5 blocks); 3: variant 2 with CTA pairs
        (cta_group::2 MMAs over two SMs, each CTA staging half of the weights); 4: 64 channels with the three taps of a filter row
        fused into one MMA (N = 192; csrc/az_resnet_wide.cu - takes variant 0's packed weights)."""
        from . import _lib

        self.lib = _lib.load()
        self.device = torch.device(device)
        self.dtype = dtype
        self.variant = variant
        self.num_blocks = model.num_res_blocks
        self.num_channels = model.num_channels
        assert variant in (0, 1, 2, 3, 4)
        assert variant in (0, 3) or self.num_channels == 64
        assert variant not in (2, 3) or self.num_blocks <= 5 or self.num_channels == 128
        pair = variant == 3
        self._pack = (lambda m, dev, dt: pack_trunk_weights_pipe(m, dev, dt, pair)) if variant != 1 else pack_trunk_weights
        self.weights, self.biases = self._pack(model, self.device, dtype)
        expect = self.lib.az_resnet_pipe_weight_bytes(self.num_blocks, self.num_channels) if variant != 1 else self.lib.az_trunk_weight_bytes(self.num_blocks)
        assert self.weights.numel() * 2 == expect
        self.heads = pack_head_weights(model, self.device, dtype, pipe=variant != 1, pair=pair, wide=variant == 4)
        hw, hb, fpw, fpb, fvw, fvb = self.heads
        self.desc = _lib.AzResnetDesc(self.num_blocks, model.num_channels, _operand_format(dtype), variant, self.weights.data_ptr(),
                                      self.biases.data_ptr(), hw.data_ptr(), hb.data_ptr(), fpw.data_ptr(), fpb.data_ptr(),
                                      fvw.data_ptr(), fvb.data_ptr())
        self._out: dict[int, Tensor] = {}
        self._lv: dict[int, tuple[Tensor, Tensor]] = {}
        self.launches = 0

    def set_weights(self, model: "ResNet") -> bool:
        """Re-pack `model`'s weights into the existing device buffers (same addresses: captured graphs stay valid)."""
        if model.num_res_blocks != self.num_blocks or model.num_channels != self.num_channels:
            return False
        w, b = self._pack(model, self.device, self.dtype)
        self.weights.copy_(w)
        self.biases.copy_(b)
        for dst, src in zip(self.heads, pack_head_weights(model, self.device, self.dtype, pipe=self.variant != 1, pair=self.variant == 3, wide=self.variant == 4)):
            dst.copy_(src)
        return True

    def forward_leaves_full(self, engine) -> tuple[Tensor, Tensor]:
        """Trunk AND heads in the one kernel -> (logits [n,7] f32, values [n,2] f32) for the engine's current leaves."""
        n = engine.n_active
        if n not in self._lv:
            self._lv[n] = (torch.zeros((n, 7), device=self.device), torch.zeros((n, 2), device=self.device))  # rows of slots without an evaluation stay zero
        logits, values = self._lv[n]
        import ctypes as C

        rc = self.lib.az_resnet_forward_leaves_v2(engine.h, C.byref(self.desc), logits.data_ptr(), values.data_ptr(),
                                                  torch.cuda.current_stream(self.device).cuda_stream)
        if rc != 0:
            raise RuntimeError(f"az_resnet_forward_leaves_v2 failed ({rc})")
        self.launches += 1
        return logits, values

    def forward_leaves(self, engine) -> Tensor:
        """-> trunk activations [n, 64, 6, 7] bf16 (channels-last memory) for the leaves of `engine.select_leaves()`."""
        assert self.dtype == torch.bfloat16 and self.variant == 1, "the trunk-only entry point belongs to the ping-pong kernel (bf16, 64 channels)"
        n = engine.n_active
        if n not in self._out:
            self._out[n] = torch.empty((n, 6, 7, 64), dtype=torch.bfloat16, device=self.device)
        out = self._out[n]
        rc = self.lib.az_trunk_forward_leaves(engine.h, self.weights.data_ptr(), self.biases.data_ptr(), self.num_blocks,
                                              out.data_ptr(), torch.cuda.current_stream(self.device).cuda_stream)
        if rc != 0:
            raise RuntimeError(f"az_trunk_forward_leaves failed ({rc})")
        self.launches += 1
        return out.permute(0, 3, 1, 2)  # NCHW view of NHWC memory == channels_last


def pack_cnn_weights(model: "CNNModel", device, dtype: torch.dtype = torch.bfloat16):
    """CNNModel's weights as operands of csrc/az_cnn.cu.  Convolutions (BatchNorm folded): pieces [9 taps][out][16 in] per K chunk -
    conv1 one piece [9][64][16] (3 -> 16 input channels), conv2 four pieces [9][128][16], conv3 eight pieces for output channels
    0..127 and eight for 128..255.  Linear 10752 -> 512: input index c * 42 + pixel (NCHW Flatten) reordered to pixel * 256 + c,
    then per chunk of 32 inputs a tile [512][32] in the MMA's canonical order.  Heads: [8][512] fp32 (7 policy rows, 1 value row)."""
    m = copy.deepcopy(model).eval().float().to(device)
    convs = [_fold_bn(m.conv_layers[0], m.conv_layers[1]), _fold_bn(m.conv_layers[3], m.conv_layers[4]), _fold_bn(m.conv_layers[6], m.conv_layers[7])]
    w0, w1, w2 = (w for w, _ in convs)
    w0 = torch.cat([w0, torch.zeros(64, 13, 3, 3, device=w0.device)], dim=1)
    parts = []

    def pieces(w):
        for ks in range(w.shape[1] // 16):
            for ky in range(3):
                for kx in range(3):
                    parts.append(_canonical_kmajor(w[:, 16 * ks:16 * ks + 16, ky, kx], dtype))

    pieces(w0)
    pieces(w1)
    pieces(w2[:128])
    pieces(w2[128:])
    conv_w = torch.cat(parts).contiguous()
    conv_b = torch.cat([b for _, b in convs]).contiguous().float()
    fc = m.shared_layers[0]
    wf = fc.weight.detach().float().reshape(512, 256, 42).permute(0, 2, 1).reshape(512, 42 * 256)  # [out][pixel * 256 + c]
    fc_w = torch.cat([_canonical_kmajor(wf[:, 32 * k:32 * k + 32], dtype) for k in range(42 * 256 // 32)]).contiguous()
    head_w = torch.cat([m.policy_head.weight.detach().float(), m.value_head[0].weight.detach().float()]).contiguous()
    head_b = torch.cat([m.policy_head.bias.detach().float(), m.value_head[0].bias.detach().float()]).contiguous()
    return conv_w, conv_b, fc_w, fc.bias.detach().float().contiguous(), head_w, head_b


class TensorCoreCNN:
    """CNNModel.forward as two tcgen05 kernels on the engine's leaves (csrc/az_cnn.cu)."""

    num_channels = 0
    variant = 0

    def __init__(self, model: "CNNModel", device: torch.device, dtype: torch.dtype = torch.bfloat16):
        from . import _lib

        self.lib = _lib.load()
        self.device = torch.device(device)
        self.dtype = dtype
        self.w = list(pack_cnn_weights(model, self.device, dtype))
        assert self.w[0].numel() * 2 == self.lib.az_cnn_conv_weight_bytes() and self.w[2].numel() * 2 == self.lib.az_cnn_fc_weight_bytes()
        self.workspace = None
        self._lv: dict[int, tuple[Tensor, Tensor]] = {}
        self.desc = None
        self.launches = 0

    def set_weights(self, model: "CNNModel") -> bool:
        for dst, src in zip(self.w, pack_cnn_weights(model, self.device, self.dtype)):
            dst.copy_(src)
        return True

    def _descriptor(self, n: int):
        from . import _lib

        need = int(self.lib.az_cnn_workspace_bytes(n))
        if self.workspace is None or self.workspace.numel() < need:
            self.workspace = torch.zeros(need, dtype=torch.uint8, device=self.device)  # conv3 activations of the evaluated leaves (21.5 KB each)
            cw, cb, fw, fb, hw, hb = self.w
            self.desc = _lib.AzCnnDesc(_operand_format(self.dtype), 0, cw.data_ptr(), cb.data_ptr(), fw.data_ptr(), fb.data_ptr(), hw.data_ptr(),
                                       hb.data_ptr(), self.workspace.data_ptr(), self.workspace.numel())
        return self.desc

    def forward_leaves_full(self, engine) -> tuple[Tensor, Tensor]:
        import ctypes as C

        n = engine.n_active
        if n not in self._lv:
            self._lv[n] = (torch.zeros((n, 7), device=self.device), torch.zeros((n, 2), device=self.device))
        logits, values = self._lv[n]
        rc = self.lib.az_cnn_forward_leaves(engine.h, C.byref(self._descriptor(n)), logits.data_ptr(), values.data_ptr(),
                                            torch.cuda.current_stream(self.device).cuda_stream)
        if rc != 0:
            raise RuntimeError(f"az_cnn_forward_leaves failed ({rc})")
        self.launches += 2
        return logits, values


class InferenceNet(nn.Module):
    """Search-time form of a `Model` (the role of `get_inference_clone()`, models/base/model.py:92-96):
    eval-mode, BatchNorm folded, conv/linear weights in `dtype` (bf16 on the hot path), activations
    channels-last.  `forward(planes) -> (logits f32 [B,7], values f32 [B,2])`, consumed directly by
    `az_expand_backup`.  BasicNN stays fp32 (config 1 parity is quoted in fp32)."""

    def __init__(self, model: Model, dtype: torch.dtype = torch.bfloat16, device: torch.device | str = "cuda",
                 use_tensor_core_kernels: bool = True, trunk_variant: int | None = None):
        super().__init__()
        self.trunk = None
        m = copy.deepcopy(model).eval().to(device)
        self.kind = type(model).__name__
        self.dtype = dtype
        self.layers: list[tuple[str, Tensor, Tensor]] = []
        self.fused = None
        if isinstance(m, BasicNN):
            self.input_layout = LAYOUT_GRID_F32
            self.net = m
            if dtype in (torch.bfloat16, torch.float16):  # hand-written tensor-core path
                self.fused = TensorCoreMLP(m, torch.device(device), dtype)
            else:
                self.dtype = torch.float32
        elif isinstance(m, (CNNModel, ResNet)):
            self.input_layout = LAYOUT_PLANES_BF16 if dtype == torch.bfloat16 else LAYOUT_PLANES_F32
            self.trunk = None
            if isinstance(m, CNNModel) and dtype in (torch.bfloat16, torch.float16) and use_tensor_core_kernels:
                self.trunk = TensorCoreCNN(m, torch.device(device), dtype)  # hand-written tcgen05 kernels (csrc/az_cnn.cu)
            if isinstance(m, ResNet) and m.num_channels in (64, 128) and m.num_res_blocks <= (9 if m.num_channels == 128 else 11) and dtype in (torch.bfloat16, torch.float16) and use_tensor_core_kernels:
                # hand-written tcgen05 kernel, trunk + heads.  64 channels, measured at 16384 positions x 4 blocks (profiles/r02_*):
                # filter rows fused into N = 192 MMAs, csrc/az_resnet_wide.cu (variant 4) 0.51 ms; layer-pipelined with two 4-position
                # CTAs per SM, csrc/az_resnet_pipe.cu (variant 2, up to 5 blocks) 0.64 ms; ping-pong, csrc/az_conv.cu (variant 1)
                # 0.70 ms; layer-pipelined with one 8-position CTA (variant 0) 0.75 ms.  128 channels only fit the layer-pipelined schedule
                auto = 4 if m.num_res_blocks >= 1 else 2
                if m.num_channels == 128:
                    variant = 3 if trunk_variant == 3 else 0
                else:
                    variant = auto if trunk_variant is None else trunk_variant
                self.trunk = TensorCoreTrunk(m, torch.device(device), dtype, variant=variant)
            self.net = self._fold(m).to(dtype).to(memory_format=torch.channels_last)
        else:
            self.input_layout = getattr(model, "input_layout", LAYOUT_PLANES_F32)
            self.net = m
            self.dtype = torch.float32
        for p in self.parameters():
            p.requires_grad_(False)

    @staticmethod
    def _fold(m: nn.Module) -> nn.Module:
        def fold_seq(seq: nn.Sequential) -> nn.Sequential:
            out, mods, i = [], list(seq), 0
            while i < len(mods):
                if isinstance(mods[i], nn.Conv2d) and i + 1 < len(mods) and isinstance(mods[i + 1], nn.BatchNorm2d):
                    w, b = _fold_bn(mods[i], mods[i + 1])
                    conv = nn.Conv2d(mods[i].in_channels, mods[i].out_channels, mods[i].kernel_size, padding=mods[i].padding)
                    conv.weight.data, conv.bias.data = w, b
                    out.append(conv)
                    i += 2
                elif isinstance(mods[i], nn.Dropout):
                    i += 1
                else:
                    out.append(mods[i])
                    i += 1
            return nn.Sequential(*out)

        if isinstance(m, CNNModel):
            m.conv_layers = fold_seq(m.conv_layers)
            m.shared_layers = fold_seq(m.shared_layers)
        else:
            m.input_conv = fold_seq(m.input_conv)
            for blk in m.residual_blocks:
                for cn, bn in (("conv1", "bn1"), ("conv2", "bn2")):
                    w, b = _fold_bn(getattr(blk, cn), getattr(blk, bn))
                    getattr(blk, cn).weight.data, getattr(blk, cn).bias.data = w, b
                    setattr(blk, bn, nn.Identity())
            m.policy_head = fold_seq(m.policy_head)
            m.value_head = fold_seq(m.value_head)
        return m

    @torch.no_grad()
    def refresh(self, model: Model) -> bool:
        """Take `model`'s weights in place (device addresses unchanged, so the CUDA graph captured around this net stays valid).
        Returns False when the architecture differs and the caller must rebuild."""
        if type(model).__name__ != self.kind:
            return False
        dev = next(self.net.parameters()).device
        if self.fused is not None:
            self.fused.set_weights(model)
            return True
        if self.trunk is not None:
            if not self.trunk.set_weights(model):
                return False
        new = copy.deepcopy(model).eval().to(dev)
        if isinstance(new, (CNNModel, ResNet)):
            new = self._fold(new)
        old_t = list(self.net.parameters()) + list(self.net.buffers())
        new_t = list(new.parameters()) + list(new.buffers())
        if len(old_t) != len(new_t) or any(a.shape != b.shape for a, b in zip(old_t, new_t)):
            return False
        for a, b in zip(old_t, new_t):
            a.copy_(b.to(a.dtype))
        return True

    @property
    def wants_leaf_compaction(self) -> bool:
        """The ResNet kernels process several waves of small batches, so skipping the ~15 % of slots whose leaf is terminal pays;
        the MLP kernel is one wave of 128-row tiles either way."""
        return self.trunk is not None

    @property
    def position_only_outputs(self) -> bool:
        """A leaf's outputs are a pure function of its position (deterministic, independent of the batch it falls in), so the
        engine's evaluation cache may serve them: k_resnet_wide (tests/test_gpu_resnet_pipe.py pins both properties)."""
        return isinstance(self.trunk, TensorCoreTrunk) and self.trunk.variant == 4

    @property
    def kernel_name(self) -> str:
        if self.fused is not None:
            return "k_mlp_fused"
        if self.trunk is not None:
            if isinstance(self.trunk, TensorCoreCNN):
                return "k_cnn_conv + k_cnn_fc"
            return {1: "k_resnet_trunk", 4: "k_resnet_wide"}.get(self.trunk.variant, "k_resnet_pipe")
        return "k_encode + cuDNN/cuBLAS (torch)"

    @torch.no_grad()
    def forward_leaves(self, engine) -> tuple[Tensor, Tensor]:
        """Evaluate the engine's current leaves without a separate gather launch (tensor-core kernels only)."""
        if self.fused is not None:
            return self.fused.forward_leaves(engine)
        return self.trunk.forward_leaves_full(engine)  # trunk + heads, one tcgen05 kernel

    @property
    def evaluates_leaves_directly(self) -> bool:
        return self.fused is not None or self.trunk is not None

    @torch.no_grad()
    def forward(self, x: Tensor) -> tuple[Tensor, Tensor]:
        if self.fused is not None:
            return self.fused(x)
        if x.dim() == 4:
            x = x.contiguous(memory_format=torch.channels_last)
        logits, values = self.net(x.to(self.dtype))
        return logits.float().contiguous(), values.float().contiguous()
