"""Policy/value networks (plain PyTorch -- the net is the only dense contraction on the path and
the only user of the tensor cores; it is library code, not the product).

``PolicyValueMLP`` is the reference's only architecture -- ``TicTacToeNet``, a 4-layer ReLU MLP
``in -> H -> H -> H -> actions`` (src/tic_tac_toe/SL/neural_networks.py:4-30, hidden 256 in
src/tic_tac_toe/SL/train.py:186) -- widened to the 8x8 board and given the value head AlphaZero
needs.  ``PolicyValueResNet`` is the usual AlphaZero tower for stronger play.

Every net maps the bf16 canonical planes written by the leaf-gather kernel to
``(policy logits [B, A], value [B] in [-1, 1])``.
"""
from __future__ import annotations

import torch
from torch import nn

N_ACTIONS = 65
TTT_ACTIONS = 9


def _swizzled_slabs(W: torch.Tensor) -> torch.Tensor:
    """[rows, K] bf16 -> uint8 [K/64 slabs, rows * 128 B]: K-major SWIZZLE_128B (16-byte chunk j of row r
    at chunk j ^ (r & 7) of its 128-byte row), the shared-memory image of a UMMA operand."""
    rows, K = W.shape
    v = W.contiguous().view(rows, K // 64, 8, 8).permute(1, 0, 2, 3).contiguous()  # [s, r, j, e]
    r = torch.arange(rows, device=W.device)[:, None]
    j = torch.arange(8, device=W.device)[None, :]
    src = (j ^ (r & 7))[None, :, :, None].expand(K // 64, rows, 8, 8)
    return torch.gather(v, 2, src).reshape(K // 64, rows * 64).view(torch.uint8)


def pack_mlp_pair_image(weights, biases) -> torch.Tensor:
    """Weight image of ``bz_mlp_forward_pair``: uint8 [2, 187712]; rank r of a CTA pair holds output rows
    r*N/2 .. (r+1)*N/2 of every layer (N = 256, 256, 256, 80), layer after layer, each layer as K/64 slabs,
    then all 848 biases as float32."""
    bias = torch.cat([b.float().reshape(-1) for b in biases]).contiguous().view(torch.uint8)
    ranks = []
    for r in range(2):
        parts = []
        for W in weights:
            h = W.shape[0] // 2
            parts.append(_swizzled_slabs(W[r * h:(r + 1) * h]).reshape(-1))
        ranks.append(torch.cat(parts + [bias]))
    return torch.stack(ranks).contiguous()


class PolicyValueMLP(nn.Module):
    """in -> H -> H -> H -> (A logits, 1 value): TicTacToeNet (neural_networks.py:4-30) + value head."""

    def __init__(self, in_features: int = 128, hidden: int = 256, n_actions: int = N_ACTIONS):
        super().__init__()
        self.fc1 = nn.Linear(in_features, hidden)
        self.fc2 = nn.Linear(hidden, hidden)
        self.fc3 = nn.Linear(hidden, hidden)
        self.policy = nn.Linear(hidden, n_actions)
        self.value = nn.Linear(hidden, 1)
        self.relu = nn.ReLU()
        self.n_actions = n_actions
        self.raw_width = (n_actions + 1 + 7) // 8 * 8  # fused head, padded so the GEMM stays aligned
        self._head = None

    def forward(self, planes: torch.Tensor):
        x = planes.reshape(planes.shape[0], -1).to(self.fc1.weight.dtype)
        x = self.relu(self.fc1(x))
        x = self.relu(self.fc2(x))
        x = self.relu(self.fc3(x))
        return self.policy(x), torch.tanh(self.value(x)).squeeze(-1)

    # -- inference fast paths -----------------------------------------------------------------------
    @torch.no_grad()
    def prepare_inference(self) -> None:
        """(Re)build the fused policy+value head and the kernels' weight images; call after every weight update.

        The buffers keep their ADDRESSES across calls (allocated once, refreshed with ``copy_``): a CUDA graph captured
        by ``BatchedMCTS`` has the device pointers of the head / weight image baked into its kernel parameters, so a
        refresh that re-allocated them would leave every graph replay reading the old (freed) weights."""
        A, H = self.n_actions, self.policy.in_features
        rows = max(self.raw_width, 80) if self.raw_width <= 80 else self.raw_width  # 80 = UMMA N of the fused kernel
        w = torch.zeros((rows, H), dtype=self.policy.weight.dtype, device=self.policy.weight.device)
        b = torch.zeros(rows, dtype=w.dtype, device=w.device)
        w[:A], w[A] = self.policy.weight, self.value.weight[0]
        b[:A], b[A] = self.policy.bias, self.value.bias[0]

        def keep(name, new):
            """store ``new`` under ``name``, in place when a buffer of the same shape / dtype / device exists"""
            old = getattr(self, name, None)
            if (isinstance(old, torch.Tensor) and old.shape == new.shape and old.dtype == new.dtype
                    and old.device == new.device):
                old.copy_(new)
                return old
            object.__setattr__(self, name, new.contiguous())
            return getattr(self, name)

        hw, hb = keep("_head_w", w), keep("_head_b", b)
        self._head_full = (hw, hb)
        self._head = (hw[: self.raw_width], hb[: self.raw_width])
        self._w = [m.weight.t() for m in (self.fc1, self.fc2, self.fc3)]  # views of the parameters themselves
        if w.is_cuda and w.dtype == torch.bfloat16 and self.fc1.in_features == 128 and self.fc1.out_features == 256 \
                and self.raw_width == 72:
            ws = [self.fc1.weight, self.fc2.weight, self.fc3.weight, hw[:80]]
            bs = [self.fc1.bias, self.fc2.bias, self.fc3.bias, hb[:80]]
            keep("_image_pair", pack_mlp_pair_image(ws, bs))
        else:
            self._image_pair = None

    def fused_kernel_ok(self, planes: torch.Tensor) -> bool:
        """the hand-written tcgen05 kernel covers exactly the Reversi shape in bf16 on a GPU"""
        return (planes.is_cuda and planes.dtype == torch.bfloat16 and self.fc1.weight.dtype == torch.bfloat16
                and self.fc1.in_features == 128 and self.fc1.out_features == 256 and self.raw_width == 72
                and not self.training)

    @torch.no_grad()
    def forward_raw(self, planes: torch.Tensor, out: torch.Tensor | None = None, fused: bool | str | None = None) -> torch.Tensor:
        """[B, raw_width]: policy logits in columns 0..A-1, PRE-tanh value in column A.

        ``fused=False``: 3 ``addmm+ReLU`` (cuBLASLt epilogue) + 1 head GEMM through PyTorch.
        ``fused="pair"``: the single-launch tcgen05 kernel on CTA pairs (``bz_mlp_forward_pair``: cta_group::2
        MMAs, each CTA keeps half of every weight matrix resident in shared memory);
        ``fused="pair2"``: the pair kernel with two ping-ponged tiles per pair (``bz_mlp_forward_pair2``).
        ``fused=None`` / ``True`` picks, for the supported shape, the pair kernel while one wave of CTA pairs
        covers the batch (<= 74 x 128 rows) and the two-tile pair kernel above that; ``None`` falls back to the
        library GEMMs for other shapes, ``True`` raises.  Both kernels give bit-identical outputs.  Measured on
        B200 per forward (graph, back to back): 4096 rows pair 6.8 us / cuBLASLt 11.8; 16 384 rows pair2 9.9 /
        19.8; 65 536 rows pair2 34.5 / 52.4 (profiles/README.md)."""
        if self._head is None:
            self.prepare_inference()
        B = planes.shape[0]
        if fused is None or fused is True:
            ok = self.fused_kernel_ok(planes) and getattr(self, "_image_pair", None) is not None
            if fused is True and not ok:
                raise RuntimeError("the tcgen05 MLP kernels cover only the bf16 128-256-256-256-(65+1) net on a GPU")
            # one wave of CTA pairs with one 128-row tile each (lowest latency) up to 74 pairs; above that every
            # pair ping-pongs two tiles (measured faster than cuBLASLt up to at least 131 072 rows)
            fused = ("pair" if B <= 74 * 128 else "pair2") if ok else False
        if fused:
            from . import _lib

            if fused not in ("pair", "pair2") or getattr(self, "_image_pair", None) is None:
                raise RuntimeError(f"unknown / unavailable MLP kernel {fused!r}")
            if out is None:
                out = torch.empty((B, self.raw_width), dtype=torch.bfloat16, device=planes.device)
            x = planes.flatten(1)  # [B, 128]; reshape(B, -1) cannot size an empty batch
            L = _lib.load()
            fn, name = ((L.bz_mlp_forward_pair2, "bz_mlp_forward_pair2") if fused == "pair2"
                        else (L.bz_mlp_forward_pair, "bz_mlp_forward_pair"))
            _lib.check(fn(_lib.dptr(x), _lib.dptr(self._image_pair), _lib.dptr(out), B, _lib.stream_ptr()), name)
            return out
        x = planes.flatten(1).to(self.fc1.weight.dtype)
        x = torch._addmm_activation(self.fc1.bias, x, self._w[0])
        x = torch._addmm_activation(self.fc2.bias, x, self._w[1])
        x = torch._addmm_activation(self.fc3.bias, x, self._w[2])
        hw, hb = self._head
        if out is None:
            return torch.addmm(hb, x, hw.t())
        return torch.addmm(hb, x, hw.t(), out=out)


class _ResBlock(nn.Module):
    def __init__(self, ch: int):
        super().__init__()
        self.c1 = nn.Conv2d(ch, ch, 3, padding=1, bias=False)
        self.b1 = nn.BatchNorm2d(ch)
        self.c2 = nn.Conv2d(ch, ch, 3, padding=1, bias=False)
        self.b2 = nn.BatchNorm2d(ch)

    def forward(self, x):
        y = torch.relu(self.b1(self.c1(x)))
        y = self.b2(self.c2(y))
        return torch.relu(x + y)


class PolicyValueResNet(nn.Module):
    """AlphaZero-style tower on [B, 2, 8, 8] planes."""

    def __init__(self, channels: int = 64, blocks: int = 4, n_actions: int = N_ACTIONS):
        super().__init__()
        self.stem = nn.Sequential(nn.Conv2d(2, channels, 3, padding=1, bias=False), nn.BatchNorm2d(channels), nn.ReLU())
        self.tower = nn.Sequential(*[_ResBlock(channels) for _ in range(blocks)])
        self.p_conv = nn.Sequential(nn.Conv2d(channels, 2, 1, bias=False), nn.BatchNorm2d(2), nn.ReLU())
        self.p_fc = nn.Linear(2 * 64, n_actions)
        self.v_conv = nn.Sequential(nn.Conv2d(channels, 1, 1, bias=False), nn.BatchNorm2d(1), nn.ReLU())
        self.v_fc = nn.Sequential(nn.Linear(64, 64), nn.ReLU(), nn.Linear(64, 1))

    def forward(self, planes: torch.Tensor):
        x = planes.reshape(-1, 2, 8, 8).to(self.p_fc.weight.dtype)
        x = self.tower(self.stem(x))
        p = self.p_fc(self.p_conv(x).flatten(1))
        v = torch.tanh(self.v_fc(self.v_conv(x).flatten(1))).squeeze(-1)
        return p, v


def make_net(kind: str = "mlp", game: str = "reversi", hidden: int = 256, channels: int = 64, blocks: int = 4,
             seed: int | None = 0, device="cuda", dtype=torch.bfloat16) -> nn.Module:
    """Random-init net (there are no checkpoints to load: the reference has no Reversi net and its
    tic-tac-toe pickles are policy-only, see SURVEY.md section 2 #13)."""
    if seed is not None:
        torch.manual_seed(seed)
    if game == "ttt":
        net = PolicyValueMLP(9, hidden, TTT_ACTIONS)  # 9 inputs: the reference's own canonical vector
    elif kind == "mlp":
        net = PolicyValueMLP(128, hidden, N_ACTIONS)
    elif kind == "resnet":
        net = PolicyValueResNet(channels, blocks, N_ACTIONS)
    else:
        raise ValueError(f"unknown net kind {kind!r}")
    return net.to(device=device, dtype=dtype).eval()


def matmul_flops_per_position(net: nn.Module) -> int:
    """2 * MACs of the Linear / Conv2d layers for one position (SURVEY.md 8d 'Net flops')."""
    total = 0
    for m in net.modules():
        if isinstance(m, nn.Linear):
            total += 2 * m.in_features * m.out_features
        elif isinstance(m, nn.Conv2d):
            k = m.kernel_size[0] * m.kernel_size[1]
            total += 2 * 64 * m.in_channels * m.out_channels * k // m.groups
    return total
