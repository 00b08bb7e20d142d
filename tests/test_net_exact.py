"""The policy/value net, bit for bit: exactly representable nets against a float64 reference.

An "exact net" has weights and biases that are small integers times a power of two per layer, with sparse rows, and is
fed 0/1 planes (the tic-tac-toe net of test_gpu_logits_path.py: 0/+-1 cells).  `check_exact` proves, on the data of each test, that every partial sum of every layer is then an
integer multiple of the layer's grid unit u far below 2^24 u: the fp32 accumulators of the tensor cores hold the exact
sum whatever the summation order, and every bf16 the kernels write must equal the float64 sum rounded to nearest even.
So the tcgen05 MLP kernels (`bz_mlp_forward_pair` / `_pair2`) and the copy of the net inside the one-launch search
(`bz_mcts_search_fused`, `bz_mcts_search_fused_entrants`) are compared with `reference_forward` by equality, not by a
tolerance.  The priors and values the searches store go through the in-kernel softmax (`ex2.approx`) and `tanhf`; they
are checked against the float64 softmax and tanh of the exact logits with the bounds of
test_gpu_mcts.py::test_logits_mode_fused_softmax_and_tanh, in every node of every tree.

The CPU tests check the premises: the generated nets are exact and round (with ties) in every layer, the reference
equals the PyTorch module, and an independent decoder recovers the weight image the kernels read."""
import numpy as np
import pytest
import torch

N_ACTIONS = 65
IMAGE_RANK_BYTES = (2 * 128 + 4 * 128 + 4 * 128 + 4 * 40) * 128 + (3 * 256 + 80) * 4  # include/betazero_b200.h
RTOL = 1e-5  # the in-kernel softmax (ex2.approx) and tanhf: the bound of test_gpu_mcts.py's logits-mode test


# ---------------------------------------------------------------------------------------------------------------------
# exact nets and the float64 reference
# ---------------------------------------------------------------------------------------------------------------------
def _sparse_ints(rows, cols, nnz, wmax, g):
    """[rows, cols] float64: nnz nonzeros per row at random columns, values in +-[1, wmax]"""
    pos = torch.rand(rows, cols, generator=g).argsort(dim=1)[:, :nnz]
    val = torch.randint(1, wmax + 1, (rows, nnz), generator=g) * (torch.randint(0, 2, (rows, nnz), generator=g) * 2 - 1)
    return torch.zeros(rows, cols, dtype=torch.float64).scatter_(1, pos, val.double())


def exact_net(seed, nnz=(24, 16, 16, 16), wmax=(7, 7, 3, 3), bias=(64, 64, 64, 64), shifts=(0, 0, 0, 12), device="cpu",
              n_in=128, n_actions=N_ACTIONS):
    """A bf16 PolicyValueMLP n_in-256-256-256-(n_actions+1) (default: the Reversi net 128-256-256-256-(65+1)) whose
    layer l (fc1, fc2, fc3, head) has nnz[l] nonzero weights per row, integers in +-[1, wmax[l]], integer biases in
    [-bias[l], bias[l]], all times 2^-shifts[l].  The value row is the head's last row.  The default head shift keeps
    the logits within about +-20 on Reversi positions."""
    from betazero_b200 import net

    g = torch.Generator().manual_seed(seed)
    m = net.PolicyValueMLP(n_in, 256, n_actions)
    shapes = ((256, n_in), (256, 256), (256, 256), (n_actions + 1, 256))
    params = []
    for l, (rows, cols) in enumerate(shapes):
        W = _sparse_ints(rows, cols, nnz[l], wmax[l], g) * 2.0 ** -shifts[l]
        b = torch.randint(-bias[l], bias[l] + 1, (rows,), generator=g).double() * 2.0 ** -shifts[l]
        params.append((W, b))
    with torch.no_grad():
        for fc, (W, b) in zip((m.fc1, m.fc2, m.fc3), params[:3]):
            fc.weight.copy_(W)
            fc.bias.copy_(b)
        W, b = params[3]
        m.policy.weight.copy_(W[:n_actions])
        m.policy.bias.copy_(b[:n_actions])
        m.value.weight.copy_(W[n_actions:])
        m.value.bias.copy_(b[n_actions:])
    return m.to(device=device, dtype=torch.bfloat16).eval()


def _layers(net):
    """[(W, b)] of fc1, fc2, fc3 and the 66-row head (policy rows, then the value row), float64 copies of the bf16
    parameters"""
    head_w = torch.cat([net.policy.weight, net.value.weight])
    head_b = torch.cat([net.policy.bias, net.value.bias])
    return [(fc.weight.double(), fc.bias.double()) for fc in (net.fc1, net.fc2, net.fc3)] + [(head_w.double(), head_b.double())]


def _unit(x):
    """the largest power of two of which every element of x is an integer multiple"""
    for s in range(-64, 200):
        y = x * 2.0 ** s
        if torch.equal(y, torch.round(y)):
            return 2.0 ** -s
    raise AssertionError("not on a power-of-two grid")


def _to_bf16(x):
    """float64 -> the nearest bf16, ties to even (the float64 -> bfloat16 conversion rounds correctly), as float64"""
    return x.to(torch.bfloat16).double()


@torch.no_grad()
def reference_forward(planes, net):
    """float64 [B, 66]: columns 0..65 of the net's raw output (65 logits, the pre-tanh value), each layer the exact sum
    plus the bias rounded once to bf16, ReLU on the hidden layers"""
    a = planes.reshape(planes.shape[0], -1).double()
    layers = _layers(net)
    for l, (W, b) in enumerate(layers):
        a = _to_bf16(a @ W.t() + b)
        if l < 3:
            a = torch.relu(a)
    return a


@torch.no_grad()
def check_exact(net, planes):
    """Assert that every layer of `net` computes exactly in fp32 on these planes, whatever the order of the sum; return
    the float64 pre-activations (sum + bias) of the four layers.

    Per layer, with u_w the weights' grid, u_a that of the layer's input activations and u_b the biases' grid: every
    product w_k * a_k is an integer multiple of u_w * u_a, so with u = min(u_w * u_a, u_b) (powers of two: the smaller
    divides the larger) every term of the sum is an integer multiple of u; and sum_k |w_k * a_k| + |b| < 2^22 u.  Then
    every partial sum, in any order and grouping, is an integer multiple of u smaller than 2^22 u, i.e. has at most 22
    significant bits, and fp32 (24 bits) holds it exactly; the spare 2 bits cover a tensor core that aligns its products to the
    largest exponent of a group before adding.  The kernels' fp32 accumulators and their fp32 bias add therefore hold
    the exact value, and the bf16 they write is that value rounded to nearest even: what `reference_forward` computes.
    Rounding a multiple of u to bf16 gives a multiple of u again, so the next layer's input grid is u."""
    a = planes.reshape(planes.shape[0], -1).double()
    u_a = 1.0
    assert torch.equal(a.abs(), (a.abs() == 1).double()), "the planes must be 0/1 (tic-tac-toe: 0/+-1)"
    pre = []
    for l, (W, b) in enumerate(_layers(net)):
        u = min(_unit(W) * u_a, _unit(b))  # every product and the bias are integer multiples of u
        assert u >= 2.0 ** -100, (l, u)  # far from fp32's subnormals
        bound = a.abs() @ W.abs().t() + b.abs()  # sum_k |w_k a_k| + |b| per row and output (exact in float64)
        assert (bound < 2.0 ** 22 * u).all(), f"layer {l}: |sum| up to {bound.max().item() / u:.0f} u, not below 2^22 u"
        x = a @ W.t() + b
        pre.append(x)
        a = _to_bf16(x)
        if l < 3:
            a = torch.relu(a)
        assert torch.equal(a / u, torch.round(a / u)), f"layer {l}: a rounded output is off the grid"
        u_a = u
    return pre


def rounding_stats(x):
    """(values bf16 rounds, exact ties among them, negative values) of float64 values exact in fp32"""
    low = x.float().view(torch.int32) & 0xFFFF  # the 16 bits bf16 drops
    return int((low != 0).sum()), int((low == 0x8000).sum()), int((x < 0).sum())


def planes_of(me, opp):
    """bf16 [n, 2, 8, 8] network input of mover-relative boards (int64 tensors holding uint64 bits): plane 0 = me,
    plane 1 = opp, bit = row * 8 + col"""
    bit = torch.arange(64, device=me.device)
    p = torch.stack([(me[:, None] >> bit) & 1, (opp[:, None] >> bit) & 1], dim=1)
    return p.reshape(-1, 2, 8, 8).to(torch.bfloat16)


def _random_planes(B, seed, device="cpu"):
    g = torch.Generator().manual_seed(seed)
    a = torch.randint(0, 3, (B, 64), generator=g)
    return torch.stack([a == 1, a == 2], dim=1).reshape(B, 2, 8, 8).to(device=device, dtype=torch.bfloat16)


# the nets of the tests: "logits" has the realistic +-20 logits of the searches; "raw" keeps the integer head (logits
# up to ~1e5); "large" has fc1 biases up to 512, so that fc1 rounds too and the hidden values are large
NET_KW = {
    "logits": dict(seed=1),
    "raw": dict(seed=2, shifts=(0, 0, 0, 0)),
    "large": dict(seed=3, bias=(512, 64, 64, 64), shifts=(0, 1, 0, 13)),
}


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the premises
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(NET_KW))
def test_exact_nets_are_exact_and_round_in_every_layer(name):
    """The nets meet check_exact on random and on reachable positions, and every layer produces what the GPU tests rely
    on: outputs bf16 rounds, exact ties, negative pre-activations (ReLU at work)."""
    from oracle import pyoracle as po

    m = exact_net(**NET_KW[name])
    B = 4096
    check_exact(m, planes_of(*(torch.from_numpy(x.view(np.int64)) for x in po.playout_boards(256, seed=7))))
    pre = check_exact(m, _random_planes(B, 11))
    for l, x in enumerate(pre):
        rounded, ties, neg = rounding_stats(x)
        n = x.numel()
        assert neg > n // 5, (l, neg, n)
        if l == 0 and name != "large":
            continue  # small fc1 biases: fc1's sums stay below 256 and need no rounding
        assert rounded > n // 20 and ties > n // 200, (l, rounded, ties, n)
    logits = _to_bf16(pre[3][:, :N_ACTIONS])
    if name != "raw":
        assert 2 < logits.abs().max() < 40, logits.abs().max()  # realistic logits: priors neither flat nor underflowing


def test_check_exact_refuses_nets_that_are_not_exact():
    m = exact_net(1)
    x = _random_planes(64, 1)
    check_exact(m, x)
    with torch.no_grad():
        m.fc2.bias[3] = 2.0 ** -20  # a finer grid: the layer's sums need more than 22 bits
    with pytest.raises(AssertionError, match="2\\^22"):
        check_exact(m, x)
    m = exact_net(1, nnz=(128, 256, 256, 256))
    with pytest.raises(AssertionError, match="2\\^22"):  # dense rows: sums too large to stay exact
        check_exact(m, x)


@pytest.mark.parametrize("name", sorted(NET_KW))
def test_reference_forward_equals_the_torch_module(name):
    """reference_forward against PolicyValueMLP.forward in bf16 on the CPU (no cuBLAS): logits bit for bit, the value
    to the precision of a bf16 tanh"""
    m = exact_net(**NET_KW[name])
    x = _random_planes(2048, 5)
    check_exact(m, x)
    ref = reference_forward(x, m)
    with torch.no_grad():
        logits, v = m(x)
    assert logits.dtype == torch.bfloat16 and torch.equal(logits.double(), ref[:, :N_ACTIONS])
    t = torch.tanh(ref[:, N_ACTIONS])
    assert ((v.double() - t).abs() <= 2.0 ** -8 * t.abs() + 1e-30).all()


def decode_pair_image(img):
    """Independent reading of the weight image of bz_mlp_forward_pair (include/betazero_b200.h, net.py): uint8 [2, R]
    -> ([W1 [256, 128], W2, W3 [256, 256], head [80, 256]] as uint16 bf16 bits, float32 biases [848]).  Rank r holds
    rows r * N / 2 .. of every layer; a layer is K / 64 slabs of N / 2 rows x 128 bytes; the 16-byte chunk j of row rr
    sits at chunk j ^ (rr & 7); after the weights come all 848 biases as float32."""
    img = np.asarray(img)
    assert img.shape == (2, IMAGE_RANK_BYTES) and img.dtype == np.uint8
    shapes = ((256, 128), (256, 256), (256, 256), (80, 256))
    Ws = [np.zeros(s, np.uint16) for s in shapes]
    for r in range(2):
        off = 0
        for W, (N, K) in zip(Ws, shapes):
            h = N // 2
            for s in range(K // 64):
                slab = img[r, off:off + h * 128].reshape(h, 8, 16)  # [row, stored chunk, byte]
                off += h * 128
                for rr in range(h):
                    for j in range(8):
                        W[r * h + rr, s * 64 + j * 8:s * 64 + j * 8 + 8] = slab[rr, j ^ (rr & 7)].view(np.uint16)
        biases = img[r, off:].view(np.float32)
        assert off + 848 * 4 == img.shape[1]
        if r == 0:
            b0 = biases.copy()
        else:
            assert np.array_equal(biases.view(np.uint32), b0.view(np.uint32)), "both ranks carry all biases"
    return Ws, b0


def test_weight_image_decodes_to_every_weight_and_bias():
    """pack_mlp_pair_image against the decoder above, twice: every weight holding a code of its row (head rows 65..79
    included, so that a misplaced value or padding row is visible), then a code of its column.  Both decode right only
    if every weight sits where the layout says.  Every bias is distinct."""
    from betazero_b200 import net

    g = torch.Generator().manual_seed(3)
    shapes = ((256, 128), (256, 256), (256, 256), (80, 256))
    bs = [torch.randn(N, generator=g) * 100 for N, _ in shapes]
    for coded in ("row", "column"):
        ws = []
        for l, (N, K) in enumerate(shapes):
            code = (torch.arange(N)[:, None] + 1).expand(N, K) if coded == "row" else -(torch.arange(K) + 1).expand(N, K)
            ws.append((code * 2.0 ** -l).to(torch.bfloat16))  # integers up to 256: distinct in bf16
        img = net.pack_mlp_pair_image(ws, bs)
        assert img.dtype == torch.uint8 and tuple(img.shape) == (2, IMAGE_RANK_BYTES)
        dw, db = decode_pair_image(img.numpy())
        for l, (w, d) in enumerate(zip(ws, dw)):
            bad = np.argwhere(w.view(torch.int16).numpy().view(np.uint16) != d)
            assert not len(bad), f"layer {l} ({coded} codes): weight [{bad[0][0]}, {bad[0][1]}] misplaced"
        assert np.array_equal(db.view(np.uint32), torch.cat(bs).float().numpy().view(np.uint32))


def test_weight_image_of_an_exact_net_decodes_to_its_parameters():
    """the image prepare_inference builds for a net: the fused head puts the policy rows, then the value row, then 14
    zero rows (and zero biases) into the 80-row head"""
    from betazero_b200 import net

    m = exact_net(4)
    hw = torch.zeros(80, 256, dtype=torch.bfloat16)
    hb = torch.zeros(80, dtype=torch.bfloat16)
    hw[:65], hw[65] = m.policy.weight, m.value.weight[0]
    hb[:65], hb[65] = m.policy.bias, m.value.bias[0]
    img = net.pack_mlp_pair_image([m.fc1.weight, m.fc2.weight, m.fc3.weight, hw], [m.fc1.bias, m.fc2.bias, m.fc3.bias, hb])
    _check_image_of(m, img)


def _check_image_of(m, img):
    dw, db = decode_pair_image(img.cpu().numpy())
    layers = _layers(m)
    for l, (W, b) in enumerate(layers):
        got = torch.from_numpy(dw[l].view(np.int16)).view(torch.bfloat16).double()
        assert torch.equal(got[: W.shape[0]], W.cpu()), l
        assert not got[W.shape[0]:].any(), l
    want_b = torch.cat([b.cpu() for _, b in layers[:3]] + [layers[3][1].cpu(), torch.zeros(80 - 66, dtype=torch.float64)])
    assert torch.equal(torch.from_numpy(db).double(), want_b)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the MLP kernels against the reference, bit for bit
# ---------------------------------------------------------------------------------------------------------------------
NAN_BITS = 0x7FC1  # a bf16 NaN: no kernel output, and never equal to anything


def _mismatch(got, ref, what):
    """assert got (bf16 [B, 66]) == ref (float64) by value (+0 == -0, NaN never), naming the first bad entry"""
    ok = got.double() == ref
    if not bool(ok.all()):
        r, c = (~ok).nonzero()[0].tolist()
        n = int((~ok).sum())
        raise AssertionError(f"{what}: {n} entries differ, first [row {r}, col {c}]: kernel {got[r, c].item()!r}, "
                             f"float64 reference {ref[r, c].item()!r}")


def _run_kernel(m, x, variant):
    """forward_raw into rows [0, B) of a NaN-filled [B + 8, 72] buffer; rows >= B must keep the pattern, rows < B must
    lose it everywhere"""
    B = x.shape[0]
    buf = torch.full((B + 8, 72), NAN_BITS, dtype=torch.int16, device="cuda").view(torch.bfloat16)
    out = m.forward_raw(x, out=buf[:B], fused=variant)
    assert out.data_ptr() == buf.data_ptr()
    torch.cuda.synchronize()
    bits = buf.view(torch.int16)
    assert (bits[B:] == NAN_BITS).all(), "a row past the batch was written"
    assert not (bits[:B] == NAN_BITS).any(), "an output element was not written"
    return buf[:B]


def _gpu_nets():
    nets = {}
    for name, kw in NET_KW.items():
        m = exact_net(device="cuda", **kw)
        m.prepare_inference()
        nets[name] = m
    return nets


@pytest.fixture(scope="module")
def gpu_nets():
    return _gpu_nets()


@pytest.mark.gpu
@pytest.mark.parametrize("variant,B", [(v, B) for v in ("pair", "pair2", True)
                                       for B in (1, 2, 127, 128, 129, 255, 256, 257, 9471, 9472, 9473, 18944, 18945)]
                         + [("pair", 20000), ("pair2", 65536)])
def test_mlp_kernels_equal_the_float64_reference(gpu_nets, variant, B):
    """bz_mlp_forward_pair / _pair2 (and the choice of fused=True, which switches kernels above 74 x 128 rows) at the
    tile and wave edges: columns 0..65 equal the float64 reference bit for bit, columns 66..71 are zero"""
    x = _random_planes(B, 1000 + B, device="cuda")
    for name, m in gpu_nets.items():
        check_exact(m, x)
        got = _run_kernel(m, x, variant)
        _mismatch(got[:, :66], reference_forward(x, m), f"{name} net, {variant}, B = {B}")
        assert (got[:, 66:] == 0).all(), "padding columns"
    if B == 1:
        for m in gpu_nets.values():
            _check_image_of(m, m._image_pair)  # the image the kernels read is the net's parameters


def _probe_net(head_block, seed):
    """Every layer a scaled 0/1 selection: fc1 row i reads input bit p1[i % 128] (x1 for i < 128, x2 above), fc2 row i
    reads fc1 unit p2[i], fc3 row i reads fc2 unit p3[i], logit c < 64 reads fc3 unit 64 * head_block + c, logit 64 and
    the value read two more units of that block.  Output column c of a row is then one known input bit (times 1 or 2):
    a misread weight, slab or rank half shows as a wrong column.  Returns the net and the source path of each column."""
    from betazero_b200 import net

    g = torch.Generator().manual_seed(seed)
    p1, p2, p3 = torch.randperm(128, generator=g), torch.randperm(256, generator=g), torch.randperm(256, generator=g)
    m = net.PolicyValueMLP(128, 256, N_ACTIONS)
    unit = 64 * head_block + torch.cat([torch.arange(64), torch.tensor([(7 * head_block + 3) % 64, (11 * head_block + 5) % 64])])
    with torch.no_grad():
        for fc in (m.fc1, m.fc2, m.fc3, m.policy, m.value):
            fc.weight.zero_()
            fc.bias.zero_()
        rows = torch.arange(256)
        m.fc1.weight[rows, p1[rows % 128]] = torch.where(rows < 128, 1.0, 2.0)
        m.fc2.weight[rows, p2] = 1.0
        m.fc3.weight[rows, p3] = 1.0
        m.policy.weight[torch.arange(65), unit[:65]] = 1.0
        m.value.weight[0, unit[65]] = 1.0
    u3 = unit
    u2 = p3[u3]
    u1 = p2[u2]
    return m.to(device="cuda", dtype=torch.bfloat16).eval(), torch.stack([u3, u2, u1, p1[u1 % 128]], dim=1)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["pair", "pair2"])
@pytest.mark.parametrize("B", [257, 9473, 18945])
def test_probe_nets_localise_a_misread_weight(variant, B):
    """Four probe nets cover all 256 hidden units of fc3 (64 per head block); on a mismatch the message names the
    output column and the fc3 / fc2 / fc1 unit and the input bit it should have read."""
    x = _random_planes(B, 77 + B, device="cuda")
    xf = x.reshape(B, -1).double()
    for block in range(4):
        m, path = _probe_net(block, seed=block + 10)
        m.prepare_inference()
        check_exact(m, x)
        ref = reference_forward(x, m)
        scale = torch.where(path[:, 2] < 128, 1.0, 2.0).double().cuda()
        assert torch.equal(ref, xf[:, path[:, 3].cuda()] * scale)  # the probe is what it claims to be
        got = _run_kernel(m, x, variant)
        bad = (got[:, :66].double() != ref).any(dim=0).nonzero().flatten().tolist()
        assert not bad, [f"column {c}: fc3 unit {path[c, 0]}, fc2 unit {path[c, 1]}, fc1 unit {path[c, 2]}, input bit "
                         f"{path[c, 3]} (head block {block})" for c in bad[:4]]
        assert (got[:, 66:] == 0).all()


@pytest.mark.gpu
def test_mlp_kernels_with_no_rows_write_nothing(gpu_nets):
    from betazero_b200 import _lib

    m = gpu_nets["logits"]
    L = _lib.load()
    x = _random_planes(8, 1, device="cuda")
    buf = torch.full((8, 72), NAN_BITS, dtype=torch.int16, device="cuda")
    for fn in (L.bz_mlp_forward_pair, L.bz_mlp_forward_pair2):
        assert fn(_lib.dptr(x), _lib.dptr(m._image_pair), _lib.dptr(buf), 0, _lib.stream_ptr()) == 0
    for variant in ("pair", "pair2", True):
        out = m.forward_raw(x[:0], out=buf.view(torch.bfloat16)[:0], fused=variant)
        assert out.shape == (0, 72)
    torch.cuda.synchronize()
    assert (buf == NAN_BITS).all()


# ---------------------------------------------------------------------------------------------------------------------
# GPU: every net evaluation inside the searches
# ---------------------------------------------------------------------------------------------------------------------
def walk_trees(pools):
    """Every expanded node of every tree, found from root_meta through the edges' meta words (action in bits 0..6, the
    child's edge count in bits 7..12, its block offset in 8-word units in bits 13..31; include/betazero_b200.h), checked
    to cover exactly arena_used units per tree.  Returns a dict of numpy arrays, one entry per node: tree, n, me, opp
    (uint64), in_N / in_W (the statistics of the edge into the node; the root has none: in_N = -1), and [nodes, 33]
    arrays act, N, W, P with `valid` marking the node's n edges."""
    T = pools.n_trees
    arena = pools.arena[: T * pools.arena_units * 8].view(T, -1).cpu().numpy().view(np.uint32)
    used = pools.arena_used[:T].cpu().numpy().astype(np.int64)
    meta = pools.root_meta[:T].cpu().numpy().view(np.uint32)
    tree, in_n_word, in_w_word = np.arange(T), np.full(T, -1), np.full(T, -1)
    e = np.arange(33)[None, :]
    found = []
    while len(tree):
        n = ((meta >> 7) & 63).astype(np.int64)
        keep = n > 0  # 0: unexpanded, terminal, or an empty tree
        tree, n, in_n_word, in_w_word = tree[keep], n[keep], in_n_word[keep], in_w_word[keep]
        base = (meta[keep] >> 13).astype(np.int64) * 8
        if not len(tree):
            break
        found.append((tree, base, n, in_n_word, in_w_word))
        valid = e < n[:, None]
        meta = arena[np.broadcast_to(tree[:, None], valid.shape)[valid], (base[:, None] + 8 + 3 * n[:, None] + e)[valid]]
        in_n_word = (base[:, None] + 8 + e)[valid]
        in_w_word = (base[:, None] + 8 + n[:, None] + e)[valid]
        tree = np.broadcast_to(tree[:, None], valid.shape)[valid]
    tree, base, n, in_n_word, in_w_word = (np.concatenate([f[i] for f in found]) if found else np.zeros(0, np.int64)
                                           for i in range(5))
    units = (8 + 4 * n + 7) // 8
    assert np.array_equal(np.bincount(tree, weights=units, minlength=T).astype(np.int64), used), "walk != arena_used"
    key = tree * (1 << 32) + base
    assert len(np.unique(key)) == len(key), "a node block is reachable twice"
    assert (base // 8 + units <= used[tree]).all()
    assert np.array_equal(arena[tree, base + 4], n), "node header n != the n its edge records"
    word = lambda w: arena[tree, w]  # noqa: E731
    me = word(base).astype(np.uint64) | (word(base + 1).astype(np.uint64) << np.uint64(32))
    opp = word(base + 2).astype(np.uint64) | (word(base + 3).astype(np.uint64) << np.uint64(32))
    valid = e < n[:, None]
    cols = np.minimum(e, n[:, None] - 1)

    def edge_field(k):
        return arena[tree[:, None], base[:, None] + 8 + k * n[:, None] + cols]

    root = in_n_word < 0
    in_N = np.where(root, -1, arena[tree, np.where(root, 0, in_n_word)].view(np.int32))
    in_W = np.where(root, 0, arena[tree, np.where(root, 0, in_w_word)]).astype(np.uint32).view(np.float32)
    return dict(tree=tree, n=n, me=me, opp=opp, in_N=in_N, in_W=in_W, valid=valid, act=edge_field(3) & 0x7F,
                N=edge_field(0).view(np.int32), W=edge_field(1).view(np.float32), P=edge_field(2).view(np.float32))


def check_search(pools, nets, tree_net, K):
    """Priors and first values of every expanded node against the float64 net of its tree (nets[tree_net[tree]]).
    Returns (nodes, nodes whose value was checked)."""
    nodes = walk_trees(pools)
    assert len(nodes["tree"]) > 0
    me = torch.from_numpy(nodes["me"].view(np.int64)).cuda()
    opp = torch.from_numpy(nodes["opp"].view(np.int64)).cuda()
    x = planes_of(me, opp)
    owner = np.asarray(tree_net)[nodes["tree"]]
    ref = torch.empty((len(owner), 66), dtype=torch.float64, device="cuda")
    for i, m in enumerate(nets):
        sel = torch.from_numpy(np.flatnonzero(owner == i)).cuda()
        if len(sel):
            check_exact(m, x[sel])
            ref[sel] = reference_forward(x[sel], m)
    ref = ref.cpu().numpy()
    valid, act = nodes["valid"], nodes["act"]
    # priors: the float64 softmax of the node's logits over its edges' actions (64 = pass)
    lg = np.where(valid, np.take_along_axis(ref, act.astype(np.int64), axis=1), -np.inf)
    p = np.exp(lg - lg.max(axis=1, keepdims=True))
    p /= p.sum(axis=1, keepdims=True)
    np.testing.assert_allclose(nodes["P"][valid], p[valid], rtol=RTOL, atol=1e-12, err_msg="priors")
    # values: a non-root node none of whose edges has been visited was reached only by the descents of the iteration
    # that expanded it, and each of them backed up -tanh(v) of its own evaluation of the node (the same row).  K = 1:
    # W_in = 0 + (-tanhf(v)) exactly.  K > 1: each descent left W -= 1 (exact: integers) and each backup stores
    # fl(fl(W + 1) - tanhf(v)); the N_in <= K backups are 2 N_in roundings of values below 2 K in magnitude, each off by
    # at most 2^-24 * 2K, so W_in / N_in is within 4 K 2^-24 of -tanhf(v).  tanhf (<= 2 ulp) is inside the 1e-5.
    leaf = (nodes["in_N"] > 0) & ~(valid & (nodes["N"] != 0)).any(axis=1)
    n_in = nodes["in_N"][leaf]
    assert (n_in <= K).all() and (K > 1 or (n_in == 1).all()), np.unique(n_in)
    t = np.tanh(ref[leaf, 65])
    w = nodes["in_W"][leaf].astype(np.float64) / n_in
    atol = 0.0 if K == 1 else 4 * K * 2.0 ** -24
    bad = np.abs(w + t) > RTOL * np.abs(t) + atol
    assert not bad.any(), f"values: {int(bad.sum())} of {len(t)} differ, e.g. W/N {w[bad][:3]} against -tanh {-t[bad][:3]}"
    return len(nodes["tree"]), int(leaf.sum())


def _roots(B, kind, size, seed):
    from betazero_b200 import env
    from oracle import pyoracle as po

    if kind == "start":
        me, opp, _ = env.reversi_init(B, size)
        return me, opp
    me_h, opp_h = po.playout_boards(B, seed=seed, size=size)  # midgame positions, forced passes, finished games
    if B == 1:  # a tree with something to search
        me_h, opp_h = po.playout_boards(64, seed=seed, size=size)
        live = int(np.flatnonzero(po.terminal(me_h, opp_h, size)[0] == 0)[0])
        me_h, opp_h = me_h[live:live + 1], opp_h[live:live + 1]
    return env.to_device_u64(me_h), env.to_device_u64(opp_h)


def _search(m, me, opp, n_sims, K, one_launch, size=8):
    from betazero_b200 import mcts

    s = mcts.BatchedMCTS(mcts.TreePools(me.numel(), n_sims, board_size=size, n_leaves=K),
                         mcts.FusedNetEvaluator(m, use_kernel=True), use_graph=not one_launch, graph_unroll=4,
                         one_launch=one_launch)
    assert s.one_launch is one_launch
    s.search(me, opp, n_sims)  # captures the per-iteration path's graph before the reset; raises on a pool overflow
    torch.cuda.synchronize()
    return s


@pytest.fixture(scope="module")
def search_net():
    m = exact_net(21, device="cuda")
    m.prepare_inference()
    return m


SEARCHES = [  # K, trees, simulations, roots, board size
    (1, 1, 64, "playout", 8), (1, 57, 64, "playout", 8), (1, 4144, 16, "playout", 8), (1, 4145, 16, "playout", 8),
    (2, 1, 64, "playout", 8), (2, 57, 64, "playout", 8), (2, 4144, 16, "playout", 8), (2, 4145, 16, "playout", 8),
    (4, 1, 64, "playout", 8), (4, 57, 96, "playout", 8), (4, 4144, 16, "playout", 8), (4, 4145, 32, "playout", 8),
    (4, 9000, 16, "playout", 8), (4, 300, 64, "start", 8), (1, 300, 48, "start", 8), (2, 300, 48, "start", 8),
    (4, 200, 48, "playout", 6), (1, 200, 32, "start", 6), (4, 200, 24, "playout", 4), (2, 100, 24, "start", 4),
]


@pytest.mark.gpu
@pytest.mark.parametrize("K,B,n_sims,roots,size", SEARCHES)
def test_one_launch_search_priors_and_values_equal_the_float64_net(search_net, K, B, n_sims, roots, size):
    """bz_mcts_search_fused: the net inside the one-launch search, checked through what it leaves in every node"""
    me, opp = _roots(B, roots, size, seed=B + K)
    s = _search(search_net, me, opp, n_sims, K, True, size)
    nodes, leaves = check_search(s.pools, [search_net], np.zeros(B, np.int64), K)
    assert nodes >= B // 2 and leaves >= B // 4, (nodes, leaves)


@pytest.mark.gpu
@pytest.mark.parametrize("K,B,n_sims", [(1, 300, 48), (2, 57, 64), (4, 300, 64), (4, 4145, 16)])
def test_per_iteration_search_priors_and_values_equal_the_float64_net(search_net, K, B, n_sims):
    """the per-iteration path: bz_mlp_forward_pair* writes the 72-wide bf16 rows, bz_mcts_step reads them"""
    me, opp = _roots(B, "playout", 8, seed=3 * B + K)
    s = _search(search_net, me, opp, n_sims, K, False)
    nodes, leaves = check_search(s.pools, [search_net], np.zeros(B, np.int64), K)
    assert nodes >= B // 2 and leaves >= B // 4, (nodes, leaves)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 4])
def test_entrant_search_evaluates_each_pair_with_its_own_net(K):
    """bz_mcts_search_fused_entrants with three exact nets and mixed budgets in one launch: the nodes of pair p are
    checked against the net of pair_entrant[p]"""
    import ctypes

    from betazero_b200 import _lib, mcts

    nets = [exact_net(30 + i, device="cuda") for i in range(3)]
    for m in nets:
        m.prepare_inference()
    budgets = [16, 48, 32]
    B = 600
    me, opp = _roots(B, "playout", 8, seed=40 + K)
    s = mcts.BatchedMCTS(mcts.TreePools(B, max(budgets), n_leaves=K), mcts.FusedNetEvaluator(nets[0]), use_graph=False,
                         one_launch=True)
    s.reset(me, opp)
    n_pairs = -(-B // 56)
    g = torch.Generator().manual_seed(K)
    pair_entrant = torch.randint(0, 3, (n_pairs,), generator=g, dtype=torch.uint8)
    pair_entrant[:3] = torch.tensor([2, 0, 1], dtype=torch.uint8)
    images = [m._image_pair.data_ptr() for m in nets]
    L = _lib.load()
    pair_entrant_d = pair_entrant.cuda()
    _lib.check(L.bz_mcts_search_fused_entrants(s.pools._ref, (ctypes.c_void_p * 3)(*images),
                                               (ctypes.c_int32 * 3)(*[n // K for n in budgets]), 3,
                                               _lib.dptr(pair_entrant_d), _lib.stream_ptr()), "entrants")
    torch.cuda.synchronize()
    s.check_errors()
    tree_net = pair_entrant.repeat_interleave(56)[:B].long().numpy()
    nodes, leaves = check_search(s.pools, nets, tree_net, K)
    assert nodes >= B and leaves >= B // 4, (nodes, leaves)
    # the check can tell the nets apart: checked against one net only, the other pairs' priors fail
    with pytest.raises(AssertionError):
        check_search(s.pools, [nets[0]], np.zeros(B, np.int64), K)
