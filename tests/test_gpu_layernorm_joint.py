"""LayerNormalization fused into the joint Gram-CTC + CTC objective (run/gram_ctc/cnn/train.py:196-198 with
``args.joint_training``): ``layernorm_gram_ctc(..., joint_ctc=True)`` against the float64 oracle (oracle/layernorm.py ->
Gram-CTC + CTC lattices on the same activations -> LayerNormalization's backward of the summed gradient), against the two
fused losses called separately, and against the unfused joint loss behind LayerNormalization written in torch ops.
Also: the shapes the fused path refuses are refused by the forward call, for every kind.

Every test but the workspace-size one needs a GPU."""
import importlib

import numpy as np
import pytest

from util import LOSS_RTOL, GRAD_ATOL

# largest label length whose backward tile fits shared memory next to 17 boxes of vocabulary (V = 4080): Gram-CTC and
# joint share one plan (csrc/layernorm_loss.cu, plan_ln_backward)
GRAM_LMAX_AT_V4080 = 63


def synth():
    return importlib.import_module("chainer-speech-recognition_b200.synth")


def make_case(B, T, V, L, seed, trained=True):
    s = synth()
    rs = np.random.RandomState(seed)
    prob = s.gram_problem(B, T, V, L, seed=seed, n_unigram=max(3, min(119, V // 3)))
    z_tbv = (rs.standard_normal((T, B, V)) * 1.7 + 0.3).astype(np.float32)
    if trained:
        s.add_alignment_bump(z_tbv, prob["labels"], prob["input_length"], prob["label_length"], bump=6.0)
    z = np.ascontiguousarray(z_tbv.transpose(1, 2, 0))
    gamma = (1.0 + 0.2 * rs.randn(V)).astype(np.float32)
    beta = (0.1 * rs.randn(V)).astype(np.float32)
    return prob, z, gamma, beta


def run_fused(pkg, kind, z, gamma, beta, prob, reduce="no", gy=None, pitch=None):
    """kind: 'joint', 'gram' or 'ctc'.  z: (B, V, T) numpy; pitch: rows of this many floats (>= T), passed as a view."""
    import torch
    dev = torch.device("cuda:0")
    B, V, T = z.shape
    if pitch is None:
        zt = torch.tensor(z, device=dev)
    else:
        buf = torch.zeros((B, V, pitch), device=dev)
        buf[:, :, :T] = torch.tensor(z, device=dev)
        zt = buf[:, :, :T]
    zin = zt.unsqueeze(2).requires_grad_(True)
    g = torch.tensor(gamma, device=dev, requires_grad=True)
    b = torch.tensor(beta, device=dev, requires_grad=True)
    lab = torch.tensor(prob["labels"], device=dev)
    il = torch.tensor(prob["input_length"], device=dev)
    ll = torch.tensor(prob["label_length"], device=dev)
    if kind == "ctc":
        out = pkg.layernorm_ctc(zin, g, b, lab, 0, il, ll, reduce=reduce)
    else:
        big = torch.tensor(prob["bigrams"], device=dev)
        out = pkg.layernorm_gram_ctc(zin, g, b, lab, big, 0, il, ll, reduce=reduce, joint_ctc=(kind == "joint"))
    up = torch.ones_like(out) if gy is None else torch.tensor(np.asarray(gy, np.float32), device=dev).reshape(out.shape)
    out.backward(up)
    torch.cuda.synchronize()
    dz = zin.grad.detach().cpu().numpy().reshape(B, V, T)
    return out.detach().cpu().numpy().astype(np.float64), dz, g.grad.cpu().numpy(), b.grad.cpu().numpy()


def run_unfused_joint(pkg, z, gamma, beta, prob):
    """LayerNormalization as torch ops + the transposed copy of asr/model/cnn.py:41-44 + gram_ctc(joint_ctc=True)."""
    import torch
    dev = torch.device("cuda:0")
    zt = torch.tensor(z, device=dev, requires_grad=True)
    g = torch.tensor(gamma, device=dev, requires_grad=True)
    b = torch.tensor(beta, device=dev, requires_grad=True)
    mean = zt.mean(dim=1, keepdim=True)
    diff = zt - mean
    std = torch.sqrt((diff * diff).sum(dim=1, keepdim=True) / z.shape[1])
    y = diff / std * g[None, :, None] + b[None, :, None]
    acts = y.permute(2, 0, 1).contiguous()
    loss = pkg.gram_ctc(acts, torch.tensor(prob["labels"], device=dev), torch.tensor(prob["bigrams"], device=dev), 0,
                        torch.tensor(prob["input_length"], device=dev), torch.tensor(prob["label_length"], device=dev),
                        reduce="no", joint_ctc=True)
    loss.sum().backward()
    torch.cuda.synchronize()
    return (loss.detach().cpu().numpy().astype(np.float64), zt.grad.cpu().numpy(), g.grad.cpu().numpy(),
            b.grad.cpu().numpy())


def run_oracle_joint(z, gamma, beta, prob, scale=None):
    """float64 LayerNormalization -> Gram-CTC + CTC on the same activations -> LayerNormalization backward of the sum.
    The NumPy lattices (float64 throughout) for small cases, the C oracle (float64 arithmetic on the activations
    rounded to float32) for large ones."""
    from oracle import layernorm, lattice, c_oracle
    acts, saved = layernorm.forward(z, gamma, beta)
    T, B, V = acts.shape
    args = (prob["input_length"], prob["label_length"])
    if B * T * V <= 2e6:
        lg, gg = lattice.gram_ctc(acts, prob["labels"], prob["bigrams"], *args, 0)
        lc, gc = lattice.ctc(acts, prob["labels"], *args, 0)
    else:
        a32 = acts.astype(np.float32)
        rg = c_oracle.run(1, a32, prob["labels"], prob["bigrams"], *args, 0)
        rc = c_oracle.run(0, a32, prob["labels"], None, *args, 0)
        lg, gg, lc, gc = rg["loss"], rg["grad"].astype(np.float64), rc["loss"], rc["grad"].astype(np.float64)
    grad = gg + gc
    if scale is not None:
        grad = grad * np.asarray(scale, np.float64).reshape(1, -1, 1)
    dz, dgamma, dbeta = layernorm.backward(grad, saved)
    return lg + lc, dz, dgamma, dbeta


def check_joint_grads(got, want, B, T, what, gmax=1.0):
    """The gradient bounds of test_gpu_layernorm.check, doubled (two losses, each good to GRAD_ATOL) and scaled by the
    largest |upstream gradient| gmax.  got, want: (dz, dgamma, dbeta)."""
    dz, dg, db = got
    dz_ref, dg_ref, db_ref = want
    assert np.abs(dz - dz_ref).max() <= 2 * gmax * GRAD_ATOL, (what, np.abs(dz - dz_ref).max())
    tol_g = 2 * (gmax * GRAD_ATOL * np.sqrt(B * T) + 1e-5 * np.abs(dg_ref))
    tol_b = 2 * (gmax * GRAD_ATOL * np.sqrt(B * T) + 1e-5 * np.abs(db_ref))
    assert np.all(np.abs(dg - dg_ref) <= tol_g), (what, np.abs(dg - dg_ref).max())
    assert np.all(np.abs(db - db_ref) <= tol_b), (what, np.abs(db - db_ref).max())


def check_joint(got, want, B, T, what):
    """test_gpu_layernorm.check for the joint objective: losses to LOSS_RTOL, gradients by check_joint_grads."""
    loss, loss_ref = got[0], want[0]
    rel = np.abs(loss - loss_ref) / np.maximum(np.abs(loss_ref), 1.0)
    assert rel.max() <= LOSS_RTOL, (what, rel.max())
    check_joint_grads(got[1:], want[1:], B, T, what)


def test_ln_workspace_bytes_joint_exceeds_gram(pkg):
    """No GPU: the fused joint workspace is Gram-CTC's plus the plain-CTC lattice's alpha/beta rows and records."""
    L = pkg._lib
    for B, T, V, Lmax in ((3, 24, 40, 5), (32, 600, 4000, 60)):
        joint = L.ln_workspace_bytes(L.KIND_JOINT, B, T, V, Lmax)
        gram = L.ln_workspace_bytes(L.KIND_GRAM, B, T, V, Lmax)
        assert joint > gram and joint % 16 == 0
        # at least the two (B, T, 2*Lmax+1) rows of (mantissa, exponent) pairs of the second lattice
        assert joint - gram >= 2 * 8 * B * T * (2 * Lmax + 1)


JOINT_SHAPES = [
    # B, T, V, L, row pitch (None: T)
    (3, 24, 40, 5, None),                         # one box
    (3, 42, 130, 6, 44),                          # T % 8 != 0, rows with a padded pitch
    (4, 96, 700, 10, None),
    (3, 120, 2000, 30, None),
    (2, 200, 4080, GRAM_LMAX_AT_V4080, None),     # 17 boxes, the longest labels the backward tile holds there
    (32, 600, 4000, 60, None),                    # BASELINE configs[2] with V cut to the fused limit
]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", JOINT_SHAPES, ids=["B%d_T%d_V%d_L%d" % s[:4] for s in JOINT_SHAPES])
def test_fused_joint_matches_oracle(pkg, shape):
    B, T, V, L, pitch = shape
    prob, z, gamma, beta = make_case(B, T, V, L, seed=71)
    got = run_fused(pkg, "joint", z, gamma, beta, prob, pitch=pitch)
    check_joint(got, run_oracle_joint(z, gamma, beta, prob), B, T, "%r" % (shape,))
    for b in range(B):
        assert not got[1][b, :, int(prob["input_length"][b]):].any()          # padded frames: exact zeros


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(4, 96, 700, 10), (3, 120, 2000, 30)])
def test_fused_joint_equals_sum_of_fused_parts(pkg, shape):
    B, T, V, L = shape
    prob, z, gamma, beta = make_case(B, T, V, L, seed=72)
    lj, dzj, dgj, dbj = run_fused(pkg, "joint", z, gamma, beta, prob)
    lg, dzg, dgg, dbg = run_fused(pkg, "gram", z, gamma, beta, prob)
    lc, dzc, dgc, dbc = run_fused(pkg, "ctc", z, gamma, beta, prob)
    assert np.allclose(lj, lg + lc, rtol=2e-6, atol=0)
    assert np.abs(dzj - (dzg + dzc)).max() <= 5e-6
    assert np.allclose(dgj, dgg + dgc, rtol=1e-4, atol=1e-4)
    assert np.allclose(dbj, dbg + dbc, rtol=1e-4, atol=1e-4)


@pytest.mark.gpu
def test_fused_joint_equals_unfused_composition(pkg):
    """The same numbers as LayerNormalization in torch ops + the transposed copy + gram_ctc(joint_ctc=True)."""
    prob, z, gamma, beta = make_case(4, 80, 500, 9, seed=73)
    fused = run_fused(pkg, "joint", z, gamma, beta, prob)
    loss, dz, dg, db = run_unfused_joint(pkg, z, gamma, beta, prob)
    assert np.allclose(fused[0], loss, rtol=2e-6)
    assert np.abs(fused[1] - dz).max() <= 1e-5                                 # two losses: twice the single-loss bound
    assert np.allclose(fused[2], dg, rtol=2e-4, atol=2e-4)
    assert np.allclose(fused[3], db, rtol=2e-4, atol=2e-4)


@pytest.mark.gpu
def test_fused_joint_reduce_mean_and_no(pkg):
    B, T = 6, 72
    prob, z, gamma, beta = make_case(B, T, 300, 8, seed=74)
    want = run_oracle_joint(z, gamma, beta, prob, scale=np.full(B, 2.5 / B))
    loss, dz, dg, db = run_fused(pkg, "joint", z, gamma, beta, prob, reduce="mean", gy=2.5)
    assert np.ndim(loss) == 0
    assert abs(loss - want[0].mean()) <= LOSS_RTOL * abs(want[0].mean())       # scale * sum_b (gram_b + ctc_b)
    check_joint_grads((dz, dg, db), want[1:], B, T, "mean gy=2.5")
    for b in range(B):
        assert not dz[b, :, int(prob["input_length"][b]):].any()
    gy = np.array([1.0, -2.0, 0.5, 3.0, 0.0, 1.5], np.float32)
    want = run_oracle_joint(z, gamma, beta, prob, scale=gy)
    loss, dz, dg, db = run_fused(pkg, "joint", z, gamma, beta, prob, reduce="no", gy=gy)
    assert np.all(np.abs(loss - want[0]) <= LOSS_RTOL * np.maximum(np.abs(want[0]), 1.0))
    check_joint_grads((dz, dg, db), want[1:], B, T, "no, per-utterance gy", gmax=3.0)     # |gy| up to 3
    for b in range(B):
        assert not dz[b, :, int(prob["input_length"][b]):].any()


@pytest.mark.gpu
def test_fused_joint_ctc_infeasible_gram_feasible(pkg):
    """Label "ab" in ONE frame: only the bigram "ab" of the Gram-CTC lattice fits, plain CTC has no alignment.  The loss is
    the Gram-CTC loss + exactly 1e10 (the reference's value for an infeasible alignment, added in float32), the gradient
    that of the unfused joint loss."""
    V, T = 10, 8
    rs = np.random.RandomState(75)
    z = (rs.standard_normal((1, V, T)) * 1.5).astype(np.float32)
    gamma = (1.0 + 0.2 * rs.randn(V)).astype(np.float32)
    beta = (0.1 * rs.randn(V)).astype(np.float32)
    prob = {"labels": np.array([[1, 2]], np.int32), "bigrams": np.array([[-1, 5]], np.int32),
            "input_length": np.array([1], np.int32), "label_length": np.array([2], np.int32)}
    lj, dzj, dgj, dbj = run_fused(pkg, "joint", z, gamma, beta, prob)
    lg = run_fused(pkg, "gram", z, gamma, beta, prob)[0]
    assert lg[0] < 1e9                                                           # Gram-CTC is feasible
    assert np.float32(lj[0]) == np.float32(np.float32(lg[0]) + np.float32(1e10))
    lu, dzu, dgu, dbu = run_unfused_joint(pkg, z, gamma, beta, prob)
    assert np.float32(lj[0]) == np.float32(lu[0])
    assert np.all(np.isfinite(dzj))
    assert np.abs(dzj - dzu).max() <= 1e-5
    assert np.allclose(dgj, dgu, rtol=2e-4, atol=2e-4) and np.allclose(dbj, dbu, rtol=2e-4, atol=2e-4)
    assert not dzj[0, :, 1:].any()


@pytest.mark.gpu
def test_fused_joint_is_deterministic(pkg):
    prob, z, gamma, beta = make_case(8, 200, 2000, 30, seed=76)
    a = run_fused(pkg, "joint", z, gamma, beta, prob)
    b = run_fused(pkg, "joint", z, gamma, beta, prob)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


# (kind, V, Lmax): the backward tile ring would hold fewer than K + 2 boxes (K = ceil(V / 240))
REFUSED = [
    ("ctc", 3500, 160),                     # 16 slots, 17 needed
    ("ctc", 4080, 120),                     # 17 of 19
    ("gram", 3500, 120),                    # 15 of 17
    ("gram", 4080, GRAM_LMAX_AT_V4080 + 1),
    ("joint", 3500, 120),
    ("joint", 4080, GRAM_LMAX_AT_V4080 + 1),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", REFUSED, ids=["%s_V%d_L%d" % c for c in REFUSED])
def test_fused_refuses_at_forward_what_backward_cannot_hold(pkg, case):
    """The forward call refuses (NotImplementedError: take the unfused path) instead of a backward that fails later."""
    import torch
    kind, V, L = case
    dev = torch.device("cuda:0")
    B, T = 1, 16
    z = torch.zeros(B, V, 1, T, device=dev, requires_grad=True)
    g, b = torch.ones(V, device=dev), torch.zeros(V, device=dev)
    lab = torch.ones(B, L, dtype=torch.int32, device=dev)
    big = torch.full((B, L), -1, dtype=torch.int32, device=dev)
    with pytest.raises(NotImplementedError):
        if kind == "ctc":
            pkg.layernorm_ctc(z, g, b, lab, 0)
        else:
            pkg.layernorm_gram_ctc(z, g, b, lab, big, 0, joint_ctc=(kind == "joint"))
