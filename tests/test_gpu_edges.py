"""-m gpu: every loss entry point on inputs synth.py never produces, against the float64 oracles (pinned in these corners
by tests/test_oracle_edges.py) at north-star tolerances:

  blank placement   blank = V-1 with V % 4 != 0 (scalar row tail), blank in the tail of a V = 20000 row, and for the
                    fused LayerNormalization path blank = 239 / 240 (either side of a 240-row box edge) and V-1 in the
                    last, partial box at V = 1213 and V = 4080;
  shared ids        labels equal to the blank, bigram ids equal to a unigram of the same utterance, V = 2 and 3;
  tight alignments  CTC at exactly L + #repeats frames and one frame short, Gram-CTC with fewer frames than characters
                    (the joint objective's CTC half is then infeasible while the Gram-CTC half is not);
  degenerate        input_length 0 (with and without labels), label_length 0 with frames, input_length 1, Lmax = 0;
  padding           label / bigram entries past label_length of -1, V + 5 or the blank give the same bits as 0;
  large logits      a common offset of +300 / +1000, scaling by 20 / 40, trained-like bumps on top; for the fused path
                    gamma ~ 8 and beta +300, and the fused greedy argmax on the same inputs.
"""
import numpy as np
import pytest

from util import run_cuda, run_oracle, assert_parity, LOSS_RTOL, GRAD_ATOL

pytestmark = pytest.mark.gpu


def synth():
    import importlib
    return importlib.import_module("chainer-speech-recognition_b200.synth")


# ---------------------------------------------------------------------------------------------------------------------
# builders
# ---------------------------------------------------------------------------------------------------------------------

def make_problem(B, T, V, L, blank, seed, in_len=None, lab_len=None, gram=False, label_pool=None, trained=False,
                 offset=0.0, scale=1.0):
    """Labels drawn from label_pool (default: every id but the blank), lengths as given (default: full), activations
    N(0,1) * scale + offset, plus a +8 bump on an even alignment when trained."""
    rs = np.random.RandomState(seed)
    in_len = np.full(B, T, np.int32) if in_len is None else np.asarray(in_len, np.int32)
    lab_len = np.full(B, L, np.int32) if lab_len is None else np.asarray(lab_len, np.int32)
    pool = np.array([v for v in range(V) if v != blank] if label_pool is None else label_pool)
    labels = np.zeros((B, L), np.int32)
    big = np.full((B, L), -1, np.int32)
    for b in range(B):
        n = int(lab_len[b])
        labels[b, :n] = rs.choice(pool, size=n)
        for i in range(1, n):
            if rs.rand() < 0.6:
                big[b, i] = rs.randint(0, V)
    x = (rs.standard_normal((T, B, V)) * scale + offset).astype(np.float32)
    if trained:
        synth().add_alignment_bump(x, labels, in_len, lab_len, blank=blank)
    prob = {"x": x, "labels": labels, "input_length": in_len, "label_length": lab_len, "blank": blank}
    if gram:
        prob["bigrams"] = big
    return prob


def check_kind(pkg, prob, kind, what):
    loss, grad, _ = run_cuda(pkg, prob, kind)
    loss_ref, grad_ref, _ = run_oracle(prob, kind)
    if kind == "joint":                     # two losses, each good to GRAD_ATOL
        rel = np.abs(loss - loss_ref) / np.maximum(np.abs(loss_ref), 1.0)
        assert rel.max() <= LOSS_RTOL, (what, loss, loss_ref)
        assert np.abs(grad - grad_ref).max() <= 2 * GRAD_ATOL, (what, np.abs(grad - grad_ref).max())
    else:
        assert_parity(loss, grad, loss_ref, grad_ref, what)
    return loss, grad, loss_ref


def check_all(pkg, prob, what, kinds=("ctc", "gram", "joint")):
    for kind in kinds:
        check_kind(pkg, prob, kind, "%s %s" % (what, kind))


# ---------------------------------------------------------------------------------------------------------------------
# plain entry points: ctc, gram_ctc, gram_ctc(joint_ctc=True)
# ---------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("V,blank", [(37, 36), (37, 0), (9, 8), (130, 129), (130, 65), (20000, 19999), (20000, 19990)])
def test_blank_placement(pkg, V, blank):
    B, T, L = 3, 40, 6
    prob = make_problem(B, T, V, L, blank, seed=V + blank, in_len=[40, 31, 23], lab_len=[6, 4, 0], gram=True,
                        label_pool=[0, 1, 2, V - 2, V - 1, V // 2] if V > 20 else None, trained=True)
    check_all(pkg, prob, "V=%d blank=%d" % (V, blank))


def test_blank_not_zero_full_size(pkg):
    """B=64, T=800, V=3500 with blank = 3499 and label id 0 an ordinary symbol."""
    B, T, V, L, blank = 64, 800, 3500, 80, 3499
    s = synth()
    base = s.ctc_problem(B, T, V, L, seed=71, trained=False)
    prob = make_problem(B, T, V, L, blank, seed=71, in_len=base["input_length"], lab_len=base["label_length"],
                        trained=True)
    prob["labels"] = np.where(prob["labels"] == 1, 0, prob["labels"]).astype(np.int32)
    check_kind(pkg, prob, "ctc", "full size blank=V-1")


@pytest.mark.parametrize("blank", [0, 5, 9])
def test_labels_equal_to_blank(pkg, blank):
    """The blank id among the labels and bigrams: the label nodes fold into the blank's merged posterior."""
    B, T, V, L = 4, 30, 10, 6
    prob = make_problem(B, T, V, L, blank, seed=blank, in_len=[30, 28, 25, 20], lab_len=[6, 5, 3, 6], gram=True,
                        label_pool=[blank, blank, 1, 2, 3] if blank not in (1, 2, 3) else None)
    prob["bigrams"][:, 2] = blank
    check_all(pkg, prob, "labels=blank %d" % blank)


def test_bigram_ids_equal_unigram_ids(pkg):
    B, T, V, L = 3, 40, 12, 8
    prob = make_problem(B, T, V, L, 11, seed=5, gram=True, label_pool=[0, 1, 2, 3])
    for b in range(B):
        for i in range(1, L):
            prob["bigrams"][b, i] = prob["labels"][b, (i + 3) % L]      # a unigram id of the same utterance
    check_all(pkg, prob, "bigram=unigram")


@pytest.mark.parametrize("V,blank", [(2, 0), (2, 1), (3, 1), (3, 2)])
def test_tiny_vocabularies(pkg, V, blank):
    B, T, L = 3, 20, 5
    prob = make_problem(B, T, V, L, blank, seed=10 * V + blank, lab_len=[5, 3, 1], gram=True,
                        label_pool=list(range(V)), trained=True)
    prob["bigrams"] = np.where(prob["bigrams"] >= 0, prob["bigrams"] % V, -1).astype(np.int32)
    check_all(pkg, prob, "V=%d blank=%d" % (V, blank))


def _min_frames(lab):
    return len(lab) + sum(int(lab[i] == lab[i - 1]) for i in range(1, len(lab)))


@pytest.mark.parametrize("blank", [0, 6])
def test_tight_alignments(pkg, blank):
    """One batch: CTC at exactly its minimum length, at the minimum - 1 (infeasible: loss exactly 1e10, gradient =
    softmax), and normal utterances next to them."""
    B, T, V, L = 5, 24, 7, 8
    prob = make_problem(B, T, V, L, blank, seed=20 + blank, lab_len=[8, 8, 8, 5, 8],
                        label_pool=[v for v in range(V) if v != blank][:3])
    prob["labels"][1] = prob["labels"][0]
    prob["labels"][2, :] = prob["labels"][2, 0]                       # all repeats: needs 2L - 1 frames
    need = [_min_frames(prob["labels"][b, :int(prob["label_length"][b])]) for b in range(B)]
    prob["input_length"] = np.array([need[0], need[1] - 1, need[2], need[3] - 1, T], np.int32)
    loss, grad, loss_ref = check_kind(pkg, prob, "ctc", "tight blank=%d" % blank)
    for b in (1, 3):
        assert loss[b] == 1e10 and loss_ref[b] == 1e10
        Tb = int(prob["input_length"][b])
        x = prob["x"][:Tb, b].astype(np.float64)
        soft = np.exp(x - x.max(axis=1, keepdims=True))
        soft /= soft.sum(axis=1, keepdims=True)
        assert np.abs(grad[:Tb, b] - soft).max() <= GRAD_ATOL
    assert loss[0] < 1e10 and loss[2] < 1e10


@pytest.mark.parametrize("blank", [0, 9])
def test_gram_shorter_than_characters(pkg, blank):
    """Gram-CTC utterances with fewer frames than characters, alignable only through bigram nodes (k = 5/6/7 edges and
    the final bigram node).  In the joint objective the CTC half is infeasible (1e10) while the Gram-CTC half is not."""
    B, T, V, L = 3, 12, 10, 8
    ids = [c for c in range(V) if c != blank]
    c, g = ids[:4], ids[4:]                                       # characters; bigram ids
    prob = make_problem(B, T, V, L, blank, seed=30 + blank, gram=True, trained=True)
    for b in range(B):
        prob["labels"][b] = [c[0], c[1], c[2], c[3], c[0], c[2], c[1], c[3]]
        prob["bigrams"][b] = [-1, g[0], g[4], g[1], -1, g[2], g[4], g[3]]   # four distinct pairs at 1, 3, 5, 7
    prob["bigrams"][2, 6] = -1
    prob["input_length"] = np.array([4, 5, 7], np.int32)          # 8 characters in 4, 5 and 7 frames
    lg, _, lg_ref = check_kind(pkg, prob, "gram", "gram short")
    assert np.all(lg < 1e10) and np.all(lg_ref < 1e10)
    lj, _, _ = check_kind(pkg, prob, "joint", "joint short")
    assert np.all(lj >= 1e10)                                     # 1e10 + the finite Gram-CTC loss


@pytest.mark.parametrize("kind", ["ctc", "gram", "joint"])
def test_degenerate_lengths(pkg, kind):
    """input_length 0 with and without labels, label_length 0 with frames (the all-blank path), input_length 1."""
    B, T, V, L = 6, 10, 11, 3
    prob = make_problem(B, T, V, L, 4, seed=40, in_len=[0, 0, 10, 1, 1, 6], lab_len=[0, 2, 0, 0, 1, 3], gram=True)
    loss, grad, loss_ref = check_kind(pkg, prob, kind, "degenerate " + kind)
    assert loss[0] == loss_ref[0] == 0.0
    assert loss[1] >= 1e10 and loss_ref[1] >= 1e10
    for b in range(B):
        assert not grad[int(prob["input_length"][b]):, b].any()


@pytest.mark.parametrize("kind", ["ctc", "gram", "joint"])
def test_no_labels_in_the_batch(pkg, kind):
    """Lmax = 0: either it works (all-blank paths) or it is refused with a Python exception."""
    import torch
    B, T, V = 3, 8, 6
    prob = make_problem(B, T, V, 0, 2, seed=41, in_len=[8, 3, 0], lab_len=[0, 0, 0], gram=True)
    try:
        loss, grad, _ = run_cuda(pkg, prob, kind)
    except (ValueError, AssertionError, NotImplementedError, IndexError, RuntimeError) as e:
        assert not isinstance(e, torch.cuda.OutOfMemoryError)
        torch.cuda.synchronize()                                  # the device is still usable
        return
    loss_ref, grad_ref, _ = run_oracle(prob, kind)
    assert np.allclose(loss, loss_ref, rtol=LOSS_RTOL, atol=LOSS_RTOL)
    assert np.abs(grad - grad_ref).max() <= 2 * GRAD_ATOL


@pytest.mark.parametrize("kind", ["ctc", "gram", "joint"])
def test_label_padding_is_ignored(pkg, kind):
    B, T, V, L = 4, 30, 25, 7
    prob = make_problem(B, T, V, L, 3, seed=42, lab_len=[7, 4, 0, 2], gram=True)
    base = run_cuda(pkg, prob, kind)
    for pad in (-1, V + 5, 3):
        p = dict(prob)
        p["labels"] = prob["labels"].copy()
        p["bigrams"] = prob["bigrams"].copy()
        for b in range(B):
            n = int(prob["label_length"][b])
            p["labels"][b, n:] = pad
            p["bigrams"][b, n:] = pad
        got = run_cuda(pkg, p, kind)
        assert np.array_equal(base[0], got[0]) and np.array_equal(base[1], got[1]), pad


LARGE = [  # (offset, scale, trained)
    (300.0, 1.0, False), (1000.0, 1.0, False), (0.0, 20.0, False), (0.0, 40.0, False),
    (300.0, 1.0, True), (1000.0, 1.0, True), (-1000.0, 1.0, True),
]


@pytest.mark.parametrize("offset,scale,trained", LARGE)
@pytest.mark.parametrize("V", [37, 500])
def test_large_logits(pkg, offset, scale, trained, V):
    """Both gradient kernels (V = 37: unaligned rows; V = 500: the row ring) at large |logits|.  The softmax must be
    as good as at small logits: the normaliser reaches the gradient as (la, scale), not as one rounded float."""
    B, T, L = 4, 60, 8
    prob = make_problem(B, T, V, L, 0, seed=int(abs(offset) + scale + V), in_len=[60, 51, 40, 33], gram=True,
                        trained=trained, offset=offset, scale=scale)
    check_all(pkg, prob, "offset=%g scale=%g trained=%s" % (offset, scale, trained))


def test_large_logits_full_size(pkg):
    B, T, V, L = 64, 800, 3500, 80
    s = synth()
    prob = s.ctc_problem(B, T, V, L, seed=72, trained=True)
    prob["x"] += np.float32(1000.0)
    check_kind(pkg, prob, "ctc", "full size +1000")


def test_host_entry_points_blank_and_tight(pkg):
    """ctc_host / gram_ctc_host on a batch with blank = V-1, a tight and an infeasible utterance."""
    B, T, V, L = 4, 20, 13, 5
    prob = make_problem(B, T, V, L, 12, seed=43, in_len=[20, 5, 4, 0], lab_len=[5, 5, 5, 0], gram=True,
                        label_pool=[0, 1, 2, 3], trained=True, offset=300.0)
    prob["labels"][1] = [0, 1, 0, 1, 2]
    prob["labels"][2] = [0, 1, 0, 1, 2]
    xb = np.ascontiguousarray(prob["x"].transpose(1, 0, 2))
    for kind in ("ctc", "gram"):
        loss_ref, grad_ref, _ = run_oracle(prob, kind)
        if kind == "ctc":
            loss, grad = pkg.ctc_host(xb, prob["labels"], 12, prob["input_length"], prob["label_length"], reduce="no",
                                      groups=2)
        else:
            loss, grad = pkg.gram_ctc_host(xb, prob["labels"], prob["bigrams"], 12, prob["input_length"],
                                           prob["label_length"], reduce="no", groups=2)
        assert_parity(np.asarray(loss, np.float64), grad.numpy().transpose(1, 0, 2), loss_ref, grad_ref, "host " + kind)
    assert loss_ref[3] == 0.0


# ---------------------------------------------------------------------------------------------------------------------
# LayerNormalization fused into the loss: layernorm_ctc, layernorm_gram_ctc (plain and joint), layernorm_greedy_argmax
# ---------------------------------------------------------------------------------------------------------------------

def run_ln(pkg, kind, z, gamma, beta, prob):
    import torch
    dev = torch.device("cuda:0")
    B, V, T = z.shape
    zin = torch.tensor(z, device=dev).unsqueeze(2).requires_grad_(True)
    g = torch.tensor(gamma, device=dev, requires_grad=True)
    b = torch.tensor(beta, device=dev, requires_grad=True)
    lab = torch.tensor(prob["labels"], device=dev)
    il = torch.tensor(prob["input_length"], device=dev)
    ll = torch.tensor(prob["label_length"], device=dev)
    if kind == "ctc":
        out = pkg.layernorm_ctc(zin, g, b, lab, prob["blank"], il, ll, reduce="no")
    else:
        out = pkg.layernorm_gram_ctc(zin, g, b, lab, torch.tensor(prob["bigrams"], device=dev), prob["blank"], il, ll,
                                     reduce="no", joint_ctc=(kind == "joint"))
    out.backward(torch.ones_like(out))
    torch.cuda.synchronize()
    return (out.detach().cpu().numpy().astype(np.float64), zin.grad.cpu().numpy().reshape(B, V, T),
            g.grad.cpu().numpy(), b.grad.cpu().numpy())


def oracle_ln(kind, z, gamma, beta, prob):
    """float64 LayerNormalization -> float64 lattice(s) -> LayerNormalization backward; also returns the activations."""
    from oracle import layernorm, lattice, c_oracle
    acts, saved = layernorm.forward(z, gamma, beta)
    args = (prob["input_length"], prob["label_length"])
    T, B, V = acts.shape
    small = B * T * V <= 2e6
    loss, grad = 0.0, 0.0
    for k in (("gram", "ctc") if kind == "joint" else (kind,)):
        if small and k == "ctc":
            l, g = lattice.ctc(acts, prob["labels"], *args, blank=prob["blank"])
        elif small:
            l, g = lattice.gram_ctc(acts, prob["labels"], prob["bigrams"], *args, blank=prob["blank"])
        else:
            r = c_oracle.run(0 if k == "ctc" else 1, acts.astype(np.float32), prob["labels"], prob.get("bigrams"), *args,
                             prob["blank"])
            l, g = r["loss"], r["grad"].astype(np.float64)
        loss, grad = loss + l, grad + g
    dz, dgamma, dbeta = layernorm.backward(grad, saved)
    return (loss, dz, dgamma, dbeta), acts, saved


def check_ln(got, want, saved, B, T, what, nloss, large=False):
    """Losses to LOSS_RTOL; dz to nloss * GRAD_ATOL (nloss = 2 for the joint objective); dgamma, dbeta as
    test_gpu_layernorm.check.  large: the activations a = gamma*n + beta reach a magnitude A where float32 cannot hold
    them to better than ulp(A)/2 -- a rounding every float32 evaluation of a makes, the reference's included.  Then:
      * |delta a| <= ulp(A)/2 moves p_v by at most p_v (1 - p_v) ulp(A) <= ulp(A)/4;
      * the fused kernel's log2 normaliser is one float near A log2 e (|la| < 4A, ulp(la) <= 4 ulp(A)), rounded to at
        most 2 ulp(A), which moves p_v by at most ln2 * 2 ulp(A) * p_v <= 1.4 ulp(A);
      so the loss gradient g w.r.t. a is within eg = nloss * (GRAD_ATOL + 1.65 ulp(A));
      * dz = rstd (gamma g - mean_v(gamma g) - n mean_v(gamma g n)) turns that into |delta dz| <= rstd max|gamma| eg
        (2 + max|n|) (mean_v |n| <= 1 for normalised n), and each per-frame term of dgamma / dbeta moves by at most
        eg max(1, |n|)."""
    loss, dz, dg, db = got
    loss_ref, dz_ref, dg_ref, db_ref = want
    rel = np.abs(loss - loss_ref) / np.maximum(np.abs(loss_ref), 1.0)
    assert rel.max() <= LOSS_RTOL, (what, rel.max())
    n, std, gamma = saved
    nmax = np.abs(n).max()
    if large:
        eg = nloss * (GRAD_ATOL + 1.65 * float(np.spacing(np.float32(large))))
        tol_dz = (1.0 / std).max() * np.abs(gamma).max() * eg * (2.0 + nmax)
        tol_g = eg * max(1.0, nmax) * np.sqrt(B * T)
    else:
        eg = tol_dz = nloss * GRAD_ATOL
        tol_g = eg * np.sqrt(B * T)
    assert np.abs(dz - dz_ref).max() <= tol_dz, (what, np.abs(dz - dz_ref).max(), tol_dz)
    assert np.all(np.abs(dg - dg_ref) <= tol_g + 1e-5 * np.abs(dg_ref)), (what, np.abs(dg - dg_ref).max())
    assert np.all(np.abs(db - db_ref) <= eg * np.sqrt(B * T) + 1e-5 * np.abs(db_ref)), (what, np.abs(db - db_ref).max())


def make_ln(B, T, V, L, blank, seed, in_len, lab_len, gamma_scale=0.2, gamma_mean=1.0, beta_mean=0.0,
            label_pool=None):
    prob = make_problem(B, T, V, L, blank, seed, in_len=in_len, lab_len=lab_len, gram=True, label_pool=label_pool,
                        trained=True, scale=1.7)
    rs = np.random.RandomState(seed + 1)
    z = np.ascontiguousarray(prob.pop("x").transpose(1, 2, 0))
    gamma = (gamma_mean + gamma_scale * rs.randn(V)).astype(np.float32)
    beta = (beta_mean + 0.1 * rs.randn(V)).astype(np.float32)
    return prob, z, gamma, beta


def ln_all(pkg, prob, z, gamma, beta, what, large=False, kinds=("ctc", "gram", "joint")):
    B, V, T = z.shape
    for kind in kinds:
        want, acts, saved = oracle_ln(kind, z, gamma, beta, prob)
        got = run_ln(pkg, kind, z, gamma, beta, prob)
        check_ln(got, want, saved, B, T, "%s %s" % (what, kind), 2 if kind == "joint" else 1,
                 large=np.abs(acts).max() if large else False)


@pytest.mark.parametrize("V,blank", [(300, 239), (300, 240), (1213, 1212), (1213, 240), (4080, 4079), (37, 36)])
def test_ln_blank_placement(pkg, V, blank):
    prob, z, gamma, beta = make_ln(3, 40, V, 6, blank, seed=V + blank, in_len=[40, 33, 17], lab_len=[6, 3, 0],
                                   label_pool=[0, 1, 238, 239, 240, 241, V - 1] if V > 242 else None)
    prob["labels"] = np.where(prob["labels"] == blank, 0, prob["labels"]).astype(np.int32) if blank != 0 else prob["labels"]
    kinds = ("ctc", "gram", "joint") if V <= 1213 else ("ctc",)
    ln_all(pkg, prob, z, gamma, beta, "LN V=%d blank=%d" % (V, blank), kinds=kinds)


def test_ln_labels_equal_to_blank_and_degenerate_lengths(pkg):
    V, blank = 130, 7
    prob, z, gamma, beta = make_ln(6, 24, V, 5, blank, seed=7, in_len=[24, 0, 0, 1, 24, 9], lab_len=[5, 0, 2, 0, 0, 3],
                                   label_pool=[blank, blank, 1, 2, 3])
    prob["bigrams"][:, 2] = blank
    ln_all(pkg, prob, z, gamma, beta, "LN labels=blank")


@pytest.mark.parametrize("gamma_mean,beta_mean", [(8.0, 0.0), (1.0, 300.0), (8.0, 300.0)])
def test_ln_large_logits(pkg, gamma_mean, beta_mean):
    """gamma ~ 8 (|a| up to several hundred) and a common beta of +300; the fused greedy argmax on the same inputs."""
    import torch
    from test_layernorm_argmax import oracle_values, assert_picks_a_maximum
    V = 1213
    prob, z, gamma, beta = make_ln(3, 40, V, 6, 5, seed=int(gamma_mean + beta_mean), in_len=[40, 29, 13], lab_len=[6, 4, 2],
                                   gamma_scale=1.0, gamma_mean=gamma_mean, beta_mean=beta_mean)
    ln_all(pkg, prob, z, gamma, beta, "LN gamma~%g beta~%g" % (gamma_mean, beta_mean), large=True)
    dev = torch.device("cuda:0")
    pick = pkg.layernorm_greedy_argmax(torch.tensor(z, device=dev).unsqueeze(2), torch.tensor(gamma, device=dev),
                                       torch.tensor(beta, device=dev)).cpu().numpy()
    y64 = oracle_values(z, gamma, beta)
    assert_picks_a_maximum(pick, y64)
    top2 = np.sort(y64, axis=2)[:, :, -2:]
    clear = top2[:, :, 1] - top2[:, :, 0] > 1e-3 * np.maximum(1.0, np.abs(top2[:, :, 1]))
    assert np.array_equal(pick[clear], y64.argmax(axis=2)[clear])


def test_ln_large_logits_full_size(pkg):
    """B=64, T=800, V=3500, blank = 3499, gamma ~ 8: the fused CTC loss on the full BASELINE configs[1] shape."""
    B, T, V, L = 64, 800, 3500, 80
    base = synth().ctc_problem(B, T, V, L, seed=73)
    prob, z, gamma, beta = make_ln(B, T, V, L, V - 1, seed=73, in_len=base["input_length"], lab_len=base["label_length"],
                                   gamma_scale=1.0, gamma_mean=8.0)
    ln_all(pkg, prob, z, gamma, beta, "LN full size", large=True, kinds=("ctc",))
