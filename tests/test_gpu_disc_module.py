"""DiscriminatorP / DiscriminatorS as modules: one forward path whether or not autograd records the call, an engine
that follows the parameters' storage, and gradient buffers that belong to the trainer that owns them."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def H():
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    import hifigan_b200
    hifigan_b200._lib.lib()
    return hifigan_b200


def _audio(b, t, seed):
    from oracle import hifigan_oracle as O
    return O.synthetic_audio(b, t, seed=seed).unsqueeze(1).cuda()


def _outputs(res):
    """every logit and feature map of an mpd / msd call, flattened into one list"""
    rs, gs, fr, fg = res
    return list(rs) + list(gs) + [f for fl in fr + fg for f in fl]


@pytest.mark.parametrize("case", ["mpd_eval", "msd_eval", "msd_train"])
def test_no_grad_call_equals_grad_mode_call(H, case):
    """A no-grad call and a grad-mode call on the same weights run the same kernels and return the same logits and
    feature maps.  In eval mode they are bit-identical.  A train-mode spectral-norm layer advances its power iteration
    on each call (two identically seeded modules see the same iteration), but the W^T u product of that iteration
    accumulates with fp32 atomics, so u, v and the outputs agree to rounding, not bit for bit."""
    def make():
        torch.manual_seed(1234)
        net = (H.MultiPeriodDiscriminator() if case == "mpd_eval" else H.MultiScaleDiscriminator()).cuda()
        return net.train(train)

    train = case == "msd_train"
    a = make()
    b = make() if train else a
    y, y_hat = _audio(2, 8192, 1), _audio(2, 8192, 2)
    with torch.no_grad():
        got_a = _outputs(a(y, y_hat))
    got_b = _outputs(b(y, y_hat))
    assert got_b[0].requires_grad
    assert len(got_a) == len(got_b)
    for x, z in zip(got_a, got_b):
        z = z.detach()
        assert x.shape == z.shape
        if train:
            assert (x - z).abs().max().item() <= 1e-2 * z.abs().max().item() + 1e-6
        else:
            assert torch.equal(x, z)
    if train:
        bufs = [(n, t) for n, t in a.named_buffers() if n.endswith(("weight_u", "weight_v"))]
        assert bufs
        other = dict(b.named_buffers())
        for n, t in bufs:
            assert torch.allclose(t, other[n], rtol=1e-4, atol=1e-5), n


def _loss(res):
    logit, fmap = res
    return logit.pow(2).mean() + sum(f.abs().mean() for f in fmap)


@pytest.mark.parametrize("move", ["data_clone", "cpu_cuda"])
@pytest.mark.parametrize("kind", ["P", "S_spectral"])
def test_engine_follows_parameter_storage(H, kind, move):
    """After `p.data = p.data.clone()` on every parameter, or `disc.cpu().cuda()`, and then loading other weights in
    place, a discriminator that was already called computes what a fresh module with those weights computes: its
    engine's job tables must not keep pointers to the old storage."""
    make = (lambda: H.DiscriminatorP(3)) if kind == "P" else (lambda: H.DiscriminatorS(use_spectral_norm=True))
    torch.manual_seed(5)
    ref = make().cuda().eval()
    torch.manual_seed(6)
    d = make().cuda().eval()
    y = _audio(2, 4000, 3)
    with torch.no_grad():
        d(y)
    _loss(d(y)).backward()                 # builds the engine's tables on the current storage
    d.zero_grad(set_to_none=True)
    if move == "data_clone":
        for p in d.parameters():
            p.data = p.data.clone()
    else:
        d.cpu().cuda()
    d.load_state_dict(ref.state_dict())    # new values into the new storage only
    with torch.no_grad():
        got, want = d(y), ref(y)
    for x, z in zip([got[0]] + got[1], [want[0]] + want[1]):
        assert torch.equal(x, z)
    _loss(d(y)).backward()
    _loss(ref(y)).backward()
    for (n, p), q in zip(d.named_parameters(), ref.parameters()):
        assert (p.grad - q.grad).norm() <= 1e-3 * q.grad.norm() + 1e-12, n


def test_module_calls_between_trainstep_build_and_step(H):
    """A grad-mode `mpd(...)` and `generator(...)` call between building a TrainStep and its first step leave every
    parameter gradient of that step as it is without them: each trainer writes into its own gradient buffers.
    Same tolerance as the autograd-vs-TrainStep test (fp32 atomics make two runs non-bit-identical)."""
    from oracle import hifigan_oracle as O
    from hifigan_b200.train import TrainStep
    h = H.AttrDict(O.config("v1"))
    ya = O.synthetic_audio(2, 8192, seed=17).cuda()
    x = H.mel_spectrogram(ya, 1024, 80, 22050, 256, 1024, 0, 8000)
    y_mel = H.mel_spectrogram(ya, 1024, 80, 22050, 256, 1024, 0, None)
    grads = []
    for interleave in (False, True):
        torch.manual_seed(1234)
        nets = (H.Generator(h), H.MultiPeriodDiscriminator(), H.MultiScaleDiscriminator())
        ts = TrainStep(*nets, h, "cuda")
        if interleave:
            G, mpd, _ = nets
            assert mpd(ya.unsqueeze(1), ya.unsqueeze(1))[0][0].requires_grad
            assert G(x).requires_grad
        ts.step(x, ya.unsqueeze(1), y_mel, update=False)
        grads.append([p.grad.detach().clone() for n in nets for p in n.parameters()])
    names = [f"{i}:{k}" for i, n in enumerate(nets) for k, _ in n.named_parameters()]
    for k, a, b in zip(names, *grads):
        assert F.cosine_similarity(a.flatten(), b.flatten(), dim=0).item() >= 0.9999, k
