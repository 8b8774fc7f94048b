"""SURVEY.md §8 f4, device side: the minibatch crop / mirror / transpose (convnet_b200_extract_patches) — the oracle pinned
to the reference's own CPU implementation (eigenmat/eigenmat.cc:2046-2090; its results stored in
tests/golden/ref_eigenmat_patches.npz, see tests/golden_ref.py), the C-ABI's argument checks, and (GPU) the kernel against
the oracle, bit for bit."""
import ctypes as ct

import numpy as np
import pytest

import golden_ref
from oracle_lib import Oracle, RefLib

CASES = [  # N, C, W, H, pw, ph
    (5, 3, 12, 10, 7, 6),
    (33, 1, 40, 36, 33, 32),
    (64, 3, 36, 36, 32, 32),
    (4, 2, 9, 9, 9, 9),           # no crop: offsets must be 0, mirror only
]


def _inputs(N, C, W, H, pw, ph, seed):
    rng = np.random.default_rng(seed)
    images = np.asfortranarray(rng.standard_normal(N * C * W * H).astype(np.float32))
    wo = np.asfortranarray(rng.integers(0, W - pw + 1, N).astype(np.float32))
    ho = np.asfortranarray(rng.integers(0, H - ph + 1, N).astype(np.float32))
    flip = np.asfortranarray((rng.random(N) > 0.5).astype(np.float32))
    return images, wo, ho, flip


def _numpy_reference(images, wo, ho, flip, N, C, W, H, pw, ph):
    src = images.reshape(N, C, H, W)
    out = np.empty((C, ph, pw, N), np.float32)
    for n in range(N):
        x0, y0 = int(wo[n]), int(ho[n])
        crop = src[n, :, y0:y0 + ph, :]
        crop = crop[:, :, ::-1][:, :, x0:x0 + pw] if flip[n] > 0.5 else crop[:, :, x0:x0 + pw]
        out[:, :, :, n] = crop
    return out.reshape(-1)


@pytest.fixture(scope="module")
def ref_patches():
    """stored results of the reference's CPU code; recording runs it live (oracle/_ref/libeigenmat_ref.so)"""
    store = golden_ref.RefStore("ref_eigenmat_patches")
    if golden_ref.RECORD and not (RefLib.available() and hasattr(RefLib().lib, "ref_extract_patches")):
        pytest.fail("recording needs oracle/_ref/libeigenmat_ref.so with the extract_patches door: run `make -C oracle`")
    yield store
    store.save()


@pytest.mark.parametrize("case", CASES)
def test_oracle_equals_the_formula_and_the_reference_cpu_code(case, ref_patches):
    N, C, W, H, pw, ph = case
    images, wo, ho, flip = _inputs(*case, seed=3)
    got = np.asfortranarray(np.full(N * C * pw * ph, np.nan, np.float32))
    assert Oracle().extract_patches(images, got, wo, ho, flip, N, C, W, H, pw, ph) == 0
    assert np.array_equal(got, _numpy_reference(images, wo, ho, flip, N, C, W, H, pw, ph))

    def live():
        ref = np.asfortranarray(np.full(N * C * pw * ph, np.nan, np.float32))
        assert RefLib().extract_patches(images, ref, wo, ho, flip, N, C, W, H, pw, ph) == 0
        return ref
    assert golden_ref.equal(got, ref_patches.reference("x".join(map(str, case)), live, exact=True))


def test_argument_checks_return_the_reference_error_code():
    """cudamat.cu:2699-2713: ERROR_INCOMPATIBLE_DIMENSIONS (-1) before anything is launched (no GPU needed)."""
    from convnet_b200 import lib
    from convnet_b200.abi import cudamat
    L = lib.load()

    def m(rows, cols):
        c = cudamat(); c.size[0], c.size[1] = rows, cols; c.data_device = None
        return ct.pointer(c)
    N, C, W, H, pw, ph = 8, 3, 12, 10, 6, 5
    img, vec = m(C * W * H, N), m(1, N)
    assert L.convnet_b200_extract_patches(img, m(N, C * pw * ph + 1), vec, vec, vec, W, H, pw, ph) == -1
    assert L.convnet_b200_extract_patches(img, m(N + 1, C * pw * ph), vec, vec, vec, W, H, pw, ph) == -1
    assert L.convnet_b200_extract_patches(img, m(N, C * pw * ph), m(1, N - 1), vec, vec, W, H, pw, ph) == -1
    assert L.convnet_b200_extract_patches(img, m(N, C * pw * ph), vec, m(2, N), vec, W, H, pw, ph) == -1
    assert L.convnet_b200_extract_patches(img, m(N, C * pw * ph), vec, vec, m(1, 1), W, H, pw, ph) == -1
    assert L.convnet_b200_extract_patches(m(C * W * H + 1, N), m(N, C * pw * ph), vec, vec, vec, W, H, pw, ph) == -1


def test_deterministic_views_follow_the_reference_rule():
    """src/datahandler.cc:547-556: view k % 5 = centre, top-left, top-right, bottom-right, bottom-left (host logic, CPU)"""
    from convnet_b200 import build, net
    build.build_host(); net.load_host()
    for mx, my in ((32, 32), (5, 9), (0, 0), (1, 7)):
        want = [(mx // 2, my // 2), (0, 0), (mx, 0), (mx, my), (0, my)]
        for k in range(12):
            assert net.view_offset(k, mx, my) == want[k % 5]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES + [(128, 3, 256, 256, 224, 224), (100, 1, 28, 28, 28, 28), (130, 3, 70, 50, 65, 33)])
def test_kernel_equals_the_oracle(case):
    import torch
    from convnet_b200 import lib
    from convnet_b200.matrix import CUDAMatrix
    L = lib.load()
    N, C, W, H, pw, ph = case
    images, wo, ho, flip = _inputs(*case, seed=11)
    want = np.asfortranarray(np.empty(N * C * pw * ph, np.float32))
    assert Oracle().extract_patches(images, want, wo, ho, flip, N, C, W, H, pw, ph) == 0
    dev = lambda a, r, c: CUDAMatrix(r, c, storage=torch.from_numpy(np.ascontiguousarray(a)).cuda())
    d_img, d_wo, d_ho, d_flip = dev(images, C * W * H, N), dev(wo, 1, N), dev(ho, 1, N), dev(flip, 1, N)
    out = CUDAMatrix(N, C * pw * ph); out.storage.fill_(float("nan"))
    rc = L.convnet_b200_extract_patches(d_img.p_mat, out.p_mat, d_wo.p_mat, d_ho.p_mat, d_flip.p_mat, W, H, pw, ph)
    assert rc == 0
    assert np.array_equal(out.storage.cpu().numpy(), want)


@pytest.mark.gpu
@pytest.mark.parametrize("translate,flip", [(True, True), (False, False)])
def test_data_iterator_fills_the_input_layer(translate, flip):
    """host/data.h DataIterator (DataHandler::GetBatch's device side): chunk upload, jitter sampling, crop / mirror into the
    net's input layer — checked against the oracle fed with the offsets the iterator reports; centre / corner crops and
    the mirror-by-multiplicity rule of src/datahandler.cc:547-567 when translate / flip are off."""
    import torch
    from convnet_b200 import lib, net
    lib.load(); net.load_host()
    batch, chunk, C, S, G = 32, 96, 8, 16, 12                    # "tiny" takes 8 x 12 x 12 inputs
    n = net.Net("tiny", batch, seed=1)
    g = torch.Generator().manual_seed(5)
    host = torch.randn(chunk, C, S, S, generator=g).pin_memory()
    it = net.DataIterator(chunk, C, S, G, translate=translate, flip=flip, seed=9)
    it.upload(host)
    for start, mult in ((0, 0), (32, 3), (64, 7)):
        it.get_batch(n, start, mult)
        torch.cuda.synchronize()
        wo, ho, fl = (np.asfortranarray(np.array(v, np.float32)) for v in it.last_noise(batch))
        if translate:
            assert wo.min() >= 0 and wo.max() <= S - G and len(set(wo.tolist())) > 1
        else:
            w, h = {0: (2, 2), 3: (4, 4), 2: (4, 0)}[mult % 5]
            assert set(wo.tolist()) == {float(w)} and set(ho.tolist()) == {float(h)}
        if not flip:
            assert set(fl.tolist()) == {float(mult // 5)}
        images = np.asfortranarray(host[start:start + batch].numpy().reshape(-1).copy())
        want = np.asfortranarray(np.empty(batch * C * G * G, np.float32))
        assert Oracle().extract_patches(images, want, wo, ho, fl, batch, C, S, S, G, G) == 0
        assert np.array_equal(n.input_tensor().cpu().numpy(), want)
    loss = n.train_step(True)                                    # and the net trains on what it was handed
    assert np.isfinite(loss)
    it.close(); n.close()
