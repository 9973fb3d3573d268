"""The float64 network reference (tests/network_reference.py) checked on its own, without a GPU: its Philox against the
C oracle's, its arithmetic against the float64 notebook network with the roundings switched off and against the fp32
emulation of tests/test_gpu_policy.py with them on, and its blob decoder against an encoder of the same layout."""
import os

import numpy as np
import pytest
import torch

import network_reference as nr
from oracle import c_oracle as co
from test_oracle_golden import PHILOX_KAT


def _fixture(golden_dir, name):
    d = np.load(os.path.join(golden_dir, name))
    return d, {k: torch.from_numpy(d[k]) for k in d.files if k.startswith("network")}


@pytest.mark.parametrize("ctr,key,out", PHILOX_KAT)
def test_numpy_philox_known_answers(ctr, key, out):
    got = nr.philox4x32_10(ctr, key)
    assert tuple(int(v) for v in got) == out == co.philox(ctr, key)


def test_numpy_philox_matches_the_oracle_on_random_counters():
    rng = np.random.default_rng(7)
    ctr = rng.integers(0, 2 ** 32, size=(4, 10_000), dtype=np.uint64)
    key = rng.integers(0, 2 ** 32, size=(2, 10_000), dtype=np.uint64)
    got = np.stack(nr.philox4x32_10(ctr, key), -1)
    ref = np.array([co.philox(tuple(int(v) for v in ctr[:, i]), tuple(int(v) for v in key[:, i])) for i in range(ctr.shape[1])],
                   dtype=np.uint32)
    assert np.array_equal(got, ref)


def test_bernoulli_uniforms_follow_the_counter_layout():
    seed, ids, steps = (5 << 32) + 9, np.array([2 ** 32 - 1, 2 ** 32, 3]), np.array([0, 2 ** 32 - 1, 2 ** 32 + 4])
    u = nr.bernoulli_uniforms(seed, ids, steps)
    for t, s in enumerate(steps):
        for i, g in enumerate(ids):
            r = co.philox((int(g) & 0xffffffff, int(g) >> 32, int(s) & 0xffffffff, 2), (seed & 0xffffffff, seed >> 32))
            assert [u[t, i, j] for j in range(3)] == [(r[j] >> 8) / 2 ** 24 for j in range(3)]


@pytest.mark.parametrize("name,head", [("policy_v1.npz", 3), ("critic_v1.npz", 1)])
def test_emulate64_without_rounding_is_the_float64_network(golden_dir, name, head):
    d, sd = _fixture(golden_dir, name)
    x = torch.from_numpy(d["obs"])
    img = nr.images_from_fold(nr.fold64(sd, head), f16=True, head=head, rounding=False)
    emu = nr.emulate64(img, x, rounding=False)["out"]
    ex = nr.exact64(sd, x, head)
    assert (emu - ex).abs().max().item() <= 1e-12 * max(1.0, ex.abs().max().item())


@pytest.mark.parametrize("f16", [True, False])
@pytest.mark.parametrize("name,head", [("policy_v1.npz", 3), ("critic_v1.npz", 1)])
def test_emulate64_agrees_with_the_fp32_emulation(golden_dir, name, head, f16):
    """The fp32 emulation of tests/test_gpu_policy.py evaluates the trunk's roundings in another summation order, which
    flips an occasional 16-bit activation.  Policy: it keeps the last hidden layer and the head in fp32 (the kernel's
    tensor-core head rounds them), so only the tolerance that test holds the kernel to applies.  Critic (same head in both):
    the acceptance rule the kernel is held to against emulate64 -- a flipped row can move by more than that test's 2e-3 of
    1 + |v| (0.14 at v = -44 in bf16, a quarter of a 16-bit ulp of its logit scale)."""
    from test_gpu_policy import _emulate16
    d, sd = _fixture(golden_dir, name)
    x = torch.from_numpy(d["obs"])
    img = nr.images_from_fold(nr.fold64(sd, head), f16=f16, head=head)
    ref = nr.emulate64(img, x)
    e32 = _emulate16(sd, x, head=head, f16=f16)
    if head == 3:
        assert (ref["out"] - e32.double()).abs().max().item() < (5e-4 if f16 else 3e-3)
    else:
        nr.assert_accepted(nr.compare(e32, ref), "fp32 emulation vs emulate64")


@pytest.mark.parametrize("f16", [True, False])
def test_decode_blob_inverts_the_encoder(f16):
    g = torch.Generator().manual_seed(3 + f16)
    img = {"fmt": "fp16" if f16 else "bf16", "head": 3}
    for name, _, N, K in nr.IMAGES:
        v = torch.randn(N, K, generator=g, dtype=torch.float64) * torch.exp2(torch.randint(-12, 8, (N, K), generator=g).double())
        img[name] = nr.rn16(v, f16)
    c = {k: (torch.randn(n, generator=g, dtype=torch.float64) * 3).float().double()
         for k, n in (("beta0", 128), ("beta1", 128), ("beta2", 64), ("b3", 4))}
    c["w3"] = torch.randn(3, 64, generator=g, dtype=torch.float64).float().double()
    img["consts"] = dict(c, fmt=img["fmt"], head=3)
    raw = nr.encode_blob(img)
    assert len(raw) == nr.BLOB_BYTES
    back = nr.decode_blob(raw)
    assert back["fmt"] == img["fmt"]
    for name, _, _, _ in nr.IMAGES:
        assert torch.equal(back[name], img[name]), name
    for k in ("beta0", "beta1", "beta2", "w3", "b3"):
        assert torch.equal(back["consts"][k], c[k]), k
    assert nr.encode_blob(back) == raw
    # the layout itself: element (n, k) of an [N][K] image at (k / 8) * N * 8 + n * 8 + k % 8
    idx = nr.image_index(128, 16)
    assert idx[0, 0] == 0 and idx[0, 7] == 7 and idx[1, 0] == 8 and idx[0, 8] == 128 * 8 and idx[127, 15] == 2047
    assert np.array_equal(np.sort(idx.ravel()), np.arange(128 * 16))
