"""The fused policy / critic network (csrc/policy_rollout.cu) against a float64 evaluation of the roundings it specifies
(tests/network_reference.py), and the sampled actions against their Philox uniforms.

The packed operand images must be the 16-bit roundings of dd_policy_pack's fold (computed here in float64); the
kernel's outputs must then match ``emulate64`` on those images under one acceptance rule (network_reference.compare):
(a) at least F of the rows agree to TAU in every logit (values: TAU (1 + |v|)), (b) no row is off by more than M_ULPS
16-bit ulps of its logit scale.  Summation order only flips an occasional 16-bit activation; a dropped low half, an extra
rounding or a wrong entry moves most rows -- the sensitivity test runs the kernel on blobs with such edits and requires
the rule to reject every one.

Calibration: TAU = 1e-5, F = 0.8, M_ULPS = 4.  Observed on a B200 (1,000 W power limit), fraction of rows agreeing to
TAU / largest row deviation in 16-bit ulps of the logit scale:

  batch                                          fp16             bf16
  policy, small shapes pooled (4,927 rows)       0.982 / 0.40     0.999 / 0.03
  policy, 200,003 rows                           0.986 / 0.70     0.999 / 0.43
  policy, magnitudes 2^-30 .. 2^15               0.876 / 0.32     0.999 / 0.23
  policy, cfg-4 buffer (16.4 M rows)             0.979 / 2.62     0.998 / 2.37
  critic, small shapes pooled                    0.994 / 0.94     0.997 / 0.06
  critic, 200,003 rows                           0.993 / 1.14     0.998 / 0.35
  critic, cfg-4 buffer                           0.999 / 0.92     0.999 / 0.56
  fp16 range check, inside edges (4,096 rows)    >= 0.964 / 2.11

(quantiles of the deviation, policy cfg-4 buffer: 50 % 0, 99 % 1.8e-4 fp16 / 0 bf16, 99.9 % 1.0e-3 / 8.7e-4 in logit
units; critic: 99 % 2.9e-7 / 1.8e-7, 99.9 % 1.0e-5 / 1.8e-6 of 1 + |v|.)  Inputs below 2^-18 make every row nearly the
same bias-only network, so one flipped activation there repeats over ~12 % of the magnitude batch: its 0.876.  The edited
blobs of the sensitivity test agree on at most 0.59 of their rows (layer-2 bias low halves zeroed, fp16), so F sits between
the two; no accepted batch came within a factor 1.5 of M_ULPS, and (b) alone rejects none of the edits.
"""
import importlib
import os
import time
import types

import numpy as np
import pytest
import torch

import network_reference as nr

pytestmark = pytest.mark.gpu

dd = importlib.import_module("reinforcement-learning-101_b200")
nv = dd.native
DEV = "cuda:0"
SMALL = (1, 127, 128, 129, 511, 512, 513)
LARGE = (148 * 512 - 1, 148 * 512, 148 * 512 + 1, 200_003)


def _load(golden_dir, name):
    d = np.load(os.path.join(golden_dir, name))
    return d, {k: torch.from_numpy(d[k]) for k in d.files if k.startswith("network")}


def _random_net(seed):
    """The random networks of test_gpu_policy.py's ragged-size test (non-trivial LayerNorm affines and biases)."""
    g = torch.Generator().manual_seed(seed)
    shapes = ((128, 15), (128,), (128,), (128,), (128, 128), (128,), (128,), (128,), (64, 128), (64,), (64,), (64,), (3, 64), (3,))
    keys = ("0.weight", "0.bias", "1.weight", "1.bias", "3.weight", "3.bias", "4.weight", "4.bias", "6.weight", "6.bias",
            "7.weight", "7.bias", "9.weight", "9.bias")
    return {"network." + k: torch.randn(s, generator=g) * (0.3 if len(s) > 1 else 0.5) + (0.0 if len(s) > 1 else 0.5)
            for k, s in zip(keys, shapes)}


def _degenerate(sd):
    sd = {k: v.clone() for k, v in sd.items()}
    for key in ("network.1.weight", "network.4.weight", "network.7.weight"):
        g = sd[key]
        g[0] = 0.0; g[1] = -0.0; g[2] = 1e-20; g[3] = -3e-15; g[4] = -1.7; g[5] = 250.0; g[6] = 1e-6
    return sd


@pytest.fixture(scope="module")
def nets(golden_dir):
    dp, sdp = _load(golden_dir, "policy_v1.npz")
    dc, sdc = _load(golden_dir, "critic_v1.npz")
    return {"policy": (sdp, 3, torch.from_numpy(dp["obs"])), "critic": (sdc, 1, torch.from_numpy(dc["obs"])),
            "random1": (_random_net(1), 3, torch.from_numpy(dp["obs"])),
            "random1000": (_random_net(1000), 3, torch.from_numpy(dp["obs"])),
            "degenerate": (_degenerate(sdp), 3, torch.from_numpy(dp["obs"]))}


def _rows(base, n, seed):
    """n observation rows drawn from a fixture's rows with a 1 % perturbation (rollout-like, O(10) at most)."""
    g = torch.Generator().manual_seed(seed)
    return base[torch.randint(0, base.shape[0], (n,), generator=g)] * (1 + 0.01 * torch.randn(n, 15, generator=g))


def _forward(blob, x):
    return dd.policy_forward(blob, x) if blob.head == 3 else dd.value_forward(blob, x)


def _check(blob, img, x, what):
    st = nr.compare(_forward(blob, x.to(DEV)), nr.emulate64(img, x.to(DEV), consts=nr.consts_dict(blob.consts, blob.head)))
    print(f"{what}: {nr.summary(st)}")
    return st


# ---- 1. the pack ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("operands", ["auto", "bf16"])
@pytest.mark.parametrize("net", ["policy", "critic", "random1", "random1000", "degenerate"])
def test_pack_images_are_the_16bit_roundings_of_the_fold(nets, net, operands):
    sd, head, _ = nets[net]
    blob = dd.PolicyBlob(sd, device=DEV, head=head, operands=operands)
    img = nr.decode_blob(blob.blob, head)
    assert img["fmt"] == blob.operand_dtype
    f16 = img["fmt"] == "fp16"
    p = 11 if f16 else 8
    sub = 2.0 ** -25 if f16 else 0.0                        # half the fp16 subnormal spacing (a low half may be that small)
    assert bytes(blob.consts) == blob.blob[nr.PAR_OFF:].cpu().numpy().tobytes()     # the launch gets the blob's constants
    assert nr.encode_blob(img) == blob.blob.cpu().numpy().tobytes()
    fold = nr.fold64(sd, head)
    for l in range(3):
        v = fold[f"img{l}"]
        # the pack evaluates s (w - fp32 mean) c in fp32: its fold sits within 2 fp32 ulps of the terms from this one
        band = 2.0 ** -22 * fold[f"img{l}_c"] * (fold[f"img{l}_mean"].abs() + (fold[f"img{l}_raw"] - fold[f"img{l}_mean"]).abs())
        if l == 0:
            hi, lo, vv, bb = img["w0"], img["w0lo"], v, band
        else:
            hi = torch.cat([img[f"w{l}"], img[f"w{l}b"][:, :1]], 1)
            lo, vv, bb = img[f"w{l}b"][:, 1], v[:, -1], band[:, -1]
            assert not img[f"w{l}b"][:, 2:].any(), f"layer {l}: bias block columns 2-15 must be 0"
        r = nr.rn16(v, f16)
        near_mid = (v - (hi + r) / 2).abs() <= band
        off = hi != r
        assert (~off | (near_mid & ((hi - r).abs() <= nr.ulp16(torch.maximum(hi.abs(), r.abs()), f16)))).all(), \
            f"layer {l}: {int(off.sum())} entries are not the rounding of the fold (first {torch.nonzero(off)[:4].tolist()})"
        h = hi if l == 0 else hi[:, -1]
        err = (h + lo - vv).abs()
        tol = 2.0 ** (-2 * p) * vv.abs() * 1.01 + bb + sub
        assert (err <= tol).all(), f"layer {l}: hi + lo misses the fold by {(err / tol).max().item():.2f} x its bound"
        print(f"{net}/{img['fmt']} layer {l}: {int(off.sum())} of {off.numel()} entries one ulp off (fold at a midpoint)")
    # the head: w3 |gamma2| in fp32 is one rounding of the float64 product; hi / lo are its split; unused rows are 0
    w32 = fold["w3"].float().double()
    assert torch.equal(img["w3"][:head], nr.rn16(w32, f16))
    assert torch.equal(img["w3"][3:3 + head], nr.rn16(w32 - img["w3"][:head], f16))
    used = torch.zeros(nr.W3_ROWS, dtype=torch.bool)
    used[:head], used[3:3 + head] = True, True
    assert not img["w3"][~used].any()
    c = nr.consts_dict(blob.consts, head)
    for l in range(3):
        ref = fold[f"beta{l}"]
        assert ((c[f"beta{l}"] - ref).abs() <= 2.0 ** -24 * ref.abs()).all(), l      # one fp32 rounding of beta / g
    assert torch.equal(c["w3"][:head], w32) and not c["w3"][head:].any()
    assert torch.equal(c["b3"][:head], fold["b3"]) and not c["b3"][head:].any()


# ---- 2. the forward pass against emulate64 ------------------------------------------------------------------------
def _magnitude_rows(seed, n=4096):
    """Rows from 2^-30 to 2^15 in magnitude: per-row scales, per-element scales, and rows of +-2^15."""
    g = torch.Generator().manual_seed(seed)
    sign = torch.where(torch.rand(n, 15, generator=g) < 0.5, -1.0, 1.0)
    mant = 1 + torch.rand(n, 15, generator=g)
    e_row = torch.randint(-30, 15, (n // 2, 1), generator=g).expand(n // 2, 15)
    e_elt = torch.randint(-30, 15, (n - n // 2 - 64, 15), generator=g)
    x = sign * mant * torch.exp2(torch.cat([e_row, e_elt, torch.full((64, 15), 14)]).float())
    x[-32:] = sign[-32:] * 2.0 ** 15
    return x.float()


@pytest.mark.parametrize("operands", ["auto", "bf16"])
@pytest.mark.parametrize("net", ["policy", "critic"])
def test_forward_matches_emulate64(nets, net, operands):
    sd, head, base = nets[net]
    blob = dd.PolicyBlob(sd, device=DEV, head=head, operands=operands)
    img = nr.decode_blob(blob.blob, head)
    what = f"{net}/{blob.operand_dtype}"
    # small shapes and unaligned starts (direct loads instead of TMA), pooled for rule (a)
    small = [_check(blob, img, _rows(base, n, n), f"{what} n={n}") for n in SMALL]
    for off in (1, 2, 3):
        n = 1000 + off
        flat = torch.empty(n * 15 + off, dtype=torch.float32, device=DEV)
        x = _rows(base, n, 77 + off)
        xs = flat[off:].view(n, 15)
        xs.copy_(x.to(DEV))
        assert xs.data_ptr() % 16 != 0
        ref = nr.emulate64(img, xs)
        small.append(nr.compare(_forward(blob, xs), ref))
        print(f"{what} unaligned +{off}: {nr.summary(small[-1])}")
    pooled = nr.pool(small)
    print(f"{what} small shapes pooled: {nr.summary(pooled)}")
    nr.assert_accepted(pooled, f"{what} small shapes")
    # the persistent path: one block per CTA, ragged, several trips per CTA
    for n in LARGE:
        x = _rows(base, n, n)
        st = _check(blob, img, x, f"{what} n={n}")
        nr.assert_accepted(st, f"{what} n={n}")
    # magnitudes from 2^-30 to 2^15 (subnormal and large hi / lo splits)
    x = _magnitude_rows(5)
    out = _forward(blob, x.to(DEV))
    assert torch.isfinite(out).all()
    st = nr.compare(out, nr.emulate64(img, x.to(DEV)))
    print(f"{what} magnitudes 2^-30..2^15: {nr.summary(st)}")
    nr.assert_accepted(st, f"{what} magnitudes")


@pytest.mark.parametrize("net", ["policy", "critic"])
def test_fp16_error_is_a_fraction_of_bf16_against_the_exact_network(nets, net):
    """DESIGN.md / include/drone_b200.h: fp16 operands give 8x lower rounding error than bf16.  Asserted: the rms error
    against the float64 network is at most a quarter of bf16's on the same (fp16-eligible) network."""
    sd, head, base = nets[net]
    x = _rows(base, 148 * 512, 3).to(DEV)
    ex = nr.exact64(sd, x, head)
    rms = {}
    for operands in ("fp16", "bf16"):
        blob = dd.PolicyBlob(sd, device=DEV, head=head, operands=operands)
        err = (_forward(blob, x).double() - ex)
        rms[operands] = err.pow(2).mean().sqrt().item()
        print(f"{net}/{operands} against exact64: max {err.abs().max().item():.3e} rms {rms[operands]:.3e}")
    print(f"{net}: bf16 / fp16 rms error ratio {rms['bf16'] / rms['fp16']:.2f}")
    assert rms["fp16"] <= rms["bf16"] / 4, rms


# ---- 3. the rule has teeth -----------------------------------------------------------------------------------------
def _edited(blob, img, case):
    """A copy of blob (device buffer + host constants) with one edit of its operands."""
    f16 = img["fmt"] == "fp16"
    e = {k: (v.clone() if isinstance(v, torch.Tensor) else v) for k, v in img.items()}
    e["consts"] = {k: (v.clone() if isinstance(v, torch.Tensor) else v) for k, v in img["consts"].items()}
    if case == "w0_lo_zeroed":
        e["w0lo"].zero_()
    elif case == "layer1_bias_lo_zeroed":
        e["w1b"][:, 1] = 0
    elif case == "layer2_bias_lo_zeroed":
        e["w2b"][:, 1] = 0
    elif case == "head_lo_zeroed":
        e["w3"][3:6] = 0
    elif case == "beta_rounded_to_16_bits":
        for k in ("beta0", "beta1", "beta2"):
            e["consts"][k] = nr.rn16(e["consts"][k], f16)
    elif case == "w1_row_one_ulp":
        r = e["w1"][5]
        e["w1"][5] = r + torch.sign(r) * nr.ulp16(r, f16)
    raw = nr.encode_blob(e)
    dev = torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(DEV)
    consts = nv.DDPolicyConsts.from_buffer_copy(nr.consts_bytes(e["consts"]))
    return types.SimpleNamespace(head=blob.head, blob=dev, consts=consts, operand_dtype=blob.operand_dtype)


SENSITIVITY = ("w0_lo_zeroed", "layer1_bias_lo_zeroed", "layer2_bias_lo_zeroed", "head_lo_zeroed",
               "beta_rounded_to_16_bits", "w1_row_one_ulp")


@pytest.mark.parametrize("case", SENSITIVITY)
@pytest.mark.parametrize("operands", ["auto", "bf16"])
def test_the_rule_rejects_a_kernel_on_edited_operands(nets, operands, case):
    sd, head, base = nets["policy"]
    blob = dd.PolicyBlob(sd, device=DEV, operands=operands)
    img = nr.decode_blob(blob.blob)
    x = torch.cat([base, _rows(base, 4096, 11)]).to(DEV)
    ref = nr.emulate64(img, x)                              # the pristine blob is the reference
    ok = nr.compare(dd.policy_forward(blob, x), ref)
    nr.assert_accepted(ok, "pristine blob")
    bad = nr.compare(dd.policy_forward(_edited(blob, img, case), x), ref)
    print(f"{case}/{blob.operand_dtype}: {nr.summary(bad)}")
    assert not nr.accepted(bad), f"{case}: the rule accepts it: {nr.summary(bad)}"


# ---- 4. the fp16 range check at its limits -------------------------------------------------------------------------
def _pm(g, N, K, scale):
    """[N][K] in +- row pairs: every column mean over the outputs is exactly 0, so the image is the weights themselves."""
    v = ((torch.rand(N // 2, K, generator=g) * 2 - 1) * scale).float()
    return torch.stack([v, -v], 1).reshape(N, K)


def _edge_base(seed=0):
    g = torch.Generator().manual_seed(seed)
    sd = {"network.0.weight": _pm(g, 128, 15, 0.5), "network.0.bias": _pm(g, 128, 1, 0.5)[:, 0],
          "network.3.weight": _pm(g, 128, 128, 0.1), "network.3.bias": _pm(g, 128, 1, 0.5)[:, 0],
          "network.6.weight": _pm(g, 64, 128, 0.1), "network.6.bias": _pm(g, 64, 1, 0.5)[:, 0],
          "network.9.weight": (torch.rand(3, 64, generator=g) - 0.5).float(), "network.9.bias": torch.zeros(3)}
    for k, n in (("1", 128), ("4", 128), ("7", 64)):
        sd[f"network.{k}.weight"] = torch.ones(n)
        sd[f"network.{k}.bias"] = (0.1 * torch.randn(n, generator=g)).float()
    return sd


def _below(v):
    return float(np.nextafter(np.float32(v), np.float32(0)))


def _above(v):
    return float(np.nextafter(np.float32(v), np.float32(np.inf)))


def _edge(bound, inside):
    sd = _edge_base()
    lin = {0: ("network.0.weight", "network.0.bias"), 1: ("network.3.weight", "network.3.bias"),
           2: ("network.6.weight", "network.6.bias")}
    if bound == "gamma_min":
        sd["network.1.weight"][7] = 2.0 ** -6 if inside else _below(2.0 ** -6)
    elif bound == "gamma_max":
        sd["network.4.weight"][7] = 64.0 if inside else _above(64.0)
    elif bound == "beta_over_gamma":
        sd["network.4.bias"][7] = 1024.0 if inside else _above(1024.0)
    elif bound.startswith("image_max"):
        l = int(bound[-1])
        m = 1024.0 if inside else _above(1024.0)
        sd[lin[l][0]][0, 3], sd[lin[l][0]][1, 3] = m, -m
    elif bound.startswith("image_min"):
        l = int(bound[-1])
        g = torch.Generator().manual_seed(l)
        w, b = lin[l]
        sd[w] = _pm(g, sd[w].shape[0], sd[w].shape[1], 2.0 ** -9)
        sd[b] = _pm(g, sd[b].shape[0], 1, 2.0 ** -9)[:, 0]
        m = 2.0 ** -8 if inside else _below(2.0 ** -8)
        sd[w][0, 3], sd[w][1, 3] = m, -m
    elif bound == "head":
        sd["network.9.weight"][1, 9] = 1024.0 if inside else _above(1024.0)
    elif bound == "beta_1024_everywhere":
        for k in ("1", "4", "7"):
            sd[f"network.{k}.bias"].fill_(1024.0)
        v = (torch.rand(3, 32, generator=torch.Generator().manual_seed(4)) - 0.5).float()
        sd["network.9.weight"] = torch.stack([v, -v], -1).reshape(3, 64)     # logits = differences of activations ~1024
    return sd


EDGES = ["gamma_min", "gamma_max", "beta_over_gamma", "image_max0", "image_max1", "image_max2",
         "image_min0", "image_min1", "image_min2", "head"]


@pytest.mark.parametrize("bound", EDGES + ["beta_1024_everywhere"])
def test_fp16_range_check_at_its_limits(nets, bound):
    _, _, base = nets["policy"]
    x = _rows(base, 4096, 21)
    sd = _edge(bound, True)
    blob = dd.PolicyBlob(sd, device=DEV)
    assert blob.operand_dtype == "fp16", bound
    img = nr.decode_blob(blob.blob)
    probs = dd.policy_forward(blob, x.to(DEV))
    assert torch.isfinite(probs).all()
    st = nr.compare(probs, nr.emulate64(img, x.to(DEV)))
    print(f"edge {bound} (inside, fp16): {nr.summary(st)}")
    nr.assert_accepted(st, f"{bound} inside")
    if bound in EDGES:
        out = _edge(bound, False)
        assert dd.PolicyBlob(out, device=DEV).operand_dtype == "bf16", bound
        with pytest.raises(nv.NativeError):
            dd.PolicyBlob(out, device=DEV, operands="fp16")


# ---- 5. sampling is its documented function ------------------------------------------------------------------------
def _bits(u, p):
    return sum(((u[..., j] < p[..., j]).astype(np.uint8) << j) for j in range(3))


def _logp_bound(prod32):
    """__logf (CUDA math docs: 2^-21.41 absolute on [0.5, 2], 3 ulps elsewhere) + the fp32 product's two roundings."""
    L = np.log(prod32.astype(np.float64))
    inner = (prod32 >= 0.5) & (prod32 <= 2)
    return np.where(inner, 2.0 ** -21.41, 3 * np.spacing(np.abs(L).astype(np.float32)).astype(np.float64)) + 2.0 ** -22


@pytest.mark.parametrize("operands", ["auto", "bf16"])
def test_sampled_actions_and_logp_are_their_philox_function(nets, operands):
    sd, _, _ = nets["policy"]
    blob = dd.PolicyBlob(sd, device=DEV, operands=operands)
    img = nr.decode_blob(blob.blob)
    seed, base, n, T = (7 << 32) + 0x1234567, 2 ** 32 - 300, 600, 12        # env ids cross 2^32: the high word carries
    kw = dict(seed=seed, randomize_drone=True, randomize_platform=True, max_steps=8, auto_reset=True,
              dtype=torch.float32, env_id_base=base)
    ids = base + np.arange(n, dtype=np.uint64)
    for t0 in (0, 777, 2 ** 32 - 5):                                      # the last wraps the step word
        env = dd.BatchedDroneEnv(n, device=DEV, **kw); env.reset()
        out = dd.policy_rollout(env, blob, T, sample=True, t0=t0, want="aplo")
        u = nr.bernoulli_uniforms(seed, ids, t0 + np.arange(T, dtype=np.uint64))
        p32 = out["probs"].cpu().numpy()
        act = out["actions"].cpu().numpy()
        assert np.array_equal(act, _bits(u, p32.astype(np.float64))), f"t0={t0}: {(act != _bits(u, p32)).sum()} actions differ"
        # logp = log of the clamped product (eps = 2^-23, 1 - q in fp32)
        eps = np.float32(2.0 ** -23)
        q = np.clip(p32, eps, np.float32(1) - eps)
        f = np.where(((act[..., None] >> np.arange(3)) & 1) == 1, q, np.float32(1) - q)
        prod32 = (f[..., 0] * f[..., 1]) * f[..., 2]
        ref = np.log(f.astype(np.float64).prod(-1))
        lp = out["logp"].cpu().numpy().astype(np.float64)
        err = np.abs(lp - ref)
        assert (err <= _logp_bound(prod32)).all(), f"t0={t0}: logp off by {err.max():.3e}"
        # tempered: against sigmoid(z_emulate64 / tau); only draws within the rule's bound of the threshold may differ
        for temp in (0.3, 2.5):
            e2 = dd.BatchedDroneEnv(n, device=DEV, **kw); e2.reset()
            o2 = dd.policy_rollout(e2, blob, T, sample=True, t0=t0, want="aplo", temperature=temp)
            ref2 = nr.emulate64(img, o2["obs"].view(-1, 15))
            inv = float(np.float32(1.0 / np.float32(temp)))
            zt = (ref2["z"] * inv).cpu().numpy().reshape(T, n, 3)
            s_ref = 1 / (1 + np.exp(-zt))
            a2 = o2["actions"].cpu().numpy()
            diff = ((a2[..., None] >> np.arange(3)) & 1) != (u < s_ref)
            margin = np.abs(u - s_ref)
            dz = (nr.M_ULPS * nr._u16(img["fmt"]) * ref2["scale"].cpu().numpy()).reshape(T, n, 1) * inv
            bound = s_ref * (1 - s_ref) * dz + 2.0 ** -22
            print(f"{blob.operand_dtype} t0={t0} temperature {temp}: {int(diff.sum())} of {diff.size} draws differ")
            assert (margin[diff] <= bound[diff]).all()
            assert diff.mean() <= 1e-3
    # the PPO-collection instantiation (exactly want="arldo") draws the same actions from the same uniforms
    env = dd.BatchedDroneEnv(n, device=DEV, **kw); env.reset()
    fast = dd.policy_rollout(env, blob, T, sample=True, t0=5, want="arldo")
    env = dd.BatchedDroneEnv(n, device=DEV, **kw); env.reset()
    gen = dd.policy_rollout(env, blob, T, sample=True, t0=5, want="ap")
    u = nr.bernoulli_uniforms(seed, ids, 5 + np.arange(T, dtype=np.uint64))
    assert np.array_equal(fast["actions"].cpu().numpy(), _bits(u, gen["probs"].cpu().numpy().astype(np.float64)))


# ---- 6. at size ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("operands", ["auto", "bf16"])
def test_whole_cfg4_buffer_matches_emulate64(nets, operands):
    """All 16.4 M rows of a cfg-4 rollout (65,536 envs x 250 steps): the rollout's own probabilities and the critic's
    values on the same rows, float64 emulation on the GPU in chunks of 1 M rows."""
    t_start = time.time()
    sdp, _, _ = nets["policy"]
    sdc, _, _ = nets["critic"]
    blob, vblob = dd.PolicyBlob(sdp, device=DEV, operands=operands), dd.ValueBlob(sdc, device=DEV, operands=operands)
    img, vimg = nr.decode_blob(blob.blob), nr.decode_blob(vblob.blob, 1)
    n, T = 65536, 250
    env = dd.BatchedDroneEnv(n, device=DEV, seed=2, randomize_drone=True, randomize_platform=True, max_steps=250,
                             auto_reset=True, dtype=torch.float32)
    env.reset()
    out = dd.policy_rollout(env, blob, T, sample=True, want="op")
    rows, probs = out["obs"].view(-1, 15), out["probs"].view(-1, 3)
    vals = dd.value_forward(vblob, out["obs"]).view(-1)
    ps, vs = [], []
    CH = 1 << 20
    for lo in range(0, rows.shape[0], CH):
        x = rows[lo:lo + CH]
        ps.append(nr.compare(probs[lo:lo + CH], nr.emulate64(img, x)))
        vs.append(nr.compare(vals[lo:lo + CH], nr.emulate64(vimg, x)))
    P, V = nr.pool(ps), nr.pool(vs)
    print(f"cfg-4 buffer, policy/{blob.operand_dtype}: {nr.summary(P)}")
    print(f"cfg-4 buffer, critic/{vblob.operand_dtype}: {nr.summary(V)}")
    print(f"cfg-4 buffer check took {time.time() - t_start:.1f} s")
    nr.assert_accepted(P, f"cfg-4 policy/{blob.operand_dtype}")
    nr.assert_accepted(V, f"cfg-4 critic/{vblob.operand_dtype}")
