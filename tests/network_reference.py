"""Float64 reference of the fused policy / critic network (``csrc/policy_rollout.cu``) -- TEST INFRASTRUCTURE.

The kernel computes a specified sequence of roundings: 16-bit operand images (fp16 or bf16, folded by
``dd_policy_pack``), a split hi + lo first layer, 16-bit hidden activations, fp32 accumulation.  This module evaluates
exactly that sequence in float64, so the only differences left between it and the kernel are the order of the fp32
sums, ``rsqrt.approx`` / ``__expf`` and the occasional 16-bit activation that those push across a rounding boundary.

* ``decode_blob`` / ``encode_blob``: the packed ``PolicyBlob`` layout (its operand images as float64, its
  ``DDPolicyConsts`` section);
* ``fold64``: ``dd_policy_pack``'s folding in float64 (what the images are roundings of);
* ``emulate64``: the kernel's arithmetic on decoded images; ``exact64``: the notebook network in float64;
* ``philox4x32_10``: the counter-based generator of the in-kernel Bernoulli uniforms, vectorised;
* ``compare`` / ``assert_accepted``: the one acceptance rule the tests apply (see ``compare``).
"""
from typing import Dict, Mapping

import numpy as np
import torch

# ---- blob layout (csrc/policy_rollout.cu, kW*Off / kParOff) -------------------------------------------------------
H1, H2, H3, IN_PAD, W3_ROWS = 128, 128, 64, 16, 16
IMAGES = (  # name, byte offset, [N][K]
    ("w0", 0, H1, IN_PAD),          # [W0 | b0] (input 15 := 1), high halves
    ("w1", 4096, H2, H1),
    ("w1b", 36864, H2, 16),         # column 0 / 1 = bias hi / lo, against a constant block of ones in columns 0, 1
    ("w2", 40960, H3, H2),
    ("w2b", 57344, H3, 16),
    ("w0lo", 59392, H1, IN_PAD),    # low halves of the layer-0 image
    ("w3", 63488, W3_ROWS, H3),     # head: rows 0-2 = hi, 3-5 = lo of w3 |gamma2|, the rest 0
)
PAR_OFF = 65536
PAR_WORDS = 520                      # DDPolicyConsts: beta0[128] beta1[128] beta2[64] w3[3][64] b3[4] operands reserved[3]
BLOB_BYTES = PAR_OFF + 4 * PAR_WORDS
OPERANDS_BF16, OPERANDS_FP16 = 1, 2
GAMMA_FLOOR = float(np.float32(1e-12))
LN_EPS = 1e-5
assert BLOB_BYTES == 67616, "the mirrored layout no longer matches DD_POLICY_BLOB_BYTES"
assert all(off + 2 * n * k <= nxt for (_, off, n, k), nxt in zip(IMAGES, [o for _, o, _, _ in IMAGES[1:]] + [PAR_OFF]))


def image_index(N: int, K: int) -> np.ndarray:
    """[N][K] array of 16-bit element indices: element (n, k) sits at (k / 8) * (N * 8) + n * 8 + k % 8."""
    n, k = np.meshgrid(np.arange(N), np.arange(K), indexing="ij")
    return (k // 8) * (N * 8) + n * 8 + k % 8


def _bits_to_f64(u16: np.ndarray, f16: bool) -> np.ndarray:
    if f16:
        return u16.view(np.float16).astype(np.float64)
    return (u16.astype(np.uint32) << 16).view(np.float32).astype(np.float64)


def rn16(t: torch.Tensor, f16: bool) -> torch.Tensor:
    """Round to the nearest fp16 / bf16 (ties to even) and back to float64; the operand is taken as fp32 first, which is
    what the kernel rounds."""
    return t.to(torch.float32).to(torch.float16 if f16 else torch.bfloat16).to(torch.float64)


def ulp16(t: torch.Tensor, f16: bool) -> torch.Tensor:
    """Spacing of the 16-bit format at |t| (subnormal spacing below the normal range)."""
    a = t.abs().clamp_min(2.0 ** -14 if f16 else 2.0 ** -126)
    return torch.exp2(torch.floor(torch.log2(a)) - (10 if f16 else 7))


def decode_blob(blob, head: int = 3) -> Dict[str, object]:
    """The operand images of a packed blob (bytes / uint8 array / tensor) as float64 [N][K] tensors, and its
    DDPolicyConsts section (``consts_dict``).  The format is the section's ``operands`` word."""
    raw = np.asarray(blob.cpu() if isinstance(blob, torch.Tensor) else bytearray(blob), dtype=np.uint8)
    assert raw.size == BLOB_BYTES, raw.size
    consts = consts_dict(raw[PAR_OFF:].tobytes(), head)
    f16 = consts["fmt"] == "fp16"
    out: Dict[str, object] = {"fmt": consts["fmt"], "head": head}
    for name, off, N, K in IMAGES:
        u16 = raw[off:off + 2 * N * K].view(np.uint16)
        out[name] = torch.from_numpy(_bits_to_f64(u16[image_index(N, K)], f16))
    out["consts"] = consts
    return out


def consts_dict(c, head: int = 3) -> Dict[str, object]:
    """A DDPolicyConsts (ctypes struct or its 2,080-byte image) as float64 tensors + the operand format."""
    raw = bytes(c)
    assert len(raw) == 4 * PAR_WORDS, len(raw)
    f = np.frombuffer(raw, dtype=np.float32).astype(np.float64)
    fmt = int(np.frombuffer(raw, dtype=np.int32)[516])
    assert fmt in (OPERANDS_BF16, OPERANDS_FP16), f"operands word {fmt}: not filled by dd_policy_pack"
    return {"beta0": torch.from_numpy(f[0:128].copy()), "beta1": torch.from_numpy(f[128:256].copy()),
            "beta2": torch.from_numpy(f[256:320].copy()), "w3": torch.from_numpy(f[320:512].reshape(3, 64).copy()),
            "b3": torch.from_numpy(f[512:516].copy()), "fmt": "fp16" if fmt == OPERANDS_FP16 else "bf16", "head": head}


def consts_bytes(consts: Mapping[str, object]) -> bytes:
    f = np.zeros(PAR_WORDS, np.float32)
    f[0:128], f[128:256], f[256:320] = consts["beta0"].numpy(), consts["beta1"].numpy(), consts["beta2"].numpy()
    f[320:512], f[512:516] = consts["w3"].reshape(-1).numpy(), consts["b3"].numpy()
    w = f.view(np.int32)
    w[516] = OPERANDS_FP16 if consts["fmt"] == "fp16" else OPERANDS_BF16
    return w.tobytes()


def encode_blob(images: Mapping[str, object]) -> bytes:
    """Inverse of decode_blob (images must hold values representable in their format)."""
    f16 = images["fmt"] == "fp16"
    raw = np.zeros(BLOB_BYTES, np.uint8)
    for name, off, N, K in IMAGES:
        v = images[name].to(torch.float64)
        assert tuple(v.shape) == (N, K), (name, tuple(v.shape))
        assert torch.equal(rn16(v, f16), v), f"{name}: values not representable in {images['fmt']}"
        if f16:
            u16 = v.numpy().astype(np.float16).view(np.uint16)
        else:
            u16 = (v.numpy().astype(np.float32).view(np.uint32) >> 16).astype(np.uint16)
        flat = np.zeros(N * K, np.uint16)
        flat[image_index(N, K)] = u16
        raw[off:off + 2 * N * K] = flat.view(np.uint8)
    raw[PAR_OFF:] = np.frombuffer(consts_bytes(images["consts"]), np.uint8)
    return raw.tobytes()


def _params64(state_dict: Mapping[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    sd = {k.replace("network.", ""): v for k, v in state_dict.items() if k.replace("network.", "")[:1].isdigit()}
    return {k: v.detach().cpu().to(torch.float32).to(torch.float64) for k, v in sd.items()}


def fold64(state_dict: Mapping[str, torch.Tensor], head: int = 3) -> Dict[str, torch.Tensor]:
    """dd_policy_pack's folding in float64.  With s = sign(gamma) (+1 for -0), g = max(|gamma|, 1e-12) and g_prev the g of
    the previous LayerNorm: image = s (W - mean over outputs) g_prev, bias = s (b - mean b), beta' = beta / g, and the last
    Linear becomes w3 g2.  Also returns the quantities the pack's fp32 evaluation rounds (``*_mean``, ``*_c``) so a test
    can bound how far the fp32 fold may sit from this one."""
    p = _params64(state_dict)
    out: Dict[str, torch.Tensor] = {}
    gam = [p["1.weight"], p["4.weight"], p["7.weight"]]
    gabs = [g.abs().clamp_min(GAMMA_FLOOR) for g in gam]
    for l, (wk, bk) in enumerate((("0.weight", "0.bias"), ("3.weight", "3.bias"), ("6.weight", "6.bias"))):
        W, b = p[wk], p[bk]
        s = torch.where(gam[l] < 0, -1.0, 1.0).to(torch.float64)
        c = gabs[l - 1] if l > 0 else torch.ones(W.shape[1], dtype=torch.float64)
        Wb = torch.cat([W, b[:, None]], 1)                        # the bias is column K (scale 1)
        cb = torch.cat([c, torch.ones(1, dtype=torch.float64)])
        mean = Wb.mean(0, keepdim=True)
        out[f"img{l}"] = s[:, None] * (Wb - mean) * cb[None, :]
        out[f"img{l}_mean"], out[f"img{l}_raw"], out[f"img{l}_c"] = mean.expand_as(Wb), Wb, cb[None, :].expand_as(Wb)
        out[f"beta{l}"] = p[("1.bias", "4.bias", "7.bias")[l]] / gabs[l]
    out["w3"] = p["9.weight"][:head] * gabs[2][None, :]
    out["b3"] = p["9.bias"][:head]
    return out


def images_from_fold(fold: Mapping[str, torch.Tensor], f16: bool, head: int = 3, rounding: bool = True) -> Dict[str, object]:
    """Operand images built in Python from ``fold64`` the way the pack builds them (hi = rn16(v), lo = rn16(v - hi));
    ``rounding=False`` keeps the exact fold in the hi images and zero low halves (the unrounded network)."""
    q = (lambda t: rn16(t, f16)) if rounding else (lambda t: t)

    def split(v):
        hi = q(v)
        return hi, (q(v - hi) if rounding else torch.zeros_like(v))

    img: Dict[str, object] = {"fmt": "fp16" if f16 else "bf16", "head": head}
    img["w0"], img["w0lo"] = split(fold["img0"])
    for l, N in ((1, H2), (2, H3)):
        img[f"w{l}"] = q(fold[f"img{l}"][:, :-1])
        bh, bl = split(fold[f"img{l}"][:, -1])
        blk = torch.zeros(N, 16, dtype=torch.float64)
        blk[:, 0], blk[:, 1] = bh, bl
        img[f"w{l}b"] = blk
    w3 = torch.zeros(W3_ROWS, H3, dtype=torch.float64)
    hi, lo = split(fold["w3"])
    w3[:head], w3[3:3 + head] = hi, lo
    img["w3"] = w3
    f32 = (lambda t: t.to(torch.float32).to(torch.float64)) if rounding else (lambda t: t)
    w3c = torch.zeros(3, H3, dtype=torch.float64)
    w3c[:head] = f32(fold["w3"])
    b3 = torch.zeros(4, dtype=torch.float64)
    b3[:head] = f32(fold["b3"])
    img["consts"] = {"beta0": f32(fold["beta0"]), "beta1": f32(fold["beta1"]), "beta2": f32(fold["beta2"]),
                     "w3": w3c, "b3": b3, "fmt": img["fmt"], "head": head}
    return img


def _ln(d: torch.Tensor, beta: torch.Tensor) -> torch.Tensor:
    """The kernel's folded LayerNorm: the accumulator is already centred, var = mean of its squares."""
    return d * torch.rsqrt((d * d).mean(-1, keepdim=True) + LN_EPS) + beta


def emulate64(images: Mapping[str, object], x: torch.Tensor, consts: Mapping[str, object] = None,
              rounding: bool = True) -> Dict[str, object]:
    """The kernel's arithmetic in float64 on the decoded images, for observation rows x [n, 15] (fp32, any device):

      x_hi = rn16(x), x_lo = rn16(x - x_hi), input 15 = 1;  D0 = x_hi W_hi + x_hi W_lo + x_lo W_hi
      D_l  = a_l W_l + ones B_l  (the bias block: hi + lo against the constant ones columns)
      y    = D rsqrt(mean D^2 + 1e-5) + beta'        a = rn16(relu(y))  (the next layer's 16-bit operand)
      policy: z_o = a3 W3[o] + a3 W3[3 + o] + b3_o, p = sigmoid(z);   critic: v = sum relu(y3) w3 + b3 (fp32 head)

    ``consts`` defaults to the blob's own section (the kernel uses the host copy handed to the launch).  ``rounding=False``
    skips the 16-bit roundings of the input and of the activations.  Returns the logits ``z`` [n, head], ``out`` (probs
    [n, 3] / values [n]), the pre-rounding activations ``y`` per hidden layer, the accumulators ``d``, and ``scale``: per
    row, the largest sum of |a_j w_j| over the head's outputs -- the logit scale a 16-bit ulp of the activations is taken
    against in the acceptance rule."""
    consts = images["consts"] if consts is None else consts
    head = consts["head"]
    f16 = images["fmt"] == "fp16"
    dev = x.device
    q = (lambda t: rn16(t, f16)) if rounding else (lambda t: t)
    g = {k: v.to(dev) for k, v in images.items() if isinstance(v, torch.Tensor)}
    c = {k: v.to(dev) for k, v in consts.items() if isinstance(v, torch.Tensor)}
    x16 = torch.cat([x.to(torch.float64), torch.ones(x.shape[0], 1, dtype=torch.float64, device=dev)], 1)
    xh = q(x16)
    xl = q(x16 - xh) if rounding else torch.zeros_like(x16)
    ones = torch.zeros(16, dtype=torch.float64, device=dev)
    ones[:2] = 1.0
    d0 = xh @ g["w0"].T + xh @ g["w0lo"].T + xl @ g["w0"].T
    y1 = _ln(d0, c["beta0"])
    d1 = q(torch.relu(y1)) @ g["w1"].T + ones @ g["w1b"].T
    y2 = _ln(d1, c["beta1"])
    d2 = q(torch.relu(y2)) @ g["w2"].T + ones @ g["w2b"].T
    y3 = _ln(d2, c["beta2"])
    if head == 3:
        a3 = q(torch.relu(y3))
        z = a3 @ g["w3"][0:3].T + a3 @ g["w3"][3:6].T + c["b3"][:3]
        scale = (a3.abs() @ g["w3"][0:3].abs().T).amax(-1)
        out = torch.sigmoid(z)
    else:
        a3 = torch.relu(y3)
        z = a3 @ c["w3"][:1].T + c["b3"][:1]
        scale = (a3.abs() @ c["w3"][:1].abs().T)[:, 0]
        out = z[:, 0]
    return {"z": z, "out": out, "y": [y1, y2, y3], "d": [d0, d1, d2], "scale": scale, "fmt": images["fmt"], "head": head}


def exact64(state_dict: Mapping[str, torch.Tensor], x: torch.Tensor, head: int = 3) -> torch.Tensor:
    """The notebook network (Linear-LayerNorm-ReLU x 3, Linear, sigmoid for the policy) in float64: probs [n, 3] or values [n]."""
    p = {k: v.to(x.device) for k, v in _params64(state_dict).items()}
    h = x.to(torch.float64)
    for lin, ln in (("0", "1"), ("3", "4"), ("6", "7")):
        h = torch.nn.functional.linear(h, p[lin + ".weight"], p[lin + ".bias"])
        h = torch.relu(torch.nn.functional.layer_norm(h, h.shape[-1:], p[ln + ".weight"], p[ln + ".bias"], eps=LN_EPS))
    z = torch.nn.functional.linear(h, p["9.weight"][:head], p["9.bias"][:head])
    return torch.sigmoid(z) if head == 3 else z[:, 0]


# ---- Philox4x32-10 (Random123), vectorised ------------------------------------------------------------------------
_M0, _M1, _W0, _W1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """ctr: 4 arrays (or ints) of uint32 words, key: 2.  Returns the 4 output words as uint32 arrays (broadcast)."""
    c = [np.asarray(v, dtype=np.uint64) & _MASK for v in ctr]
    k0, k1 = (np.asarray(v, dtype=np.uint64) & _MASK for v in key)
    c0, c1, c2, c3 = np.broadcast_arrays(*c)
    k0, k1 = np.broadcast_to(k0, c0.shape), np.broadcast_to(k1, c0.shape)
    for r in range(10):
        if r:
            k0, k1 = (k0 + _W0) & _MASK, (k1 + _W1) & _MASK
        p0, p1 = _M0 * c0, _M1 * c2                        # < 2^64: exact in uint64
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _MASK, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _MASK)
    return tuple(v.astype(np.uint32) for v in (c0, c1, c2, c3))


def bernoulli_uniforms(seed: int, env_ids: np.ndarray, steps: np.ndarray) -> np.ndarray:
    """The Bernoulli uniforms of include/drone_b200.h: r = Philox((id lo, id hi, step mod 2^32, 2), (seed lo, seed hi)),
    u_j = (r_j >> 8) 2^-24 for lanes j = 0, 1, 2 (DD_ACT_MAIN / LEFT / RIGHT).  env_ids [N], steps [T] -> u [T, N, 3]."""
    ids = np.asarray(env_ids, dtype=np.uint64)[None, :]
    t = (np.asarray(steps, dtype=np.uint64) & _MASK)[:, None]
    r = philox4x32_10((ids & _MASK, ids >> np.uint64(32), t, 2), (seed & 0xFFFFFFFF, seed >> 32))
    return np.stack([(r[j] >> 8).astype(np.float64) * 2.0 ** -24 for j in range(3)], -1)


# ---- the acceptance rule ------------------------------------------------------------------------------------------
# Accumulation order and systematic error look different.  A different summation order (tensor cores against a float64
# sum) occasionally pushes a 16-bit activation across a rounding boundary: rare rows move, by at most a few 16-bit ulps
# of the logit scale.  A dropped low half, an extra rounding, a wrong constant or a wrong column moves most rows.  So:
#   (a) at least a fraction F of the rows agree with emulate64 to within TAU in every logit (values: TAU (1 + |v|));
#   (b) no row is off by more than M_ULPS 16-bit ulps (2^-11 fp16, 2^-8 bf16) of its logit scale (emulate64's ``scale``).
# Probabilities carry the logit only to the fp32 resolution of the sigmoid: a row whose sigmoid evaluation error, in logit
# units, exceeds TAU says nothing about (a) and counts in (b) only, with that error allowed on top.
TAU = 1e-5
F = 0.8
M_ULPS = 4.0


def _quantiles(t: torch.Tensor) -> Dict[float, float]:
    """0.5 / 0.9 / 0.99 / 0.999 quantiles (by sorting: torch.quantile refuses inputs beyond 2^24 elements)."""
    if t.numel() == 0:
        return {q: 0.0 for q in (0.5, 0.9, 0.99, 0.999)}
    s = torch.sort(t.reshape(-1).double()).values
    return {q: float(s[min(int(q * s.numel()), s.numel() - 1)].item()) for q in (0.5, 0.9, 0.99, 0.999)}


def _u16(fmt: str) -> float:
    return 2.0 ** -11 if fmt == "fp16" else 2.0 ** -8


def compare(kernel_out: torch.Tensor, ref: Mapping[str, object], worst: int = 5) -> Dict[str, object]:
    """Per-row deviation of a kernel output (probs [n, 3] or values [n]) from emulate64's ``ref``.

    ``d``: per row, the largest logit deviation (probabilities: |p - sigmoid(z)| / sigmoid'(z), less the fp32 sigmoid's own
    error) or |v - v_ref| / (1 + |v_ref|) for values, in units of TAU's scale.  ``ulps``: the same row's deviation in
    16-bit ulps of its logit scale (rule (b)).  Returns those with their quantiles, the fraction of informative rows
    within TAU and the worst rows."""
    k = kernel_out.to(torch.float64).reshape(ref["out"].shape).to(ref["out"].device)
    if ref["head"] == 3:
        z = ref["z"]
        p = torch.sigmoid(z)
        dsig = torch.exp(-z.abs()) / (1 + torch.exp(-z.abs())) ** 2
        # the fp32 sigmoid's own error in logit units: __expf (2 + 1.17 |x| ulps), the rounding of 1 + e^-z and the MUFU
        # reciprocal (p near 1 is resolved only to 2^-24, i.e. 2^-24 / (1 - p) in the logit); below z = -87 the kernel's p
        # is 0 (__expf overflows, __fdividef flushes), so an absolute 2^-126 is allowed too
        allow = 2.0 ** -24 * (6 + 2 * z.abs() + 3 / (1 - p).clamp_min(1e-300)) + 2.0 ** -126 / dsig.clamp_min(1e-300)
        dev = ((k - p).abs() / dsig - allow).clamp_min(0.0)
        absdev = dev.amax(-1)
        inf_logit = allow <= TAU
        informative = inf_logit.any(-1)
        rel = torch.where(inf_logit, dev, torch.zeros_like(dev)).amax(-1)     # (a) over the logits that can tell
    else:
        absdev = (k - ref["out"]).abs()
        rel = absdev / (1 + ref["out"].abs())
        informative = torch.ones_like(rel, dtype=torch.bool)
    ulps = absdev / (_u16(ref["fmt"]) * ref["scale"])
    ri = rel[informative]
    order = torch.argsort(ulps, descending=True)[:worst]
    return {
        "n": int(rel.numel()), "informative": int(informative.sum().item()),
        "agree": float((ri <= TAU).double().mean().item()) if ri.numel() else 1.0,
        "quantiles": _quantiles(ri), "max": float(rel.max().item()) if rel.numel() else 0.0,
        "max_ulps": float(ulps.max().item()) if ulps.numel() else 0.0,
        "worst": [(int(i), float(rel[i]), float(ulps[i])) for i in order.tolist()],
        "rel": rel.cpu(), "ulps": ulps.cpu(), "informative_mask": informative.cpu(),
    }


def pool(stats) -> Dict[str, object]:
    """Several compare() results as one batch (rule (a) over all of their rows)."""
    rel = torch.cat([s["rel"] for s in stats])
    ulps = torch.cat([s["ulps"] for s in stats])
    inf = torch.cat([s["informative_mask"] for s in stats])
    ri = rel[inf]
    return {"n": int(rel.numel()), "informative": int(inf.sum().item()),
            "agree": float((ri <= TAU).double().mean().item()) if ri.numel() else 1.0, "quantiles": _quantiles(ri),
            "max": float(rel.max().item()), "max_ulps": float(ulps.max().item()),
            "worst": [], "rel": rel, "ulps": ulps, "informative_mask": inf}


def accepted(stats: Mapping[str, object], min_informative: int = 500) -> bool:
    """Rule (a) (when the batch has enough informative rows to mean something) and rule (b)."""
    a = stats["informative"] < min_informative or stats["agree"] >= F
    return a and stats["max_ulps"] <= M_ULPS


def summary(stats: Mapping[str, object]) -> str:
    q = stats["quantiles"]
    return (f"n={stats['n']} informative={stats['informative']} agree={stats['agree']:.4f} "
            f"q50/90/99/99.9={q[0.5]:.2e}/{q[0.9]:.2e}/{q[0.99]:.2e}/{q[0.999]:.2e} max={stats['max']:.2e} "
            f"max_ulps={stats['max_ulps']:.3f} worst={stats['worst'][:3]}")


def assert_accepted(stats: Mapping[str, object], what: str = "", min_informative: int = 500) -> None:
    assert accepted(stats, min_informative), f"{what}: {summary(stats)} (rule: agree >= {F} within {TAU}, max_ulps <= {M_ULPS})"
