"""The batch imager of device-resident diagrams without a GPU: tlc_pimg_batch_dev / tlc_pimg_batch_grad_dev reject bad
arguments before any CUDA call, api.persistence_images checks its tensors before touching CUDA, and the pure-torch
restatement of the imager that the GPU tests use as their reference (values and autograd) is pinned here against the
oracle, itself pinned against the real imager."""
import ctypes as C
import math
import os

import numpy as np
import pytest
import torch

import oracle as orc
from helpers import GOLDEN, rel_err
from tlc_b200 import _lib as L
from tlc_b200 import api


def torch_images(poff, birth, death, kind=None, img_mask=None, resolution=5):
    """PersistenceImager(resolution).transform of every diagram of a ragged batch, in torch (differentiable): the imager
    of include/tlc_b200.h stated with torch.special.erfc, torch.clamp and the mesh i * step, one [points, res, res]
    outer product summed per diagram."""
    res = int(resolution)
    dev = birth.device
    po = poff.to("cpu", torch.int64)
    D = po.numel() - 1
    lo, hi = int(po[0]), int(po[-1])
    seg = torch.repeat_interleave(torch.arange(D, device=dev), (po[1:] - po[:-1]).clamp(min=0).to(dev))
    b, p = birth[lo:hi], death[lo:hi] - birth[lo:hi]
    w = torch.clamp(p, 0.0, 1.0)
    if kind is not None:
        k = kind[lo:hi].to(torch.int64)
        w = w * (((torch.full_like(k, img_mask) >> k.clamp(max=31)) & 1) * (k < 32)).to(w.dtype)
    step = ((1.0 + 1.0 / res) - 0.0) / (res + 1)
    x = torch.arange(res + 1, dtype=torch.float64, device=dev) * step

    def cdf(z):
        return torch.special.erfc(-z / math.sqrt(2.0)) * 0.5

    cb, cp = cdf(x[None, :] - b[:, None]), cdf(x[None, :] - p[:, None])
    a_, b_ = cb[:, 1:] - cb[:, :-1], cp[:, 1:] - cp[:, :-1]
    terms = (w[:, None, None] * a_[:, :, None] * b_[:, None, :]).reshape(-1, res * res)
    return torch.zeros((D, res * res), dtype=torch.float64, device=dev).index_add(0, seg, terms)


def golden_diagrams():
    """[(diagram [K, 2], resolution, stored image)] of pimg_vectors.npz"""
    z = np.load(os.path.join(GOLDEN, "pimg_vectors.npz"))
    out = [(z["PD"], 5, z["img"])] + [(z["rnd%d" % k], 5, z["img%d" % k]) for k in range(4)]
    return out + [(z["rnd2"], 7, z["img2_res7"])], z["gt4"]


def test_restatement_equals_the_oracle_on_the_golden_vectors():
    cases, gt4 = golden_diagrams()
    for dgm, res, img in cases:
        t = torch.from_numpy(np.ascontiguousarray(dgm, dtype=np.float64))
        mine = torch_images(torch.tensor([0, len(dgm)]), t[:, 0].contiguous(), t[:, 1].contiguous(), resolution=res)
        ref = orc.pimg_transform(dgm, res).reshape(-1)
        assert rel_err(mine.numpy()[0], ref) < 1e-12, (len(dgm), res)
        assert rel_err(mine.numpy()[0], img) < 1e-5
    pd = torch.from_numpy(cases[0][0])
    assert np.max(np.abs(torch_images(torch.tensor([0, 46]), pd[:, 0], pd[:, 1]).numpy()[0] - gt4)) < 6e-5


def test_restatement_batches_masks_and_empty_segments():
    rng = np.random.default_rng(3)
    dgms = [rng.uniform(-0.3, 1.4, size=(k, 2)) for k in (0, 5, 0, 9, 1, 0)]
    kinds = [rng.integers(0, 5, size=len(d)) for d in dgms]
    poff = torch.tensor(np.concatenate([[2], 2 + np.cumsum([len(d) for d in dgms])]))
    allp = np.concatenate([np.zeros((2, 2))] + dgms + [np.zeros((3, 2))])
    kind = torch.from_numpy(np.concatenate([np.zeros(2, np.int64)] + kinds + [np.zeros(3, np.int64)]).astype(np.uint8))
    mask = (1 << L.K_UP) | (1 << L.K_ONE)
    out = torch_images(poff, torch.from_numpy(allp[:, 0].copy()), torch.from_numpy(allp[:, 1].copy()), kind, mask).numpy()
    for t, (d, k) in enumerate(zip(dgms, kinds)):
        keep = np.isin(k, (L.K_UP, L.K_ONE))
        assert rel_err(out[t], orc.pimg_transform(d[keep], 5).reshape(-1)) < 1e-12, t


BAD_BATCH = [  # (D, poff, birth, death, resolution, word the message names)
    (-1, 1, 1, 1, 5, "D"),
    (1 << 31, 1, 1, 1, 5, "D"),
    (2, 1, 1, 1, 0, "resolution"),
    (2, 1, 1, 1, 17, "resolution"),
    (2, 0, 1, 1, 5, "dev_poff"),
    (2, 1, 0, 1, 5, "dev_birth"),
    (2, 1, 1, 0, 5, "dev_death"),
]


def test_batch_entry_points_reject_bad_arguments():
    lib = L.lib()
    fake = C.create_string_buffer(64)  # never dereferenced: every check below fails first
    ptr = C.addressof(fake)
    for D, po, b, d, res, word in BAD_BATCH:
        args = (0, D, ptr if po else None, ptr if b else None, ptr if d else None, None, 1, res)
        assert lib.tlc_pimg_batch_dev(*args, ptr, None) == L.E_INVALID, word
        assert word in lib.tlc_last_error().decode(), word
        assert lib.tlc_pimg_batch_grad_dev(*args, ptr, ptr, ptr, None) == L.E_INVALID, word
        assert word in lib.tlc_last_error().decode(), word
    assert lib.tlc_pimg_batch_dev(0, 2, ptr, ptr, ptr, None, 1, 5, None, None) == L.E_INVALID
    assert "dev_out" in lib.tlc_last_error().decode()
    assert lib.tlc_pimg_batch_grad_dev(0, 2, ptr, ptr, ptr, None, 1, 5, None, ptr, ptr, None) == L.E_INVALID
    assert "dev_grad_out" in lib.tlc_last_error().decode()
    # nothing to do: no CUDA call, so these succeed without a device
    assert lib.tlc_pimg_batch_dev(0, 0, None, None, None, None, 1, 5, None, None) == 0
    assert lib.tlc_pimg_batch_grad_dev(0, 0, None, None, None, None, 1, 5, None, None, None, None) == 0
    assert lib.tlc_pimg_batch_grad_dev(0, 2, ptr, ptr, ptr, None, 1, 5, ptr, None, None, None) == 0


def cpu_inputs(P=6):
    return (torch.tensor([0, 2, P]), torch.rand(P, dtype=torch.float64), torch.rand(P, dtype=torch.float64),
            torch.zeros(P, dtype=torch.uint8))


@pytest.mark.parametrize("case", ["cpu", "poff_dtype", "birth_dtype", "death_dtype", "kind_dtype", "death_shape",
                                  "kind_shape", "birth_2d", "poff_empty", "death_strided", "mask_without_kind",
                                  "resolution"])
def test_persistence_images_checks_its_tensors_before_cuda(case, monkeypatch):
    def no_cuda(*a, **k):
        raise AssertionError("a CUDA call was made")
    monkeypatch.setattr(api, "_images_fn", no_cuda)
    poff, b, d, k = cpu_inputs()
    kw = dict(kind=k, img_mask=1)
    err = ValueError
    if case == "poff_dtype":
        poff, err = poff.to(torch.int32), TypeError
    elif case == "birth_dtype":
        b, err = b.float(), TypeError
    elif case == "death_dtype":
        d, err = d.float(), TypeError
    elif case == "kind_dtype":
        kw["kind"], err = k.to(torch.int32), TypeError
    elif case == "death_shape":
        d = d[:5]
    elif case == "kind_shape":
        kw["kind"] = torch.zeros(7, dtype=torch.uint8)
    elif case == "birth_2d":
        b = b.reshape(2, 3)
    elif case == "poff_empty":
        poff = torch.zeros(0, dtype=torch.int64)
    elif case == "death_strided":
        d = torch.rand(12, dtype=torch.float64)[::2]
    elif case == "mask_without_kind":
        kw = dict(img_mask=1)
    elif case == "resolution":
        kw["resolution"] = 17
    with pytest.raises(err):
        api.persistence_images(poff, b, d, **kw)
