"""bench.py --dump-outputs on CPU stand-ins for the sub-batch pipelines: the seeded sample reads image bytes only (never
the alignment gaps between images), in batch order, the same positions on every run, within 64 MB of float32."""
import types

import numpy as np
import torch

import bench

GAP = 255


def _pipe(shapes, first_image):
    """Image k of the sub-batch is filled with its batch index; the 16-byte alignment gaps hold GAP."""
    offs, end = [], 0
    for s in shapes:
        end = (end + 15) & ~15
        offs.append(end)
        end += int(np.prod(s))
    out = torch.full((end,), GAP, dtype=torch.uint8)
    for k, (o, s) in enumerate(zip(offs, shapes)):
        out[o:o + int(np.prod(s))] = first_image + k
    coef = torch.arange(64 * 5, dtype=torch.int16).reshape(5, 64) + 1000 * first_image
    err = torch.arange(first_image, first_image + len(shapes), dtype=torch.int32)
    geom = types.SimpleNamespace(out_offsets=offs, out_shapes=shapes)
    return types.SimpleNamespace(out=out, coef=coef, err=err, plan=types.SimpleNamespace(geom=geom))


def test_dump_outputs_samples_images_in_batch_order(tmp_path):
    pipes = [_pipe([(3, 5, 3), (2, 7)], 0), _pipe([(1, 1, 3), (4, 3, 3), (2, 2)], 2)]
    sizes = [45, 14, 3, 36, 4]
    bench.dump_outputs(tmp_path / "a", pipes)
    bench.dump_outputs(tmp_path / "b", pipes)
    names = ("pixels", "coefficients", "errors")
    a = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in names}
    for n in names:
        assert a[n].dtype == np.float32
        assert np.array_equal(a[n], np.load(tmp_path / "b" / f"{n}.npy"))
    assert sum((tmp_path / "a" / f"{n}.npy").stat().st_size for n in names) <= 64 << 20

    px = a["pixels"]
    assert not (px == GAP).any()
    assert (np.diff(px) >= 0).all()
    counts = np.bincount(px.astype(np.int64), minlength=len(sizes))
    assert np.allclose(counts / len(px), np.array(sizes) / sum(sizes), atol=2e-3)

    coef = np.concatenate([p.coef.reshape(-1).numpy() for p in pipes]).astype(np.float32)
    assert np.isin(a["coefficients"], coef).all() and (np.diff(a["coefficients"]) >= 0).all()
    assert np.array_equal(a["errors"], np.arange(5, dtype=np.float32))
