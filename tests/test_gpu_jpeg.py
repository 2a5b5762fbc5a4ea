"""GPU JPEG decode (csrc/jpeg.cu via rajni_vit_b200.jpeg): frames equal Pillow's on a mixed batch, malformed streams come
back as statuses with Pillow's result in their slots, and --gpu_decode feeds the model exactly what --gpu_preprocess does."""
import io
import json
import os
import re

import numpy as np
import pytest
import torch
from PIL import Image

from rajni_vit_b200 import jpeg
from tests import jpeg_cases as jc

pytestmark = pytest.mark.gpu


def _pillow(data: bytes) -> np.ndarray:
    return np.asarray(Image.open(io.BytesIO(data)).convert("RGB"))


def _frames(out, meta):
    out, meta = out.cpu(), meta.cpu()
    return [out[o:o + h * w * 3].reshape(h, w, 3).numpy() for o, h, w in meta.tolist()]


def test_mixed_batch_equals_pillow():
    """Every supported kind and size, the fallbacks Pillow decodes, and a frame a worker decoded, in one batch."""
    cases = jc.supported_small() + jc.supported_large()
    cases += [(n, d) for n, d in jc.fallbacks() if n in ("progressive", "cmyk", "440", "411", "png")]
    items = [d for _, d in cases]
    pre = torch.from_numpy(jc.content(37, 53, "texture", seed=3))
    items.insert(5, pre)
    out, meta, max_h, status = jpeg.decode_batch(items, "cuda", return_status=True)
    got = _frames(out, meta)
    assert max_h == max(f.shape[0] for f in got)
    names = [n for n, _ in cases]
    names.insert(5, "pre-decoded")
    for i, (name, item) in enumerate(zip(names, items)):
        ref = item.numpy() if isinstance(item, torch.Tensor) else _pillow(item)
        np.testing.assert_array_equal(got[i], ref, err_msg=name)
        expect = jpeg.OK if not isinstance(item, torch.Tensor) and jpeg.parse(item).gpu else jpeg.SKIPPED
        assert status[i] == expect, (name, status[i])


def test_malformed_streams_are_statuses_with_pillows_result():
    cases = dict(jc.malformed())
    good = jc.pil_jpeg(jc.content(48, 40, "grad"), quality=90)
    items = [good, cases["cut-scan"], cases["bad-code"]]
    out, meta, _, status = jpeg.decode_batch(items, "cuda", return_status=True)
    assert status == [jpeg.OK, jpeg.TRUNCATED, jpeg.BAD_CODE]
    for f, d in zip(_frames(out, meta), items):
        np.testing.assert_array_equal(f, _pillow(d))


def test_truncated_file_raises_pillows_error():
    trunc = dict(jc.fallbacks())["truncated-scan"]
    with pytest.raises(OSError) as ref:
        _pillow(trunc)
    with pytest.raises(type(ref.value), match=re.escape(str(ref.value))):
        jpeg.decode_batch([jc.pil_jpeg(jc.content(16, 16, "grad")), trunc], "cuda")


def _folder(root):
    """An ImageFolder of ImageNet-like files: 4:2:0, 4:4:4, 4:2:2 with restarts, grayscale, progressive, a PNG named .JPEG."""
    files = []
    sizes = [(375, 500), (500, 375), (333, 500), (224, 224), (400, 260), (256, 300)]
    for i in range(24):
        h, w = sizes[i % len(sizes)]
        a = jc.content(h, w, "texture", seed=200 + i)
        kind = i % 6
        if kind == 4:
            data = jc.pil_jpeg(a, quality=85, progressive=True)
        elif kind == 5 and i == 5:
            b = io.BytesIO()
            Image.fromarray(a).save(b, "PNG")
            data = b.getvalue()
        else:
            data = jc.pil_jpeg(a, gray=kind == 3, quality=(90, 75, 95, 80, 0, 60)[kind], subsampling=(2, 0, 1, 2, 2, 2)[kind],
                               restart_marker_blocks=4 if kind == 2 else 0)
        d = os.path.join(root, f"n{i % 2:08d}")
        os.makedirs(d, exist_ok=True)
        with open(os.path.join(d, f"img_{i:03d}.JPEG"), "wb") as f:
            f.write(data)
        files.append(data)
    return files


def test_gpu_decode_loader_matches_gpu_preprocess_loader(tmp_path):
    import torchvision.datasets as datasets
    import torchvision.transforms as T
    import rajni_vit_b200 as pkg
    from rajni_vit_b200 import run
    from rajni_vit_b200.data import GpuDecodeLoader, GpuPreprocessLoader, collate_frames, decode_only, read_for_gpu_decode
    from rajni_vit_b200.vit import create_model
    _folder(str(tmp_path))
    kw = dict(batch_size=10, shuffle=False, num_workers=2, collate_fn=collate_frames)
    dec = GpuDecodeLoader(torch.utils.data.DataLoader(datasets.ImageFolder(str(tmp_path), loader=read_for_gpu_decode), **kw), "cuda")
    pre = GpuPreprocessLoader(torch.utils.data.DataLoader(datasets.ImageFolder(str(tmp_path), decode_only), **kw), "cuda")
    assert len(dec) == len(pre) == 3 and dec.rajni_sharded is False
    tf = T.Compose([T.Resize(256, interpolation=T.InterpolationMode.BICUBIC), T.CenterCrop(224), T.ToTensor(),
                    T.Normalize(mean=run.IMAGENET_MEAN, std=run.IMAGENET_STD)])
    ref_ds = datasets.ImageFolder(str(tmp_path), tf)
    model = pkg.RAJNIViTWrapper(create_model("vit_tiny_patch16_224", seed=0), {3: {"keep_ratio": 0.8}}).cuda().eval()
    model_u8 = pkg.RAJNIViTWrapper(create_model("vit_tiny_patch16_224", seed=0), {3: {"keep_ratio": 0.8}}).cuda().eval()
    model_u8.set_input_normalization(run.IMAGENET_MEAN, run.IMAGENET_STD)
    start = 0
    for (c_dec, l_dec), (c_pre, l_pre) in zip(dec, pre):
        assert torch.equal(c_dec, c_pre) and torch.equal(l_dec, l_pre)
        n = c_dec.shape[0]
        ref = torch.stack([ref_ds[start + i][0] for i in range(n)])
        start += n
        assert torch.equal(model_u8(c_dec), model(ref.cuda()))
    assert start == 24


def test_run_gpu_decode_gives_the_gpu_preprocess_accuracy(tmp_path):
    from rajni_vit_b200 import run
    _folder(str(tmp_path / "data"))
    sched = tmp_path / "s.json"
    sched.write_text(json.dumps({"3": {"keep_ratio": 0.8}}))
    common = ["--data_path", str(tmp_path / "data"), "--schedule", str(sched), "--model", "vit_tiny_patch16_224",
              "--batch_size", "8", "--num_workers", "2", "--warmup", "0"]
    a = run.main(common + ["--gpu_decode"])
    b = run.main(common + ["--gpu_preprocess"])
    assert a["rajni"][0] == b["rajni"][0]
