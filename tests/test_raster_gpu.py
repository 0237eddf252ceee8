"""GPU parity of the rasterizer / correspondence kernels (through the C ABI) against
  * the reference's own CUDA kernels compiled for sm_100a (oracle/_ref, bit-exact fim): SHA-256 digests of their outputs
    on the inputs of REF_FACES / REF_CASES, stored by tests/golden/make_raster_golden.py, and
  * the C restatement (oracle/raster_ref.c) + torch glue restatement (oracle/nmr_ref.py)."""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

from impersonator_b200 import kernels as K
from impersonator_b200 import synthetic as S
from oracle import nmr_ref, raster

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def run_mine(faces, size, flip=False, want_inv=True):
    B, F = faces.shape[:2]
    dev = faces.device
    fim = torch.full((B, size, size), -1, dtype=torch.int32, device=dev)
    wim = torch.zeros((B, size, size, 3), dtype=torch.float32, device=dev)
    depth = torch.full((B, size, size), 100.0, dtype=torch.float32, device=dev)
    finv = torch.zeros((B, F, 3, 3), dtype=torch.float32, device=dev) if want_inv else None
    K.raster_forward_face_index_map(faces, fim, wim, depth, size, faces_inv=finv, flip_rows=flip)
    torch.cuda.synchronize()
    return fim, wim, depth, finv


def digest(t):
    return hashlib.sha256(t.detach().cpu().contiguous().numpy().tobytes()).hexdigest()


def compare_with_gpu_ref(case, faces, size):
    """Bitwise comparison with the outputs of the reference kernels for the faces of REF_FACES[case] at ``size``."""
    want = json.load(open(os.path.join(GOLD, "raster_ref.json")))["%s@%d" % (case, size)]
    assert digest(faces) == want["faces"], "the faces differ from those the reference kernels were run on"
    fim, wim, depth, finv = run_mine(faces, size)
    covered = int((fim >= 0).sum())
    print("covered %d (reference %d)" % (covered, want["covered"]))
    assert digest(finv) == want["faces_inv"], "faces_inv differs bitwise from the reference kernel_1"
    assert covered == want["covered"] and digest(fim) == want["fim"], "face_index_map differs from the reference kernel_2"
    assert digest(wim) == want["wim"] and digest(depth) == want["depth"]
    return fim


def sphere_faces(B, seed, dev):
    v, f = S.uv_sphere()
    cam, verts = S.synthetic_frames(B, seed=seed, base_verts=v)
    return nmr_ref.project_to_faces(cam, verts, f).to(dev).contiguous(), cam, verts, f


def test_sphere_bit_exact_vs_reference_kernels(cuda):
    faces, _, _, _ = sphere_faces(3, 1234, cuda)
    for size in (256, 64):
        fim = compare_with_gpu_ref("sphere_b3_seed1234", faces, size)
        assert int((fim >= 0).sum()) > 100


def test_sphere_512_bit_exact(cuda):
    faces, _, _, _ = sphere_faces(2, 77, cuda)
    compare_with_gpu_ref("sphere_b2_seed77", faces, 512)


def teapot_batch_faces():
    """tests/utils.py:11-27 (to_minibatch): the teapot sits in slot 2 of a batch of 4, the other
    three meshes are all-zero vertices -> every face degenerate (whole-image scan path)."""
    g = np.load(os.path.join(GOLD, "teapot.npz"))
    tp = torch.from_numpy(g["faces"])
    zero_v = torch.zeros(1, 1292, 3)
    # the all-zero mesh after look_at + perspective (look_at.py:57-60, perspective.py:13-20)
    z = zero_v[..., 2] - nmr_ref.EYE_Z
    width = torch.tan(torch.tensor(30. / 180 * np.pi))
    zv = torch.stack((zero_v[..., 0] / z / width, zero_v[..., 1] / z / width, z), dim=2)
    zf = zv[0][torch.zeros(tp.shape[0], 3, dtype=torch.long)]
    return torch.stack([zf, zf, tp, zf]).contiguous()


def test_teapot_batch_with_degenerate_meshes(cuda):
    g = np.load(os.path.join(GOLD, "teapot.npz"))
    fim = compare_with_gpu_ref("teapot_batch", teapot_batch_faces().to(cuda), 256)
    sil = np.unpackbits(g["silhouette"]).reshape(256, 256).astype(bool)
    mine = (fim[2].flip(0) >= 0).cpu().numpy()
    assert (mine != sil).sum() == 0                      # test_rasterize_silhouettes.py:16-35
    assert int((fim[[0, 1, 3]] >= 0).sum()) == 0


def random_soup(B, F, seed):
    g = torch.Generator().manual_seed(seed)
    c = torch.rand(B, F, 1, 2, generator=g) * 2.4 - 1.2
    size = torch.rand(B, F, 1, 1, generator=g) ** 3 * 0.8 + 0.002
    xy = c + (torch.rand(B, F, 3, 2, generator=g) - 0.5) * size
    z = 1.0 + torch.rand(B, F, 3, 1, generator=g) * 3
    faces = torch.cat([xy, z], dim=-1)
    faces[:, 1::7] = faces[:, 0::7][:, :faces[:, 1::7].shape[1]]          # exact duplicates -> depth ties
    faces[:, 5::11, :, 2] = 2.0                                           # coplanar constant depth -> many ties
    faces[:, 3::50, 1] = faces[:, 3::50, 0]                               # two identical vertices (zero area)
    faces[:, 4::53] = faces[:, 4::53, :1]                                 # all three identical
    faces[:, 9::61, :, 0] = faces[:, 9::61, :1, 0]                        # vertical collinear
    faces[0, 7::97, 0, 2] = 0.05                                          # vertices nearer than `near`
    faces[0, 8::89, :, :2] *= 30                                          # huge triangles
    return faces.float().contiguous()


def test_random_triangle_soup_bit_exact(cuda):
    for seed, size in ((1, 128), (2, 256), (3, 96)):
        compare_with_gpu_ref("soup_seed%d" % seed, random_soup(2, 3000, seed).to(cuda), size)


def big_faces():
    g = torch.Generator().manual_seed(11)
    B, F = 2, 1500
    c = torch.rand(B, F, 1, 2, generator=g) * 1.6 - 0.8
    size = 0.2 + torch.rand(B, F, 1, 1, generator=g) * 1.2                 # 25..180 px wide at 256^2
    xy = c + (torch.rand(B, F, 3, 2, generator=g) - 0.5) * size
    z = 1.0 + torch.rand(B, F, 3, 1, generator=g) * 3
    return torch.cat([xy, z], dim=-1).float().contiguous()


def test_big_faces_bit_exact_and_grid_wide(cuda):
    """Many faces covering thousands of pixels each (boxes > kBigBox go to the grid-wide scan instead of one warp): bit-exact
    against the reference kernels, and not a straggler."""
    faces = big_faces().to(cuda)
    compare_with_gpu_ref("big_faces", faces, 256)
    for _ in range(3):
        run_mine(faces, 256, want_inv=False)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        run_mine(faces, 256, want_inv=False)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    print("3000 large faces (avg box ~10^4 px) @256^2: %.3f ms" % ms)
    assert ms < 5.0


# the inputs (CPU faces) and image sizes the bit-exact tests above compare on
REF_FACES = {"sphere_b3_seed1234": lambda: sphere_faces(3, 1234, "cpu")[0], "sphere_b2_seed77": lambda: sphere_faces(2, 77, "cpu")[0],
             "teapot_batch": teapot_batch_faces, "big_faces": big_faces,
             **{"soup_seed%d" % s: (lambda s=s: random_soup(2, 3000, s)) for s in (1, 2, 3)}}
REF_CASES = [("sphere_b3_seed1234", 256), ("sphere_b3_seed1234", 64), ("sphere_b2_seed77", 512), ("teapot_batch", 256),
             ("soup_seed1", 128), ("soup_seed2", 256), ("soup_seed3", 96), ("big_faces", 256)]


def test_flip_rows_matches_torch_flip(cuda):
    faces, _, _, _ = sphere_faces(2, 5, cuda)
    a = run_mine(faces, 256, flip=False, want_inv=False)
    b = run_mine(faces, 256, flip=True, want_inv=False)
    assert torch.equal(a[0].flip(1), b[0]) and torch.equal(a[1].flip(1), b[1]) and torch.equal(a[2].flip(1), b[2])


def test_raster_matches_c_oracle(cuda):
    faces, _, _, _ = sphere_faces(2, 99, cuda)
    fim, wim, depth, finv = run_mine(faces, 256)
    ofim, owim, odepth, ofinv = raster.forward_face_index_map_cpu(faces.cpu().numpy(), 256)
    assert int((fim.cpu().numpy() != ofim).sum()) == 0
    assert np.array_equal(finv.cpu().numpy().view(np.int32), ofinv.view(np.int32))
    assert np.abs(wim.cpu().numpy() - owim).max() == 0
    assert np.abs(depth.cpu().numpy() - odepth).max() == 0


@pytest.mark.parametrize("align_corners", [False, True])
def test_correspond_matches_oracle(cuda, align_corners):
    """lwb_correspond vs the restated torch glue (models/imitator.py:251-260)."""
    v, f = S.uv_sphere()
    cam, verts = S.synthetic_frames(3, seed=42, base_verts=v)
    tabs = S.synthetic_tables()
    src_img = S.synthetic_source(256)
    f2v_src, _, _ = nmr_ref.render_fim_wim(cam[:1], verts[:1], f, 256)
    p2v = nmr_ref.src_p2verts(f2v_src)
    ref = nmr_ref.correspond(cam[1:], verts[1:], f, tabs["map_fn"], p2v, src_img, 256, align_corners)
    out = K.correspond(cam[1:].to(cuda).contiguous(), verts[1:].to(cuda).contiguous(), f.to(cuda), 256,
                       tabs["map_fn"].to(cuda), p2v.to(cuda).contiguous(), src_img.to(cuda),
                       align_corners=align_corners, want_f2verts=True)
    torch.cuda.synchronize()
    assert torch.equal(out["f2verts"].cpu(), ref["f2verts"])
    assert int((out["fim"].cpu() != ref["fim"]).sum()) == 0
    for k, tol in (("wim", 1e-6), ("T", 1e-5), ("cond", 0.0), ("tsf_img", 2e-5), ("tsf_inputs", 2e-5)):
        d = (out[k].cpu() - ref[k]).abs().max().item()
        print(k, d)
        assert d <= tol, (k, d)


def test_correspond_source_pass_matches_render_fim_wim(cuda):
    """personalize-side use (models/imitator.py:100-107): f2verts / fim / wim only."""
    v, f = S.uv_sphere()
    cam, verts = S.synthetic_frames(1, seed=8, base_verts=v)
    tabs = S.synthetic_tables()
    f2v, fim, wim = nmr_ref.render_fim_wim(cam, verts, f, 256)
    p2v = nmr_ref.src_p2verts(f2v)
    out = K.correspond(cam.to(cuda), verts.to(cuda), f.to(cuda), 256, tabs["map_fn"].to(cuda), p2v.to(cuda).contiguous(),
                       None, want_f2verts=True)
    assert torch.equal(out["fim"].cpu(), fim)
    assert (out["wim"].cpu() - wim).abs().max().item() <= 1e-6
    # self-correspondence: T of the source onto itself reproduces pixel centres (sanity of cal_bc_transform)
    T = out["T"].cpu()
    cov = fim[0] >= 0
    ys, xs = torch.meshgrid(torch.arange(256), torch.arange(256), indexing="ij")
    gx = (2.0 * xs + 1 - 256) / 256
    assert (T[0][cov][:, 0] - gx[cov]).abs().max().item() < 2e-2


def test_self_correspondence_is_the_identity_warp(cuda):
    """Round trip through lwb_correspond at the full 256^2 / 512^2 sizes: frame 0 corresponded with itself gives
    T = pixel centres and tsf_img = src_img on covered pixels, -2 / 0 elsewhere (no oracle involved).  The image identity
    holds in the align_corners=False sampling convention (pixel centres are the rasterizer's sample points); the default
    torch-1.2 convention shifts the sample by <= half a pixel, exactly as the reference did."""
    v, f = S.uv_sphere()
    tabs = S.synthetic_tables()
    for size in (256, 512):
        cam, verts = S.synthetic_frames(2, seed=8, base_verts=v)
        ys, xs = torch.meshgrid(torch.arange(size, dtype=torch.float32), torch.arange(size, dtype=torch.float32), indexing="ij")
        gx, gy = (2 * xs + 1 - size) / size, (2 * ys + 1 - size) / size
        src = torch.stack([torch.sin(3 * gx) * torch.cos(2 * gy), gx * gy, torch.cos(4 * gx + gy)])[None]
        from impersonator_b200.nmr import SMPLRenderer
        r = SMPLRenderer(image_size=size, faces=f.numpy(), map_fn=tabs["map_fn"]).to(cuda)
        src_pass = r.correspond(cam[:1].to(cuda), verts[:1].to(cuda), None, None, want_f2verts=True)     # personalize side
        p2v = src_pass["f2verts"][:, :, :, 0:2].clone()
        p2v[:, :, :, 1] *= -1                                                  # models/imitator.py:105-107
        out = r.correspond(cam.to(cuda), verts.to(cuda), p2v.contiguous(), src.to(cuda), align_corners=False)
        torch.cuda.synchronize()
        fim, T, img = out["fim"][0].cpu(), out["T"][0].cpu(), out["tsf_img"][0].cpu()
        cov = fim >= 0
        assert 0.05 < cov.float().mean() < 0.6
        # a quarter of a pixel at most (worst on sliver faces, where the reference's clamped barycentrics are least exact)
        assert (T[..., 0] - gx)[cov].abs().max() < 0.5 / size and (T[..., 1] - gy)[cov].abs().max() < 0.5 / size
        assert (T[..., 0] - gx)[cov].abs().mean() < 2e-5
        assert torch.all(T[~cov] == -2) and torch.all(img[:, ~cov] == 0)
        assert (img - src[0])[:, cov].abs().max() < 5e-3
