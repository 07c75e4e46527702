"""Host-side piece preparation for the puzzle grid (SURVEY 8a rows a1-a3): crop geometry, LAB->RGB, resize, normalise.

The reference redoes this work 2*N*(N-1) times inside DataLoader workers (data/datasets/pieces_dataset.py:34-56); it
is deterministic per piece, so here it runs once per piece (O(N)) with the same cv2 / PIL / torchvision calls and the
result is uploaded once. Integer geometry is bit-exact with paikin_tal_solver/puzzle_importer.py:182-232, :430-446.
"""
import math

import numpy as np
import torch


def grid_geometry(img_h, img_w, piece_width):
    """(numb_rows, numb_cols, top, left): floor grid, centred (puzzle_importer.py:196-213)."""
    numb_cols = int(math.floor(img_w / piece_width))
    numb_rows = int(math.floor(img_h / piece_width))
    if numb_cols == 0 or numb_rows == 0:
        raise ValueError("Image size is too small for the image.  Check your setup")
    top = (img_h - numb_rows * piece_width) // 2
    left = (img_w - numb_cols * piece_width) // 2
    return numb_rows, numb_cols, top, left


def erosion_crop(piece_width, erosion):
    """(eroded side, offset): ceil(w*(1-e)) and Python-round centre crop (puzzle_importer.py:224, :430-446)."""
    side = math.ceil(piece_width * (1 - erosion))
    side = side if side < piece_width else piece_width
    off = int(round((piece_width - side) / 2.0))
    return side, off


def make_pieces_lab(img_bgr, piece_width, erosion=0.0):
    """BGR uint8 image -> (list of eroded LAB uint8 pieces in row-major piece-id order, (rows, cols)).
    Mirrors Puzzle._load_puzzle_image + make_pieces (puzzle_importer.py:136-156, :182-232)."""
    import cv2
    lab = cv2.cvtColor(img_bgr, cv2.COLOR_BGR2LAB)
    h, w = img_bgr.shape[:2]
    rows, cols, top, left = grid_geometry(h, w, piece_width)
    side, off = erosion_crop(piece_width, erosion)
    pieces = []
    for r in range(rows):
        for c in range(cols):
            y0 = top + r * piece_width + off
            x0 = left + c * piece_width + off
            pieces.append(lab[y0:y0 + side, x0:x0 + side, :])
    return pieces, (rows, cols)


def piece_to_tensor(lab_piece, img_size):
    """LAB uint8 [s,s,3] -> fp32 [3,S,S] in [-1,1]; same calls as PiecesDataset.__getitem__ + TwoImgSyncEval
    (pieces_dataset.py:35-46, data/transforms.py:14-18)."""
    import cv2
    from torchvision import transforms
    rgb = cv2.cvtColor(np.ascontiguousarray(lab_piece), cv2.COLOR_LAB2RGB)
    pil = transforms.ToPILImage()(rgb)
    norm = transforms.Compose([
        transforms.Resize(img_size),
        transforms.ToTensor(),
        transforms.Normalize((0.5, 0.5, 0.5), (0.5, 0.5, 0.5)),
    ])
    return norm(pil)


def pieces_to_batch(lab_pieces, img_size):
    """[N,3,S,S] fp32 (CPU); upload once with .cuda()."""
    return torch.stack([piece_to_tensor(p, img_size) for p in lab_pieces], dim=0)


def fragment_to_tensor(pil_image, img_size=512):
    """Hisfrag20 test-time prep (SURVEY 8a row a6): CenterCrop(img_size) -> ToTensor -> Normalize(.5, .5), the
    transform of hisfrag.py:89-93 applied by HisFrag20Test.__getitem__ (hisfrag_dataset.py:181-191)."""
    from torchvision import transforms
    tf = transforms.Compose([
        transforms.CenterCrop(img_size),
        transforms.ToTensor(),
        transforms.Normalize((0.5, 0.5, 0.5), (0.5, 0.5, 0.5)),
    ])
    return tf(pil_image)


def prepare_pieces_device(img_bgr, piece_width, erosion, img_size, device='cuda'):
    """BGR uint8 image [H, W, 3] -> (CUDA fp32 [N, 3, S, S] in piece-id order, (rows, cols)).

    The device replacement of ``make_pieces_lab`` + ``pieces_to_batch`` (SURVEY 8f row 2): the image is converted to
    LAB once on the host as Puzzle._load_puzzle_image does (puzzle_importer.py:136-156) and uploaded as bytes; crop,
    Lab -> sRGB, the PIL bilinear resize and the normalisation run in one kernel (C-ABI ``vited_prepare_pieces``) and
    give bit-identical floats to the per-piece cv2 / PIL / torchvision calls of pieces_dataset.py:35-46."""
    import ctypes

    import cv2
    from . import _lib
    lab = cv2.cvtColor(np.ascontiguousarray(img_bgr), cv2.COLOR_BGR2LAB)
    h, w = lab.shape[:2]
    rows, cols, _, _ = grid_geometry(h, w, piece_width)
    side, off = erosion_crop(piece_width, erosion)
    dev = torch.device(device)
    with torch.cuda.device(dev):
        lab_d = torch.from_numpy(lab).to(dev)
        out = torch.empty((rows * cols, 3, img_size, img_size), dtype=torch.float32, device=dev)
        n = ctypes.c_int(0)
        stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        _lib.check(_lib.lib.vited_prepare_pieces(ctypes.c_void_p(lab_d.data_ptr()), h, w, piece_width, side, off, img_size,
                                                 ctypes.c_void_p(out.data_ptr()), ctypes.byref(n), stream),
                   'vited_prepare_pieces')
    assert n.value == rows * cols
    return out, (rows, cols)


def center_crop_u8(img, size):
    """torchvision CenterCrop(size) on an [H, W, 3] uint8 array (transforms/functional.py center_crop): zero padding
    when the image is smaller than the crop, then offsets ``int(round((dim - size) / 2.0))`` (Python banker's round)."""
    img = np.asarray(img)
    h, w = img.shape[:2]
    if size > w or size > h:
        pl = (size - w) // 2 if size > w else 0
        pt = (size - h) // 2 if size > h else 0
        pr = (size - w + 1) // 2 if size > w else 0
        pb = (size - h + 1) // 2 if size > h else 0
        img = np.pad(img, ((pt, pb), (pl, pr), (0, 0)))
        h, w = img.shape[:2]
    top = int(round((h - size) / 2.0))
    left = int(round((w - size) / 2.0))
    return img[top:top + size, left:left + size]


def fragments_to_u8_device(images, img_size=512, device='cuda'):
    """List of PIL images / [H, W, 3] uint8 arrays -> CUDA uint8 [N, S, S, 3]: the CenterCrop of the Hisfrag20
    test-time preparation done on the bytes, then one upload. ``model.score_grid`` and ``grid.score_fragments`` take
    this directly and normalise inside the patch embedding: a quarter of the device memory of the fp32 batch that
    ``fragments_to_batch_device`` returns, identical scores."""
    from . import _lib
    crops = np.stack([center_crop_u8(np.asarray(im), img_size) for im in images])
    if crops.dtype != np.uint8 or crops.shape[1:] != (img_size, img_size, 3):
        raise _lib.VitedError(f'fragments_to_u8_device: expected uint8 RGB images, got {crops.dtype} {crops.shape}')
    return torch.from_numpy(np.ascontiguousarray(crops)).to(torch.device(device))


def fragments_to_batch_device(images, img_size=512, device='cuda'):
    """List of PIL images / [H, W, 3] uint8 arrays -> CUDA fp32 [N, 3, S, S]: the Hisfrag20 test-time preparation
    (SURVEY 8a row a6; ``fragment_to_tensor`` is the per-image host version) with the crop done on the bytes and
    ToTensor + Normalize on the device (C-ABI ``vited_normalize_u8``): a quarter of the upload, identical floats."""
    import ctypes

    from . import _lib
    dev = torch.device(device)
    with torch.cuda.device(dev):
        src = fragments_to_u8_device(images, img_size, dev)
        out = torch.empty((src.shape[0], 3, img_size, img_size), dtype=torch.float32, device=dev)
        _lib.check(_lib.lib.vited_normalize_u8(ctypes.c_void_p(src.data_ptr()), src.shape[0], img_size,
                                               ctypes.c_void_p(out.data_ptr()),
                                               ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)),
                   'vited_normalize_u8')
    return out
