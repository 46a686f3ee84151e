"""numpy model of the device APNG writer (include/rtclj_b200.h, rtclj_ctx_encode_apng; DESIGN.md section 4.14).

Built from png_model, frame by frame: every frame's data chunks are those of png_model.encode on that frame (its
filtered stream, its segments from png_model.encode_segment, its Adler-32), as IDATs in frame 0 and as fdATs with a
sequence number after it; an acTL after IHDR, an fcTL before every frame, IEND at the end."""
from __future__ import annotations

import struct
import zlib

import numpy as np

import png_model as P


def frame_chunks(rgb8: np.ndarray) -> list:
    """The data of one frame's IDAT chunks in its own PNG: the zlib header, one per segment, the Adler-32."""
    F, _ = P.filter_rows(np.ascontiguousarray(rgb8, dtype=np.uint8))
    N = len(F)
    out = [b"\x78\x01"]
    for a in range(0, N, P.SEG):
        out.append(P.encode_segment(F[a:a + P.SEG], a + P.SEG >= N)[0])
    out.append(struct.pack(">I", zlib.adler32(F.tobytes()) & 0xFFFFFFFF))
    return out


def fctl(seq: int, W: int, H: int, delay) -> bytes:
    return P._chunk(b"fcTL", struct.pack(">IIIIIHHBB", seq, W, H, 0, 0, delay[0], delay[1], 0, 0))


def encode(frames: np.ndarray, delay=(1, 30), plays: int = 0) -> bytes:
    frames = np.ascontiguousarray(frames, dtype=np.uint8)
    K, H, W, _ = frames.shape
    return assemble([frame_chunks(frames[f]) for f in range(K)], W, H, delay, plays)


def assemble(per_frame: list, W: int, H: int, delay=(1, 30), plays: int = 0) -> bytes:
    """The file from every frame's frame_chunks."""
    K = len(per_frame)
    out = [P.SIG, P._chunk(b"IHDR", struct.pack(">IIBBBBB", W, H, 8, 2, 0, 0, 0)),
           P._chunk(b"acTL", struct.pack(">II", K, plays))]
    seq = 0
    for f in range(K):
        out.append(fctl(seq, W, H, delay))
        seq += 1
        for data in per_frame[f]:
            if f == 0:
                out.append(P._chunk(b"IDAT", data))
            else:
                out.append(P._chunk(b"fdAT", struct.pack(">I", seq) + data))
                seq += 1
    out.append(P._chunk(b"IEND", b""))
    return b"".join(out)


def nseg(W: int, H: int) -> int:
    return -(-(H * (1 + 3 * W)) // P.SEG)


def stored_bound(W: int, H: int, K: int) -> int:
    """The sizing call's answer, the header's closed formula: B + 58 + (K - 1)(B + 4 nseg + 1)."""
    B = P.stored_bound(W, H)
    return B + 58 + (K - 1) * (B + 4 * nseg(W, H) + 1)


def stored_size(W: int, H: int, K: int) -> int:
    """The file's size when every segment of every frame is stored, counted chunk by chunk."""
    N = H * (1 + 3 * W)
    data = sum(P.stored_bytes(min(P.SEG, N - a)) for a in range(0, N, P.SEG))
    ns = nseg(W, H)
    frame0 = 38 + 14 + 12 * ns + data + 16
    later = 38 + 18 + 16 * ns + data + 20
    return 33 + 20 + frame0 + (K - 1) * later + 12


# ---- the inputs the CPU and GPU tests share

def cpu_cases() -> dict:
    """name -> (frames [K,H,W,3], delay, plays)."""
    rng = np.random.default_rng(21)
    cases = P.cpu_cases()
    main = cases["scene_main"]
    shifted = np.stack([np.roll(main, 7 * k, axis=1) for k in range(3)])
    noise = rng.integers(0, 256, (40, 50, 3), dtype=np.uint8)
    return {
        "K1_main": (main[None], (1, 30), 0),
        "K3_main_shifted": (shifted, (1, 30), 0),
        "1x1_K4": (rng.integers(0, 256, (4, 1, 1, 3), dtype=np.uint8), (1, 30), 0),
        # H (1 + 3W) = 65536 and 65537: the filtered stream ends on a segment boundary, or one byte past it
        "F_1x65536_K3": ((rng.integers(0, 2, (3, 256, 85, 3)) * 40).astype(np.uint8), (1, 30), 0),
        "F_3x65536_plus_1_K2": (np.stack([(np.arange(65536 * 3) % 251).astype(np.uint8).reshape(1, 65536, 3),
                                  (np.arange(65536 * 3) % 13).astype(np.uint8).reshape(1, 65536, 3)]), (1, 30), 0),
        "noise_and_constant": (np.stack([noise, np.full_like(noise, 77), rng.integers(0, 256, noise.shape, dtype=np.uint8),
                                         np.full_like(noise, 3)]), (1, 30), 0),
        "delay_0_0": (shifted[:2], (0, 0), 3),
        "delay_65535": (shifted[:2], (65535, 65535), 65535),
        "wide_K2": (np.stack([cases["wide_30000"], cases["wide_30000"][:, ::-1]]), (2, 25), 1),
    }
