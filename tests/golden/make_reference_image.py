"""Generates tests/golden/cornell256_refstream_4096spp.npz: the Cornell box at 256x256, 4096 spp, depth 50 rendered by
the CPU oracle in its reference-stream mode (MODE_FORWARD_BURN: per-pixel persistent RNG state, dead paths burn the
draws the reference still consumes -- the trajectories of the reference's own render, which tests/test_ref_harness.py
pins to the reference's worklets).  bench.py's image_check and tests/test_gpu_parity.py compare GPU renders against it.

Stored: mean linear radiance per pixel (float16 [256*256, 3], NaN where the reference's sum is NaN-poisoned) as two
independent halves of 2048 spp (so the fixture also carries its own Monte-Carlo noise estimate); rendered in eight
chunks of 512 spp with disjoint per-pixel streams.  float16 keeps the file under 1 MB; its rounding (5e-4 relative,
6e-8 absolute below 6e-5) is far below the Monte-Carlo noise of 2048 spp.
~15 minutes on 8 cores.  usage: python tests/golden/make_reference_image.py"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import oracle as O  # noqa: E402

W, SPP, DEPTH, CHUNK = 256, 4096, 50, 512
O.build()
sc, cam = O.cornell_scene(), O.Camera(W, W)
parts = []
for k in range(SPP // CHUNK):
    # chunk k continues nothing: every chunk is an independent reference-stream render with its own seed offset (the
    # reference seeds pixel i with i; offset k*W*W gives chunk k a disjoint set of per-pixel streams)
    img, st = O.render(sc, cam, CHUNK, DEPTH, mode=O.MODE_FORWARD_BURN, seed_offset=k * W * W)
    parts.append((img[:, :3] / CHUNK).astype(np.float32))
    print("chunk", k, "paths", st.paths, "nan pixels", int(np.isnan(img[:, :3]).any(1).sum()), flush=True)
halves = np.stack(parts).astype(np.float64).reshape(2, SPP // CHUNK // 2, W * W, 3).mean(1).astype(np.float32).astype(np.float16)
np.savez_compressed(os.path.join(ROOT, "tests", "golden", "cornell256_refstream_4096spp.npz"),
                    parts=halves, spp_per_part=SPP // 2, depth=DEPTH, width=W)
