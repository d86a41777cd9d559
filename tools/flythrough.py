#!/usr/bin/env python
"""The reference's render loop with its fly camera, headless: a script of key presses and mouse moves instead of GLFW
events (main.cpp:77-150), one PNG / PPM per frame instead of glfwSwapBuffers.

    python tools/flythrough.py --scene atrium --grid 256 --size 1280x720 --script "W*30 D*10 M(120,0) W*20 S(-10)" --out fly_%04d.png
    python tools/flythrough.py --script "W*3 M(90,0) E*2" --dry-run        # camera path only, no device needed
    python tools/flythrough.py --scene atrium --grid 256 --voxels 2 --out vox_%04d.png   # mip level 2 as cubes instead

Script tokens (each yields one frame; `*n` repeats): W S A D = forward / back / left / right as main.cpp:136-143 binds
them, E Q = the enum's UP / DOWN (Camera.h:16-17; the reference binds no key to them) -- ProcessKeyBoard with
deltaTime = --dt; M(dx,dy) = mouse move in pixels (mouse_callback -> ProcessMouseMovement), S(dy) with an argument =
scroll (scroll_callback -> ProcessMouseScroll, changes the field of view)."""
import argparse
import os
import re
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import vct_b200  # noqa: E402
from vct_b200 import images, renderer, scenes  # noqa: E402

KEYS = {"W": renderer.FORWARD, "S": renderer.BACKWARD, "A": renderer.LEFT, "D": renderer.RIGHT, "E": renderer.UP, "Q": renderer.DOWN}


def parse_script(text):
    """-> list of ("key", direction) / ("mouse", dx, dy) / ("scroll", dy), one entry per frame"""
    out = []
    for tok in text.split():
        m = re.fullmatch(r"([WSADEQM])(?:\(([-\d.]+)(?:,([-\d.]+))?\))?(?:\*(\d+))?", tok)
        if not m:
            raise ValueError(f"bad script token {tok!r}")
        k, a, b, n = m.group(1), m.group(2), m.group(3), int(m.group(4) or 1)
        if k == "M":
            ev = ("mouse", float(a), float(b or 0.0))
        elif k == "S" and a is not None:
            ev = ("scroll", float(a))
        else:
            ev = ("key", KEYS[k])
        out.extend([ev] * n)
    return out


def apply(cam, ev, dt):
    if ev[0] == "key":
        cam.ProcessKeyBoard(ev[1], dt)
    elif ev[0] == "mouse":
        cam.ProcessMouseMovement(ev[1], ev[2])
    else:
        cam.ProcessMouseScroll(ev[1])


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--scene", default="cornell", choices=["cornell", "atrium", "knot"])
    ap.add_argument("--grid", type=int, default=128)
    ap.add_argument("--size", default="1280x720")
    ap.add_argument("--script", default="W*5")
    ap.add_argument("--dt", type=float, default=1.0 / 60.0 * 20, help="deltaTime handed to ProcessKeyBoard per frame (seconds)")
    ap.add_argument("--out", default="fly_%04d.png", help="printf pattern; .png or .ppm")
    ap.add_argument("--dry-run", action="store_true", help="print the camera path and exit (no CUDA device needed)")
    ap.add_argument("--voxels", type=int, default=None, metavar="LEVEL",
                    help="write voxel views of mip LEVEL (the grid drawn as cubes, vct_render_voxels) instead of frames")
    a = ap.parse_args(argv)
    w, h = (int(x) for x in a.size.lower().split("x"))
    sc = {"cornell": scenes.cornell, "atrium": scenes.atrium, "knot": scenes.dynamic_knot}[a.scene]()
    cam = renderer.Camera(sc.camera_pos, sc.yaw, sc.pitch, sc.fov_deg)
    events = parse_script(a.script)
    if a.dry_run:
        for k, ev in enumerate(events):
            apply(cam, ev, a.dt)
            print(f"frame {k}: position {np.round(cam.position, 3).tolist()} yaw {cam.Yaw:.2f} pitch {cam.Pitch:.2f} zoom {cam.Zoom:.1f}")
        return cam
    r = vct_b200.Voxel_Cone_Tracing(w, h, None, device=0, VoxelDimensions=a.grid, camera=cam)
    r.init_voxel_cone_tracing(sc)
    frame = np.empty((h, w, 4), dtype=np.uint8)
    for k, ev in enumerate(events):
        apply(cam, ev, a.dt)
        if a.voxels is None:
            r.Render(frame)                            # reads camera.GetViewMatrix() / Zoom, as Render() does (:161-165)
        else:
            r.RenderVoxels(a.voxels, frame)            # same camera, the pyramid's level instead of the shaded frame
        path = a.out % k
        top_down = np.ascontiguousarray(frame[::-1, :, :3])    # GL rows run bottom-up
        (images.save_pnm if path.endswith((".ppm", ".pgm")) else images.save_png)(top_down, path)
    print(f"{len(events)} {'frames' if a.voxels is None else f'voxel views of level {a.voxels}'} -> {a.out}")
    return cam


if __name__ == "__main__":
    main()
