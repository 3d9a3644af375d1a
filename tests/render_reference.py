"""Rolling-shutter fisheye frames of a purely rotating camera, rendered from a procedural texture on the
sphere, with the true correspondence of any point.

The camera model is synth's: the gyro track of synth.make_workload (angular_velocity, integrate_gyro,
QuatTrack), its rotation convention (a ray r of a row exposed at time t sees the world direction
conj(q(t + delay)) r conj(q)^-1), its Hero6 lens through pixel_to_ray / ray_to_pixel, and its row timing
ts = frame_ts + readout * (y / height).  The lens is scaled to the image size: fx, cx by width / 2704,
fy, cy by height / 2028, which maps a pixel (x, y) to synth's pixel (x / sx, y / sy).

The texture is 48 seeded sinusoids of the world direction d, 127.5 + 40 sum a_i sin(k_i . d + phi_i) /
sqrt(sum a_i^2 / 2), clipped to [0, 255] and rounded; the wave numbers |k_i| give wavelengths of 15 to 80
pixels at the image's focal length.  A pixel shows the texture at its own centre (integer coordinates),
the convention of the tracker and of cv2's Lucas-Kanade."""
from __future__ import annotations

import importlib

import numpy as np

synth = importlib.import_module("rs-sync_b200.synth")


def lens_for(width, height, readout=synth.READOUT):
    """rssync_lens fields of synth's lens scaled to a width x height image"""
    sx, sy = width / synth.WIDTH, height / synth.HEIGHT
    return (readout, synth.FX * sx, synth.FY * sy, synth.CX * sx, synth.CY * sy, synth.K1, synth.K2, synth.K3, synth.K4)


class Clip:
    """n_images frames starting at frame number first_frame of a fps clip; image j starts its exposure at
    (first_frame + j) / fps seconds and its gyro orientation is the track's at that time + delay"""

    def __init__(self, width, height, n_images, *, first_frame=600, fps=60.0, delay=0.037, readout=synth.READOUT,
                 seed=1, gyro_rate=1000.0):
        self.width, self.height, self.n_images = int(width), int(height), int(n_images)
        self.first_frame, self.fps, self.delay, self.readout = int(first_frame), float(fps), float(delay), float(readout)
        self.sx, self.sy = self.width / synth.WIDTH, self.height / synth.HEIGHT
        t_first = first_frame / fps
        t_last = (first_frame + n_images) / fps + readout
        pad = 1.2 + abs(delay)
        g0 = np.floor((t_first - pad) * gyro_rate) / gyro_rate
        ng = int(np.ceil((t_last + pad - g0) * gyro_rate)) + 1
        tg = g0 + np.arange(ng) / gyro_rate
        self.gyro_rate, self.gyro_t0 = gyro_rate, float(g0)
        self.quats = synth.integrate_gyro(synth.angular_velocity(tg, seed), np.full(ng, 1.0 / gyro_rate))
        self.track = synth.QuatTrack(self.quats, gyro_rate, g0)
        rng = np.random.default_rng([seed, 4242, self.width, self.height])
        fx = synth.FX * self.sx
        lam = rng.uniform(15.0, 80.0, 48)
        direction = rng.normal(size=(48, 3))
        direction /= np.linalg.norm(direction, axis=1, keepdims=True)
        self.k = direction * (2 * np.pi * fx / lam)[:, None]
        self.phase = rng.uniform(0, 2 * np.pi, 48)
        self.amp = rng.uniform(0.5, 1.0, 48)
        self.norm = np.sqrt(np.sum(self.amp ** 2) / 2.0)
        self._rays = None

    # ---- geometry --------------------------------------------------------------------------
    def lens(self):
        return lens_for(self.width, self.height, self.readout)

    def image_ts(self):
        return (self.first_frame + np.arange(self.n_images)) / self.fps

    def frame_ids(self):
        return self.first_frame + np.arange(self.n_images - 1, dtype=np.int64)

    def pixel_to_ray(self, x, y):
        return synth.pixel_to_ray(np.asarray(x, dtype=np.float64) / self.sx, np.asarray(y, dtype=np.float64) / self.sy)

    def ray_to_pixel(self, r):
        x, y = synth.ray_to_pixel(r)
        return x * self.sx, y * self.sy

    def orientation(self, j, y):
        """gyro quaternion of row y of image j"""
        t = self.image_ts()[j] + self.readout * (np.asarray(y, dtype=np.float64) / self.height)
        return self.track(t + self.delay)

    def world(self, j, x, y):
        return synth.quat_rotate(synth.quat_conj(self.orientation(j, y)), self.pixel_to_ray(x, y))

    def true_b(self, j, points, iters=10):
        """the true position in image j + 1 of points (n, 2) of image j: the rolling-shutter fixed point
        (the row fixes the exposure time of the second observation), as synth's generator solves it"""
        p = np.asarray(points, dtype=np.float64).reshape(-1, 2)
        w = self.world(j, p[:, 0], p[:, 1])
        xb, yb = p[:, 0].copy(), p[:, 1].copy()
        for _ in range(iters):
            cam = synth.quat_rotate(self.orientation(j + 1, yb), w)
            xb, yb = self.ray_to_pixel(cam)
        return np.stack([xb, yb], axis=-1)

    # ---- rendering -------------------------------------------------------------------------
    def texture(self, d):
        s = np.zeros(d.shape[:-1])
        for i in range(self.k.shape[0]):
            s += self.amp[i] * np.sin(d @ self.k[i] + self.phase[i])
        return 127.5 + 40.0 * s / self.norm

    def _pixel_rays(self):
        if self._rays is None:
            ys, xs = np.meshgrid(np.arange(self.height, dtype=np.float64), np.arange(self.width, dtype=np.float64),
                                 indexing="ij")
            self._rays = self.pixel_to_ray(xs, ys)
        return self._rays

    def _row_rotations(self, j):
        """(height, 3, 3): the matrices of r -> conj(q) r q for every row of image j"""
        q = synth.quat_conj(self.orientation(j, np.arange(self.height)))
        eye = np.eye(3)
        return np.stack([synth.quat_rotate(q, np.broadcast_to(eye[c], q.shape[:-1] + (3,))) for c in range(3)], axis=-1)

    def render(self, j):
        """image j as a (height, width) uint8 array (numpy)"""
        d = np.einsum("yij,yxj->yxi", self._row_rotations(j), self._pixel_rays())
        return np.clip(np.rint(self.texture(d)), 0, 255).astype(np.uint8)

    def render_torch(self, j, device):
        """image j as a (height, width) uint8 CUDA tensor, the same values as render(j) up to the rounding of
        sin on the device (float64)"""
        import torch
        if not hasattr(self, "_rays_t") or self._rays_t.device != torch.device(device):
            self._rays_t = torch.from_numpy(self._pixel_rays()).to(device)
            self._k_t = torch.from_numpy(self.k).to(device)
            self._ph_t = torch.from_numpy(self.phase).to(device)
            self._amp_t = torch.from_numpy(self.amp).to(device)
        rot = torch.from_numpy(self._row_rotations(j)).to(device)
        out = torch.empty((self.height, self.width), dtype=torch.uint8, device=device)
        step = max(1, (1 << 22) // (self.width * 48))
        for y0 in range(0, self.height, step):
            d = torch.einsum("yij,yxj->yxi", rot[y0:y0 + step], self._rays_t[y0:y0 + step])
            s = (torch.sin(d @ self._k_t.T + self._ph_t) * self._amp_t).sum(-1)
            out[y0:y0 + step] = torch.clamp(torch.round(127.5 + 40.0 * s / self.norm), 0, 255).to(torch.uint8)
        return out

    def render_all(self, device=None):
        if device is None:
            return np.stack([self.render(j) for j in range(self.n_images)])
        import torch
        return torch.stack([self.render_torch(j, device) for j in range(self.n_images)])
