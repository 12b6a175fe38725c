"""Blender-synthetic scene reader with the reference's conventions (dataloader.py:10-56):
transforms_{phase}.json, frames[i].file_path + ".png", image resized to img_size x img_size and
converted to RGB float32 / 255, pose = transform_matrix, focal_length = 0.5 / tan(0.5 *
camera_angle_x) in normalised pixel units.  Host-side data format only; no kernels.
white_background=True loads the RGBA images and composites them onto white, rgb * a + (1 - a), the NeRF paper's setup
for these scenes (train and render with background=(1, 1, 1) to match)."""
import json
import os

import numpy as np


class BlenderScene:
    def __init__(self, root_dir, img_size=64, phase="train", white_background=False):
        self.root_dir, self.img_size, self.phase = root_dir, int(img_size), phase
        self.white_background = bool(white_background)
        with open(os.path.join(root_dir, "transforms_%s.json" % phase)) as fh:
            tr = json.load(fh)
        self.camera_angle_x = float(tr["camera_angle_x"])
        self.focal_length = 0.5 / np.tan(0.5 * self.camera_angle_x)
        self.frames = [(os.path.join(root_dir, f["file_path"] + ".png"), np.array(f["transform_matrix"], np.float64))
                       for f in tr["frames"]]

    def __len__(self):
        return len(self.frames)

    @property
    def normalized_K(self):
        """Intrinsics in normalised [0,1] pixel coordinates as train_nerf.py builds them from the
        focal length (principal point at the image centre)."""
        f = self.focal_length
        return np.array([[f, 0.0, 0.5], [0.0, f, 0.5], [0.0, 0.0, 1.0]])

    def __getitem__(self, idx):
        from PIL import Image
        path, pose = self.frames[idx]
        if self.white_background:
            rgba = np.asarray(Image.open(path).resize((self.img_size, self.img_size)).convert("RGBA"), dtype=np.float32) / 255.0
            image = rgba[..., :3] * rgba[..., 3:] + (1.0 - rgba[..., 3:])
        else:
            img = Image.open(path).resize((self.img_size, self.img_size)).convert("RGB")
            image = np.asarray(img, dtype=np.float32) / 255.0
        return {"image": image, "pose": pose, "focal_length": self.focal_length}
