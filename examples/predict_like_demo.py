"""The reference's `CognitiveAimInference.predict` flow (reference demo.py:300-405) on the B200 path.

    python examples/predict_like_demo.py IMAGE.jpg [--instruction center] [--image-size 224] [--overlay out.npy]
    python examples/predict_like_demo.py --image-dir DIR [--instruction center] [--image-size 224]
    python examples/predict_like_demo.py IMAGE.jpg --interactive < instructions.txt

What demo.py does per image and what runs here instead:
    Image.open(path).convert('RGB')                    -> nvJPEG decode on the GPU              (model.preprocess_jpeg)
    Resize((S, S)) / ToTensor / Normalize              -> exact-Pillow resample + normalise     (same call)
    default EXIF 50 mm, f/2.8, ISO 100, camera 0       -> the same defaults                    (demo.py:271-277)
    delattr(model, '_last_attention_weights')          -> the same                              (demo.py:334-335)
    model.forward_with_guidance(x, exif, instruction)  -> the same call                         (demo.py:344-346)
    numpy / scipy heat-map overlay                     -> model.focus_map((h, w)) on the GPU    (demo.py:530-563)
`--instruction all` (demo_results/: one photograph under all nine instructions) runs ONE instruction sweep
(`Predictor.predict_all`, model.forward_with_guidance_sweep) instead of nine calls, with the same printed results.
`--image-dir` (demo.py:406-432 `predict_batch`, one call per file there) decodes every JPEG of the folder in one batched
nvJPEG call and runs the photographs, whatever their sizes, through ONE forward (`Predictor.predict_batch`).
`--interactive` encodes the photograph once (`Predictor.encode`, model.encode: decode, backbone, focal stream) and then
reads instructions from stdin, one per line, printing for each the line `predict` prints (`Predictor.predict_scene`,
model.guide); the results equal successive `predict` calls on the same photograph.
Weights: random init (seed 0, the reference's own construction order) unless --checkpoint names a reference state_dict.
"""
from __future__ import annotations

import argparse
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from cognitive_aim_depth_estimation_b200 import ops  # noqa: E402
from cognitive_aim_depth_estimation_b200.model import create_model  # noqa: E402

INSTRUCTIONS = ["center", "left", "right", "top", "bottom", "top-left", "top-right", "bottom-left", "bottom-right"]
CONFIG = {"cognitive_modules": ["ambient_stream", "iterative_focal_stream", "exif_prior_database"],  # demo.py:46-52
          "model": {"exif_config": {"num_cameras": 71}}}


class Predictor:
    """Counterpart of demo.py's CognitiveAimInference: one model on one GPU, `predict(jpeg bytes, instruction)`."""

    def __init__(self, state_dict=None, device="cuda:0", image_size=224):
        self.device, self.image_size = torch.device(device), image_size
        self.model = create_model(CONFIG, {"num_cameras": 71}, device=self.device)  # demo.py:56-68
        self.model.input_size = image_size  # lists of photographs are resized to it
        if state_dict is not None:
            self.model.load_state_dict(state_dict, strict=False)                    # demo.py:89-150
        self.model.eval()

    def default_exif(self, n=1):
        """demo.py:271-277: no EXIF in the file -> 50 mm, f/2.8, ISO 100, camera index 0."""
        f = dict(device=self.device, dtype=torch.float32)
        return {"focal_length": torch.full((n,), 50.0, **f), "aperture": torch.full((n,), 2.8, **f),
                "iso": torch.full((n,), 100.0, **f), "camera_idx": torch.zeros(n, device=self.device, dtype=torch.long)}

    @torch.no_grad()
    def predict(self, jpeg_bytes: bytes, instruction=None, exif=None, overlay_size=None):
        """-> (depth, confidence, metadata) like demo.py:300-405; metadata carries the attention arg-max cell and, when
        `overlay_size` = (h, w) is given, the overlay heat map demo.py would paint."""
        x = self.model.preprocess_jpeg([jpeg_bytes], self.image_size)
        exif = exif if exif is not None else self.default_exif(1)
        if hasattr(self.model, "_last_attention_weights"):
            delattr(self.model, "_last_attention_weights")
        if instruction is not None:
            depth, conf = self.model.forward_with_guidance(x, exif, instruction)
        else:
            depth, conf = self.model(x, exif)
        att = self.model.get_attention_weights()
        g = self.image_size // 14
        cell = int(att[0].argmax())
        meta = {"processed_size": (self.image_size, self.image_size), "instruction": instruction,
                "attention_cell": (cell // g, cell % g),
                "model_status": {"ambient": self.model.use_ambient, "focal": self.model.use_focal, "exif": self.model.use_exif}}
        if overlay_size is not None:
            meta["overlay"] = self.model.focus_map(overlay_size)[0]
        return float(depth.squeeze()), float(conf.squeeze()), meta

    @torch.no_grad()
    def predict_all(self, jpeg_bytes: bytes, instructions, exif=None, overlay_size=None):
        """`[predict(jpeg_bytes, ins, exif, overlay_size) for ins in instructions]` — demo_results/' one photograph under
        every instruction — as ONE instruction sweep: the image is decoded and run through the backbone and the focal
        stream once.  Same results, bit for bit, and the same model state afterwards."""
        x = self.model.preprocess_jpeg([jpeg_bytes], self.image_size)
        exif = exif if exif is not None else self.default_exif(1)
        if hasattr(self.model, "_last_attention_weights"):
            delattr(self.model, "_last_attention_weights")
        depth, conf, heat = self.model.forward_with_guidance_sweep(x, exif, list(instructions), return_attention=True)
        g = self.image_size // 14
        out = []
        for k, ins in enumerate(instructions):
            cell = int(heat[k, 0].argmax())
            meta = {"processed_size": (self.image_size, self.image_size), "instruction": ins,
                    "attention_cell": (cell // g, cell % g),
                    "model_status": {"ambient": self.model.use_ambient, "focal": self.model.use_focal,
                                     "exif": self.model.use_exif}}
            if overlay_size is not None:
                meta["overlay"] = self.model.focus_map(overlay_size, attention=heat[k])[0]
            out.append((float(depth[k].squeeze()), float(conf[k].squeeze()), meta))
        return out

    @torch.no_grad()
    def predict_batch(self, jpeg_files, instruction=None, exifs=None):
        """demo.py:406-432 `predict_batch`: a list of JPEG files (bytes) of any sizes -> [(depth, confidence, metadata)]
        per file.  `instruction`: one for every file, or a list of one per file.  The files are decoded in one batched
        nvJPEG call and go through ONE forward as a list of photographs (resized to image_size on the GPU, bit-exact
        Pillow).  The reference calls `predict` per file, so each file there gets its own per-call random projection
        (src/model.py:1421); here the batch shares one, like any batched call."""
        imgs = self.model_images(jpeg_files)
        n = len(imgs)
        exif = exifs if exifs is not None else self.default_exif(n)
        if hasattr(self.model, "_last_attention_weights"):
            delattr(self.model, "_last_attention_weights")
        if instruction is not None:
            depth, conf = self.model.forward_with_guidance(imgs, exif, instruction)
        else:
            depth, conf = self.model(imgs, exif)
        heat = self.model.get_attention_weights()
        g = self.image_size // 14
        out = []
        for i in range(n):
            cell = int(heat[i].argmax())
            ins = instruction[i] if isinstance(instruction, (list, tuple)) else instruction
            meta = {"processed_size": (self.image_size, self.image_size), "instruction": ins,
                    "attention_cell": (cell // g, cell % g),
                    "model_status": {"ambient": self.model.use_ambient, "focal": self.model.use_focal,
                                     "exif": self.model.use_exif}}
            out.append((float(depth[i].squeeze()), float(conf[i].squeeze()), meta))
        return out

    @torch.no_grad()
    def encode(self, jpeg_bytes: bytes, exif=None):
        """Decode and encode one photograph for any number of later instructions (`predict_scene`)."""
        x = self.model.preprocess_jpeg([jpeg_bytes], self.image_size)
        return self.model.encode(x, exif if exif is not None else self.default_exif(1))

    @torch.no_grad()
    def predict_scene(self, scene, instruction, overlay_size=None):
        """`predict(jpeg_bytes, instruction, exif, overlay_size)` for the photograph `scene` was encoded from, bit for bit
        (the backbone and the focal stream are not run again)."""
        depth, conf, heat = self.model.guide(scene, instruction, return_attention=True)
        g = self.image_size // 14
        cell = int(heat[0].argmax())
        meta = {"processed_size": (self.image_size, self.image_size), "instruction": instruction,
                "attention_cell": (cell // g, cell % g),
                "model_status": {"ambient": self.model.use_ambient, "focal": self.model.use_focal, "exif": self.model.use_exif}}
        if overlay_size is not None:
            meta["overlay"] = self.model.focus_map(overlay_size, attention=heat)[0]
        return float(depth.squeeze()), float(conf.squeeze()), meta

    def model_images(self, jpeg_files):
        """JPEG files (bytes) -> list of decoded uint8 [H_i, W_i, 3] CUDA tensors (one nvjpegDecodeBatched call)."""
        with torch.cuda.device(self.device):
            return ops.jpeg_decode_batch(list(jpeg_files), self.device)


def result_line(ins, depth, conf, meta):
    return f"{str(ins):13s} depth {depth:.4f}  confidence {conf:.4f}  attention cell {meta['attention_cell']}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("image", nargs="?")
    ap.add_argument("--image-dir", default=None, help="predict every .jpg / .jpeg of DIR in one batched call")
    ap.add_argument("--instruction", default=None, help="one of %s, or 'all'" % ", ".join(INSTRUCTIONS))
    ap.add_argument("--image-size", type=int, default=224)  # configs/experiment_B.yaml:87
    ap.add_argument("--checkpoint", default=None)
    ap.add_argument("--overlay", default=None, help="write the overlay heat map of the last instruction as .npy")
    ap.add_argument("--interactive", action="store_true",
                    help="encode IMAGE once, then read instructions from stdin, one per line")
    args = ap.parse_args()
    if (args.image is None) == (args.image_dir is None):
        ap.error("give IMAGE or --image-dir DIR")
    # without a checkpoint: the reference's own random init (demo.py:148-150 "continuing with randomly initialized
    # weights") — create_model draws it from the global generator exactly like the reference's constructor
    sd = torch.load(args.checkpoint, map_location="cpu") if args.checkpoint else None
    torch.manual_seed(0)
    p = Predictor(sd, image_size=args.image_size)
    if args.image_dir:
        if args.instruction == "all" or args.overlay:
            ap.error("--image-dir takes one instruction and no --overlay")
        names = sorted(f for f in os.listdir(args.image_dir) if f.lower().endswith((".jpg", ".jpeg")))
        if not names:
            ap.error(f"no JPEG files in {args.image_dir}")
        files = [open(os.path.join(args.image_dir, f), "rb").read() for f in names]
        for depth, conf, meta in p.predict_batch(files, args.instruction):  # one line per file, sorted by name
            print(result_line(args.instruction, depth, conf, meta))
        return
    data = open(args.image, "rb").read()
    if args.interactive:
        if args.instruction or args.overlay:
            ap.error("--interactive reads its instructions from stdin and takes no --overlay")
        scene = p.encode(data)
        for line in sys.stdin:
            ins = line.strip()
            if ins:
                print(result_line(ins, *p.predict_scene(scene, ins)), flush=True)
        return
    overlay_size = (480, 640) if args.overlay else None
    if args.instruction == "all":  # every instruction in one sweep (backbone and focal pass once)
        results = zip(INSTRUCTIONS, p.predict_all(data, INSTRUCTIONS, overlay_size=overlay_size))
    else:
        results = [(args.instruction, p.predict(data, args.instruction, overlay_size=overlay_size))]
    for ins, (depth, conf, meta) in results:
        print(result_line(ins, depth, conf, meta))
    if args.overlay:
        import numpy as np
        np.save(args.overlay, meta["overlay"].cpu().numpy())


if __name__ == "__main__":
    main()
