"""TEST INFRASTRUCTURE ONLY.  Run in the build container (needs /root/reference):

    python -m oracle.make_golden

1. builds the UNMODIFIED reference Videoseal for each card via oracle/ref_import.py,
2. loads the seeded synthetic checkpoint of oracle/restate.py::synth_state_dict into it
   (`load_state_dict(strict=False)` exactly like utils/cfg.py:148-149),
3. checks oracle/restate.py against the reference outputs on seeded inputs (pins the oracle),
4. writes small fixtures to tests/golden/<card>.pt: full logits, strided samples + global
   statistics of the image-sized outputs, so the fixtures stay small.  The samples of the
   six video-mode runs (case D) go to tests/golden/<card>_video_modes.pt so that no
   fixture file exceeds 1 MB.
"""
import math
import os
import sys
import time

import torch
import yaml

from oracle import ref_import, restate

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CARDS = ["videoseal_1.0", "pixelseal", "videoseal_0.0", "chunkyseal"]
SEED = 1234
# per-card case sizes: chunkyseal costs ~3.5 TFLOP per embed+detect frame on the CPU, so its cases are single frames
CASES = {
    "default":    {"A": 2, "B_hw": (384, 480), "C": (10, 320, 288, 2, 4)},
    "chunkyseal": {"A": 1, "B_hw": (288, 320), "C": (5, 272, 304, 1, 4)},
}


def sample(t: torch.Tensor, stride: int = 8) -> torch.Tensor:
    return t[..., ::stride, ::stride].contiguous().clone()


def stats(t: torch.Tensor) -> dict:
    t = t.double()
    return {"mean": t.mean().item(), "absmean": t.abs().mean().item(), "std": t.std().item(),
            "min": t.min().item(), "max": t.max().item()}


def structured_image(h: int, w: int, seed: int = 5) -> torch.Tensor:
    """Deterministic [1,3,h,w] image with natural-image-like statistics for the JND branches the uniform-noise cases never reach:
    near-black and near-white flat regions (background luminance far below / above 127), smooth gradients (zero contrast
    masking), hard edges and fine texture (large Sobel responses).  Procedural on purpose: no reference asset is copied."""
    g = torch.Generator().manual_seed(seed)
    yy, xx = torch.meshgrid(torch.linspace(0, 1, h), torch.linspace(0, 1, w), indexing="ij")
    base = 0.5 + 0.45 * torch.sin(2.3 * math.pi * xx + 0.7) * torch.cos(1.7 * math.pi * yy)
    img = torch.stack([base, 0.5 + 0.45 * torch.sin(3.1 * math.pi * yy), 0.5 + 0.4 * torch.cos(2.0 * math.pi * (xx + yy))])
    img[:, : h // 5, : w // 4] = 0.01                                   # dark flat block
    img[:, -h // 5:, -w // 3:] = 0.99                                   # bright flat block
    disc = ((yy - 0.55) ** 2 + (xx - 0.35) ** 2) < 0.03
    img[:, disc] = torch.tensor([0.95, 0.9, 0.2])[:, None]              # saturated disc with a hard edge
    img[:, h // 2: h // 2 + h // 6, w // 2: w // 2 + w // 5] = (torch.rand(3, h // 6, w // 5, generator=g) > 0.5).float()   # binary texture
    img = img + 0.02 * torch.randn(3, h, w, generator=g)
    return img.clamp(0, 1).unsqueeze(0)


def main(cards=None):
    torch.manual_seed(0)
    torch.set_num_threads(os.cpu_count() or 8)
    for card_name in (cards or CARDS):
        cs = CASES.get(card_name, CASES["default"])
        t0 = time.time()
        ref, cfg = ref_import.build_reference_model(card_name)
        card = yaml.safe_load(open(os.path.join(ref_import.REF_ROOT, "videoseal/cards", card_name + ".yaml")))
        spec = restate.spec_from_card(card)
        sd = restate.synth_state_dict(spec, seed=SEED)
        msg = ref.load_state_dict(sd, strict=False)
        assert not msg.unexpected_keys, msg.unexpected_keys
        missing = [k for k in msg.missing_keys if not k.startswith("attenuation.")]
        assert not missing, missing
        orc = restate.OracleModel(spec, sd)
        out = {"card": card_name, "seed": SEED, "torch": str(torch.__version__), "spec": spec, "cases": {}}

        g = torch.Generator().manual_seed(0)
        # case A: image mode @ processing size, B=2
        imgs = torch.rand(cs["A"], 3, 256, 256, generator=g)
        msgs = torch.randint(0, 2, (cs["A"], spec["nbits"]), generator=g)
        with torch.no_grad():
            r = ref.embed(imgs, msgs, is_video=False)
            d = ref.detect(r["imgs_w"], is_video=False)
            o = orc.embed(imgs, msgs, is_video=False)
            od = orc.detect(o["imgs_w"], is_video=False)
            # raw network seams (embedder.py:151 / extractor.py:154)
            x_e = ref.rgb2yuv(imgs)[:, 0:1] if ref.embedder.yuv else imgs
            delta = ref.embedder(x_e, msgs)
            hm = ref.attenuation.heatmaps(imgs) if ref.attenuation is not None else torch.zeros(cs["A"], 1, 256, 256)
        errs = {
            "imgs_w": (r["imgs_w"] - o["imgs_w"]).abs().max().item(),
            "preds_w": (r["preds_w"] - o["preds_w"]).abs().max().item(),
            "preds": (d["preds"] - od["preds"]).abs().max().item(),
            "delta": (delta - orc.embedder(imgs, msgs)).abs().max().item(),
            "hmaps": (hm - orc.heatmaps(imgs)).abs().max().item() if ref.attenuation is not None else 0.0,
        }
        print(card_name, "A", errs)
        assert errs["imgs_w"] < 1e-5 and errs["preds"] < 1e-4 and errs["delta"] < 1e-4 and errs["hmaps"] < 1e-6, errs
        out["cases"]["img256"] = {
            "gen_seed": 0, "B": cs["A"], "H": 256, "W": 256,
            "imgs_w_s": sample(r["imgs_w"]), "preds_w_s": sample(r["preds_w"]), "delta_s": sample(delta),
            "hmaps_s": sample(hm), "preds": d["preds"].clone(),
            "imgs_w_stats": stats(r["imgs_w"]), "delta_stats": stats(delta),
            "psnr": restate.psnr(r["imgs_w"], imgs), "oracle_vs_ref": errs,
        }

        # case B: image mode, non-square input needing AA-resize, B=1
        g = torch.Generator().manual_seed(1)
        bh, bw = cs["B_hw"]
        imgs = torch.rand(1, 3, bh, bw, generator=g)
        msgs = torch.randint(0, 2, (1, spec["nbits"]), generator=g)
        with torch.no_grad():
            r = ref.embed(imgs, msgs, is_video=False)
            d = ref.detect(r["imgs_w"], is_video=False)
            o = orc.embed(imgs, msgs, is_video=False)
            od = orc.detect(o["imgs_w"], is_video=False)
        errs = {"imgs_w": (r["imgs_w"] - o["imgs_w"]).abs().max().item(),
                "preds_w": (r["preds_w"] - o["preds_w"]).abs().max().item(),
                "preds": (d["preds"] - od["preds"]).abs().max().item()}
        print(card_name, "B", errs)
        assert errs["imgs_w"] < 1e-5 and errs["preds"] < 1e-4, errs
        out["cases"]["img_resized"] = {
            "gen_seed": 1, "B": 1, "H": bh, "W": bw,
            "imgs_w_s": sample(r["imgs_w"]), "preds_w_s": sample(r["preds_w"]), "preds": d["preds"].clone(),
            "imgs_w_stats": stats(r["imgs_w"]), "oracle_vs_ref": errs,
        }

        # case C: video mode, e.g. 10 frames @ 320x288 (ragged tail: not a multiple of step_size),
        # small chunk so the chunk loop runs more than once
        g = torch.Generator().manual_seed(2)
        nf, vh, vw, vchunk, vstep = cs["C"]
        vid = torch.rand(nf, 3, vh, vw, generator=g)
        msgs = torch.randint(0, 2, (1, spec["nbits"]), generator=g)
        ref.chunk_size, orc.chunk_size = vchunk, vchunk
        ref.step_size, orc.step_size = vstep, vstep
        with torch.no_grad():
            r = ref.embed(vid, msgs, is_video=True)
            d = ref.detect(r["imgs_w"], is_video=True)
            o = orc.embed(vid, msgs, is_video=True)
            od = orc.detect(o["imgs_w"], is_video=True)
            em = ref.extract_message(r["imgs_w"])
            oem = orc.extract_message(o["imgs_w"])
        errs = {"imgs_w": (r["imgs_w"] - o["imgs_w"]).abs().max().item(),
                "preds": (d["preds"] - od["preds"]).abs().max().item(),
                "extract_equal": bool((em == oem).all())}
        print(card_name, "C", errs)
        assert errs["imgs_w"] < 1e-5 and errs["preds"] < 1e-4 and errs["extract_equal"], errs
        out["cases"]["vid"] = {
            "gen_seed": 2, "F": nf, "H": vh, "W": vw, "chunk_size": vchunk, "step_size": vstep,
            "imgs_w_s": sample(r["imgs_w"]), "preds": d["preds"].clone(), "extract": em.clone(),
            "imgs_w_stats": stats(r["imgs_w"]), "oracle_vs_ref": errs,
        }
        # case D (cards with an attenuation, cheap ones only): the other video modes, low-resolution attenuation, and every
        # extract_message aggregation (SURVEY 8(f)2: videoseal.py:80-118, wam.py:177-180, videoseal.py:390-428)
        if ref.attenuation is not None and card_name != "chunkyseal":
            g = torch.Generator().manual_seed(3)
            vid = torch.rand(11, 3, 288, 272, generator=g)
            msgs = torch.randint(0, 2, (1, spec["nbits"]), generator=g)
            ref.chunk_size, orc.chunk_size = 2, 2
            ref.step_size, orc.step_size = 4, 4
            dcase = {"gen_seed": 3, "F": 11, "H": 288, "W": 272, "chunk_size": 2, "step_size": 4, "modes": {}}
            for mode in ("alternate", "interpolate", "repeat"):
                for lowres in (False, True):
                    ref.video_mode, orc.video_mode = mode, mode
                    with torch.no_grad():
                        r = ref.embed(vid, msgs, is_video=True, lowres_attenuation=lowres)
                        o = orc.embed(vid, msgs, is_video=True, lowres_attenuation=lowres)
                    e = (r["imgs_w"] - o["imgs_w"]).abs().max().item()
                    print(card_name, "D", mode, "lowres" if lowres else "fullres", e)
                    assert e < 1e-6, (mode, lowres, e)
                    dcase["modes"][f"{mode}/{int(lowres)}"] = {"imgs_w_s": sample(r["imgs_w"]), "imgs_w_stats": stats(r["imgs_w"]), "err": e}
            ref.video_mode, orc.video_mode = "repeat", "repeat"
            with torch.no_grad():
                r = ref.embed(vid, msgs, is_video=True)
                aggs = {}
                for agg in ("avg", "squared_avg", "l1norm_avg", "l2norm_avg"):
                    a_ref = ref.extract_message(r["imgs_w"], aggregation=agg)
                    a_orc = orc.extract_message(r["imgs_w"], aggregation=agg)
                    assert (a_ref == a_orc).all(), agg
                    aggs[agg] = a_ref.clone()
            dcase["aggregations"] = aggs
            # image mode with low-resolution attenuation (wam.py:177-180) and a non-default interpolation (antialias off)
            with torch.no_grad():
                nointerp = {"mode": "bilinear", "align_corners": False, "antialias": False}
                r = ref.embed(vid[:2], msgs.repeat(2, 1), is_video=False, lowres_attenuation=True, interpolation=nointerp)
                o = orc.embed(vid[:2], msgs.repeat(2, 1), is_video=False, lowres_attenuation=True, interpolation=nointerp)
            e = max((r["imgs_w"] - o["imgs_w"]).abs().max().item(), (r["preds_w"] - o["preds_w"]).abs().max().item())
            print(card_name, "D image lowres no-aa", e)
            assert e < 1e-6, e
            dcase["img_lowres_noaa"] = {"imgs_w_s": sample(r["imgs_w"]), "preds_w_s": sample(r["preds_w"]), "err": e}
            out["cases"]["vid_modes"] = dcase
        # case E: structured image (dark / bright flats, gradients, edges, texture), image mode at a non-processing size
        if ref.attenuation is not None and card_name != "chunkyseal":
            imgs = structured_image(352, 416)
            g = torch.Generator().manual_seed(6)
            msgs = torch.randint(0, 2, (1, spec["nbits"]), generator=g)
            with torch.no_grad():
                r = ref.embed(imgs, msgs, is_video=False)
                d = ref.detect(r["imgs_w"], is_video=False)
                o = orc.embed(imgs, msgs, is_video=False)
                od = orc.detect(o["imgs_w"], is_video=False)
                hm = ref.attenuation.heatmaps(imgs)
            errs = {"imgs_w": (r["imgs_w"] - o["imgs_w"]).abs().max().item(), "preds": (d["preds"] - od["preds"]).abs().max().item(),
                    "hmaps": (hm - orc.heatmaps(imgs)).abs().max().item()}
            print(card_name, "E", errs, "hmap range", hm.min().item(), hm.max().item())
            assert errs["imgs_w"] < 1e-6 and errs["preds"] < 1e-5 and errs["hmaps"] < 1e-7, errs
            out["cases"]["structured"] = {"H": 352, "W": 416, "msg_seed": 6, "imgs_w_s": sample(r["imgs_w"], 4), "hmaps_s": sample(hm, 4),
                                          "preds": d["preds"].clone(), "hmaps_stats": stats(hm), "oracle_vs_ref": errs}
        path = os.path.join(ROOT, "tests", "golden", card_name + ".pt")
        if "vid_modes" in out["cases"]:
            modes_path = os.path.join(ROOT, "tests", "golden", card_name + "_video_modes.pt")
            torch.save({"card": card_name, "seed": SEED, "modes": out["cases"]["vid_modes"].pop("modes")}, modes_path)
            print(card_name, "->", modes_path, os.path.getsize(modes_path) // 1024, "KiB")
        torch.save(out, path)
        print(card_name, "->", path, os.path.getsize(path) // 1024, "KiB", f"{time.time()-t0:.1f}s")


if __name__ == "__main__":
    if not ref_import.available():
        sys.exit("needs the reference tree at " + ref_import.REF_ROOT)
    main(sys.argv[1:] or None)
