"""Generate the reference goldens that need a B200, by executing the UNMODIFIED reference modules of ``oracle/_ref``.

Run from the repository root on a B200, after ``__graft_entry__.build()`` has packed ``oracle/_ref`` from a checkout of the
reference:  ``python oracle/gen_golden_gpu.py [OUT_DIR]``  (default tests/golden).  Writes

  fullsize_reference.pt   the reference at full size on the synthetic weights and inputs of tests/test_fullsize_gpu.py:
                          Flux.forward for workloads B, C, D, E, the 4- and 30-point cfg-B trajectories, the 30-point trajectory's
                          decoded query row and the AutoEncoder decode (fp32 and bf16) -- each as the fixed, seeded sample
                          ``test_fullsize_gpu._sample`` of its elements, in the dtype the reference returned
  pipeline_small.pt       the oracle composition of tests/test_pipeline_gpu.py (its reference ``prepare_modified`` included):
                          the sampler inputs and the final images of process_images and of upsampling
"""
from __future__ import annotations

import dataclasses
import os
import sys

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [REPO, os.path.join(REPO, "tests")]

import test_fullsize_gpu as tf      # noqa: E402
import test_pipeline_gpu as tp      # noqa: E402
from oracle import ref_runner as rr  # noqa: E402


@torch.no_grad()
def gen_fullsize(out_dir: str) -> None:
    ours, P = tf._model()
    ref = rr.build_flux(dataclasses.asdict(P), 256, dict(ours.state_dict()))
    res = {}
    for workload, t in (("B", 0.63), ("C", 0.41), ("D", 0.41), ("E", 0.41)):
        inp, _, _ = tf._eval_inputs(workload, t)
        res[f"forward_{workload}"] = tf._sample(rr.flux_forward(ref, **inp)).cpu()
    x, kw, _, _ = tf._inputs("B")
    xg, kwg = x.cuda(), tf._cuda(kw)
    traj = rr.sample_ode(ref, xg, kwg, num_steps=4, do_shift=True, time_shifting_factor=1)
    res["traj4_final"], res["traj4_step1"] = tf._sample(traj[-1]).cpu(), tf._sample(traj[1]).cpu()
    traj = rr.sample_ode(ref, xg, kwg, num_steps=30, do_shift=True, time_shifting_factor=1)
    res["traj30_final"], res["traj30_point15"] = tf._sample(traj[-1]).cpu(), tf._sample(traj[15]).cpu()
    del ref, ours
    dec, z = tf._vae_decoder_and_latent()
    res["traj30_row_image"] = tf._sample(tf._row_image(dec, traj[-1].float()), tf.IMAGE_SAMPLE).cpu()
    p = dec.params
    kw = dict(resolution=256, in_channels=3, ch=p.ch, out_ch=p.out_ch, ch_mult=list(p.ch_mult), num_res_blocks=p.num_res_blocks,
              z_channels=p.z_channels, scale_factor=p.scale_factor, shift_factor=p.shift_factor)
    ae = rr.build_autoencoder(kw, dict(dec.state_dict()), "cuda", torch.float32)
    res["vae_decode_fp32"] = tf._sample(ae.decode(z).float(), tf.IMAGE_SAMPLE).cpu()
    res["vae_decode_bf16"] = tf._sample(ae.to(torch.bfloat16).decode(z.to(torch.bfloat16)).float(), tf.IMAGE_SAMPLE).cpu()
    torch.save(res, os.path.join(out_dir, "fullsize_reference.pt"))


@torch.no_grad()
def gen_pipeline(out_dir: str) -> None:
    rig = tp._rig()
    torch.save({"process_images": tp.oracle_process_images(rig), "upsampling": tp.oracle_upsampling(rig)},
               os.path.join(out_dir, "pipeline_small.pt"))


if __name__ == "__main__":
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(REPO, "tests", "golden")
    os.makedirs(out, exist_ok=True)
    assert torch.cuda.is_available() and rr.available(), "needs a GPU and oracle/_ref"
    gen_pipeline(out)
    gen_fullsize(out)
    for f in ("pipeline_small.pt", "fullsize_reference.pt"):
        print(f, os.path.getsize(os.path.join(out, f)))
