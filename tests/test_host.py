"""Host-side logic of the drop-in boundary: config loading, define_G surface, state_dict
compatibility, schedule buffers, loud failure without a GPU, C-ABI exports.  CPU only."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import fastdiffsr_b200 as F
from fastdiffsr_b200 import _lib
from fastdiffsr_b200.config import default_config, load_config, NoneDict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# a checkout of the original FastDiffSR repository (test_reference_DDPM_wrapper_runs_on_patched_define_G)
REF_ROOT = os.environ.get("FASTDIFFSR_REFERENCE", "")


def test_config_comment_stripping(tmp_path):
    p = tmp_path / "c.json"
    p.write_text('{\n "phase": "val", // train or val\n "gpu_ids": [0, 1],\n // whole line\n "model": {"x": 1}\n}\n')
    opt = load_config(str(p), phase="val")
    assert opt["gpu_ids"] == [0, 1] and opt["distributed"] is True
    assert isinstance(opt["model"], NoneDict) and opt["model"]["missing"] is None
    # README names a file that does not exist; the alias resolves to infer_x4 (SURVEY F4)
    (tmp_path / "sr_fastdiffsr_infer_x4.json").write_text('{"datasets": {"val": {"l_resolution": 128}}}\n')
    assert load_config(str(tmp_path / "sr_fastdiffsr_infer_128_512.json"))["datasets"]["val"]["l_resolution"] == 128


def test_default_configs_cover_reference_names():
    for name in ("sr_fastdiffsr_test_64_256", "sr_fastdiffsr_test_32_256", "sr_fastdiffsr_infer_x4",
                 "sr_fastdiffsr_infer_128_512.json"):
        opt = default_config(name)
        assert opt["model"]["which_model_G"] == "fastdiffsr"
        assert opt["model"]["beta_schedule"]["val"]["n_timestep"] == 20
    assert default_config("sr_fastdiffsr_infer_x4")["datasets"]["val"]["r_resolution"] == 512


def test_define_G_surface_and_state_dict(oracle, golden_dir):
    opt = default_config()
    netG = F.define_G(opt)
    assert isinstance(netG, torch.nn.Module) and netG.conditional and netG.channels == 3 and netG.image_size == 256
    keys = [(k, tuple(v.shape)) for k, v in netG.state_dict().items()]
    spec = [(k, s) for k, s, _, _ in oracle.state_dict_spec(oracle.DEFAULT_UNET)]
    assert keys == spec
    netG.set_loss("cpu")
    netG.set_new_noise_schedule(opt["model"]["beta_schedule"]["val"], "cpu")
    assert netG.num_timesteps == 20 and netG.betas.device.type == "cpu"
    g = np.load(os.path.join(golden_dir, "schedule_T20.npz"))
    for k in g.files:
        if k == "sqrt_alphas_cumprod_prev":
            assert np.array_equal(netG.sqrt_alphas_cumprod_prev, g[k])
        else:
            assert np.array_equal(getattr(netG, k).numpy(), g[k]), k
    assert len(netG.state_dict()) == 317 + 12
    # a reference-style checkpoint (weights + the 12 buffers) loads strictly
    sd = oracle.make_state_dict(oracle.DEFAULT_UNET, seed=3)
    for k in g.files:
        if k != "sqrt_alphas_cumprod_prev":
            sd[k] = torch.from_numpy(g[k])
    netG.load_state_dict(sd, strict=True)
    assert torch.equal(netG.denoise_fn.downs[0].weight, sd["denoise_fn.downs.0.weight"])
    netG.set_new_noise_schedule(opt["model"]["beta_schedule"]["val"], "cpu")  # re-entrant like the reference


def test_sr3_define_G_surface_and_configs(oracle):
    """which_model_G = 'ddpm' (the SR3 baseline): config defaults, state_dict surface equals the reference's (421
    tensors incl. the time_mlp.0.inv_freq buffer), no CPU fallback."""
    for name in ("sr_ddpm_test_64_256", "sr_ddpm_test_32_256", "sr_ddpm_infer_x4"):
        mine = default_config(name)
        assert mine["model"]["which_model_G"] == "ddpm" and mine["model"]["beta_schedule"]["val"]["n_timestep"] == 1000
    opt =default_config("sr_ddpm_test_64_256")
    netG = F.define_G(opt)
    assert isinstance(netG.denoise_fn, F.SR3UNet) and netG.sr3
    keys = [(k, tuple(v.shape)) for k, v in netG.state_dict().items()]
    assert keys == [(k, s) for k, s, _, _ in oracle.sr3_state_dict_spec(oracle.SR3_UNET, 256)] and len(keys) == 421
    sd = oracle.make_state_dict(oracle.SR3_UNET, seed=3, spec=oracle.sr3_state_dict_spec(oracle.SR3_UNET, 256))
    assert torch.equal(sd["denoise_fn.time_mlp.0.inv_freq"], netG.state_dict()["denoise_fn.time_mlp.0.inv_freq"])
    netG.load_state_dict(sd, strict=True)
    netG.set_new_noise_schedule(opt["model"]["beta_schedule"]["val"], "cpu")
    assert netG.num_timesteps == 1000
    tab = oracle.schedule_tables(oracle.make_beta_schedule(**oracle.SR3_SCHEDULE))
    assert np.array_equal(netG.posterior_mean_coef1.numpy(), tab["posterior_mean_coef1"].astype(np.float32))
    with pytest.raises(F.FdsrError):
        netG.super_resolution(torch.zeros(1, 3, 64, 64), False)


def test_other_generators_and_training_rejected():
    opt = default_config()
    opt["model"]["which_model_G"] = "tesr"
    with pytest.raises(NotImplementedError):
        F.define_G(opt)
    with pytest.raises(NotImplementedError):
        F.define_G(default_config(phase="train"))
    with pytest.raises(NotImplementedError):
        F.make_beta_schedule("nope", 20)


def test_no_cpu_fallback():
    opt = default_config()
    netG = F.define_G(opt)
    netG.set_new_noise_schedule(opt["model"]["beta_schedule"]["val"], "cpu")
    with pytest.raises(F.FdsrError):
        netG.super_resolution(torch.zeros(1, 3, 64, 64), False)
    with pytest.raises(NotImplementedError):
        netG({"HR": None, "SR": None})


def test_beta_schedules_match_oracle(oracle):
    for name in ("linear", "quad", "const", "jsd", "warmup10", "warmup50", "linear_cosine"):
        a = F.make_beta_schedule(name, 20, 1e-6, 1e-2)
        assert np.array_equal(a, oracle.make_beta_schedule(name, 20, 1e-6, 1e-2)), name


def test_cabi_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "fdsr.h")).read()
    declared = sorted(set(re.findall(r"\b(fdsr_[a-z0-9_]+)\s*\(", hdr)))
    assert len(declared) >= 20
    assert os.path.exists(_lib.LIB_PATH), "build first: python -c 'import __graft_entry__ as g; g.build()'"
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for sym in declared:
        assert hasattr(lib, sym), sym
    assert sorted(_lib.EXPORTS) == declared  # the Python binding covers exactly the header
    # error path that needs no GPU: creating a context without a device fails loudly
    if not torch.cuda.is_available():
        cfg = _lib.FdsrConfig()
        h = ctypes.c_void_p()
        l = _lib.load()
        assert l.fdsr_create(ctypes.byref(cfg), ctypes.byref(h)) < 0
        assert b"no CPU fallback" in l.fdsr_global_error() or b"CUDA" in l.fdsr_global_error()


def test_cabi_from_plain_c(tmp_path):
    """include/fdsr.h compiles as C and links against libfdsr.so from a C program (no C++ / torch types at the
    boundary); without a GPU fdsr_create reports FDSR_E_CUDA instead of falling back."""
    import shutil
    import subprocess
    from fastdiffsr_b200._lib import LIB_PATH
    if shutil.which("gcc") is None or not os.path.exists(LIB_PATH):
        pytest.skip("gcc or libfdsr.so missing")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "abi_check")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(root, "include"),
                    os.path.join(root, "tests", "c_abi", "abi_check.c"), "-o", exe, LIB_PATH,
                    "-Wl,-rpath," + os.path.dirname(LIB_PATH)], check=True)
    res = subprocess.run([exe], capture_output=True, text=True)
    assert res.returncode == 0, (res.returncode, res.stdout, res.stderr)


def test_reference_checkpoint_with_schedule_buffers_loads_through_load_network(oracle, tmp_path):
    """ADVICE r1 (high): the reference saves netG.state_dict() AFTER set_new_noise_schedule (model/model.py:126-146),
    so a real `*_gen.pth` carries the 12 schedule buffers.  evaluate.load_network must accept it strictly both in the
    reference's call order (schedule registered first, model/model.py:19-41) and on a net without the buffers."""
    from fastdiffsr_b200 import evaluate
    opt = default_config()
    donor = F.define_G(opt)
    donor.load_state_dict(oracle.make_state_dict(oracle.DEFAULT_UNET, seed=4), strict=False)
    donor.set_new_noise_schedule(opt["model"]["beta_schedule"]["train"], "cpu")
    full = donor.state_dict()
    assert len(full) == 317 + 12 and "betas" in full
    torch.save(full, str(tmp_path / "I1_E1_gen.pth"))
    opt["path"] = {"resume_state": str(tmp_path / "I1_E1")}
    opt["model"]["finetune_norm"] = False
    # reference order: buffers exist at load time -> strict load of all 329 keys
    net1 = F.define_G(opt)
    net1.set_loss("cpu")
    net1.set_new_noise_schedule(opt["model"]["beta_schedule"]["train"], "cpu")
    assert evaluate.load_network(net1, opt)
    # buffer-less net (schedule not yet set): the buffers of the checkpoint are dropped, the denoiser loads strictly
    net2 = F.define_G(opt)
    assert evaluate.load_network(net2, opt)
    for net in (net1, net2):
        assert torch.equal(net.denoise_fn.downs[0].weight, full["denoise_fn.downs.0.weight"])
        assert torch.equal(net.state_dict()["denoise_fn.final_conv.block.3.bias"], full["denoise_fn.final_conv.block.3.bias"])
    # a checkpoint that lacks a denoiser tensor still fails loudly under strict loading
    broken = {k: v for k, v in full.items() if k != "denoise_fn.downs.0.weight"}
    torch.save(broken, str(tmp_path / "I2_E2_gen.pth"))
    opt["path"] = {"resume_state": str(tmp_path / "I2_E2")}
    with pytest.raises(RuntimeError):
        evaluate.load_network(F.define_G(opt), opt)


@pytest.mark.skipif(not REF_ROOT, reason="imports and runs the original FastDiffSR's own model/ package, which is not part "
                                          "of this repository and cannot be stored as test data; runs when "
                                          "FASTDIFFSR_REFERENCE names a checkout of that repository")
def test_reference_DDPM_wrapper_runs_on_patched_define_G(oracle, tmp_path):
    """INTEGRATION.md's one-line patch, exercised with the reference's OWN wrapper: `model.networks.define_G` replaced
    by fastdiffsr_b200.define_G, then the unmodified `model.model.DDPM` (model/model.py:12-42) is constructed — set_device,
    set_loss, set_new_noise_schedule('train'), strict load_network of a reference-style checkpoint (148-160),
    print_network — and switched to the 'val' schedule as sr_mfe.py:93-94 does.  `thop` (imported by base_model.py but
    never called on this path) is stubbed.  On this CPU-only container DDPM.test() must fail loudly (no fallback)."""
    import sys
    import types
    saved_path, saved_mods = list(sys.path), set(sys.modules)
    try:
        thop = types.ModuleType("thop")
        thop.profile = thop.clever_format = lambda *a, **k: None
        sys.modules["thop"] = thop
        sys.path.insert(0, REF_ROOT)
        import model as RefModel
        import model.networks as ref_networks
        ref_define_G = ref_networks.define_G
        ref_networks.define_G = F.define_G                      # <- the integration patch
        opt = default_config()
        opt["gpu_ids"] = None                                   # BaseModel: device = cpu
        donor = ref_define_G(default_config())                   # a checkpoint written by the REFERENCE's own netG
        donor.set_new_noise_schedule(opt["model"]["beta_schedule"]["train"], "cpu")
        ckpt = {k: v.cpu() for k, v in donor.state_dict().items()}   # model/model.py:131-137
        assert len(ckpt) == 317 + 12
        torch.save(ckpt, str(tmp_path / "I9_E9_gen.pth"))
        opt["path"] = {"resume_state": str(tmp_path / "I9_E9")}
        m = RefModel.create_model(opt)                          # the reference's DDPM.__init__
        assert type(m).__module__ == "model.model" and isinstance(m.netG, F.GaussianDiffusion)
        assert m.netG.num_timesteps == 20 and m.schedule_phase == "train"
        for k, v in ckpt.items():
            assert torch.equal(m.netG.state_dict()[k], v), k
        m.set_new_noise_schedule(opt["model"]["beta_schedule"]["val"], schedule_phase="val")
        assert m.schedule_phase == "val"
        s, n = m.get_network_description(m.netG)
        assert n == 23802277                                    # SURVEY section 6: total parameters
        m.feed_data({"HR": torch.zeros(1, 3, 64, 64), "SR": torch.zeros(1, 3, 64, 64), "Index": None})
        with pytest.raises(F.FdsrError):
            m.test(continous=False)
    finally:
        sys.path[:] = saved_path
        for name in set(sys.modules) - saved_mods:
            del sys.modules[name]


def test_documented_results_match_the_committed_records(tmp_path):
    """Measurement hygiene (VERDICT r1 item 6): the result tables of README.md / DESIGN.md are generated from the bench
    records under profiles/r2, and traffic.json (what bench.py's roofline.traffic quotes) from the raw ncu pages —
    a hand-edited number or a stale table fails here."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "tools/fill_tables.py", "--check"], cwd=root, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    out = tmp_path / "traffic.json"
    r = subprocess.run([sys.executable, "tools/extract_traffic.py", "profiles/r2", str(out)], cwd=root, capture_output=True,
                       text=True)
    assert r.returncode == 0, r.stderr
    assert json.load(open(out))["launches"] == json.load(open(os.path.join(root, "profiles", "r2", "traffic.json")))["launches"]
