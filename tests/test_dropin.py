"""The drop-in boundary, driven the way the reference's own scripts drive it (CPU; needs a checkout of the reference,
singer-yang/Aberration-Aware-Depth-from-Focus, named by the environment variable AADFF_REFERENCE).

Two integration modes (INTEGRATION.md):
  shadow  -- this repo's site directory in front of the reference checkout on sys.path: the import block of
             2_aber_aware_dff_aif.py:23-25 and get_lens(args) from configs/aber_aware_dff_aif.yml must work, with
             PSFNet / get_lens / select_focus_dist coming from here and everything else from the reference;
  install -- the reference imported first, then aadff_b200.install() grafts the CUDA-backed methods onto it.

Optional packages the reference imports but this container lacks (matplotlib, lpips, skimage, wandb) are
stubbed in the child process; they are never touched on the path.
"""
import os
import subprocess
import sys
import textwrap

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHADOW = os.path.join(ROOT, "aberration-aware-depth-from-focus_b200")
REF = os.environ.get("AADFF_REFERENCE", "")

pytestmark = pytest.mark.skipif(not os.path.isdir(REF), reason="needs a reference checkout (set AADFF_REFERENCE)")

STUBS = textwrap.dedent("""
    import sys, types
    for name in ["matplotlib", "matplotlib.pyplot", "lpips", "skimage", "skimage.metrics", "skimage.morphology",
                 "skimage.filters", "wandb"]:
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    sys.modules["skimage.metrics"].peak_signal_noise_ratio = lambda *a, **k: 0
    sys.modules["skimage.metrics"].structural_similarity = lambda *a, **k: 0
    sys.modules["skimage.morphology"].disk = sys.modules["skimage.morphology"].closing = lambda *a, **k: None
    import scipy.ndimage
    sys.modules.setdefault("scipy.ndimage.interpolation", scipy.ndimage)
""")


def run_child(body, path):
    code = STUBS + f"\nimport os\nos.chdir({REF!r})\nREF_ROOT = os.path.realpath({REF!r}) + os.sep\nsys.path[:0] = {path!r}\n" + \
        textwrap.dedent(body)
    env = dict(os.environ, PYTHONPATH="")
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    return res.stdout


def test_shadow_runs_the_training_scripts_import_block_and_get_lens():
    out = run_child("""
        import yaml, torch
        # ---- 2_aber_aware_dff_aif.py:23-25, verbatim
        from deeplens.utils import set_seed, set_logger
        from deeplens.psfnet import *
        from dff import *
        import deeplens, dff, deeplens.utils, deeplens.psfnet, dff.utils, dff.AiFNet, dff.dataset
        here = lambda m: os.path.realpath(m.__file__)
        assert here(deeplens.utils).startswith(REF_ROOT), here(deeplens.utils)
        assert here(dff.AiFNet).startswith(REF_ROOT) and here(dff.dataset).startswith(REF_ROOT)
        assert not here(deeplens.psfnet).startswith(REF_ROOT)
        assert not here(dff.utils).startswith(REF_ROOT)
        assert PSFNet.__module__ == 'aadff_lens' and ThinLens.__module__ == 'aadff_lens'
        assert select_focus_dist.__module__ == 'aadff_focus' and get_lens.__module__ == 'aadff_factory'
        AiFDepthNet, get_dataset, Middlebury, mask_mae, local_psf_render          # names the scripts use
        set_seed(126)
        # ---- config() + get_lens(args) of 2_aber_aware_dff_aif.py:27-57 (device as config() picks it on this box)
        with open('configs/aber_aware_dff_aif.yml') as f:
            args = yaml.load(f, Loader=yaml.FullLoader)
        args['device'] = torch.device('cuda' if torch.cuda.is_available() else 'cpu')
        train_lens, test_lens = get_lens(args)
        assert type(train_lens).__module__ == 'aadff_lens' and train_lens.kernel_size == 11
        sd = torch.load(args['train']['psfnet_path'], map_location='cpu')
        for k, v in train_lens.psfnet.state_dict().items():
            assert torch.equal(v.cpu(), sd[k]), k
        net = AiFDepthNet(n_stack=args['n_stack'])                                  # the reference's network, untouched
        # the thin-lens branch of get_lens (configs/*.yml, commented alternative)
        args['train'] = dict(args['train'], lens='thinlens', foc_len=50.0, fnum=1.8, sensor_size=['36', '24'])
        tl, _ = get_lens(args)
        assert type(tl).__name__ == 'ThinLens' and abs(tl.ps - 36.0 / 480) < 1e-9
        if not torch.cuda.is_available():
            try:
                train_lens.render(torch.zeros(1, 3, 8, 8), torch.zeros(1, 1, 8, 8), torch.tensor([-1000.]))
            except RuntimeError as e:
                assert 'no CPU path' in str(e)
            else:
                raise AssertionError('render must fail loudly without a GPU')
        print('SHADOW-OK')
    """, [SHADOW, REF])
    assert "SHADOW-OK" in out


def test_install_patches_an_already_imported_reference():
    out = run_child("""
        import torch
        import deeplens.psfnet as ref_psfnet              # the REFERENCE (its root precedes the shadow dir)
        import deeplens.render_psf
        ref_render = sys.modules['deeplens.render_psf']   # (the attribute deeplens.render_psf is a function there)
        import dff.utils as ref_dff_utils
        assert os.path.realpath(ref_psfnet.__file__).startswith(REF_ROOT)
        ref_render_fn, ref_gather, ref_select = ref_psfnet.PSFNet.render, ref_render.local_psf_render, ref_dff_utils.select_focus_dist
        sys.path.insert(0, %r)
        import aadff_b200
        assert aadff_b200.PSFNet.__module__ == 'aadff_lens'          # own classes, not the imported reference's
        assert aadff_b200.install() is True
        import aadff_lens, aadff_render, aadff_focus
        assert ref_psfnet.PSFNet.render is aadff_lens.PSFNet.render and ref_psfnet.PSFNet.pred is aadff_lens.PSFNet.pred
        assert hasattr(ref_psfnet.PSFNet, 'render_stack') and hasattr(ref_psfnet.PSFNet, 'simulate_focal_stack')
        assert ref_psfnet.ThinLens.render is aadff_lens.ThinLens.render
        assert ref_render.local_psf_render is aadff_render.local_psf_render
        assert ref_psfnet.local_psf_render is aadff_render.local_psf_render
        assert ref_dff_utils.select_focus_dist is aadff_focus.select_focus_dist
        aadff_b200.uninstall()
        assert ref_psfnet.PSFNet.render is ref_render_fn and not hasattr(ref_psfnet.PSFNet, 'render_stack')
        assert ref_render.local_psf_render is ref_gather and ref_dff_utils.select_focus_dist is ref_select
        print('INSTALL-OK')
    """ % ROOT, [REF])
    assert "INSTALL-OK" in out
