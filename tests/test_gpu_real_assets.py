"""Full real-asset regression (SURVEY 8(f2)): all 40 scenes of the reference's demo assets against the template set of
their object with the notebook's parameters (notebooks/pose_extimation_example.ipynb:216-226): DT3 planes, hypothesis
list, every match and the penalised top-10 bit-exact against the oracle."""
import glob
import os

import numpy as np
import pytest

import openfdcm_b200 as fdcm
from oracle import fdcm_oracle as orc
from tests.helpers import ASSETS, load_object

pytestmark = pytest.mark.gpu


def test_assets_complete():
    n_t = sum(len(glob.glob(os.path.join(ASSETS, o, "templates", "*.tmpl"))) for o in ("obj_01", "obj_02", "obj_03", "obj_04"))
    n_s = len(glob.glob(os.path.join(ASSETS, "obj_0*", "scene_*", "camera_0.scene")))
    assert (n_t, n_s) == (421, 40)


@pytest.mark.parametrize("obj", ["obj_01", "obj_02", "obj_03", "obj_04"])
def test_real_scenes_bit_exact(obj):
    tmpls, scenes = load_object(obj)
    assert len(scenes) == 10 and len(tmpls) > 80
    tset = fdcm.TemplateSet(tmpls)
    lengths = orc.template_lengths(tmpls)
    s_, o_, p_ = fdcm.DefaultSearch(4, 10), fdcm.BatchOptimize(10), fdcm.ExponentialPenalty(1.5)
    fm = None
    for i, scene in enumerate(scenes):
        params = fdcm.Dt3CudaParameters(30, 5.0, 1.0, fdcm.distance.L2)
        if fm is None:
            fm = fdcm.build_cuda_featuremap(scene, params)
        else:
            fm.rebuild(scene)
        c = orc.Dt3Cpu(scene, 30, 5.0, 1.0)
        assert (fm.width, fm.height) == (c.W, c.H)
        for d in (0, 8, 15, 23, 29):
            assert np.array_equal(fm.plane(d), c.plane(d)), f"{obj} scene {i} plane {d}"
        got = fdcm.search_all(fm, tset, scene, s_, o_)
        want, hyp = c.search(tmpls, scene, 4, 10, batch=10, want_hyp=True)
        assert np.array_equal(fm.last_hypotheses(), hyp), f"{obj} scene {i}: hypothesis list"
        assert len(got) == len(want)
        assert np.array_equal(got["tmpl_idx"], want["tmpl_idx"]) and np.array_equal(got["transform"], want["transform"])
        assert np.array_equal(got["score"], want["score"]), f"{obj} scene {i}: scores"
        top = fdcm.search_topk(fm, tset, None, s_, o_, p_, k=10)
        pen = orc.penalize(1, 1.5, want, lengths)
        assert np.array_equal(top, pen[np.lexsort((np.arange(len(pen)), pen["score"]))[:10]]), f"{obj} scene {i}: top-10"
