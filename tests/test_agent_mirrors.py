"""Agent-boundary mirrors against outputs of the reference itself (tests/golden/agent_golden.json, made by make_agent_golden.py),
and integration.patch_reference applied to the REAL reference classes when MSC_REFERENCE_SRC names the original project's src/ directory."""
import inspect
import json
import os
import sys

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLD = json.load(open(os.path.join(GOLDEN, "agent_golden.json")))
REF_SRC = os.environ.get("MSC_REFERENCE_SRC", "")  # src/ of a checkout of the original project, which this repository does not carry


# the methods whose parameter lists the mirrors share with the reference's classes (SURVEY.md section 8(b))
SHARED_METHODS = {"LiDARAgent": ("_preprocess_point_cloud", "_segment_ground", "_generate_multi_layer_bev", "_generate_cluster_visualization",
                                 "_detect_objects_3d", "_extract_semantic_features", "_generate_structured_report", "process",
                                 "_classify_batch_with_llm"),
                  "SceneGraphAgent": ("_parse_annotations", "_categorize_objects", "_build_spatial_zones", "process", "_generate_scene_graph",
                                      "_generate_summary"),
                  "CameraAgent": ("process",)}


def mirror_signatures():
    """Parameter names of the shared methods on the mirror classes (tests/golden/interface_golden.json records them)."""
    from msc_geom.camera_agent import CameraAgent
    from msc_geom.lidar_agent import LiDARAgent
    from msc_geom.scenegraph_agent import SceneGraphAgent
    classes = {"LiDARAgent": LiDARAgent, "SceneGraphAgent": SceneGraphAgent, "CameraAgent": CameraAgent}
    return {c: {n: list(inspect.signature(getattr(classes[c], n)).parameters) for n in names} for c, names in SHARED_METHODS.items()}


def test_mirror_signatures_equal_the_recorded_interface():
    """The parameter lists test_patch_reference_on_the_real_reference_classes compares with the reference's own classes, against the
    record of them: a change to the interface the reference's callers use fails here without the reference at hand."""
    rec = json.load(open(os.path.join(GOLDEN, "interface_golden.json")))["signatures"]
    assert mirror_signatures() == rec
    from msc_geom import integration                                                   # the patch leaves the LLM half and process alone
    assert not set(integration._LIDAR_METHODS) & {"_classify_batch_with_llm", "_extract_semantic_features", "_generate_structured_report", "process"}
    assert set(integration._SCENE_METHODS) <= set(rec["SceneGraphAgent"]) - {"process", "_categorize_objects"}


def test_fallback_scene_graph_and_summary_equal_reference():
    from msc_geom.scenegraph_agent import SceneGraphAgent, fallback_scene_graph
    ref = GOLD["scenegraph_fallback"]["result"]
    graph = fallback_scene_graph(len(GOLD["scenegraph_fallback"]["annotations"]))
    assert graph == ref["scene_graph"]
    assert SceneGraphAgent._generate_summary(None, graph) == ref["observations"]


def test_summary_of_a_populated_graph_equals_reference():
    from msc_geom.scenegraph_agent import SceneGraphAgent
    ref = GOLD["scenegraph_llm"]["result"]
    assert SceneGraphAgent._generate_summary(None, ref["scene_graph"]) == ref["observations"]


def test_camera_agent_mirror_equals_reference():
    from msc_geom.camera_agent import CameraAgent, split_camera_sections
    g = GOLD["camera"]
    cams = g["camera_names"]
    imgs = [np.full((6, 8, 3), 10 * i, np.uint8) for i in range(len(cams))]
    for name, reply in g["replies"].items():
        seen = {}

        def llm(messages, temperature=0.7, **kw):
            seen["messages"], seen["temperature"] = messages, temperature
            return reply
        out = CameraAgent(object(), "m", "CameraAgent", llm=llm).process(imgs, cams, context=g["context"] if name == "sectioned" else None)
        assert out == g["results"][name], name
        assert split_camera_sections(reply, cams) == g["results"][name]["observations"]
        assert seen["temperature"] == 0.3
        if name == "sectioned":  # the evidence enters the prompt exactly where and how the reference puts any context
            content = seen["messages"][-1]["content"]
            assert content[0]["text"] == GOLD["camera_context_text"] and content[1]["text"] == GOLD["camera_prompt_text"]
            assert content[3]["image_url"]["url"] == GOLD["camera_first_image_url"]


@pytest.mark.skipif(not os.path.isdir(REF_SRC), reason="needs the original project's src/ directory in MSC_REFERENCE_SRC")
def test_patch_reference_on_the_real_reference_classes():
    """Names, signatures and attributes: everything the patch replaces exists on the reference's own classes with the same parameters,
    what it must leave alone is left alone, and the patched methods reach the engine they were given (a recorder; no GPU here)."""
    sys.dont_write_bytecode = True
    if REF_SRC not in sys.path:
        sys.path.insert(0, REF_SRC)
    import importlib
    ref_lidar = importlib.import_module("agents.content_transform.lidar_agent")
    ref_scene = importlib.import_module("agents.content_transform.scenegraph_agent")
    ref_cam = importlib.import_module("agents.content_transform.camera_agent")
    from msc_geom import integration
    from msc_geom import lidar_agent as la
    from msc_geom import scenegraph_agent as sg

    def params(fn):
        return [p for p in inspect.signature(fn).parameters]

    # reference-side signatures the mirrors promise (SURVEY.md section 8(b))
    for name in ("_preprocess_point_cloud", "_segment_ground", "_generate_multi_layer_bev", "_generate_cluster_visualization", "_detect_objects_3d",
                 "_extract_semantic_features", "_generate_structured_report", "process"):
        assert params(getattr(ref_lidar.LiDARAgent, name)) == params(getattr(la.LiDARAgent, name)), name
    assert params(ref_lidar.LiDARAgent._classify_batch_with_llm) == params(la.LiDARAgent._classify_batch_with_llm)
    for name in ("_parse_annotations", "_categorize_objects", "_build_spatial_zones", "process", "_generate_scene_graph", "_generate_summary"):
        assert params(getattr(ref_scene.SceneGraphAgent, name)) == params(getattr(sg.SceneGraphAgent, name)), name
    from msc_geom.camera_agent import CameraAgent
    assert params(ref_cam.CameraAgent.process) == params(CameraAgent.process)[:4]       # + the additive `sample`

    # patch copies of the real classes (subclasses, so the imported modules stay pristine for other tests)
    L = type("LiDARAgent", (ref_lidar.LiDARAgent,), {})
    S = type("SceneGraphAgent", (ref_scene.SceneGraphAgent,), {})
    C = type("CameraAgent", (ref_cam.CameraAgent,), {})
    untouched = {n: getattr(L, n) for n in ("_classify_batch_with_llm", "_extract_semantic_features", "_generate_structured_report", "process", "call_llm")}

    class Recorder:  # stands in for GeometryEngine: the patched methods must go through it (and nothing else) for their numerics
        pass
    eng = integration.patch_reference(L, S, engine=Recorder(), camera_cls=C)
    assert isinstance(eng, Recorder)
    for n in integration._LIDAR_METHODS:
        assert getattr(L, n) is not getattr(ref_lidar.LiDARAgent, n, None), n
    for n, fn in untouched.items():
        assert getattr(L, n) is fn, n                                                  # the LLM half stays the reference's
    for n in integration._SCENE_METHODS:
        assert getattr(S, n) is not getattr(ref_scene.SceneGraphAgent, n), n
    assert S._categorize_objects is ref_scene.SceneGraphAgent._categorize_objects and S.process is ref_scene.SceneGraphAgent.process
    a = L(object(), "m", "LiDARAgent")
    for attr, v in (("dbscan_eps", 0.5), ("dbscan_min_samples", 10), ("bev_resolution", 800), ("bev_range", 50)):
        assert getattr(a, attr) == v                                                   # the attributes _params() reads (lidar_agent.py:43-49)
    p = a._params()
    assert (p.bev_res, p.bev_range, p.range_max, p.ground_z) == (800, 50.0, 50.0, -1.4)
    with pytest.raises(AttributeError):                                                # Recorder has no CUDA library behind it: the call got there
        a._preprocess_point_cloud(np.zeros((4, 4), np.float32))
    assert a.engine is eng
    assert a._detect_objects_3d(np.zeros((3, 4), np.float32)) == []                    # fewer than dbscan_min_samples points (lidar_agent.py:144-145)
    s = S(object(), "m", "SceneGraphAgent")
    assert set(s.spatial_zones) == set(sg.ZONE_NAMES)                                  # zone table the kernel hard-codes (scenegraph_agent.py:136-146)
    assert "sample" in params(C.process)
