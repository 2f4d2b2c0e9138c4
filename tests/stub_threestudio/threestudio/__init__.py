"""Minimal stand-in for the reference's `threestudio` package -- TEST INFRASTRUCTURE, written for this repo.

pytorch_lightning / omegaconf / diffusers / nvdiffrast are absent on the build and GPU boxes, so the reference package
cannot be imported there.  This stub restates only the INTERFACE the five plugins of dreammat_b200.threestudio_plugin
touch (registry, BaseObject / BaseModule construction protocol, Updateable walk, BaseLift3DSystem wiring, parse_optimizer)
so that `threestudio.find("dreammat-system")(cfg)` can be driven end to end.  tests/test_plugin_registry.py pins its
behaviour against the reference's own code (the event log recorded in tests/golden/threestudio_protocol.json).

Registry: threestudio/__init__.py:1-13 of the reference (module-level dict, last writer wins).
"""
__modules__ = {}


def register(name):
    def deco(cls):
        __modules__[name] = cls
        return cls
    return deco


def find(name):
    return __modules__[name]


def info(*a, **k):
    pass


debug = warn = info

from . import systems, utils  # noqa: E402,F401
