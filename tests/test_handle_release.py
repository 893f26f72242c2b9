"""Handles released while a CUDA graph is being captured are destroyed after the capture, not inside it (_lib.release)."""
import importlib

_lib = importlib.import_module("sgmm_b200._lib")


class FakeLib:
    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        return lambda h: self.calls.append((name, h.value))


def test_release_defers_during_a_capture_and_drains_after(monkeypatch):
    fake = FakeLib()
    monkeypatch.setattr(_lib, "lib", lambda: fake)
    monkeypatch.setattr(_lib, "_DEFERRED", [])
    monkeypatch.setattr(_lib, "_capturing", lambda: True)
    _lib.release("sgmm_bundle_destroy", 0x1000)
    _lib.release("sgmm_ga_destroy", 0x2000)
    _lib.release("sgmm_bundle_destroy", 0)                  # a closed handle is ignored
    assert fake.calls == [] and len(_lib._DEFERRED) == 2
    monkeypatch.setattr(_lib, "_capturing", lambda: False)
    _lib.release("sgmm_bundle_destroy", 0x3000)
    assert sorted(fake.calls) == [("sgmm_bundle_destroy", 0x1000), ("sgmm_bundle_destroy", 0x3000), ("sgmm_ga_destroy", 0x2000)]
    assert _lib._DEFERRED == []
