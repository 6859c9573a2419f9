"""Engines of pending autograd forwards.

An engine keeps the activations its backward reads, so two forwards of one shape whose backward has not run yet
(the reference's loop runs a whole rollout, or two, before its single ``loss.backward()``) need two engines.
``EnginePool`` hands out an engine per shape key and leases it to the autograd node of a forward: the lease is a
token tensor the node saves for backward, and the slot returns to the pool when that token dies -- when the node's
saved tensors are freed after its backward (without ``retain_graph``), or when the graph is dropped unused.

Slot 0 of a key is the module's existing engine (``make(key, 0)``), so code with at most one pending forward per
shape runs on exactly the engine it ran on before, and shares it with the agents' direct engine use."""
import weakref

import torch


class EnginePool:
    def __init__(self, make):
        """``make(key, slot)``: the engine of ``slot`` (0, 1, ...) for shape ``key``, created on first use."""
        self._make = make
        self._busy = set()               # (key, slot) leased to a pending forward

    def _first_free(self, key):
        slot = 0
        while (key, slot) in self._busy:
            slot += 1
        return slot

    def busy(self, key=None):
        """The leased slots (of ``key``), sorted."""
        return sorted(s for k, s in self._busy if key is None or k == key)

    def free(self, key):
        """An engine of ``key`` that no pending forward holds, not leased: for a forward that records no autograd
        node (``torch.no_grad()``), whose outputs are copies and whose engine is done with when it returns."""
        return self._make(key, self._first_free(key))

    def lease(self, key):
        """``(engine, token)``: an engine of ``key`` held until ``token`` dies.  The autograd function stores the
        token with ``ctx.save_for_backward``."""
        slot = self._first_free(key)
        eng = self._make(key, slot)
        self._busy.add((key, slot))
        token = torch.empty(0)
        weakref.finalize(token, self._busy.discard, (key, slot)).atexit = False
        return eng, token

    def acquire(self, key, hold):
        """``lease(key)`` when ``hold``, else ``(free(key), None)``."""
        return self.lease(key) if hold else (self.free(key), None)


def lease_slot(slot):
    """The engine-cache slot of pool slot ``slot``: 0 stays 0 (the existing engine); later slots get names of their
    own, apart from the numbered slots the agents pick for their rollouts."""
    return 0 if slot == 0 else ("lease", slot)
