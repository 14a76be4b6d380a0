"""``torch.use_deterministic_algorithms`` as seen by this library.

The flag is read per call.  Under it the backward of the op takes the bit-reproducible kernels
(``msda_backward_det_*``); an operation without a deterministic implementation raises like a torch op does, or warns and
runs the normal path under ``warn_only=True``.  With the flag off nothing changes.
"""
from __future__ import annotations

import warnings

import torch

OFF, ON, WARN = "off", "on", "warn"


def mode() -> str:
    """OFF when deterministic algorithms are not requested, ON when they are, WARN when they are with warn_only."""
    if not torch.are_deterministic_algorithms_enabled():
        return OFF
    return WARN if torch.is_deterministic_algorithms_warn_only_enabled() else ON


def alert_not_deterministic(caller: str) -> None:
    """For an operation that has no deterministic implementation: raise (ON) or warn (WARN), in PyTorch's wording."""
    m = mode()
    if m == OFF:
        return
    msg = (f"{caller} does not have a deterministic implementation, but you set "
           "'torch.use_deterministic_algorithms(True)'. You can turn off determinism just for this operation, or you "
           "can use the 'warn_only=True' option, if that's acceptable for your application.")
    if m == ON:
        raise RuntimeError(msg)
    warnings.warn(msg, UserWarning, stacklevel=3)
