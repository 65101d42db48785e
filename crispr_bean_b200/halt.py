"""What every SVI engine shares to halt a fit at its first non-finite step (include/bean_b200.h: `nonfinite_step`).

The kernels record, in one device int32 word, the first step whose loss or any ClippedAdam input was NaN or inf.  An engine
reads it after a batch of steps (`nonfinite_step`), and can set itself back to the start of the batch (`snapshot` /
`restore`) to re-run the steps before the bad one: runs are deterministic, so that gives exactly the parameters the bad step
started from.
"""
from __future__ import annotations

from typing import Optional

import torch

INT32_MAX = 2 ** 31 - 1


class NonfiniteWatch:
    """Mixin.  The engine calls `_init_nonfinite()` once (it returns the word's device address for the C state) and lists, in
    `_snapshot_tensors()`, every tensor a later step reads that an earlier step wrote; `_snapshot_extra` / `_restore_extra`
    carry host-side state."""

    def _init_nonfinite(self) -> int:
        self.nonfinite = torch.full((1,), INT32_MAX, dtype=torch.int32, device=self.device)
        return self.nonfinite.data_ptr()

    def nonfinite_step(self) -> Optional[int]:
        """First step that went non-finite since the last `restore` (None: none).  Synchronises."""
        t = int(self.nonfinite.item())
        return None if t == INT32_MAX else t

    def snapshot(self) -> dict:
        """Device-side copy of the state the next steps start from."""
        snap = {"tensors": [t.detach().clone() for t in self._snapshot_tensors()], "step": self.step}
        snap.update(self._snapshot_extra())
        return snap

    def restore(self, snap: dict) -> None:
        """Back to `snap`, with the non-finite word cleared."""
        with torch.no_grad():
            for t, saved in zip(self._snapshot_tensors(), snap["tensors"]):
                t.copy_(saved)
        self.step = snap["step"]
        self._restore_extra(snap)
        self.nonfinite.fill_(INT32_MAX)

    def _snapshot_extra(self) -> dict:
        return {}

    def _restore_extra(self, snap: dict) -> None:
        pass
