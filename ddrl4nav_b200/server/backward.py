"""Backward module compute body -- USTC_lab/server/backward.py:182-209.

``BackwardModule.train_on(exp)`` = ``train_data.to_tensor(...)`` + ``for ... in net.learn(train_data)``;
the Redis / logger / checkpoint lines stay with the reference thread."""
from typing import Dict, List

import torch


class BackwardModule:
    """``prefetch(next_batch)`` is the device half of the reference's BackwardGetDataThread (backward.py:104-160 runs
    concurrently with the train thread): it starts the NEXT batch's host->device copies on a side stream while the
    current batch trains; ``train_on`` of that batch then only waits for the copy event."""

    def __init__(self, net, device="cuda", tensortype=torch.float32):
        self.net = net
        self.device = device
        self.tensortype = tensortype
        self.data_len = 0
        self._copy_stream = None
        self._prefetched = None

    def prefetch(self, train_data) -> None:
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(torch.device(self.device))
        with torch.cuda.stream(self._copy_stream):
            train_data.to_tensor(dtype=self.tensortype, device=self.device)
            ev = torch.cuda.Event()
            ev.record(self._copy_stream)
        self._prefetched = (train_data, ev)

    def train_on(self, train_data) -> List[Dict[str, float]]:
        if self._prefetched is not None and self._prefetched[0] is train_data:
            main = torch.cuda.current_stream(torch.device(self.device))
            main.wait_event(self._prefetched[1])
            extra = [train_data.old_values] if getattr(train_data, "old_values", None) is not None else []
            for t in list(train_data.states) + [train_data.advs, train_data.actions, train_data.old_logps, train_data.values] + extra:
                t.record_stream(main)
            self._prefetched = None
        else:
            train_data.to_tensor(dtype=self.tensortype, device=self.device)
        self.data_len += len(train_data)
        logs = []
        for loss_items, update_time, last in self.net.learn(train_data):
            logs.append(dict(loss_items, update_time=update_time))
        return logs
