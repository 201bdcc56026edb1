"""sihl_b200 — B200-native (sm_100a) implementation of the dense tail of sihl's
``ObjectDetection`` head: anchor grid, CIoU top-k label assignment, loss reductions (+backward),
top-k decode and (extension) dense decode + class-aware NMS, behind the C ABI of
``include/sihl_od.h``.  ``sihl_b200.heads.ObjectDetection`` is the drop-in head."""

__version__ = "0.1.2"
