// Test-only: compiles diou_pair of sihl_b200/csrc/od_math.h (the DIoU-NMS suppression test of every DIoU kernel) for the
// HOST, so it can be checked bit for bit against torchvision.ops.distance_box_iou where no GPU exists.
// Never part of the product library.
#include "../sihl_b200/csrc/od_math.h"

// out[i * nb + j] = diou(a_i, b_j); areas as the kernels compute them
extern "C" void shim_diou_matrix(const float *a, int na, const float *b, int nb, float *out)
{
    for (int i = 0; i < na; ++i) {
        const sihl::Box4 bi{a[4 * i], a[4 * i + 1], a[4 * i + 2], a[4 * i + 3]};
        const float ai = (bi.x2 - bi.x1) * (bi.y2 - bi.y1);
        for (int j = 0; j < nb; ++j) {
            const sihl::Box4 bj{b[4 * j], b[4 * j + 1], b[4 * j + 2], b[4 * j + 3]};
            const float aj = (bj.x2 - bj.x1) * (bj.y2 - bj.y1);
            out[(long)i * nb + j] = sihl::diou_pair(bi, ai, bj, aj);
        }
    }
}
