/* Test infrastructure, not product code.
 *
 * Plain-C restatement of one image of multi-label NMS: upstream YOLOv9's candidate set
 * (utils/general.py, non_max_suppression(..., multi_label=True): `i, j = (x[:, 5:mi] > conf_thres).nonzero().T`)
 * on top of yolo-re's algorithm (src/yolo/utils/nms.py:61-92 and torchvision.ops.nms), as oracle/nms_ref.c restates
 * the single-label one.  Candidates are every (anchor a, class c) with score > conf_thres (and c in the class list),
 * in row-major order; ties of the descending score sort go to the lower candidate.  Exists because a full-size image has
 * up to 2.69 M candidates.  Build with -ffp-contract=off so that every fp32 operation is rounded separately.
 */
#include <stdint.h>
#include <stdlib.h>

typedef struct { float score; int32_t idx; } cand_t;

static int cmp_cand(const void* a, const void* b) {
    const cand_t* x = (const cand_t*)a; const cand_t* y = (const cand_t*)b;
    if (x->score > y->score) return -1;
    if (x->score < y->score) return 1;
    return (x->idx > y->idx) - (x->idx < y->idx);
}

static inline float fmax2(float a, float b) { return a > b ? a : b; }
static inline float fmin2(float a, float b) { return a < b ? a : b; }

static int wanted(int c, const int32_t* classes, int n_classes) {
    if (n_classes < 0) return 1;
    for (int k = 0; k < n_classes; ++k) if (classes[k] == c) return 1;
    return 0;
}

/* pred [A][4+nc] fp32; det [max_det][6]; keep_anchor [max_det].  Returns the number of detections, < 0 on error. */
int yre_oracle_nms_image_multi_label(const float* pred, int A, int nc, float conf_thres, double iou_thres, int max_det,
                                     const int32_t* classes, int n_classes, int agnostic,
                                     float* det, int64_t* keep_anchor)
{
    const int ch = 4 + nc;
    size_t n = 0;
    for (int a = 0; a < A; ++a)
        for (int c = 0; c < nc; ++c)
            if (pred[(size_t)a * ch + 4 + c] > conf_thres && wanted(c, classes, n_classes)) ++n;
    if (n == 0) return 0;
    cand_t* cd = (cand_t*)malloc(sizeof(cand_t) * n);
    int32_t* anc = (int32_t*)malloc(sizeof(int32_t) * n);
    int32_t* cls = (int32_t*)malloc(sizeof(int32_t) * n);
    float* box = (float*)malloc(sizeof(float) * 4 * n);    /* un-offset xyxy */
    float* nb = (float*)malloc(sizeof(float) * 4 * n);     /* offset xyxy   */
    float* area = (float*)malloc(sizeof(float) * n);
    uint8_t* dead = (uint8_t*)calloc(n, 1);
    if (!cd || !anc || !cls || !box || !nb || !area || !dead) {
        free(cd); free(anc); free(cls); free(box); free(nb); free(area); free(dead); return -1;
    }

    size_t q = 0;
    float max_coord = 0.f; int have_max = 0;
    for (int a = 0; a < A; ++a) {
        const float* row = pred + (size_t)a * ch;
        for (int c = 0; c < nc; ++c) {
            if (!(row[4 + c] > conf_thres) || !wanted(c, classes, n_classes)) continue;   /* strict > */
            const float hw = row[2] / 2.f, hh = row[3] / 2.f;
            float* b = box + 4 * q;
            b[0] = row[0] - hw; b[1] = row[1] - hh; b[2] = row[0] + hw; b[3] = row[1] + hh;
            for (int k = 0; k < 4; ++k) if (!have_max || b[k] > max_coord) { max_coord = b[k]; have_max = 1; }
            anc[q] = a; cls[q] = c;
            cd[q].score = row[4 + c]; cd[q].idx = (int32_t)q; ++q;
        }
    }
    const float scale = max_coord + 1.f;
    for (size_t i = 0; i < n; ++i) {
        const float off = agnostic ? 0.f : (float)cls[i] * scale;
        const float* b = box + 4 * i; float* o = nb + 4 * i;
        if (agnostic) { o[0] = b[0]; o[1] = b[1]; o[2] = b[2]; o[3] = b[3]; }
        else { o[0] = b[0] + off; o[1] = b[1] + off; o[2] = b[2] + off; o[3] = b[3] + off; }
        area[i] = (o[2] - o[0]) * (o[3] - o[1]);
    }
    qsort(cd, n, sizeof(cand_t), cmp_cand);

    int kept = 0;
    for (size_t p = 0; p < n && kept < max_det; ++p) {
        const int i = cd[p].idx;
        if (dead[i]) continue;
        const float* bi = box + 4 * (size_t)i;
        det[6 * kept + 0] = bi[0]; det[6 * kept + 1] = bi[1]; det[6 * kept + 2] = bi[2]; det[6 * kept + 3] = bi[3];
        det[6 * kept + 4] = cd[p].score; det[6 * kept + 5] = (float)cls[i];
        keep_anchor[kept] = anc[i]; ++kept;
        if (kept == max_det) break;
        const float* oi = nb + 4 * (size_t)i; const float ai = area[i];
        for (size_t r = p + 1; r < n; ++r) {
            const int j = cd[r].idx;
            if (dead[j]) continue;
            const float* oj = nb + 4 * (size_t)j;
            const float w = fmax2(0.f, fmin2(oi[2], oj[2]) - fmax2(oi[0], oj[0]));
            const float h = fmax2(0.f, fmin2(oi[3], oj[3]) - fmax2(oi[1], oj[1]));
            const float inter = w * h;
            const float iou = inter / (ai + area[j] - inter);
            if ((double)iou > iou_thres) dead[j] = 1;   /* fp32 IoU vs DOUBLE threshold, as torchvision's CPU kernel */
        }
    }
    free(cd); free(anc); free(cls); free(box); free(nb); free(area); free(dead);
    return kept;
}
