// Host-side construction of the body-model tables from the raw model arrays (no Python, no device work).
//
//   bf_model_build_blob(const BfModelDesc*, void** blob, int64_t* nbytes)  ->  the same image PreparedModel.save_blob writes
//   bf_model_create(const BfModelDesc*, BfModel** out)                     ->  build + bf_model_load_memory (one upload)
//
// What is built (and from which reference code it follows):
//   * Bm: ONE blend matrix [Kp, 3 n_pad] = posedirs | shapedirs^T | v_template, for the full vertex set and for the ACTIVE
//     set (the vertices the keypoint term can touch)                                  smplx.lbs blend_shapes / pose offsets
//   * Jt / Jd: J_regressor folded into template / shape directions (fp64 accumulation)  smplx.lbs vertices2joints
//   * kinematic tree tables (depth, levels, children)                                   smplx.lbs batch_rigid_transform
//   * ELL skinning weights + CSR joint->vertex lists                                    smplx.lbs (W @ A)
//   * the output-joint table: chain joints, picked vertices, barycentric landmarks, yaw-dependent contour landmarks,
//     regressed extra joints, re-indexed by the OpenPose / SPIN joint maps              models/smpl.py:56-83, models/utils.py:32-141
//   * its inverse by target, the per-contour-row "live" lists and 16-vertex block masks  (this implementation's kernels)
//   * the GMM pose prior: symmetrised precisions, log weights, the K-major GEMM operand   smplify/prior.py:127-174
// The Python builder (bodyfitting_b200/model.py) is the same algorithm; tests/test_host.py compares the two blobs table by table.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <set>
#include <vector>

namespace bfb {

static inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

struct Arrays {                                    // array section of the blob; pointer fields hold (offset + 1), 0 = NULL
    std::vector<char> bytes;
    void* put_raw(const void* p, size_t n) {
        const size_t off = bytes.size();
        const char* c = (const char*)p;
        bytes.insert(bytes.end(), c, c + n);
        bytes.resize((bytes.size() + 15) & ~(size_t)15, 0);
        return (void*)(uintptr_t)(off + 1);
    }
    template <class T> const T* put(const std::vector<T>& v) { return (const T*)put_raw(v.data(), v.size() * sizeof(T)); }
    // numpy's pad1: an empty table is stored as one zero so that the pointer is never NULL
    template <class T> const T* put1(const std::vector<T>& v) {
        if (!v.empty()) return put(v);
        std::vector<T> z(1, T(0));
        return put(z);
    }
};

// hi = round-to-nearest-away TF32 of x (what cvt.rna.tf32.f32 gives), lo = x - hi exactly representable remainder
static inline void split_tf32(const std::vector<float>& x, std::vector<float>& hi, std::vector<float>& lo) {
    hi.resize(x.size()); lo.resize(x.size());
    for (size_t i = 0; i < x.size(); ++i) {
        uint32_t u; memcpy(&u, &x[i], 4);
        u = (u + 0x1000u) & 0xFFFFE000u;
        float h; memcpy(&h, &u, 4);
        hi[i] = h; lo[i] = x[i] - h;
    }
}

struct JointEntry { int kind; int src[3]; float w[3]; };   // 0 chain joint, 1 vertices (pick / barycentric), 2 contour slot, 3 regressed

// OpenPose (coco25) <- model joints, models/utils.py:32-141 (only the two variants the fitting path uses)
static inline std::vector<int> openpose_map(bool smplx) {
    static const int body_tail[14] = {12, 17, 19, 21, 16, 18, 20, 0, 2, 5, 8, 1, 4, 7};
    std::vector<int> out;
    out.push_back(smplx ? 55 : 24);
    for (int i = 0; i < 14; ++i) out.push_back(body_tail[i]);
    const int toes0 = smplx ? 56 : 25;
    for (int i = 0; i < 10; ++i) out.push_back(toes0 + i);
    if (!smplx) return out;
    // hands: wrist, then per finger (thumb, index, middle, ring, pinky) three chain joints and the tip vertex joint
    static const int firsts[2][5] = {{37, 25, 28, 34, 31}, {52, 40, 43, 49, 46}};
    static const int wrist[2] = {20, 21}, tip0[2] = {66, 71};
    for (int h = 0; h < 2; ++h) {
        out.push_back(wrist[h]);
        for (int f = 0; f < 5; ++f) {
            out.push_back(firsts[h][f]); out.push_back(firsts[h][f] + 1); out.push_back(firsts[h][f] + 2); out.push_back(tip0[h] + f);
        }
    }
    for (int i = 0; i < 51 + 17; ++i) out.push_back(76 + i);      // face landmarks + contour
    return out;
}
// [constants.JOINT_MAP[n] for n in constants.JOINT_NAMES] of the reference (constants.py:13-89): 25 OpenPose + 24 GT joints
static const int kSpinJointMap[49] = {24, 12, 17, 19, 21, 16, 18, 20, 0, 2, 5, 8, 1, 4, 7, 25, 26, 27, 28, 29, 30, 31, 32, 33, 34,
                                      8, 5, 45, 46, 4, 7, 21, 19, 17, 16, 18, 20, 47, 48, 49, 50, 51, 52, 53, 24, 26, 25, 28, 27};
// smplx.vertex_ids (the official model files do not carry them)
static const int kExtraVidsSmpl[21] = {332, 6260, 2800, 4071, 583, 3216, 3226, 3387, 6617, 6624, 6787,
                                       2746, 2319, 2445, 2556, 2673, 6191, 5782, 5905, 6016, 6133};
static const int kExtraVidsSmplx[21] = {9120, 9929, 9448, 616, 6, 5770, 5780, 8846, 8463, 8474, 8635,
                                        5361, 4933, 5058, 5169, 5286, 8079, 7669, 7794, 7905, 8022};

// in-place inverse and determinant of an n x n matrix (double, partial pivoting); returns false when singular
static inline bool invert(std::vector<double>& a, int n, double* det_out) {
    std::vector<double> inv((size_t)n * n, 0.0);
    for (int i = 0; i < n; ++i) inv[(size_t)i * n + i] = 1.0;
    double det = 1.0;
    for (int c = 0; c < n; ++c) {
        int piv = c;
        for (int r = c + 1; r < n; ++r) if (std::fabs(a[(size_t)r * n + c]) > std::fabs(a[(size_t)piv * n + c])) piv = r;
        if (a[(size_t)piv * n + c] == 0.0) return false;
        if (piv != c) {
            for (int k = 0; k < n; ++k) { std::swap(a[(size_t)piv * n + k], a[(size_t)c * n + k]); std::swap(inv[(size_t)piv * n + k], inv[(size_t)c * n + k]); }
            det = -det;
        }
        const double d = a[(size_t)c * n + c];
        det *= d;
        for (int k = 0; k < n; ++k) { a[(size_t)c * n + k] /= d; inv[(size_t)c * n + k] /= d; }
        for (int r = 0; r < n; ++r) {
            if (r == c) continue;
            const double fct = a[(size_t)r * n + c];
            if (fct == 0.0) continue;
            for (int k = 0; k < n; ++k) { a[(size_t)r * n + k] -= fct * a[(size_t)c * n + k]; inv[(size_t)r * n + k] -= fct * inv[(size_t)c * n + k]; }
        }
    }
    a.swap(inv);
    if (det_out) *det_out = det;
    return true;
}

struct Builder {
    const BfModelDesc& d;
    Arrays arr;
    int V, J, P, NB, NS, Kp, NP, K_used;
    bool smplx, tc;
    std::vector<float> vt;                   // [V,3]
    std::vector<float> sd;                   // [V,3,NS]
    std::vector<float> Bm_rows;              // [Kp, 3V]
    std::vector<float> xr;                   // J_regressor_extra [n_xr, V] (SMPL) or empty
    int n_xr = 0;
    std::vector<int> dyn_faces;              // [rows, n_dyn, 3] vertex ids
    int dyn_rows = 0, n_dyn = 0;
    std::vector<JointEntry> joint_table, ori_table;
    const char* err = nullptr;
    char msg[128] = "";                      // room for an error text with numbers in it (err points here)

    explicit Builder(const BfModelDesc& desc) : d(desc) {}

    struct Entry { int target, k; float w; };

    bool build_vset(const std::vector<int>& vids, const std::vector<JointEntry>& table, bool live, BfVSet* vs) {
        memset(vs, 0, sizeof(*vs));
        const int n = (int)vids.size();
        const int n_pad = round_up(std::max(n, 1), 32);
        std::vector<int> pos(V, -1);
        for (int i = 0; i < n; ++i) pos[vids[i]] = i;
        // blend matrix columns of the set
        std::vector<float> Bm((size_t)Kp * 3 * n_pad, 0.f);
        for (int k = 0; k < Kp; ++k)
            for (int i = 0; i < n; ++i)
                for (int c = 0; c < 3; ++c) Bm[(size_t)k * 3 * n_pad + 3 * i + c] = Bm_rows[(size_t)k * 3 * V + 3 * vids[i] + c];
        // ELL skinning weights: non-zero joints first (joint order kept), padded with (joint 0, weight 0)
        const float* W = d.weights;
        int nnz = 1;
        for (int i = 0; i < n; ++i) {
            int c = 0;
            for (int j = 0; j < J; ++j) c += W[(size_t)vids[i] * J + j] != 0.f;
            nnz = std::max(nnz, c);
        }
        std::vector<int32_t> ell_j((size_t)n_pad * nnz, 0);
        std::vector<float> ell_w((size_t)n_pad * nnz, 0.f);
        for (int i = 0; i < n; ++i) {
            int c = 0;
            for (int j = 0; j < J && c < nnz; ++j) {
                const float w = W[(size_t)vids[i] * J + j];
                if (w != 0.f) { ell_j[(size_t)i * nnz + c] = j; ell_w[(size_t)i * nnz + c] = w; ++c; }
            }
        }
        // CSR joint -> vertices of the set
        std::vector<int32_t> jv_ptr(J + 1, 0), jv_vid;
        std::vector<float> jv_w;
        for (int j = 0; j < J; ++j) {
            for (int i = 0; i < n; ++i) {
                const float w = W[(size_t)vids[i] * J + j];
                if (w != 0.f) { jv_vid.push_back(i); jv_w.push_back(w); }
            }
            jv_ptr[j + 1] = (int32_t)jv_vid.size();
        }
        // output joints
        const int K_out = (int)table.size();
        std::vector<int32_t> kj_kind(K_out, 0), kj_src((size_t)K_out * 3, 0);
        std::vector<float> kj_w((size_t)K_out * 3, 0.f);
        std::vector<int32_t> dyn_src;                       // [rows, n_dyn, 3] positions in the set
        std::vector<float> dyn_w;
        if (dyn_rows > 0) {
            dyn_src.resize(dyn_faces.size());
            for (size_t i = 0; i < dyn_faces.size(); ++i) dyn_src[i] = pos[dyn_faces[i]];
            dyn_w.assign(d.dynamic_lmk_bary_coords, d.dynamic_lmk_bary_coords + dyn_faces.size());
        }
        std::vector<int32_t> xr_ptr, xr_vid;
        std::vector<float> xr_w;
        bool has3 = false;
        for (const JointEntry& e : table) has3 |= e.kind == 3;
        int n_extra = 0;
        if (n_xr > 0 && has3) {
            n_extra = n_xr;
            xr_ptr.push_back(0);
            for (int r = 0; r < n_xr; ++r) {
                for (int v = 0; v < V; ++v) {
                    const float w = xr[(size_t)r * V + v];
                    if (w != 0.f) {
                        if (pos[v] < 0) { err = "extra joint regressor references a vertex outside the set"; return false; }
                        xr_vid.push_back(pos[v]); xr_w.push_back(w);
                    }
                }
                xr_ptr.push_back((int32_t)xr_vid.size());
            }
        }
        std::vector<Entry> entries;                          // static entries only: contour landmarks are scattered per yaw row
        std::vector<int32_t> dyn_k;
        for (int k = 0; k < K_out; ++k) {
            const JointEntry& e = table[k];
            kj_kind[k] = e.kind;
            if (e.kind == 0) {
                kj_src[3 * k] = e.src[0];
                entries.push_back({e.src[0], k, 1.0f});
            } else if (e.kind == 1) {
                for (int i = 0; i < 3; ++i) {
                    const int p = pos[e.src[i]];
                    if (p < 0) { err = "an output joint references a vertex outside the set"; return false; }
                    kj_src[3 * k + i] = p; kj_w[3 * k + i] = e.w[i];
                    if (e.w[i] != 0.f) entries.push_back({J + p, k, e.w[i]});
                }
            } else if (e.kind == 2) {
                kj_src[3 * k] = e.src[0];
                for (int a = 0; a < dyn_rows; ++a)
                    for (int i = 0; i < 3; ++i)
                        if (dyn_src[((size_t)a * n_dyn + e.src[0]) * 3 + i] < 0) { err = "a contour landmark references a vertex outside the set"; return false; }
                dyn_k.push_back(k);
            } else {
                const int r = e.src[0];
                kj_src[3 * k] = r;
                for (int q = xr_ptr[r]; q < xr_ptr[r + 1]; ++q) entries.push_back({J + xr_vid[q], k, xr_w[q]});
            }
        }
        std::stable_sort(entries.begin(), entries.end(), [](const Entry& a, const Entry& b) { return a.target != b.target ? a.target < b.target : a.k < b.k; });
        const int ntg = J + n;
        std::vector<int32_t> tg_ptr(ntg + 1, 0), tg_k, tg_a;
        std::vector<float> tg_w;
        for (const Entry& e : entries) { tg_ptr[e.target + 1]++; tg_k.push_back(e.k); tg_a.push_back(-1); tg_w.push_back(e.w); }
        for (int i = 0; i < ntg; ++i) tg_ptr[i + 1] += tg_ptr[i];

        vs->Bm = arr.put(Bm);
        vs->ell_j = arr.put(ell_j); vs->ell_w = arr.put(ell_w);
        vs->jv_ptr = arr.put(jv_ptr); vs->jv_vid = arr.put1(jv_vid); vs->jv_w = arr.put1(jv_w);
        vs->kj_kind = arr.put(kj_kind); vs->kj_src = arr.put(kj_src); vs->kj_w = arr.put(kj_w);
        vs->tg_ptr = arr.put(tg_ptr); vs->tg_k = arr.put1(tg_k); vs->tg_a = arr.put1(tg_a); vs->tg_w = arr.put1(tg_w);
        vs->n = n; vs->n_pad = n_pad; vs->ldn = 3 * n_pad; vs->nnz = nnz; vs->K_out = K_out; vs->n_dyn = 0; vs->n_extra = n_extra;
        if (tc) {
            std::vector<float> hi, lo, Bt((size_t)Kp * 3 * n_pad);
            split_tf32(Bm, hi, lo);
            vs->Bm_hi = arr.put(hi); vs->Bm_lo = arr.put(lo);
            for (int k = 0; k < Kp; ++k)
                for (int c = 0; c < 3 * n_pad; ++c) Bt[(size_t)c * Kp + k] = Bm[(size_t)k * 3 * n_pad + c];
            split_tf32(Bt, hi, lo);
            vs->Bt_hi = arr.put(hi); vs->Bt_lo = arr.put(lo);
        }
        const bool use_dyn = dyn_rows > 0 && !dyn_k.empty();
        if (use_dyn) {
            for (size_t s = 0; s < dyn_k.size(); ++s)
                if (table[dyn_k[s]].src[0] != (int)s) { err = "contour slots must appear in order"; return false; }
            if ((int)dyn_k.size() != n_dyn) { err = "every contour slot must be an output joint"; return false; }
            vs->dyn_src = arr.put(dyn_src); vs->dyn_w = arr.put(dyn_w); vs->dyn_k = arr.put(dyn_k);
            vs->n_dyn = n_dyn;
        }
        std::vector<int32_t> nzj;
        for (int j = 0; j < J; ++j) if (jv_ptr[j + 1] > jv_ptr[j]) nzj.push_back(j);
        vs->jv_nz = arr.put1(nzj);
        vs->n_nz = (int)nzj.size();
        if (live) build_live(n, entries, use_dyn ? &dyn_src : nullptr, dyn_w, dyn_k, vids, nzj, vs);
        if (!xr_ptr.empty()) { vs->xr_ptr = arr.put(xr_ptr); vs->xr_vid = arr.put1(xr_vid); vs->xr_w = arr.put1(xr_w); }
        return true;
    }

    // per contour row: live vertices, their gradient gather lists, the joint -> live-vertex skinning lists, block masks
    void build_live(int n, const std::vector<Entry>& entries, const std::vector<int32_t>* dyn_src, const std::vector<float>& dyn_w,
                    const std::vector<int32_t>& dyn_k, const std::vector<int>& vids, const std::vector<int32_t>& nzj, BfVSet* vs) {
        typedef std::vector<std::pair<int, float> > KW;
        const int rows = dyn_src ? dyn_rows : 1;
        std::map<int, KW> stat;
        for (const Entry& e : entries) if (e.target >= J) stat[e.target - J].push_back(std::make_pair(e.k, e.w));
        std::vector<std::map<int, KW> > per_row(rows, stat);
        if (dyn_src)
            for (int a = 0; a < rows; ++a)
                for (size_t s = 0; s < dyn_k.size(); ++s)
                    for (int i = 0; i < 3; ++i) {
                        const size_t q = ((size_t)a * n_dyn + s) * 3 + i;
                        per_row[a][(*dyn_src)[q]].push_back(std::make_pair((int)dyn_k[s], dyn_w[q]));
                    }
        size_t mx = 0;
        for (int a = 0; a < rows; ++a) mx = std::max(mx, per_row[a].size());
        const int lmax = round_up((int)mx, 32);
        const int nnzj = std::max(1, (int)nzj.size());
        std::vector<int32_t> lv_n(rows, 0), lv_vid((size_t)rows * lmax, 0), lt_ptr((size_t)rows * (lmax + 1), 0), lt_k;
        std::vector<int32_t> lj_ptr((size_t)rows * (nnzj + 1), 0), lj_vid;
        std::vector<float> lt_w, lj_w;
        std::vector<uint32_t> lv_blk(rows, 0u);
        const float* W = d.weights;
        for (int a = 0; a < rows; ++a) {
            std::vector<int> livev;
            for (std::map<int, KW>::const_iterator it = per_row[a].begin(); it != per_row[a].end(); ++it) livev.push_back(it->first);   // ascending
            const int L = (int)livev.size();
            lv_n[a] = L;
            for (int i = 0; i < L; ++i) {
                lv_vid[(size_t)a * lmax + i] = livev[i];
                lt_ptr[(size_t)a * (lmax + 1) + i] = (int32_t)lt_k.size();
                const KW& kw = per_row[a][livev[i]];
                for (size_t e = 0; e < kw.size(); ++e) { lt_k.push_back(kw[e].first); lt_w.push_back(kw[e].second); }
            }
            for (int i = L; i <= lmax; ++i) lt_ptr[(size_t)a * (lmax + 1) + i] = (int32_t)lt_k.size();
            for (size_t jn = 0; jn < nzj.size(); ++jn) {
                lj_ptr[(size_t)a * (nnzj + 1) + jn] = (int32_t)lj_vid.size();
                for (int i = 0; i < L; ++i) {
                    const float w = W[(size_t)vids[livev[i]] * J + nzj[jn]];
                    if (w != 0.f) { lj_vid.push_back(i); lj_w.push_back(w); }
                }
            }
            for (int jn = (int)nzj.size(); jn <= nnzj; ++jn) lj_ptr[(size_t)a * (nnzj + 1) + jn] = (int32_t)lj_vid.size();
            if ((n + 15) / 16 > 32) lv_blk[a] = 0xFFFFFFFFu;
            else for (int i = 0; i < L; ++i) lv_blk[a] |= 1u << (livev[i] / 16);
        }
        vs->lv_n = arr.put(lv_n); vs->lv_vid = arr.put(lv_vid); vs->lt_ptr = arr.put(lt_ptr);
        vs->lt_k = arr.put1(lt_k); vs->lt_w = arr.put1(lt_w);
        vs->lj_ptr = arr.put(lj_ptr); vs->lj_vid = arr.put1(lj_vid); vs->lj_w = arr.put1(lj_w);
        vs->lv_blk = arr.put(lv_blk);
        vs->lmax = lmax; vs->n_rows = rows;
    }

    bool run(BfModel* m) {
        memset(m, 0, sizeof(*m));
        smplx = d.is_smplx != 0; tc = d.tensor_cores != 0;
        V = d.V; J = d.J;
        if (!d.v_template || !d.shapedirs || !d.posedirs || !d.J_regressor || !d.weights || !d.parents || V <= 0 || J <= 1 || J > 64) {
            err = "v_template / shapedirs / posedirs / J_regressor / weights / parents are required (1 < J <= 64)"; return false;
        }
        for (int j = 1; j < J; ++j) if (d.parents[j] < 0 || d.parents[j] >= j) { err = "kinematic tree must be topologically sorted"; return false; }
        P = (J - 1) * 9;
        NB = d.num_betas;
        const int NE = smplx ? d.num_expression : 0;
        if (NB < 1 || NE < 0) { err = "num_betas must be at least 1 and num_expression not negative"; return false; }
        if (d.face_params && !smplx) { err = "face parameters (jaw pose, expression) apply to SMPL-X only"; return false; }
        const bool face = smplx && d.face_params != 0;
        const int S = d.n_shape_dirs;
        vt.assign(d.v_template, d.v_template + (size_t)V * 3);
        // shape directions: [V,3,NB] (+ the kid direction) (+ NE expression directions; official files keep them after 300)
        std::vector<float> kid;
        if (d.kid_template) {
            if (smplx) { err = "the kid template applies to SMPL only (smplify/smplify.py:50-56)"; return false; }
            if (S < NB) { err = "shapedirs has fewer directions than num_betas"; return false; }
            float mean[3] = {0.f, 0.f, 0.f};                 // float32 running sums, as numpy reduces the leading axis
            for (int v = 0; v < V; ++v) for (int c = 0; c < 3; ++c) mean[c] += d.kid_template[3 * v + c];
            for (int c = 0; c < 3; ++c) mean[c] = (float)((double)mean[c] / (double)V);
            kid.resize((size_t)V * 3);
            for (int v = 0; v < V; ++v)
                for (int c = 0; c < 3; ++c) {
                    const float centred = d.kid_template[3 * v + c] - mean[c];
                    kid[3 * v + c] = centred - vt[3 * v + c];
                }
        }
        const int NBk = NB + (kid.empty() ? 0 : 1);
        NS = NBk + NE;
        const bool official = smplx && S >= 300 + NE;
        if (!official && S < NB + NE) { err = "shapedirs has too few directions"; return false; }
        sd.resize((size_t)V * 3 * NS);
        for (int i = 0; i < V * 3; ++i) {
            for (int l = 0; l < NB; ++l) sd[(size_t)i * NS + l] = d.shapedirs[(size_t)i * S + l];
            if (!kid.empty()) sd[(size_t)i * NS + NB] = kid[i];
            for (int l = 0; l < NE; ++l) sd[(size_t)i * NS + NBk + l] = d.shapedirs[(size_t)i * S + (official ? 300 : NB) + l];
        }
        NB = NBk;
        const int Kdim = P + NS + 1;
        Kp = round_up(Kdim, 16);
        NP = 7 + (smplx ? 63 : 69) + NB + (smplx ? 18 : 0);
        // the kernels' per-frame limits (BF_MAXNS / BF_MAXNP), checked here so that such a model fails when it is built rather
        // than at its first launch; the Python builder raises the same text.  The 100-entry limit applies to the row without
        // the face block; that block (3 + NE entries) is bounded by the shape limit, so a face row has at most 111 entries.
        if (NS > BF_MAXNS) { snprintf(msg, sizeof(msg), "%d shape coefficients (betas + expression) exceed the limit of %d", NS, BF_MAXNS); err = msg; return false; }
        if (NP > BF_MAXNP) { snprintf(msg, sizeof(msg), "%d theta entries exceed the limit of %d", NP, BF_MAXNP); err = msg; return false; }
        if (face) NP += 3 + NE;                          // [jaw 3 | expression NE] after the right-hand PCA

        // kinematic tree
        std::vector<int32_t> parents(J), depth(J, 0), child_ptr(J + 1, 0), child_idx;
        parents[0] = -1;
        for (int j = 1; j < J; ++j) { parents[j] = d.parents[j]; depth[j] = depth[parents[j]] + 1; }
        for (int j = 0; j < J; ++j) {
            for (int c = 1; c < J; ++c) if (parents[c] == j) child_idx.push_back(c);
            child_ptr[j + 1] = (int32_t)child_idx.size();
        }
        child_idx.push_back(0);
        int max_depth = 0;
        for (int j = 0; j < J; ++j) max_depth = std::max(max_depth, (int)depth[j]);
        std::vector<int32_t> lvl_j(J), lvl_ptr(max_depth + 2, 0);
        for (int j = 0; j < J; ++j) lvl_j[j] = j;
        std::stable_sort(lvl_j.begin(), lvl_j.end(), [&](int a, int b) { return depth[a] < depth[b]; });
        for (int j = 0; j < J; ++j) lvl_ptr[depth[j] + 1]++;
        for (int l = 0; l <= max_depth; ++l) lvl_ptr[l + 1] += lvl_ptr[l];
        // regressor folded into template / shape directions (fp64 accumulation, rounded once)
        std::vector<float> Jt((size_t)J * 3), Jd((size_t)J * 3 * NS);
        {
            std::vector<double> acc(3 + 3 * NS);
            for (int j = 0; j < J; ++j) {
                std::fill(acc.begin(), acc.end(), 0.0);
                for (int v = 0; v < V; ++v) {
                    const double r = d.J_regressor[(size_t)j * V + v];
                    if (r == 0.0) continue;
                    for (int c = 0; c < 3; ++c) acc[c] += r * (double)vt[3 * v + c];
                    const float* s = &sd[(size_t)v * 3 * NS];
                    for (int q = 0; q < 3 * NS; ++q) acc[3 + q] += r * (double)s[q];
                }
                for (int c = 0; c < 3; ++c) Jt[3 * j + c] = (float)acc[c];
                for (int q = 0; q < 3 * NS; ++q) Jd[(size_t)j * 3 * NS + q] = (float)acc[3 + q];
            }
        }
        std::vector<float> pose_mean(3 * J, 0.f), hand_l, hand_r;
        if (smplx) {
            if (!d.hands_meanl || !d.hands_meanr || !d.hands_componentsl || !d.hands_componentsr || 3 * J < 165) { err = "SMPL-X needs the hand PCA tables"; return false; }
            for (int i = 0; i < 45; ++i) { pose_mean[75 + i] = d.hands_meanl[i]; pose_mean[120 + i] = d.hands_meanr[i]; }
            hand_l.assign(d.hands_componentsl, d.hands_componentsl + 6 * 45);
            hand_r.assign(d.hands_componentsr, d.hands_componentsr + 6 * 45);
        }

        // output joint table before the joint map
        std::vector<JointEntry> pre;
        for (int j = 0; j < J; ++j) pre.push_back({0, {j, 0, 0}, {1.f, 0.f, 0.f}});
        const int n_xv = d.extra_vids ? d.n_extra_vids : 21;
        for (int i = 0; i < n_xv; ++i) {
            const int v = d.extra_vids ? d.extra_vids[i] : (smplx ? kExtraVidsSmplx[i] : kExtraVidsSmpl[i]);
            if (v < 0 || v >= V) { err = "vertex-picked joint ids outside the mesh"; return false; }
            pre.push_back({1, {v, v, v}, {1.f, 0.f, 0.f}});
        }
        std::vector<int> jmap;
        if (smplx) {
            if (!d.faces || !d.lmk_faces_idx || !d.lmk_bary_coords || !d.dynamic_lmk_faces_idx || !d.dynamic_lmk_bary_coords) { err = "SMPL-X needs faces and the landmark tables"; return false; }
            if (d.F <= 0 || d.n_lmk < 0 || d.n_dyn_rows <= 0 || d.n_dyn <= 0) { err = "SMPL-X needs F, n_dyn_rows, n_dyn > 0"; return false; }
            for (int i = 0; i < d.n_lmk; ++i)
                if (d.lmk_faces_idx[i] < 0 || d.lmk_faces_idx[i] >= d.F) { err = "lmk_faces_idx outside the face list"; return false; }
            for (size_t i = 0; i < (size_t)d.n_dyn_rows * d.n_dyn; ++i)
                if (d.dynamic_lmk_faces_idx[i] < 0 || d.dynamic_lmk_faces_idx[i] >= d.F) { err = "dynamic_lmk_faces_idx outside the face list"; return false; }
            for (size_t i = 0; i < (size_t)d.F * 3; ++i)
                if (d.faces[i] < 0 || d.faces[i] >= V) { err = "faces reference a vertex outside the mesh"; return false; }
            for (int i = 0; i < d.n_lmk; ++i) {
                const int32_t* fc = d.faces + 3 * (size_t)d.lmk_faces_idx[i];
                const float* b = d.lmk_bary_coords + 3 * (size_t)i;
                pre.push_back({1, {fc[0], fc[1], fc[2]}, {b[0], b[1], b[2]}});
            }
            dyn_rows = d.n_dyn_rows; n_dyn = d.n_dyn;
            dyn_faces.resize((size_t)dyn_rows * n_dyn * 3);
            for (size_t i = 0; i < (size_t)dyn_rows * n_dyn; ++i)
                for (int c = 0; c < 3; ++c) dyn_faces[3 * i + c] = d.faces[3 * (size_t)d.dynamic_lmk_faces_idx[i] + c];
            for (int s = 0; s < n_dyn; ++s) pre.push_back({2, {s, 0, 0}, {0.f, 0.f, 0.f}});
            jmap = openpose_map(true);
            K_used = (int)jmap.size();
        } else {
            if (d.J_regressor_extra && d.n_regressor_extra > 0) {
                n_xr = d.n_regressor_extra;
                xr.assign(d.J_regressor_extra, d.J_regressor_extra + (size_t)n_xr * V);
                for (int r = 0; r < n_xr; ++r) pre.push_back({3, {r, 0, 0}, {0.f, 0.f, 0.f}});
                jmap.assign(kSpinJointMap, kSpinJointMap + 49);
            } else {
                jmap = openpose_map(false);
            }
            K_used = 25;
        }
        for (size_t i = 0; i < jmap.size(); ++i) {
            if (jmap[i] < 0 || jmap[i] >= (int)pre.size()) { err = "joint map exceeds the model's joint list"; return false; }
            joint_table.push_back(pre[jmap[i]]);
        }
        if (!smplx) ori_table.assign(pre.begin(), pre.begin() + J + n_xv);

        // GMM prior (smplify/prior.py:127-174)
        int n_gmm = 0;
        if (d.gmm_means && d.gmm_covars && d.gmm_weights && d.n_gmm > 0) {
            n_gmm = d.n_gmm;
            const int D = 69;
            std::vector<float> means(d.gmm_means, d.gmm_means + (size_t)n_gmm * D), psym((size_t)n_gmm * D * 72, 0.f), logw(n_gmm);
            std::vector<double> sqrdet(n_gmm);
            std::vector<std::vector<float> > prec(n_gmm);
            for (int c = 0; c < n_gmm; ++c) {
                std::vector<double> a((size_t)D * D);
                for (int i = 0; i < D * D; ++i) a[i] = (double)d.gmm_covars[(size_t)c * D * D + i];
                double det = 0.0;
                if (!invert(a, D, &det) || !(det > 0.0)) { err = "GMM covariance is not positive definite"; return false; }
                sqrdet[c] = std::sqrt(det);
                prec[c].resize((size_t)D * D);
                for (int i = 0; i < D * D; ++i) prec[c][i] = (float)a[i];
            }
            double mn = sqrdet[0];
            for (int c = 1; c < n_gmm; ++c) mn = std::min(mn, sqrdet[c]);
            const double cst = std::pow(2.0 * 3.14159265358979323846, 69 / 2.0);
            for (int c = 0; c < n_gmm; ++c) {
                const float nllw = (float)((double)d.gmm_weights[c] / (cst * (sqrdet[c] / mn)));
                logw[c] = std::log(nllw);
                for (int i = 0; i < D; ++i)
                    for (int j = 0; j < D; ++j)
                        psym[((size_t)c * D + i) * 72 + j] = (prec[c][(size_t)i * D + j] + prec[c][(size_t)j * D + i]) * 0.5f;
            }
            m->gmm_mean = arr.put(means); m->gmm_psym = arr.put(psym); m->gmm_logw = arr.put(logw);
            if (tc && (n_gmm * 72) % 192 == 0) {
                std::vector<float> bt((size_t)n_gmm * 72 * 80, 0.f), hi, lo;
                for (int c = 0; c < n_gmm; ++c)
                    for (int i = 0; i < D; ++i) {
                        double dot = 0.0;
                        for (int j = 0; j < D; ++j) {
                            const float p = psym[((size_t)c * D + i) * 72 + j];
                            bt[((size_t)c * 72 + i) * 80 + j] = p;
                            dot += (double)p * (double)means[(size_t)c * D + j];
                        }
                        bt[((size_t)c * 72 + i) * 80 + 69] = -(float)dot;
                    }
                split_tf32(bt, hi, lo);
                m->gmm_bt_hi = arr.put(hi); m->gmm_bt_lo = arr.put(lo);
            }
        }

        // blend matrix rows over all vertices
        Bm_rows.assign((size_t)Kp * 3 * V, 0.f);
        for (int i = 0; i < 3 * V; ++i) {
            for (int p = 0; p < P; ++p) Bm_rows[(size_t)p * 3 * V + i] = d.posedirs[(size_t)i * P + p];
            for (int l = 0; l < NS; ++l) Bm_rows[(size_t)(P + l) * 3 * V + i] = sd[(size_t)i * NS + l];
            Bm_rows[(size_t)(P + NS) * 3 * V + i] = vt[i];
        }
        // active set: vertices every frame uses (ascending), then contour candidates by the first yaw row that uses them
        std::set<int> stat;
        for (int k = 0; k < K_used; ++k) {
            const JointEntry& e = joint_table[k];
            if (e.kind == 1) { for (int i = 0; i < 3; ++i) if (e.w[i] != 0.f) stat.insert(e.src[i]); }
            else if (e.kind == 3) { for (int v = 0; v < V; ++v) if (xr[(size_t)e.src[0] * V + v] != 0.f) stat.insert(v); }
        }
        std::map<int, int> first_row;
        for (int k = 0; k < K_used; ++k) {
            const JointEntry& e = joint_table[k];
            if (e.kind != 2) continue;
            for (int a = 0; a < dyn_rows; ++a)
                for (int i = 0; i < 3; ++i) {
                    const int x = dyn_faces[((size_t)a * n_dyn + e.src[0]) * 3 + i];
                    if (stat.count(x)) continue;
                    std::map<int, int>::iterator it = first_row.find(x);
                    if (it == first_row.end()) first_row[x] = a; else it->second = std::min(it->second, a);
                }
        }
        std::vector<int> active(stat.begin(), stat.end());
        {
            std::vector<std::pair<int, int> > cand;           // (first row, vertex)
            for (std::map<int, int>::const_iterator it = first_row.begin(); it != first_row.end(); ++it) cand.push_back(std::make_pair(it->second, it->first));
            std::sort(cand.begin(), cand.end());
            for (size_t i = 0; i < cand.size(); ++i) active.push_back(cand[i].second);
        }

        m->parents = arr.put(parents); m->depth = arr.put(depth); m->lvl_ptr = arr.put(lvl_ptr); m->lvl_j = arr.put(lvl_j);
        m->child_ptr = arr.put(child_ptr); m->child_idx = arr.put(child_idx);
        m->Jt = arr.put(Jt); m->Jd = arr.put(Jd); m->pose_mean = arr.put(pose_mean);
        if (smplx) { m->hand_l = arr.put(hand_l); m->hand_r = arr.put(hand_r); }
        std::vector<int> all(V);
        for (int v = 0; v < V; ++v) all[v] = v;
        std::vector<JointEntry> full_table(joint_table);
        full_table.insert(full_table.end(), ori_table.begin(), ori_table.end());
        if (!build_vset(all, full_table, false, &m->full)) return false;
        std::vector<JointEntry> act_table(joint_table.begin(), joint_table.begin() + K_used);
        if (!build_vset(active, act_table, true, &m->act)) return false;
        m->J = J; m->P = P; m->NS = NS; m->NB = NB; m->Kp = Kp; m->NP = NP; m->is_smplx = smplx ? 1 : 0;
        m->max_depth = max_depth; m->K_used = K_used; m->n_gmm = n_gmm; m->face = face ? 1 : 0;
        return true;
    }
};

}  // namespace bfb
