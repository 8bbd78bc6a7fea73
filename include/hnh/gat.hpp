// hnh/gat.hpp -- multi-head graph attention on top of a Distributed_Sparse object: the forward pass (the second
// application that benchmark_algorithm can run, app == "gat"), and a backward pass with a plain SGD step for
// training.  Class and member names follow the reference (GATLayer, GAT{d_ops, layers, buffers, leaky_relu_alpha,
// computeSelfAttentionHead, forwardPass}: gat.hpp:26-113; used at benchmark_dist.cpp:88-94,133-135) so that its
// callers compile; the reference stops at the forward pass (its backward pass is marked work in progress).
//
// One head of one layer:
//     H      = X_in * W                       dense projection          (hnh_dgemm_f64: own fp64 DMMA kernel)
//     e_uv   = <H_u, H_v> for every edge      SDDMM through d_ops       (K1)
//     e_uv   = LeakyReLU(e_uv)                                           (hnh_leaky_relu_f64)
//     Z      = E * H                          SpMM through d_ops        (K2)
//     X_out[:, head window] = ReLU(Z)                                    (hnh_relu_cols_f64)
// All operands stay in HBM between the steps.  The weights are whatever the caller stores in
// layers[i].wMats[j]; the reference leaves them zero and never assigns leaky_relu_alpha (reading it is
// undefined there) -- this implementation defaults alpha to 0.2.
//
// Backward pass of one head, given Ybar = dL/d(layer output), with Y the layer output and w the head's column window:
//     G      = Ybar[:, w] o [Y[:, w] > 0]                                (hnh_relu_cols_backward_f64; ReLU'(0) = 0)
//     ebar   = <G_u, H_v> * LReLU'(e_uv) on every edge                  SDDMM with the slope as S values
//     Hbar   = ebar H (rows) + ebar^T H + a^T G (columns)                one spmmA + two spmmB
//     Wbar   = X^T Hbar, summed over all ranks                          (hnh_dgemm_tn_f64, one world all-reduce)
//     Xbar  += Hbar W^T over the heads                                   (hnh_dgemm_nt_f64)
// H and e are recomputed from `buffers` rather than kept from the forward pass, which therefore stays as it is and
// needs no extra memory.  The A-mode operations work in S-value order and the B-mode ones in ST-value order, so the
// edge values are computed once in each order.
#pragma once
#include <string>
#include <vector>

#include "hnh/15D_dense_shift.hpp"
#include "hnh/distributed_sparse.h"
#include "hnh_b200.h"

class GATLayer {
public:
    int input_features;
    int features_per_head;
    int num_heads;

    vector<DenseMatrix> wMats;  // one input_width x head_width projection per head
    VectorXd a1;                // attention vectors: declared by the reference, unused by its forward pass
    VectorXd a2;

    GATLayer(int in_width, int head_width, int heads)
        : input_features(in_width), features_per_head(head_width), num_heads(heads) {}
    int output_features() const { return features_per_head * num_heads; }
};

class GAT {
public:
    Distributed_Sparse *d_ops;
    vector<GATLayer> layers;
    vector<DenseMatrix> buffers;  // [0] network input (B-shaped), [i + 1] output of layer i (A-shaped)
    double leaky_relu_alpha = 0.2;
    vector<vector<DenseMatrix>> wGrads;  // [layer][head]: dL/d wMats, identical on every rank (backwardPass)
    DenseMatrix input_grad;              // dL/d buffers[0], this rank's rows (backwardPass)

    GAT(vector<GATLayer> &l_input, Distributed_Sparse *ops) : d_ops(ops), layers(l_input) {
        if (layers.empty()) throw hnh::Error(-1, "GAT: no layers");
        for (size_t i = 1; i < layers.size(); i++)
            if (layers[i].input_features != layers[i - 1].output_features())
                throw hnh::Error(-1, "GAT: layer " + std::to_string(i) + " does not take the width layer " +
                                         std::to_string(i - 1) + " produces");
        // Shapes come from the algorithm object at the R in force, as in the reference (gat.hpp:60-79):
        // the input is B-shaped at R = input width, layer outputs are A-shaped at R = heads * head width,
        // a head's projection maps the previous buffer's local columns onto localAcols at R = head width.
        d_ops->setRValue(layers.front().input_features);
        buffers.push_back(d_ops->like_B_matrix(0.0));
        for (GATLayer &layer : layers) {
            const int64_t in_cols = buffers.back().cols();
            d_ops->setRValue(layer.output_features());
            buffers.push_back(d_ops->like_A_matrix(0.0));
            d_ops->setRValue(layer.features_per_head);
            layer.wMats.clear();
            for (int h = 0; h < layer.num_heads; h++)
                layer.wMats.push_back(DenseMatrix::Constant(in_cols, d_ops->localAcols, 0.0));
        }
    }

    // head j of layer i: reads buffers[i], writes its column window of buffers[i + 1]
    void computeSelfAttentionHead(int i, int j) {
        GATLayer &layer = layers.at((size_t)i);
        DenseMatrix &input = buffers[(size_t)i], &output = buffers[(size_t)i + 1];
        d_ops->setRValue(layer.features_per_head);

        DenseMatrix projected = input * layer.wMats.at((size_t)j);
        DenseMatrix neighbours = projected;  // the same projection in the role of the other SDDMM operand
        d_ops->de_shift(&neighbours, nullptr, k_spmmA);

        VectorXd pattern = d_ops->like_S_values(1.0);
        VectorXd scores = d_ops->like_S_values(1.0);
        d_ops->algorithm(projected, neighbours, pattern, &scores, k_sddmmA, true);
        scores.leakyRelu(leaky_relu_alpha);

        projected.setZero();  // becomes the SpMM accumulator
        d_ops->algorithm(projected, neighbours, scores, nullptr, k_spmmA, false);
        output.setMiddleColsRelu((int64_t)j * projected.cols(), projected);
    }

    void forwardPass() {
        for (size_t i = 0; i < layers.size(); i++)
            for (int j = 0; j < layers[i].num_heads; j++) computeSelfAttentionHead((int)i, j);
    }

    // Why backwardPass cannot run on this layout, or "" when it can.  The backward pass is the derivative of the
    // global GAT formula, so it runs where the forward pass computes that formula: any algorithm on one rank, the
    // 1.5D dense-shift algorithm with fusion 1 at any c and with fusion 2 at c = 1, square matrices only.
    string backwardUnsupportedReason() const {
        if (d_ops->M != d_ops->N) return "the backward pass needs a square matrix (M != N)";
        if (d_ops->localArows != d_ops->localBrows) return "the A and B row blocks of this layout differ";
        if (d_ops->p == 1) return "";
        const Sparse15D_Dense_Shift *ds = dynamic_cast<const Sparse15D_Dense_Shift *>(d_ops);
        if (!ds)
            return "on more than one rank the backward pass needs the 1.5D dense-shift algorithm (" + d_ops->algorithm_name +
                   " splits the dense operands differently)";
        if (ds->fusionApproach == 2 && ds->c > 1)
            return "1.5D fusion 2 with c > 1 accumulates its SpMM onto the gathered projection (as the reference does), so "
                   "its forward pass is not the GAT formula";
        return "";
    }
    bool supportsBackward() const { return backwardUnsupportedReason().empty(); }

    // Gradients of L with respect to every weight (wGrads) and to the network input (input_grad), given
    // output_grad = dL/d buffers.back() (this rank's rows).  Assumes `buffers` hold the forward pass for the current
    // weights.  Overwrites the gradients (no accumulation); stream-ordered on the compute stream like forwardPass.
    // Throws hnh::Error(HNH_E_INVALID) before enqueuing anything where supportsBackward() is false.
    void backwardPass(const DenseMatrix &output_grad) {
        const string why = backwardUnsupportedReason();
        if (!why.empty()) throw hnh::Error(HNH_E_INVALID, "GAT::backwardPass: " + why);
        if (output_grad.rows() != buffers.back().rows() || output_grad.cols() != buffers.back().cols())
            throw hnh::Error(HNH_E_INVALID, "GAT::backwardPass: the output gradient must have the shape of buffers.back()");
        wGrads.resize(layers.size());
        DenseMatrix upstream;  // dL/d buffers[i + 1] for i < layers.size() - 1
        for (size_t i = layers.size(); i-- > 0;) {
            const DenseMatrix &grad_out = i + 1 == layers.size() ? output_grad : upstream;
            DenseMatrix grad_in(buffers[i].rows(), buffers[i].cols());
            wGrads[i].resize((size_t)layers[i].num_heads);
            for (int j = 0; j < layers[i].num_heads; j++) computeSelfAttentionHeadBackward((int)i, j, grad_out, grad_in);
            upstream = std::move(grad_in);
        }
        input_grad = std::move(upstream);
        if (d_ops->p > 1) {
            // every rank owns distinct rows of the graph: the weight gradients are the sum over ranks
            hnh::Comm &world = *hnh::Comm::world();
            for (vector<DenseMatrix> &heads : wGrads)
                for (DenseMatrix &g : heads) world.allreduce_sum_f64(g.data(), (size_t)g.size(), hnh::Runtime::get().compute_stream());
        }
    }

    // Plain SGD: wMats[i][j] -= learning_rate * wGrads[i][j], on the compute stream.
    void applyGradients(double learning_rate) {
        if (wGrads.size() != layers.size()) throw hnh::Error(HNH_E_INVALID, "GAT::applyGradients: no gradients (run backwardPass first)");
        for (size_t i = 0; i < layers.size(); i++)
            for (size_t j = 0; j < layers[i].wMats.size(); j++) {
                DenseMatrix &w = layers[i].wMats[j];
                hnh::abi_check(hnh_axpby_f64(w.data(), 1.0, w.data(), -learning_rate, wGrads[i][j].data(), w.size(),
                                             hnh::Runtime::get().compute_stream()),
                               "GAT::applyGradients");
            }
    }

    // head j of layer i: wGrads[i][j] = X^T Hbar (this rank's rows), grad_in (+)= Hbar W^T (overwritten by head 0)
    void computeSelfAttentionHeadBackward(int i, int j, const DenseMatrix &grad_out, DenseMatrix &grad_in) {
        GATLayer &layer = layers.at((size_t)i);
        DenseMatrix &input = buffers[(size_t)i], &output = buffers[(size_t)i + 1];
        DenseMatrix &weights = layer.wMats.at((size_t)j);
        const int64_t f = layer.features_per_head;
        cudaStream_t s = hnh::Runtime::get().compute_stream();
        d_ops->setRValue(layer.features_per_head);

        // the forward quantities, recomputed as computeSelfAttentionHead makes them
        DenseMatrix projected = input * weights;
        DenseMatrix neighbours = projected;
        d_ops->de_shift(&neighbours, nullptr, k_spmmA);
        VectorXd ones_S = d_ops->like_S_values(1.0), ones_T = d_ops->like_ST_values(1.0);
        VectorXd slope_S = d_ops->like_S_values(0.0), scores_T = d_ops->like_ST_values(0.0);
        d_ops->sddmmA(projected, neighbours, ones_S, slope_S);
        d_ops->sddmmB(projected, neighbours, ones_T, scores_T);
        VectorXd slope_T(scores_T.size());
        hnh::abi_check(hnh_leaky_relu_slope_f64(slope_S.data(), slope_S.data(), slope_S.size(), leaky_relu_alpha, s), "slope");
        hnh::abi_check(hnh_leaky_relu_slope_f64(slope_T.data(), scores_T.data(), scores_T.size(), leaky_relu_alpha, s), "slope");
        scores_T.leakyRelu(leaky_relu_alpha);  // the attention values a, in ST order

        // G: the gradient of the head's pre-ReLU output
        DenseMatrix g(output.rows(), f);
        hnh::abi_check(hnh_relu_cols_backward_f64(g.data(), grad_out.data(), output.data(), output.cols(), (int64_t)j * f,
                                                  output.rows(), f, s),
                       "relu_cols_backward");
        // edge gradients: each SDDMM result is SValues o dot, so the LeakyReLU slope rides in as the S values
        VectorXd edge_S = d_ops->like_S_values(0.0), edge_T = d_ops->like_ST_values(0.0);
        d_ops->sddmmA(g, neighbours, slope_S, edge_S);
        d_ops->sddmmB(g, neighbours, slope_T, edge_T);

        // Hbar: row side of the SDDMM, column side of the SDDMM, and the SpMM
        DenseMatrix h_grad = d_ops->like_A_matrix(0.0);
        DenseMatrix from_spmm = d_ops->like_B_matrix(0.0), from_cols = d_ops->like_B_matrix(0.0);
        d_ops->spmmA(h_grad, neighbours, edge_S);
        d_ops->spmmB(g, from_spmm, scores_T);
        d_ops->spmmB(projected, from_cols, edge_T);
        h_grad += from_spmm;
        h_grad += from_cols;

        DenseMatrix &w_grad = wGrads[(size_t)i][(size_t)j];
        w_grad.resize(weights.rows(), weights.cols());
        hnh::abi_check(hnh_dgemm_tn_f64(w_grad.data(), input.data(), h_grad.data(), input.rows(), f, weights.rows(), s),
                       "dgemm_tn");
        hnh::abi_check(hnh_dgemm_nt_f64(grad_in.data(), h_grad.data(), weights.data(), h_grad.rows(), weights.rows(), f,
                                        j == 0 ? 0.0 : 1.0, s),
                       "dgemm_nt");
    }
};
