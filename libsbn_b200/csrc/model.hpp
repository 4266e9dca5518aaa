// Host-side phylogenetic model tables: what FatBeagle::SetParameters ->
// PhyloModel::SetParameters -> UpdatePhyloModelInBeagle produces per tree
// (reference src/fat_beagle.cpp:43-46, 273-300), as flat POD the kernels read.
#ifndef SBNB_MODEL_HPP_
#define SBNB_MODEL_HPP_

#include <map>
#include <string>
#include <utility>
#include <vector>

namespace sbnb {

enum class SubstitutionKind { kJC69, kGTR, kHKY };
enum class SiteKind { kConstant, kWeibull, kGamma };
enum class ClockKind { kNone, kStrict };

// Layout of one row of the phylo_model_params matrix: the reference's
// BlockSpecification (src/block_specification.cpp, src/phylo_model.cpp:11-13).
struct ModelSpec {
  SubstitutionKind substitution = SubstitutionKind::kJC69;
  SiteKind site = SiteKind::kConstant;
  ClockKind clock = ClockKind::kNone;
  int category_count = 1;
  // "<site>+I": a proportion of invariable sites, the last entry of the "entire site" block
  bool invariant = false;
  int param_count = 0;
  // key -> (start, length); same keys the python block map shows.
  std::map<std::string, std::pair<int, int>> blocks;

  static ModelSpec Parse(const std::string& substitution, const std::string& site,
                         const std::string& clock);
  std::pair<int, int> Block(const std::string& key) const;
  // Number of stick-breaking coordinates the finite-difference substitution
  // gradient runs over (GTR: 5 rates + 3 frequencies; fat_beagle.cpp:440-465).
  int SubstitutionGradientSize() const;
  // Entries of one tree's "site_model" gradient row: the shape (Weibull, Gamma), then the
  // proportion invariant (+I); 1 for a constant site model without +I (always 0).
  int SiteGradientSize() const;
};

// The fused tree walk gives every rate category of a site pattern its own lane, so a
// pattern takes at most one warp of categories.
constexpr int kMaxCategories = 32;

// Everything the kernels need to know about the substitution + site model of
// one (virtual) tree.  Row-major 4x4 blocks, as BEAGLE receives them
// (fat_beagle.cpp:289-293).
struct ModelTables {
  double evec[16];      // V
  double ivec[16];      // V^-1
  double eval[4];       // Lambda
  double freqs[4];      // pi
  double q[16];         // rate matrix Q (unit expected rate)
  double rates[kMaxCategories];     // category rates r_c           (first category_count used)
  double weights[kMaxCategories];   // category proportions p_c
  double drates[kMaxCategories];    // d r_c / d shape (Weibull, Gamma; 0 for a constant site model)
  double pinv;                      // proportion of invariable sites (+I; 0 otherwise).  rates and
                                    // drates are then divided by 1 - pinv: the mean rate stays 1
};

// substitution_model.cpp:17-80 (GTR), substitution_model.hpp:59-74 (JC69).
// `params` points at the "entire substitution" block of a row.
void BuildSubstitution(const ModelSpec& spec, const double* params, ModelTables* out);
// site_model.cpp:37-62 (Weibull median discretisation) / constant / discrete Gamma
// (an addition: the reference has no Gamma site model; same median discretisation).
// `params` points at the "entire site" block of a row.
void BuildSite(const ModelSpec& spec, const double* params, ModelTables* out);
// Whole row -> tables.
void BuildModelTables(const ModelSpec& spec, const double* row, ModelTables* out);

// Analytic substitution-parameter gradient (SURVEY.md 8f-1), host part.  With
// P = exp(Q tau) = V exp(Lambda tau) V^-1,
//     d P / d theta = V [ (V^-1 dQ/dtheta V) o Phi(tau) ] V^-1,
//     Phi_kl = (e^{lambda_k tau} - e^{lambda_l tau}) / (lambda_k - lambda_l)   (tau e^{lambda_k tau} when equal),
// so  d logL / d theta = < W, B_theta > + d pi / d theta . R  with  B_theta = V^-1 dQ/dtheta V  and the
// device sums  W_kl = sum over edges, categories, patterns of  w/lik (V^T T)_k (V^-1 L)_l Phi_kl,
// R_j = sum of w/lik p_c L_root,j.  theta runs over the reference's gradient coordinates
// (fat_beagle.cpp:440-465): GTR -> 5 stick-breaking coordinates of the rates, then 3 of the
// frequencies; HKY -> kappa, then 3 of the frequencies.
struct SubstitutionDerivatives {
  int count = 0;
  double b[8][16];      // B_theta, row-major
  double dfreqs[8][4];  // d pi / d theta
};
void BuildSubstitutionDerivatives(const ModelSpec& spec, const double* row, const ModelTables& tables,
                                  SubstitutionDerivatives* out);
// d x / d y of the stick-breaking transform: jacobian[m * (simplex_size - 1) + k] = d x_m / d y_k.
void StickBreakingJacobian(const double* y, int simplex_size, double* jacobian);

// stick_breaking_transform.cpp:20-43: simplex <-> unconstrained coordinates.
void StickBreaking(const double* y, int simplex_size, double* x);
void StickBreakingInverse(const double* x, int simplex_size, double* y);

// Cyclic Jacobi eigensolver for a symmetric 4x4 (row-major); eigenvectors in the
// columns of `vectors`.  P(t) is invariant to eigenvector order and sign, so any
// accurate solver reproduces Eigen::SelfAdjointEigenSolver's P(t).
void SymmetricEigen4(const double* matrix, double* values, double* vectors);

// Regularized lower incomplete gamma function P(a, x) and its inverse in x
// (the quantile function of a unit-scale Gamma distribution with shape a).
double RegularizedGammaP(double a, double x);
double InverseRegularizedGammaP(double a, double p);

}  // namespace sbnb

#endif  // SBNB_MODEL_HPP_
