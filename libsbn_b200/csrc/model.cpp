#include "model.hpp"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <sstream>
#include <vector>

#include "common.hpp"

namespace sbnb {

namespace {

void AppendBlock(ModelSpec* spec, const std::string& entire_key,
                 const std::vector<std::pair<std::string, int>>& sub_blocks) {
  // The reference keeps ParamCounts in a std::map, so sub-blocks are laid out
  // in key order (block_specification.cpp:10-21): "GTR rates" < "frequencies".
  std::vector<std::pair<std::string, int>> sorted = sub_blocks;
  std::sort(sorted.begin(), sorted.end());
  const int start = spec->param_count;
  for (const auto& [key, length] : sorted) {
    spec->blocks[key] = {spec->param_count, length};
    spec->param_count += length;
  }
  spec->blocks[entire_key] = {start, spec->param_count - start};
}

// One lane of a warp per rate category in the fused tree walk: 1 to 32.
void CheckCategoryCount(const ModelSpec& spec, const std::string& site) {
  if (spec.category_count < 1 || spec.category_count > kMaxCategories)
    Fail(SBNB_ERR_INVALID_ARGUMENT,
         "Site model category count out of range [1," + std::to_string(kMaxCategories) + "]: " + site +
             " (the fused tree walk gives each rate category one lane of a warp; libhmsbeagle_b200.so, the "
             "BEAGLE-compatible device library behind the unmodified FatBeagle, takes any number)");
}

// "weibull" / "gamma" (4 categories) or "weibull+K" / "gamma+K" with K all digits.
int CategoryCount(const std::string& base, const std::string& name, const std::string& site) {
  if (base == name) return 4;
  const std::string digits = base.substr(std::min(base.size(), name.size() + 1));
  if (base.compare(0, name.size() + 1, name + "+") != 0 || digits.empty() || digits.size() > 9 ||
      digits.find_first_not_of("0123456789") != std::string::npos)
    Fail(SBNB_ERR_INVALID_ARGUMENT, "Site model not known: " + site);
  return std::stoi(digits);
}

// The "entire site" block: the shape (if any), then "proportion invariant" for +I.
void AppendSiteBlock(ModelSpec* spec, const char* shape_key) {
  std::vector<std::pair<std::string, int>> sub_blocks;
  if (shape_key) sub_blocks.push_back({shape_key, 1});
  const int start = spec->param_count;
  AppendBlock(spec, "entire site", sub_blocks);
  if (spec->invariant) {
    spec->blocks["proportion invariant"] = {spec->param_count, 1};
    spec->param_count += 1;
    spec->blocks["entire site"] = {start, spec->param_count - start};
  }
}

}  // namespace

ModelSpec ModelSpec::Parse(const std::string& substitution, const std::string& site,
                           const std::string& clock) {
  ModelSpec spec;
  if (substitution == "JC69") {
    spec.substitution = SubstitutionKind::kJC69;
    AppendBlock(&spec, "entire substitution", {});
  } else if (substitution == "GTR") {
    spec.substitution = SubstitutionKind::kGTR;
    AppendBlock(&spec, "entire substitution", {{"GTR rates", 6}, {"frequencies", 4}});
  } else if (substitution == "HKY") {
    spec.substitution = SubstitutionKind::kHKY;
    AppendBlock(&spec, "entire substitution", {{"kappa", 1}, {"frequencies", 4}});
  } else {
    // substitution_model.cpp:14
    Fail(SBNB_ERR_INVALID_ARGUMENT, "Substitution model not known: " + substitution);
  }
  // "<site>+I": the suffix is split off before the category count is read, so that
  // "weibull+4+I" is Weibull with 4 categories and a proportion invariant.
  const bool invariant = site.size() >= 2 && site.compare(site.size() - 2, 2, "+I") == 0;
  const std::string base = invariant ? site.substr(0, site.size() - 2) : site;
  spec.invariant = invariant;
  if (base == "constant") {
    spec.site = SiteKind::kConstant;
    spec.category_count = 1;
    AppendSiteBlock(&spec, nullptr);
  } else if (site.rfind("weibull", 0) == 0) {
    // site_model.cpp:15-22: "weibull" (4 categories) or "weibull+K".
    spec.site = SiteKind::kWeibull;
    spec.category_count = CategoryCount(base, "weibull", site);
    CheckCategoryCount(spec, site);
    AppendSiteBlock(&spec, "Weibull shape");
  } else if (site.rfind("gamma", 0) == 0) {
    // Not in the reference (its "Gamma-4" is weibull+4): "gamma" (4 categories) or "gamma+K".
    spec.site = SiteKind::kGamma;
    spec.category_count = CategoryCount(base, "gamma", site);
    CheckCategoryCount(spec, site);
    AppendSiteBlock(&spec, "Gamma shape");
  } else {
    Fail(SBNB_ERR_INVALID_ARGUMENT, "Site model not known: " + site);
  }
  if (clock == "none") {
    spec.clock = ClockKind::kNone;
    AppendBlock(&spec, "entire clock", {});
  } else if (clock == "strict") {
    spec.clock = ClockKind::kStrict;
    AppendBlock(&spec, "entire clock", {{"clock rate", 1}});
  } else {
    Fail(SBNB_ERR_INVALID_ARGUMENT, "Clock model not known: " + clock);
  }
  spec.blocks["entire"] = {0, spec.param_count};
  return spec;
}

std::pair<int, int> ModelSpec::Block(const std::string& key) const {
  auto it = blocks.find(key);
  if (it == blocks.end())
    Fail(SBNB_ERR_INVALID_ARGUMENT, "Can't find block key: " + key);
  return it->second;
}

int ModelSpec::SiteGradientSize() const {
  const int entries = (site == SiteKind::kConstant ? 0 : 1) + (invariant ? 1 : 0);
  return entries > 0 ? entries : 1;
}

int ModelSpec::SubstitutionGradientSize() const {
  switch (substitution) {
    case SubstitutionKind::kGTR:
      return 8;
    case SubstitutionKind::kHKY:
      return 4;  // kappa (linear) + 3 frequency coordinates
    default:
      return 0;
  }
}

void SymmetricEigen4(const double* matrix, double* values, double* vectors) {
  double a[4][4], v[4][4];
  for (int i = 0; i < 4; i++)
    for (int j = 0; j < 4; j++) {
      a[i][j] = 0.5 * (matrix[i * 4 + j] + matrix[j * 4 + i]);
      v[i][j] = (i == j) ? 1.0 : 0.0;
    }
  for (int sweep = 0; sweep < 64; sweep++) {
    double off = 0.0, diag = 0.0;
    for (int i = 0; i < 4; i++)
      for (int j = 0; j < 4; j++) (i == j ? diag : off) += a[i][j] * a[i][j];
    if (off <= 1e-40 * (diag + 1e-300)) break;
    for (int p = 0; p < 3; p++)
      for (int q = p + 1; q < 4; q++) {
        if (a[p][q] == 0.0) continue;
        const double theta = (a[q][q] - a[p][p]) / (2.0 * a[p][q]);
        const double t = (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
        const double c = 1.0 / std::sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < 4; k++) {
          const double akp = a[k][p], akq = a[k][q];
          a[k][p] = c * akp - s * akq;
          a[k][q] = s * akp + c * akq;
        }
        for (int k = 0; k < 4; k++) {
          const double apk = a[p][k], aqk = a[q][k];
          a[p][k] = c * apk - s * aqk;
          a[q][k] = s * apk + c * aqk;
        }
        for (int k = 0; k < 4; k++) {
          const double vkp = v[k][p], vkq = v[k][q];
          v[k][p] = c * vkp - s * vkq;
          v[k][q] = s * vkp + c * vkq;
        }
      }
  }
  // Ascending eigenvalue order (what Eigen's solver returns); order is
  // immaterial to P(t) but makes the tables reproducible.
  int order[4] = {0, 1, 2, 3};
  std::sort(order, order + 4, [&a](int x, int y) { return a[x][x] < a[y][y]; });
  for (int k = 0; k < 4; k++) {
    values[k] = a[order[k]][order[k]];
    for (int i = 0; i < 4; i++) vectors[i * 4 + k] = v[i][order[k]];
  }
}

namespace {

void CheckSimplex(const double* x, int count, const char* what) {
  double sum = 0;
  for (int i = 0; i < count; i++) sum += x[i];
  if (!(std::fabs(sum - 1.0) < 0.001)) {
    // substitution_model.cpp:21-35
    std::ostringstream oss;
    oss << "GTR " << what << " do not sum to 1 +/- 0.001! vector: (";
    for (int i = 0; i < count; i++) oss << (i ? "," : "") << x[i];
    oss << ")";
    Fail(SBNB_ERR_MODEL, oss.str());
  }
}

// Q from six exchangeabilities (order AC,AG,AT,CG,CT,GT) and four frequencies,
// scaled to one expected substitution per unit time; then the Felsenstein
// p.206 symmetrisation (substitution_model.cpp:39-80).
void GeneralTimeReversible(const double* rates, const double* freqs, ModelTables* out) {
  double q[4][4];
  int rate_index = 0;
  for (int i = 0; i < 4; i++)
    for (int j = i + 1; j < 4; j++) {
      const double rate = rates[rate_index++];
      q[i][j] = rate * freqs[j];
      q[j][i] = rate * freqs[i];
    }
  double total = 0;
  for (int i = 0; i < 4; i++) {
    double row_sum = 0;
    for (int j = 0; j < 4; j++)
      if (i != j) row_sum += q[i][j];
    q[i][i] = -row_sum;
    total += row_sum * freqs[i];
  }
  for (int i = 0; i < 4; i++)
    for (int j = 0; j < 4; j++) q[i][j] /= total;
  double sqrt_f[4], sym[16];
  for (int i = 0; i < 4; i++) sqrt_f[i] = std::sqrt(freqs[i]);
  for (int i = 0; i < 4; i++)
    for (int j = 0; j < 4; j++) sym[i * 4 + j] = sqrt_f[i] * q[i][j] / sqrt_f[j];
  double vectors[16];
  SymmetricEigen4(sym, out->eval, vectors);
  for (int i = 0; i < 4; i++)
    for (int k = 0; k < 4; k++) {
      out->evec[i * 4 + k] = vectors[i * 4 + k] / sqrt_f[i];
      out->ivec[k * 4 + i] = vectors[i * 4 + k] * sqrt_f[i];
    }
  for (int i = 0; i < 4; i++) {
    out->freqs[i] = freqs[i];
    for (int j = 0; j < 4; j++) out->q[i * 4 + j] = q[i][j];
  }
}

}  // namespace

void BuildSubstitution(const ModelSpec& spec, const double* params, ModelTables* out) {
  switch (spec.substitution) {
    case SubstitutionKind::kJC69: {
      // substitution_model.hpp:59-74: closed-form tables, no parameters.
      const double evec[16] = {1.0, 2.0, 0.0, 0.5, 1.0, -2.0, 0.5, 0.0,
                               1.0, 2.0, 0.0, -0.5, 1.0, -2.0, -0.5, 0.0};
      const double ivec[16] = {0.25, 0.25, 0.25, 0.25, 0.125, -0.125, 0.125, -0.125,
                               0.0, 1.0, 0.0, -1.0, 1.0, 0.0, -1.0, 0.0};
      std::memcpy(out->evec, evec, sizeof(evec));
      std::memcpy(out->ivec, ivec, sizeof(ivec));
      out->eval[0] = 0.0;
      for (int k = 1; k < 4; k++) out->eval[k] = -1.3333333333333333;
      for (int i = 0; i < 4; i++) {
        out->freqs[i] = 0.25;
        for (int j = 0; j < 4; j++) out->q[i * 4 + j] = (i == j) ? -1.0 : 1.0 / 3.0;
      }
      break;
    }
    case SubstitutionKind::kGTR: {
      const auto rates = spec.Block("GTR rates");
      const auto freqs = spec.Block("frequencies");
      const int base = spec.Block("entire substitution").first;
      CheckSimplex(params + freqs.first - base, 4, "frequencies");
      CheckSimplex(params + rates.first - base, 6, "rates");
      GeneralTimeReversible(params + rates.first - base, params + freqs.first - base, out);
      break;
    }
    case SubstitutionKind::kHKY: {
      const auto kappa = spec.Block("kappa");
      const auto freqs = spec.Block("frequencies");
      const int base = spec.Block("entire substitution").first;
      CheckSimplex(params + freqs.first - base, 4, "frequencies");
      const double k = params[kappa.first - base];
      if (!(k > 0)) Fail(SBNB_ERR_MODEL, "HKY kappa must be positive.");
      // Transitions are A<->G and C<->T.
      const double rates[6] = {1.0, k, 1.0, 1.0, k, 1.0};
      GeneralTimeReversible(rates, params + freqs.first - base, out);
      break;
    }
  }
}

// P(a, x): power series for x < a + 1, Lentz continued fraction for Q = 1 - P otherwise.
double RegularizedGammaP(double a, double x) {
  if (!(x > 0.0)) return 0.0;
  const double log_prefactor = a * std::log(x) - x - std::lgamma(a);
  if (x < a + 1.0) {
    double term = 1.0 / a, sum = term, denominator = a;
    for (int n = 0; n < 10000; n++) {
      denominator += 1.0;
      term *= x / denominator;
      sum += term;
      if (std::fabs(term) < std::fabs(sum) * 1e-17) break;
    }
    return sum * std::exp(log_prefactor);
  }
  const double tiny = 1e-300;
  double b = x + 1.0 - a, c = 1.0 / tiny, d = 1.0 / b, fraction = d;
  for (int n = 1; n < 10000; n++) {
    const double an = -n * (n - a);
    b += 2.0;
    d = an * d + b;
    if (std::fabs(d) < tiny) d = tiny;
    c = b + an / c;
    if (std::fabs(c) < tiny) c = tiny;
    d = 1.0 / d;
    const double delta = d * c;
    fraction *= delta;
    if (std::fabs(delta - 1.0) < 1e-16) break;
  }
  return 1.0 - std::exp(log_prefactor) * fraction;
}

// Solves P(a, x) = p for x: a small-x / Wilson-Hilferty starting point, then
// Halley steps on P (pdf and its log-derivative are closed form), kept positive.
double InverseRegularizedGammaP(double a, double p) {
  if (!(p > 0.0)) return 0.0;
  if (!(p < 1.0)) return INFINITY;
  const double log_gamma = std::lgamma(a);
  double x;
  // small-x asymptote P ~ x^a / Gamma(a + 1)
  const double small = std::exp((std::log(p) + log_gamma + std::log(a)) / a);
  if (small < 0.3 * (a + 1.0)) {
    x = small;
  } else {
    // Wilson-Hilferty: (x / a)^(1/3) is nearly normal with mean 1 - 1/(9a), variance 1/(9a)
    const double t = std::sqrt(-2.0 * std::log(p < 0.5 ? p : 1.0 - p));
    double z = t - (2.30753 + 0.27061 * t) / (1.0 + t * (0.99229 + 0.04481 * t));
    if (p < 0.5) z = -z;
    const double cube = 1.0 - 1.0 / (9.0 * a) + z / (3.0 * std::sqrt(a));
    x = a * cube * cube * cube;
    if (!(x > 0.0)) x = small;
  }
  for (int iteration = 0; iteration < 100; iteration++) {
    const double error = RegularizedGammaP(a, x) - p;
    const double pdf = std::exp((a - 1.0) * std::log(x) - x - log_gamma);
    if (!(pdf > 0.0)) break;
    const double newton = error / pdf;
    // Halley correction with d log pdf / dx = (a - 1) / x - 1, limited to a factor 2
    const double curvature = newton * ((a - 1.0) / x - 1.0);
    double step = newton / (1.0 - 0.5 * std::min(1.0, std::max(-1.0, curvature)));
    double next = x - step;
    if (!(next > 0.0)) next = 0.5 * x;
    step = x - next;
    x = next;
    if (std::fabs(step) <= 1e-16 * x) break;
  }
  return x;
}

namespace {

void BuildRateCategories(const ModelSpec& spec, const double* params, ModelTables* out) {
  const int count = spec.category_count;
  for (int c = 0; c < kMaxCategories; c++) {
    out->rates[c] = 1.0;
    out->weights[c] = 0.0;
    out->drates[c] = 0.0;
  }
  if (spec.site == SiteKind::kConstant) {
    out->weights[0] = 1.0;
    return;
  }
  const double shape = params[0];
  double mean_rate = 0, mean_derivative = 0;
  double unscaled_derivative[kMaxCategories];
  if (spec.site == SiteKind::kGamma) {
    // Median discretisation of Gamma(shape, rate = shape) (Yang 1994), the same
    // scheme the reference uses for its Weibull model: category i sits at the
    // quantile (2i+1)/(2C) and the rates are divided by their mean -- the 1/shape
    // scale cancels, so the unit-scale quantile g_i = P^-1(shape, q_i) is enough.
    // d g / d shape by implicit differentiation of P(shape, g) = q:
    //   dg/da = -(dP/da) / pdf(g),  dP/da by central differences of P (smooth in a).
    if (!(shape > 0)) Fail(SBNB_ERR_MODEL, "Gamma shape must be positive.");
    const double h = 1e-5 * std::max(shape, 1.0);
    for (int i = 0; i < count; i++) {
      const double quantile = (2.0 * i + 1.0) / (2.0 * count);
      const double g = InverseRegularizedGammaP(shape, quantile);
      out->rates[i] = g;
      mean_rate += g;
      const double dP_da = (RegularizedGammaP(shape + h, g) - RegularizedGammaP(shape - h, g)) / (2.0 * h);
      const double log_pdf = (shape - 1.0) * std::log(g) - g - std::lgamma(shape);
      unscaled_derivative[i] = -dP_da / std::exp(log_pdf);
      mean_derivative += unscaled_derivative[i];
    }
  } else {
    if (!(shape > 0)) Fail(SBNB_ERR_MODEL, "Weibull shape must be positive.");
    // site_model.cpp:37-62
    for (int i = 0; i < count; i++) {
      const double quantile = (2.0 * i + 1.0) / (2.0 * count);
      out->rates[i] = std::pow(-std::log(1.0 - quantile), 1.0 / shape);
      mean_rate += out->rates[i];
      unscaled_derivative[i] =
          -out->rates[i] * std::log(-std::log(1.0 - quantile)) / (shape * shape);
      mean_derivative += unscaled_derivative[i];
    }
  }
  mean_rate /= count;
  mean_derivative /= count;
  for (int i = 0; i < count; i++) {
    out->drates[i] = (unscaled_derivative[i] * mean_rate - out->rates[i] * mean_derivative) /
                     (mean_rate * mean_rate);
    out->rates[i] /= mean_rate;
    out->weights[i] = 1.0 / count;  // site_model.hpp:57-59
  }
}

}  // namespace

void BuildSite(const ModelSpec& spec, const double* params, ModelTables* out) {
  BuildRateCategories(spec, params, out);
  out->pinv = 0.0;
  if (!spec.invariant) return;
  const double p = params[spec.Block("proportion invariant").first - spec.Block("entire site").first];
  if (!(p >= 0.0 && p < 1.0)) Fail(SBNB_ERR_MODEL, "Proportion invariant must lie in [0, 1).");
  out->pinv = p;
  if (p == 0.0) return;  // (bitwise the tables of the site model without +I)
  // The variable sites carry the whole substitution rate: mean rate over all sites 1.
  for (int c = 0; c < spec.category_count; c++) {
    out->rates[c] /= 1.0 - p;
    out->drates[c] /= 1.0 - p;
  }
}

void BuildModelTables(const ModelSpec& spec, const double* row, ModelTables* out) {
  BuildSubstitution(spec, row + spec.Block("entire substitution").first, out);
  BuildSite(spec, row + spec.Block("entire site").first, out);
}

void StickBreaking(const double* y, int simplex_size, double* x) {
  double stick = 1.0;
  for (int k = 0; k < simplex_size - 1; k++) {
    const double z = 1.0 / (1.0 + std::exp(-(y[k] - std::log(double(simplex_size - k - 1)))));
    x[k] = stick * z;
    stick -= x[k];
  }
  x[simplex_size - 1] = stick;
}

void StickBreakingJacobian(const double* y, int simplex_size, double* jacobian) {
  const int coords = simplex_size - 1;
  double stick = 1.0;
  std::vector<double> dstick(coords, 0.0);  // d stick / d y_j
  for (int k = 0; k < coords; k++) {
    const double z = 1.0 / (1.0 + std::exp(-(y[k] - std::log(double(simplex_size - k - 1)))));
    for (int j = 0; j < coords; j++) {
      // x_k = stick z_k
      const double dx = dstick[j] * z + (j == k ? stick * z * (1.0 - z) : 0.0);
      jacobian[k * coords + j] = dx;
      dstick[j] -= dx;
    }
    stick -= stick * z;
  }
  for (int j = 0; j < coords; j++) jacobian[coords * coords + j] = dstick[j];  // x_last = the rest of the stick
}

void BuildSubstitutionDerivatives(const ModelSpec& spec, const double* row, const ModelTables& tables,
                                  SubstitutionDerivatives* out) {
  out->count = 0;
  if (spec.substitution == SubstitutionKind::kJC69) return;
  const bool gtr = spec.substitution == SubstitutionKind::kGTR;
  const double* freqs = row + spec.Block("frequencies").first;
  double rates[6];
  if (gtr) {
    std::copy(row + spec.Block("GTR rates").first, row + spec.Block("GTR rates").first + 6, rates);
  } else {
    const double kappa = row[spec.Block("kappa").first];
    const double hky[6] = {1.0, kappa, 1.0, 1.0, kappa, 1.0};
    std::copy(hky, hky + 6, rates);
  }
  // exchangeability of the pair (i, j), order AC AG AT CG CT GT
  int pair_a[6], pair_b[6], index = 0;
  double r[4][4] = {};
  for (int i = 0; i < 4; i++)
    for (int j = i + 1; j < 4; j++) {
      pair_a[index] = i, pair_b[index] = j;
      r[i][j] = r[j][i] = rates[index++];
    }
  double mu = 0.0;  // the expected rate the unnormalised matrix is divided by
  for (int i = 0; i < 4; i++)
    for (int j = 0; j < 4; j++)
      if (i != j) mu += freqs[i] * r[i][j] * freqs[j];
  // d Q / d (one exchangeability), d Q / d (one frequency): Q = Qu / mu.
  auto finish = [&](double (&dqu)[16], double dmu, double* dq) {
    for (int e = 0; e < 16; e++) dq[e] = (dqu[e] - tables.q[e] * dmu) / mu;
  };
  double dq_rate[6][16], dq_freq[4][16];
  for (int m = 0; m < 6; m++) {
    const int a = pair_a[m], b = pair_b[m];
    double dqu[16] = {};
    dqu[a * 4 + b] = freqs[b];
    dqu[b * 4 + a] = freqs[a];
    dqu[a * 4 + a] = -freqs[b];
    dqu[b * 4 + b] = -freqs[a];
    finish(dqu, 2.0 * freqs[a] * freqs[b], dq_rate[m]);
  }
  for (int k = 0; k < 4; k++) {
    double dqu[16] = {};
    double dmu = 0.0;
    for (int i = 0; i < 4; i++) {
      if (i == k) continue;
      dqu[i * 4 + k] = r[i][k];
      dqu[i * 4 + i] = -r[i][k];
      dmu += 2.0 * r[k][i] * freqs[i];
    }
    finish(dqu, dmu, dq_freq[k]);
  }
  // chain rule through the parametrisation
  double dq[8][16] = {};
  auto add = [](double* to, const double* from, double factor) {
    for (int e = 0; e < 16; e++) to[e] += factor * from[e];
  };
  int count = 0;
  if (gtr) {
    double y[5], jacobian[6 * 5];
    StickBreakingInverse(rates, 6, y);
    StickBreakingJacobian(y, 6, jacobian);
    for (int k = 0; k < 5; k++, count++) {
      for (int m = 0; m < 6; m++) add(dq[count], dq_rate[m], jacobian[m * 5 + k]);
      std::fill(out->dfreqs[count], out->dfreqs[count] + 4, 0.0);
    }
  } else {
    add(dq[count], dq_rate[1], 1.0);  // kappa multiplies the two transitions A<->G, C<->T
    add(dq[count], dq_rate[4], 1.0);
    std::fill(out->dfreqs[count], out->dfreqs[count] + 4, 0.0);
    count++;
  }
  {
    double y[3], jacobian[4 * 3];
    StickBreakingInverse(freqs, 4, y);
    StickBreakingJacobian(y, 4, jacobian);
    for (int k = 0; k < 3; k++, count++) {
      for (int m = 0; m < 4; m++) {
        add(dq[count], dq_freq[m], jacobian[m * 3 + k]);
        out->dfreqs[count][m] = jacobian[m * 3 + k];
      }
    }
  }
  // B = V^-1 dQ V
  for (int t = 0; t < count; t++) {
    double left[16];
    for (int k = 0; k < 4; k++)
      for (int j = 0; j < 4; j++) {
        double sum = 0.0;
        for (int i = 0; i < 4; i++) sum += tables.ivec[k * 4 + i] * dq[t][i * 4 + j];
        left[k * 4 + j] = sum;
      }
    for (int k = 0; k < 4; k++)
      for (int l = 0; l < 4; l++) {
        double sum = 0.0;
        for (int j = 0; j < 4; j++) sum += left[k * 4 + j] * tables.evec[j * 4 + l];
        out->b[t][k * 4 + l] = sum;
      }
  }
  out->count = count;
}

void StickBreakingInverse(const double* x, int simplex_size, double* y) {
  double sum = 0;
  for (int k = 0; k < simplex_size - 1; k++) {
    const double z = x[k] / (1.0 - sum);
    y[k] = std::log(z / (1.0 - z)) + std::log(double(simplex_size - k - 1));
    sum += x[k];
  }
}

}  // namespace sbnb
