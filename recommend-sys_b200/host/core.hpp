// core.hpp — C++ host mirror of the reference's Go package `core` for the KNN hot path, over
// the C ABI (include/rs_knn.h) and the host helpers (rs_host.h).  The reference is compiled
// code (Go) whose toolchain is absent from the build image, so this header is the compiled
// host side: same names, argument meaning and error behaviour (a non-zero status throws, where
// Go panics).  Header-only; link with -lrs_knn_b200 -lrs_host.
//
//   reference                              here
//   core/base.go:14-57   Parameters        core::Parameters (typed getters throw on a wrong type)
//   core/data.go:21-105  DataSet           core::DataSet (KFold, SubSet, Predict)
//   core/data.go:109-216 TrainSet          core::TrainSet / NewTrainSet
//   core/base.go:108-163 BaseLine          core::BaseLine (host SGD)
//   core/knn.go          KNN + 4 ctors     core::KNN, NewKNN, NewKNNWithMean, NewKNNWithZScore, NewKNNBaseLine
//   core/eval.go:18-67   CrossValidate     core::CrossValidate (intended 6-argument form)
//   core/utils.go:160-180 RMSE / MAE       core::RMSE / core::MAE on (predictions, truth)
#pragma once

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <functional>
#include <map>
#include <memory>
#include <numeric>
#include <random>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <variant>
#include <vector>

#include "rs_host.h"
#include "rs_knn.h"

namespace core {

constexpr int newID = -1;  // core/data.go:129

enum class Sim { Cosine = RS_SIM_COSINE, MSD = RS_SIM_MSD, Pearson = RS_SIM_PEARSON,
                 PearsonBaseline = RS_SIM_PEARSON_BASELINE };

// core/base.go:14-57
class Parameters {
  public:
    using Value = std::variant<int, bool, double, std::string, Sim>;
    Parameters() = default;
    Parameters(std::initializer_list<std::pair<const std::string, Value>> init) : m_(init) {}
    Parameters Copy() const { return *this; }
    void Set(const std::string &k, Value v) { m_[k] = std::move(v); }
    int GetInt(const std::string &k, int d) const { return get<int>(k, d, "int"); }
    bool GetBool(const std::string &k, bool d) const { return get<bool>(k, d, "bool"); }
    double GetFloat64(const std::string &k, double d) const { return get<double>(k, d, "float64"); }
    std::string GetString(const std::string &k, const std::string &d) const { return get<std::string>(k, d, "string"); }
    Sim GetSim(const std::string &k, Sim d) const { return get<Sim>(k, d, "core.Sim"); }

  private:
    template <typename T> T get(const std::string &k, const T &d, const char *what) const {
        auto it = m_.find(k);
        if (it == m_.end()) return d;
        if (!std::holds_alternative<T>(it->second))  // Go: val.(T) panics (core/base.go:26-54)
            throw std::runtime_error("interface conversion: Parameters[\"" + k + "\"] is not " + what);
        return std::get<T>(it->second);
    }
    std::map<std::string, Value> m_;
};

// core/data.go:21-47
struct DataSet {
    std::vector<double> Ratings;
    std::vector<int64_t> Users, Items;
    size_t Length() const { return Ratings.size(); }
    DataSet SubSet(const std::vector<size_t> &idx) const {
        DataSet d;
        for (size_t i : idx) { d.Users.push_back(Users[i]); d.Items.push_back(Items[i]); d.Ratings.push_back(Ratings[i]); }
        return d;
    }
};

// core/data.go:109-182
struct TrainSet : DataSet {
    double GlobalMean = NAN;
    int UserCount = 0, ItemCount = 0;
    std::vector<int32_t> innerUsers, innerItems;  // per rating row, dataset order
    std::unordered_map<int64_t, int32_t> InnerUserIDs, InnerItemIDs;
    int ConvertUserID(int64_t u) const { auto it = InnerUserIDs.find(u); return it == InnerUserIDs.end() ? newID : it->second; }
    int ConvertItemID(int64_t i) const { auto it = InnerItemIDs.find(i); return it == InnerItemIDs.end() ? newID : it->second; }
};

inline TrainSet NewTrainSet(const DataSet &rowSet) {  // core/data.go:131-154
    TrainSet s;
    static_cast<DataSet &>(s) = rowSet;
    double sum = 0.0;
    for (double r : s.Ratings) sum += r;
    s.GlobalMean = sum / (double)s.Ratings.size();  // stat.Mean, core/data.go:134
    s.innerUsers.resize(s.Length());
    s.innerItems.resize(s.Length());
    s.UserCount = (int)rs_host_inner_ids(s.Users.data(), (int64_t)s.Length(), s.innerUsers.data());
    s.ItemCount = (int)rs_host_inner_ids(s.Items.data(), (int64_t)s.Length(), s.innerItems.data());
    for (size_t i = 0; i < s.Length(); i++) {
        s.InnerUserIDs.emplace(s.Users[i], s.innerUsers[i]);
        s.InnerItemIDs.emplace(s.Items[i], s.innerItems[i]);
    }
    return s;
}

// The TrainSet of t's rows followed by rowSet's: NewTrainSet of the concatenation (inner ids continue the order of
// first appearance, GlobalMean is the concatenation's).
inline TrainSet Extend(const TrainSet &t, const DataSet &rowSet) {
    DataSet d = t;
    d.Users.insert(d.Users.end(), rowSet.Users.begin(), rowSet.Users.end());
    d.Items.insert(d.Items.end(), rowSet.Items.begin(), rowSet.Items.end());
    d.Ratings.insert(d.Ratings.end(), rowSet.Ratings.begin(), rowSet.Ratings.end());
    return NewTrainSet(d);
}

// core/data.go:49-70 — the reference's permutation is unseeded (SURVEY.md hazard 3); here mt19937_64(seed).
inline void KFold(const DataSet &d, int k, int64_t seed, std::vector<TrainSet> &trains, std::vector<DataSet> &tests) {
    const size_t n = d.Length();
    std::vector<size_t> perm(n);
    std::iota(perm.begin(), perm.end(), 0);
    std::mt19937_64 rng((uint64_t)seed);
    std::shuffle(perm.begin(), perm.end(), rng);
    const size_t fold = n / k;
    size_t begin = 0, end = 0;
    for (int i = 0; i < k; i++) {
        end += fold;
        if ((size_t)i < n % k) end++;
        std::vector<size_t> te(perm.begin() + begin, perm.begin() + end), tr(perm.begin(), perm.begin() + begin);
        tr.insert(tr.end(), perm.begin() + end, perm.end());
        tests.push_back(d.SubSet(te));
        trains.push_back(NewTrainSet(d.SubSet(tr)));
        begin = end;
    }
}

struct Estimator {  // core/base.go:8-12
    Parameters Params;
    virtual ~Estimator() = default;
    virtual void SetParams(const Parameters &p) { Params = p; }
    virtual double Predict(int64_t userId, int64_t itemId) = 0;
    virtual void Fit(const TrainSet &trainSet) = 0;
    virtual std::vector<double> PredictBatch(const std::vector<int64_t> &users, const std::vector<int64_t> &items) {
        std::vector<double> out(users.size());
        for (size_t j = 0; j < users.size(); j++) out[j] = Predict(users[j], items[j]);  // core/data.go:98-105
        return out;
    }
    virtual std::unique_ptr<Estimator> Clone() const = 0;  // stands in for the gob Copy (core/eval.go:29-30)
};

inline void rs_check(int32_t rc);

// core/base.go:108-163
struct BaseLine : Estimator {
    std::vector<double> userBias, itemBias;
    double globalBias = 0.0;
    const TrainSet *trainSet = nullptr;
    explicit BaseLine(const Parameters &p = {}) { Params = p; }
    void Fit(const TrainSet &t) override {
        trainSet = &t;
        userBias.assign(t.UserCount, 0.0);
        itemBias.assign(t.ItemCount, 0.0);
        if (Params.GetString("baseline", "sgd") == "als") {   // EXTENSION: ALS baselines on the device
            rs_check(rs_baseline_als(Params.GetInt("device", -1), t.innerUsers.data(), t.innerItems.data(),
                                     t.Ratings.data(), (int64_t)t.Length(), t.UserCount, t.ItemCount, t.GlobalMean,
                                     Params.GetFloat64("regU", 15.0), Params.GetFloat64("regI", 10.0),
                                     Params.GetInt("nEpochs", 10), userBias.data(), itemBias.data()));
            globalBias = t.GlobalMean;
            return;
        }
        rs_host_baseline_sgd(t.innerUsers.data(), t.innerItems.data(), t.Ratings.data(), (int64_t)t.Length(), t.UserCount,
                             t.ItemCount, Params.GetFloat64("reg", 0.02), Params.GetFloat64("lr", 0.005),
                             Params.GetInt("nEpochs", 20), userBias.data(), itemBias.data(), &globalBias);
    }
    double Predict(int64_t u, int64_t i) override {
        double ret = globalBias;
        const int iu = trainSet->ConvertUserID(u), ii = trainSet->ConvertItemID(i);
        if (iu != newID) ret += userBias[iu];
        if (ii != newID) ret += itemBias[ii];
        return ret;
    }
    std::unique_ptr<Estimator> Clone() const override { return std::make_unique<BaseLine>(Params); }
};

inline void rs_check(int32_t rc) {
    if (rc != RS_OK) throw std::runtime_error(std::string("rs_knn error ") + std::to_string(rc) + ": " + rs_last_error());
}

// core/knn.go
struct KNN : Estimator {
    std::string KNNType;
    double GlobalMean = NAN;
    std::vector<double> Means, StdDevs, Bias;
    const TrainSet *Data = nullptr;

    KNN(std::string type, const Parameters &p) : KNNType(std::move(type)) { Params = p; }
    ~KNN() override { Close(); }
    void Close() { if (h_) { rs_knn_destroy(h_); h_ = nullptr; } }

    void Fit(const TrainSet &t) override {  // core/knn.go:143-217
        const Sim sim = Params.GetSim("sim", Sim::MSD);
        userBased_ = Params.GetBool("userBased", true);
        Data = &t;
        GlobalMean = t.GlobalMean;
        const auto &left = userBased_ ? t.innerUsers : t.innerItems;
        const auto &right = userBased_ ? t.innerItems : t.innerUsers;
        nLeft_ = userBased_ ? t.UserCount : t.ItemCount;
        const int nRight = userBased_ ? t.ItemCount : t.UserCount;
        const double *lb = nullptr, *rb = nullptr;
        double gb = 0.0;
        BaseLine bl(Params);
        if (KNNType == "baseline" || sim == Sim::PearsonBaseline) {  // core/knn.go:179-187
            bl.Fit(t);
            lb = (userBased_ ? bl.userBias : bl.itemBias).data();
            if (sim == Sim::PearsonBaseline) rb = (userBased_ ? bl.itemBias : bl.userBias).data();
            gb = bl.globalBias;
            if (KNNType == "baseline") Bias = userBased_ ? bl.userBias : bl.itemBias;
        }
        Close();
        rs_knn_params p;
        rs_check(rs_knn_params_default(&p));
        p.sim = (int32_t)sim;
        p.knn_type = KNNType == "basic" ? RS_KNN_BASIC : KNNType == "centered" ? RS_KNN_CENTERED
                   : KNNType == "zscore" ? RS_KNN_ZSCORE : RS_KNN_BASELINE;
        p.k = Params.GetInt("k", 40);
        p.min_k = Params.GetInt("mink", 1);
        p.device = Params.GetInt("device", -1);
        p.pearson_mode = Params.GetString("pearsonMode", "exact") == "sums" ? RS_PEARSON_SUMS : RS_PEARSON_EXACT;
        const std::string path = Params.GetString("simPath", "auto");
        p.sim_path = path == "tensor" ? RS_PATH_TENSOR : path == "stream" ? RS_PATH_STREAM : RS_PATH_AUTO;
        p.store = Params.GetString("store", "matrix") == "topk" ? RS_STORE_TOPK : RS_STORE_MATRIX;
        p.topk = Params.GetInt("topk", p.k);
        p.row_begin = Params.GetInt("rowBegin", 0);
        p.row_end = Params.GetInt("rowEnd", 0);
        p.shrinkage = Params.GetFloat64("shrinkage", 0.0);
        p.shard_count = Params.GetInt("shardCount", 0);      // one estimator per GPU: see rs_knn.h
        p.shard_index = Params.GetInt("shardIndex", 0);
        rs_check(rs_knn_create(&p, &h_));
        k_ = p.k;
        minK_ = p.min_k;
        rs_check(rs_knn_fit(h_, left.data(), right.data(), t.Ratings.data(), (int64_t)t.Length(), nLeft_, nRight,
                            t.GlobalMean, lb, rb, gb));
        extended_.reset();
        ReadStats();
    }

    // Adds the ratings of `rowSet` (raw user, raw item, rating; users and items may be new) to the fitted model
    // without a refit (rs_knn_update): the model becomes the Fit of Extend(*Data, rowSet), bit for bit, and Data that
    // TrainSet (owned by the estimator).
    void Update(const DataSet &rowSet) {
        auto t = std::make_shared<const TrainSet>(Extend(*Data, rowSet));
        const size_t n0 = Data->Length();
        const auto &left = userBased_ ? t->innerUsers : t->innerItems;
        const auto &right = userBased_ ? t->innerItems : t->innerUsers;
        const int nLeft = userBased_ ? t->UserCount : t->ItemCount, nRight = userBased_ ? t->ItemCount : t->UserCount;
        rs_check(rs_knn_update(h_, left.data() + n0, right.data() + n0, t->Ratings.data() + n0,
                               (int64_t)(t->Length() - n0), nLeft, nRight, t->GlobalMean));
        extended_ = t;
        Data = t.get();
        GlobalMean = t->GlobalMean;
        nLeft_ = nLeft;
        ReadStats();
    }

    std::vector<double> PredictBatch(const std::vector<int64_t> &users, const std::vector<int64_t> &items) override {
        std::vector<int32_t> l(users.size()), r(users.size());
        for (size_t j = 0; j < users.size(); j++) {
            const int32_t iu = Data->ConvertUserID(users[j]), ii = Data->ConvertItemID(items[j]);
            l[j] = userBased_ ? iu : ii;
            r[j] = userBased_ ? ii : iu;
        }
        SyncK();
        std::vector<double> out(users.size());
        rs_check(rs_knn_predict_batch(h_, l.data(), r.data(), (int64_t)l.size(), out.data()));
        return out;
    }
    double Predict(int64_t u, int64_t i) override { return PredictBatch({u}, {i})[0]; }  // core/knn.go:75-141

    // The n best items each user has not rated, as raw item ids ranked by (score desc, inner item id asc) with their
    // scores (Predict(user, item) bit for bit): [users.size()][n] row-major, unused slots newID with score NaN.
    void Recommend(const std::vector<int64_t> &users, int n, std::vector<int64_t> &items, std::vector<double> &scores) {
        std::vector<int32_t> q(users.size()), ids(users.size() * (size_t)n);
        for (size_t j = 0; j < users.size(); j++) q[j] = Data->ConvertUserID(users[j]);
        SyncK();
        scores.assign(ids.size(), 0.0);
        if (!users.empty())
            rs_check(rs_knn_recommend(h_, userBased_ ? RS_SIDE_LEFT : RS_SIDE_RIGHT, q.data(), (int64_t)q.size(), n,
                                      ids.data(), scores.data()));
        std::vector<int64_t> raw(Data->ItemCount);          // inner -> raw: the order of first appearance
        for (size_t j = 0; j < Data->Length(); j++) raw[Data->innerItems[j]] = Data->Items[j];
        items.resize(ids.size());
        for (size_t j = 0; j < ids.size(); j++) items[j] = ids[j] >= 0 ? raw[ids[j]] : newID;
    }

    // Recommend for users whose ratings are given in `given` (raw user, raw item, rating) instead of taken from the
    // train set (rs_knn_recommend_given, not a refit): users in order of first appearance, each user's ratings in
    // dataset order, items the train set does not know dropped; the given items are never listed.
    void RecommendGiven(const DataSet &given, int n, std::vector<int64_t> &users, std::vector<int64_t> &items,
                        std::vector<double> &scores) {
        std::unordered_map<int64_t, size_t> group;
        std::vector<std::vector<size_t>> rows;
        users.clear();
        for (size_t j = 0; j < given.Length(); j++) {
            auto it = group.find(given.Users[j]);
            if (it == group.end()) {
                it = group.emplace(given.Users[j], users.size()).first;
                users.push_back(given.Users[j]);
                rows.emplace_back();
            }
            if (Data->ConvertItemID(given.Items[j]) != newID) rows[it->second].push_back(j);
        }
        std::vector<int64_t> ptr(1, 0);
        std::vector<int32_t> ids;
        std::vector<double> vals;
        for (const auto &r : rows) {
            for (size_t j : r) { ids.push_back(Data->ConvertItemID(given.Items[j])); vals.push_back(given.Ratings[j]); }
            ptr.push_back((int64_t)ids.size());
        }
        if (ids.empty()) { ids.push_back(0); vals.push_back(0.0); }   // every list empty: valid pointers all the same
        SyncK();
        std::vector<int32_t> top(users.size() * (size_t)n);
        scores.assign(top.size(), 0.0);
        if (!users.empty())
            rs_check(rs_knn_recommend_given(h_, userBased_ ? RS_SIDE_LEFT : RS_SIDE_RIGHT, ptr.data(), ids.data(),
                                            vals.data(), (int64_t)users.size(), n, top.data(), scores.data()));
        std::vector<int64_t> raw(Data->ItemCount);          // inner -> raw: the order of first appearance
        for (size_t j = 0; j < Data->Length(); j++) raw[Data->innerItems[j]] = Data->Items[j];
        items.resize(top.size());
        for (size_t j = 0; j < top.size(); j++) items[j] = top[j] >= 0 ? raw[top[j]] : newID;
    }

    std::vector<double> SimsRows(int64_t row0, int64_t nrows) {  // backs KNN.Sims (core/knn.go:21)
        std::vector<double> out((size_t)nrows * nLeft_);
        rs_check(rs_knn_sims_rows(h_, row0, nrows, out.data()));
        return out;
    }
    rs_knn_profile Profile() { rs_knn_profile p; rs_check(rs_knn_profile_get(h_, &p)); return p; }
    int NLeft() const { return nLeft_; }
    std::unique_ptr<Estimator> Clone() const override { return std::make_unique<KNN>(KNNType, Params); }

  private:
    void ReadStats() {
        if (KNNType == "centered" || KNNType == "zscore") { Means.resize(nLeft_); rs_check(rs_knn_means(h_, Means.data())); }
        if (KNNType == "zscore") { StdDevs.resize(nLeft_); rs_check(rs_knn_stddevs(h_, StdDevs.data())); }
    }

    // core/knn.go:80-81 reads k / mink in Predict: SetParams after Fit takes effect at the next call
    void SyncK() {
        const int k = Params.GetInt("k", 40), minK = Params.GetInt("mink", 1);
        if (k != k_ || minK != minK_) { rs_check(rs_knn_set_k(h_, k, minK)); k_ = k; minK_ = minK; }
    }

    rs_knn *h_ = nullptr;
    std::shared_ptr<const TrainSet> extended_;   // Data after an Update
    int k_ = 40, minK_ = 1;   // what the handle currently holds
    bool userBased_ = true;
    int nLeft_ = 0;
};

inline std::unique_ptr<KNN> NewKNN(const Parameters &p = {}) { return std::make_unique<KNN>("basic", p); }
inline std::unique_ptr<KNN> NewKNNWithMean(const Parameters &p = {}) { return std::make_unique<KNN>("centered", p); }
inline std::unique_ptr<KNN> NewKNNWithZScore(const Parameters &p = {}) { return std::make_unique<KNN>("zscore", p); }
inline std::unique_ptr<KNN> NewKNNBaseLine(const Parameters &p = {}) { return std::make_unique<KNN>("baseline", p); }

// core/slope_one.go (SURVEY.md §8 f-2): deviation matrix on the device (RS_SIM_SLOPE_ONE), Predict as a
// batch gather.  Fit with left = items, right = users.
struct SlopeOne : Estimator {
    const TrainSet *Data = nullptr;
    explicit SlopeOne(const Parameters &p = {}) { Params = p; }
    ~SlopeOne() override { Close(); }
    void Close() { if (h_) { rs_knn_destroy(h_); h_ = nullptr; } }
    void Fit(const TrainSet &t) override {  // core/slope_one.go:47-93
        Data = &t;
        Close();
        rs_knn_params p;
        rs_check(rs_knn_params_default(&p));
        p.sim = RS_SIM_SLOPE_ONE;
        p.device = Params.GetInt("device", -1);
        rs_check(rs_knn_create(&p, &h_));
        rs_check(rs_knn_fit(h_, t.innerItems.data(), t.innerUsers.data(), t.Ratings.data(), (int64_t)t.Length(),
                            t.ItemCount, t.UserCount, t.GlobalMean, nullptr, nullptr, 0.0));
    }
    std::vector<double> PredictBatch(const std::vector<int64_t> &users, const std::vector<int64_t> &items) override {
        std::vector<int32_t> l(users.size()), r(users.size());
        for (size_t j = 0; j < users.size(); j++) {
            l[j] = Data->ConvertItemID(items[j]);
            r[j] = Data->ConvertUserID(users[j]);
        }
        std::vector<double> out(users.size());
        rs_check(rs_knn_predict_batch(h_, l.data(), r.data(), (int64_t)l.size(), out.data()));
        return out;
    }
    double Predict(int64_t u, int64_t i) override { return PredictBatch({u}, {i})[0]; }  // core/slope_one.go:22-45
    std::vector<double> DevRows(int64_t row0, int64_t nrows) {  // backs SlopeOne.dev (core/slope_one.go:13)
        std::vector<double> out((size_t)nrows * Data->ItemCount);
        rs_check(rs_knn_sims_rows(h_, row0, nrows, out.data()));
        return out;
    }
    std::unique_ptr<Estimator> Clone() const override { return std::make_unique<SlopeOne>(Params); }

  private:
    rs_knn *h_ = nullptr;
};
inline std::unique_ptr<SlopeOne> NewSlopeOne(const Parameters &p = {}) { return std::make_unique<SlopeOne>(p); }

// core/utils.go:160-180 with the intended ([]float64, []float64) signature (SURVEY.md §4.3)
using Evaluator = std::function<double(const std::vector<double> &, const std::vector<double> &)>;
inline double RMSE(const std::vector<double> &p, const std::vector<double> &t) {
    double s = 0.0;
    for (size_t j = 0; j < t.size(); j++) s += (p[j] - t[j]) * (p[j] - t[j]);
    return std::sqrt(s / (double)t.size());
}
inline double MAE(const std::vector<double> &p, const std::vector<double> &t) {
    double s = 0.0;
    for (size_t j = 0; j < t.size(); j++) s += std::fabs(p[j] - t[j]);
    return s / (double)t.size();
}

struct CrossValidateResult { std::vector<double> Trains, Tests; };

// core/eval.go:18-67 (6-argument form): every fold works on its own estimator copy whose Params
// are REPLACED by `params` (core/eval.go:34).
inline std::vector<CrossValidateResult> CrossValidate(const Estimator &estimator, const DataSet &dataSet,
                                                      const std::vector<Evaluator> &metrics, int cv, int64_t seed,
                                                      const Parameters &params) {
    std::vector<CrossValidateResult> ret(metrics.size());
    for (auto &r : ret) { r.Trains.assign(cv, 0.0); r.Tests.assign(cv, 0.0); }
    std::vector<TrainSet> trains;
    std::vector<DataSet> tests;
    KFold(dataSet, cv, seed, trains, tests);
    for (int i = 0; i < cv; i++) {
        auto cp = estimator.Clone();
        cp->SetParams(params);
        cp->Fit(trains[i]);
        const auto pred = cp->PredictBatch(tests[i].Users, tests[i].Items);
        for (size_t j = 0; j < metrics.size(); j++) ret[j].Tests[i] = metrics[j](pred, tests[i].Ratings);
    }
    return ret;
}

}  // namespace core
