// knn.go — drop-in replacement of the reference's core/knn.go: same type, constructors,
// Parameters keys and results, with Fit/Predict running on the B200 through bridge.go.
// Everything that is not the hot path (Parameters, TrainSet, BaseLine, CrossValidate,
// CandidateSet's ordering contract) is the reference's own code and stays untouched.
package core

const (
	basic    = "basic"
	centered = "centered"
	zScore   = "zscore"
	baseline = "baseline"
)

// KNN keeps ALL of the reference's exported fields (core/knn.go:17-27), so gob Save/Load
// (core/dump.go:11-36) writes the same record.  Sims is no longer filled by Fit: the N x N matrix
// lives in HBM and MaterializeSims copies it out on demand (e.g. before Save).  LeftRatings /
// RightRatings are the TrainSet's adjacency lists exactly as the reference assigns them
// (core/knn.go:154-162; the left ones id-sorted in place by `sorts`, core/data.go:236-243) — slice
// headers onto the TrainSet's own storage, no copy.
type KNN struct {
	Base
	KNNType      string
	GlobalMean   float64
	Sims         [][]float64
	LeftRatings  [][]IDRating
	RightRatings [][]IDRating
	Means        []float64
	StdDevs      []float64
	Bias         []float64

	dev       *deviceKNN // unexported: invisible to gob, so Copy() never aliases a device handle
	userBased bool
	nLeft     int
	kk        [2]int // k, mink the handle currently holds
}

func NewKNN(params Parameters) *KNN          { return &KNN{Base: Base{Params: params}, KNNType: basic} }
func NewKNNWithMean(params Parameters) *KNN  { return &KNN{Base: Base{Params: params}, KNNType: centered} }
func NewKNNWithZScore(params Parameters) *KNN { return &KNN{Base: Base{Params: params}, KNNType: zScore} }
func NewKNNBaseLine(params Parameters) *KNN  { return &KNN{Base: Base{Params: params}, KNNType: baseline} }

// Close releases the device memory (also done by a finalizer).
func (K *KNN) Close() {
	if K.dev != nil {
		K.dev.close()
		K.dev = nil
	}
}

// Fit replaces core/knn.go:143-217.  The host part is only marshalling: inner ids in dataset
// order (the order Means / StdDevs are accumulated in) narrowed to int32.
func (K *KNN) Fit(trainSet TrainSet) {
	sim := K.Params.GetSim("sim", MSD)
	K.userBased = K.Params.GetBool("userBased", true)
	K.Data = trainSet
	K.GlobalMean = trainSet.GlobalMean
	n := trainSet.Length()
	left := make([]int32, n)
	right := make([]int32, n)
	for i := 0; i < n; i++ {
		u := int32(trainSet.ConvertUserID(trainSet.Users[i]))
		it := int32(trainSet.ConvertItemID(trainSet.Items[i]))
		if K.userBased {
			left[i], right[i] = u, it
		} else {
			left[i], right[i] = it, u
		}
	}
	nLeft, nRight := trainSet.UserCount, trainSet.ItemCount
	if !K.userBased {
		nLeft, nRight = nRight, nLeft
	}
	var leftBias, rightBias []float64
	globalBias := 0.0
	isPB := simEnum(sim) == simEnum(PearsonBaseline)
	if K.KNNType == baseline || isPB {
		baseLine := NewBaseLine(K.Params) // core/knn.go:179-187: sequential SGD stays on the host
		if K.Params.GetString("baseline", "sgd") == "als" { // EXTENSION: ALS baselines on the device
			iu, ii := make([]int32, trainSet.Length()), make([]int32, trainSet.Length())
			for i := 0; i < trainSet.Length(); i++ {
				iu[i] = int32(trainSet.ConvertUserID(trainSet.Users[i]))
				ii[i] = int32(trainSet.ConvertItemID(trainSet.Items[i]))
			}
			baseLine.userBias, baseLine.itemBias = baselineALS(K.Params.GetInt("device", -1), iu, ii,
				trainSet.Ratings, trainSet.UserCount, trainSet.ItemCount, trainSet.GlobalMean,
				K.Params.GetFloat64("regU", 15), K.Params.GetFloat64("regI", 10), K.Params.GetInt("nEpochs", 10))
			baseLine.globalBias = trainSet.GlobalMean
		} else {
			baseLine.Fit(trainSet)
		}
		if K.userBased {
			leftBias, rightBias = baseLine.userBias, baseLine.itemBias
		} else {
			leftBias, rightBias = baseLine.itemBias, baseLine.userBias
		}
		globalBias = baseLine.globalBias
		if K.KNNType == baseline {
			K.Bias = leftBias
		}
		if !isPB {
			rightBias = nil
		}
	}
	if K.userBased { // core/knn.go:154-162
		K.LeftRatings, K.RightRatings = trainSet.UserRatings(), trainSet.ItemRatings()
	} else {
		K.LeftRatings, K.RightRatings = trainSet.ItemRatings(), trainSet.UserRatings()
	}
	sorts(K.LeftRatings) // core/knn.go:190 sorts the TrainSet's cached rows in place; callers may rely on it
	K.Close()
	K.dev = newDeviceKNN(K.Params, K.KNNType)
	K.dev.fit(left, right, trainSet.Ratings, nLeft, nRight, trainSet.GlobalMean, leftBias, rightBias, globalBias)
	K.nLeft = nLeft
	K.kk = [2]int{K.Params.GetInt("k", 40), K.Params.GetInt("mink", 1)}
	if K.KNNType == centered || K.KNNType == zScore {
		K.Means = K.dev.means(nLeft)
	}
	if K.KNNType == zScore {
		K.StdDevs = K.dev.stddevs(nLeft)
	}
}

// Update adds the ratings of rowSet (raw user, raw item, rating; users and items may be new) to the fitted model
// without a refit (rs_knn_update, an extension: the reference has none).  The model becomes the Fit of NewTrainSet of
// the training rows followed by rowSet's, bit for bit, and Data that TrainSet; only the rows of the users (items) the
// ratings touch are recomputed.  A pair the model holds already, KNNBaseline, PearsonBaseline, Pearson in sums mode,
// row shards and top-k-only stores are refused (a panic, as every refused call).
func (K *KNN) Update(rowSet DataSet) {
	n0 := K.Data.Length()
	trainSet := NewTrainSet(DataSet{
		Users:   append(append([]int{}, K.Data.Users...), rowSet.Users...),
		Items:   append(append([]int{}, K.Data.Items...), rowSet.Items...),
		Ratings: append(append([]float64{}, K.Data.Ratings...), rowSet.Ratings...),
	})
	n := trainSet.Length() - n0
	left := make([]int32, n)
	right := make([]int32, n)
	for i := 0; i < n; i++ {
		u := int32(trainSet.ConvertUserID(trainSet.Users[n0+i]))
		it := int32(trainSet.ConvertItemID(trainSet.Items[n0+i]))
		if K.userBased {
			left[i], right[i] = u, it
		} else {
			left[i], right[i] = it, u
		}
	}
	nLeft, nRight := trainSet.UserCount, trainSet.ItemCount
	if !K.userBased {
		nLeft, nRight = nRight, nLeft
	}
	K.dev.update(left, right, trainSet.Ratings[n0:], nLeft, nRight, trainSet.GlobalMean)
	K.Data = trainSet
	K.GlobalMean = trainSet.GlobalMean
	if K.userBased {
		K.LeftRatings, K.RightRatings = trainSet.UserRatings(), trainSet.ItemRatings()
	} else {
		K.LeftRatings, K.RightRatings = trainSet.ItemRatings(), trainSet.UserRatings()
	}
	sorts(K.LeftRatings)
	K.nLeft = nLeft
	if K.KNNType == centered || K.KNNType == zScore {
		K.Means = K.dev.means(nLeft)
	}
	if K.KNNType == zScore {
		K.StdDevs = K.dev.stddevs(nLeft)
	}
}

// PredictBatch implements BatchPredictor: DataSet.Predict (core/data.go:98-105) hands the
// whole test set over in one cgo call.
func (K *KNN) PredictBatch(userIDs, itemIDs []int) []float64 {
	left := make([]int32, len(userIDs))
	right := make([]int32, len(userIDs))
	for i := range userIDs {
		u := int32(K.Data.ConvertUserID(userIDs[i])) // newID = -1 -> GlobalMean on the device
		it := int32(K.Data.ConvertItemID(itemIDs[i]))
		if K.userBased {
			left[i], right[i] = u, it
		} else {
			left[i], right[i] = it, u
		}
	}
	K.syncK()
	return K.dev.predictBatch(left, right)
}

// syncK: core/knn.go:80-81 reads k / mink in Predict, so SetParams after Fit takes effect at the next call.
func (K *KNN) syncK() {
	if kk := [2]int{K.Params.GetInt("k", 40), K.Params.GetInt("mink", 1)}; kk != K.kk {
		K.dev.setK(kk[0], kk[1])
		K.kk = kk
	}
}

// Recommend returns, for each user, the n best items the user has not rated: items[u][x] are raw item ids ranked
// by (score desc, inner item id asc), scores[u][x] the scores, which are Predict(user, item) bit for bit.
// Unused slots are newID (-1) with score NaN; an unknown user scores GlobalMean everywhere.
func (K *KNN) Recommend(userIDs []int, n int) ([][]int, [][]float64) {
	q := make([]int32, len(userIDs))
	for i, u := range userIDs {
		q[i] = int32(K.Data.ConvertUserID(u))
	}
	K.syncK()
	side := sideLeft // user-based: the users are the left side
	if !K.userBased {
		side = sideRight
	}
	ids, sc := K.dev.recommend(side, q, n)
	raw := make([]int, K.Data.ItemCount) // inner -> raw: the order of first appearance
	for _, it := range K.Data.Items {
		raw[K.Data.ConvertItemID(it)] = it
	}
	items := make([][]int, len(userIDs))
	scores := make([][]float64, len(userIDs))
	for i := range userIDs {
		items[i] = make([]int, n)
		for x := 0; x < n; x++ {
			items[i][x] = newID
			if id := ids[i*n+x]; id >= 0 {
				items[i][x] = raw[id]
			}
		}
		scores[i] = sc[i*n : (i+1)*n]
	}
	return items, scores
}

// RecommendGiven is Recommend for users whose ratings are given in dataSet (raw user, raw item, rating) instead of
// taken from the train set: users who signed up or rated after Fit, or held-out ratings (core/eval.go NewAUC).  The
// rows are grouped by user in order of first appearance, each user's ratings kept in dataset order; items the train
// set does not know are dropped (they have no row or column of the model).  users[u] are the raw user ids, items /
// scores as in Recommend; the given items are never listed.  The model is not refitted: the given ratings enter
// neither the similarities between the train set's rows, nor its means, nor GlobalMean.
func (K *KNN) RecommendGiven(dataSet DataSet, n int) ([]int, [][]int, [][]float64) {
	group := map[int]int{}
	var users []int
	var lists [][]int
	for j, u := range dataSet.Users {
		g, ok := group[u]
		if !ok {
			g = len(users)
			group[u] = g
			users = append(users, u)
			lists = append(lists, nil)
		}
		if K.Data.ConvertItemID(dataSet.Items[j]) != newID {
			lists[g] = append(lists[g], j)
		}
	}
	ptr := make([]int64, len(users)+1)
	var ids []int32
	var vals []float64
	for g, rows := range lists {
		for _, j := range rows {
			ids = append(ids, int32(K.Data.ConvertItemID(dataSet.Items[j])))
			vals = append(vals, dataSet.Ratings[j])
		}
		ptr[g+1] = int64(len(ids))
	}
	K.syncK()
	side := sideLeft // user-based: the users are the left side, the lists hold right (item) ids
	if !K.userBased {
		side = sideRight
	}
	top, sc := K.dev.recommendGiven(side, ptr, ids, vals, n)
	raw := make([]int, K.Data.ItemCount) // inner -> raw: the order of first appearance
	for _, it := range K.Data.Items {
		raw[K.Data.ConvertItemID(it)] = it
	}
	items := make([][]int, len(users))
	scores := make([][]float64, len(users))
	for i := range users {
		items[i] = make([]int, n)
		for x := 0; x < n; x++ {
			items[i][x] = newID
			if id := top[i*n+x]; id >= 0 {
				items[i][x] = raw[id]
			}
		}
		scores[i] = sc[i*n : (i+1)*n]
	}
	return users, items, scores
}

// Predict replaces core/knn.go:75-141 (a one-element batch).
func (K *KNN) Predict(userID int, itemID int) float64 {
	return K.PredictBatch([]int{userID}, []int{itemID})[0]
}

// MaterializeSims fills the exported Sims field from HBM (NaN = unset, core/utils.go:110-120).
func (K *KNN) MaterializeSims() {
	flat := K.dev.simsRows(0, K.nLeft, K.nLeft)
	K.Sims = make([][]float64, K.nLeft)
	for i := range K.Sims {
		K.Sims[i] = flat[i*K.nLeft : (i+1)*K.nLeft]
	}
}

// TopK returns the per-row neighbour lists (idx -1 / sim NaN for unused slots).
func (K *KNN) TopK(k int) ([]int32, []float64) { return K.dev.topK(k, K.nLeft) }
